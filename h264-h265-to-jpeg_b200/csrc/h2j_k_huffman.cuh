// K3: optimal Huffman tables (mjpegenc_huffman.c) + code tables + JPEG header (mjpegenc_common.c).
// One CTA of 128 threads per table (DC luma, DC chroma, AC luma, AC chroma) and frame.
//
// What is sequential and why: AV_QSORT is not stable and the order of equal counts / equal lengths decides the
// DHT bytes, so both sorts are replayed step for step by one thread of the group (in shared memory).
// What is parallel: the package-merge.  Level t of ff_mjpegenc_huffman_compute_bits is a merge of two sorted
// lists -- the symbols and the pairwise sums ("packages") of level t-1 -- with packages winning ties.  Every
// item finds its rank in the other list with a binary search, so a level costs a handful of dependent
// shared-memory reads instead of ~500 serial steps.  Per level only the item probabilities and, for every
// prefix of the merged list, the number of symbols in it are kept; that is enough to recover the code lengths
// (symbols are consumed in sorted order, packages in pairs) and gives the same answer as the reference's
// list-copying formulation.
#pragma once
#include "h2j_common.cuh"

namespace h2j {

struct __align__(8) HuffPair { int a, b; };  // {value, prob} or {code, length}

// tools/microbench/k3_phases.cu: cycle stamps of one table's phases (thread 0 of the CTA that builds table 2 of frame 0)
#ifdef H2J_K3_CLOCKS
__device__ long long g_k3_clocks[16];
#define K3_STAMP(i) do { if (gt == 0 && S->stamp_on) g_k3_clocks[i] = clock64(); } while (0)
#else
#define K3_STAMP(i) do { } while (0)
#endif

// ---- AV_QSORT (libavutil/qsort.h), replayed ---------------------------------------------------------------
// The reference's sort is an explicit-stack quicksort: median of three, partition around the middle element, a shortcut
// for ranges that turn out sorted, then one of the two remaining ranges goes on the stack and the loop continues with the
// other.  It is not stable, and where equal counts / equal lengths end up decides the DHT bytes, so every comparison and
// swap of it is reproduced.  What is NOT reproduced is the order in which the ranges are taken: the two ranges a
// partition leaves are disjoint and nothing outside a range is read or written while it is being sorted, so they can be
// sorted at the same time -- by two threads -- with the result the sequential order gives.  qsort_range() is the
// reference's loop body for one range; qsort_replay() runs the ranges of one recursion depth side by side, a round per
// depth (~2 log2 n rounds instead of ~n/2 partitions one after the other: 20 us -> ~2 us for an AC table of 60 symbols).
constexpr int kQsortMaxRanges = 136;  // ranges of one depth: at most num / 2 + 1 with num <= 257

__device__ __forceinline__ void qsort_range(HuffPair *p, int start, int end, unsigned short (*next)[2], int *n_next)
{
    if (start >= end - 1) {  // two elements
        const HuffPair a = p[start], b = p[end];
        if (a.b > b.b) { p[start] = b; p[end] = a; }
        return;
    }
    int checksort = 0;
    int right = end - 2, left = start + 1;
    const int mid = start + ((end - start) >> 1);
    HuffPair ps = p[start], pm = p[mid], pe = p[end];  // (start < mid < end: three different elements)
    auto swp = [](HuffPair &x, HuffPair &y) { const HuffPair t = x; x = y; y = t; };
    if (ps.b > pe.b) {
        if (pe.b > pm.b) swp(ps, pm);
        else swp(ps, pe);
    } else {
        if (ps.b > pm.b) swp(ps, pm);
        else checksort = 1;
    }
    if (pm.b > pe.b) {
        swp(pm, pe);
        checksort = 0;
    }
    p[start] = ps;
    p[end] = pe;
    if (start == end - 2) {
        p[mid] = pm;
        return;
    }
    // SWAP(end[-1], *mid): the pivot waits at end - 1 (mid <= end - 2 here)
    p[mid] = p[end - 1];
    p[end - 1] = pm;
    const int pivot = pm.b;
    // The two scans visit the elements in the reference's order and stop where it stops; only the LOADS differ: four
    // keys are requested at once (a scan is a chain of shared-memory round trips otherwise).  Keys past `right` / below
    // `left` are only looked at under the reference's own bounds test, and the addresses stay inside the array
    // (start <= left, right <= end - 2, elements up to p[num + 2] exist).
    while (left <= right) {
        for (;;) {
            const int k0 = p[left].b, k1 = p[left + 1].b, k2 = p[left + 2].b, k3 = p[left + 3].b;
            if (!(left <= right && k0 < pivot)) break;
            left++;
            if (!(left <= right && k1 < pivot)) break;
            left++;
            if (!(left <= right && k2 < pivot)) break;
            left++;
            if (!(left <= right && k3 < pivot)) break;
            left++;
        }
        for (;;) {
            const int k0 = p[right].b, k1 = p[max(right - 1, start)].b, k2 = p[max(right - 2, start)].b, k3 = p[max(right - 3, start)].b;
            if (!(left <= right && k0 > pivot)) break;
            right--;
            if (!(left <= right && k1 > pivot)) break;
            right--;
            if (!(left <= right && k2 > pivot)) break;
            right--;
            if (!(left <= right && k3 > pivot)) break;
            right--;
        }
        if (left <= right) {
            const HuffPair x = p[left], y = p[right];
            p[left] = y;
            p[right] = x;
            left++;
            right--;
        }
    }
    {  // SWAP(end[-1], *left)
        const HuffPair x = p[end - 1], y = p[left];
        p[end - 1] = y;
        p[left] = x;
    }
    if (checksort && (mid == left - 1 || mid == left)) {
        int m = start;
        while (m < end && p[m].b <= p[m + 1].b) m++;
        if (m == end) return;
    }
    if (start < right) {
        const int i = atomicAdd(n_next, 1);
        next[i][0] = (unsigned short)start;
        next[i][1] = (unsigned short)right;
    }
    if (left + 1 < end) {
        const int i = atomicAdd(n_next, 1);
        next[i][0] = (unsigned short)(left + 1);
        next[i][1] = (unsigned short)end;
    }
}

struct QsortRounds {
    unsigned short range[2][kQsortMaxRanges][2];
    int count[3];  // ranges of this round / the next one / the one after (being cleared)
};

__device__ __forceinline__ void group_sync(int group) { asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(128) : "memory"); }

// Measured and dropped: ranges of 24 and more keys partitioned by a whole warp (the stoppers of both scans as ballots, the
// k-th from the left swapped with the k-th from the right, all pairs at once -- exact, it passed the whole suite): an AC
// table of 60 symbols took 10.6 + 10.8 us for its two sorts instead of 10.9 + 7.3 (finding the k-th set bit per lane and
// the extra warp synchronisations cost what the shorter scans saved).
// all kHuffGroup threads of the group call this; p[0 .. num + 2] must exist
__device__ void qsort_replay(HuffPair *p, int num, QsortRounds *Q, int gt, int group)
{
    if (gt == 0) {
        Q->range[0][0][0] = 0;
        Q->range[0][0][1] = (unsigned short)(num - 1);
        Q->count[0] = num > 1 ? 1 : 0;
        Q->count[1] = 0;
        Q->count[2] = 0;
    }
    group_sync(group);
    // range i goes to thread (i % 4) * 32 + i / 4: the first ranges of a round land in different warps (threads of one warp
    // that sort different ranges take turns at every divergent step)
    const int my_first = ((gt & 31) << 2) | (gt >> 5);
    for (int round = 0;; round++) {
        const int n = Q->count[round % 3];
        if (n == 0) break;
        if (gt == 0) Q->count[(round + 2) % 3] = 0;
        for (int i = my_first; i < n; i += kHuffGroup)
            qsort_range(p, Q->range[round & 1][i][0], Q->range[round & 1][i][1], Q->range[(round + 1) & 1], &Q->count[(round + 1) % 3]);
        group_sync(group);
#ifdef H2J_K3_CLOCKS
        if (gt == 0) g_k3_clocks[15] = round + 1;  // rounds of the last sort
#endif
    }
}

constexpr int kPmMaxItems = 516;  // a level holds at most 257 + 258/2 items; rounded up
struct HuffScratch {
    HuffPair sorted[264];                        // {value, count}, then sorted by count (+ room for the scans' look-ahead)
    HuffPair distinct[264];                      // {value, code length}, then sorted by length
    QsortRounds rounds;
    __align__(8) int prob[2][kPmMaxItems];
    __align__(8) int symcnt[2 * 264];            // {count of sorted symbol i, 0}: the symbols in the shape of the package pairs
    unsigned short leaves[17][kPmMaxItems + 2];  // leaves[t][p] = number of symbols among the first p items of level t
    int nl[17];                                  // symbols counted at each level by the back-trace
    unsigned char nbits_by_value[260];
    int warp_tot[4];
    int first_code[18], first_index[18];
    unsigned int bits_cnt[17];
#ifdef H2J_K3_CLOCKS
    int stamp_on;
#endif
};


// exclusive prefix sum of `v` over the 128 threads of a group; *total receives the group sum
__device__ __forceinline__ int group_excl_scan(int v, int gt, int group, int *warp_tot, int *total)
{
    const int lane = gt & 31, w = gt >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    group_sync(group);  // protects warp_tot against the previous use
    if (lane == 31) warp_tot[w] = incl;
    group_sync(group);
    int off = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        if (i < w) off += warp_tot[i];
        tot += warp_tot[i];
    }
    *total = tot;
    return off + incl - v;
}

// One table, executed by the 128 threads of `group` (gt = thread index inside the group).
__device__ void build_one_table(const unsigned int *__restrict__ hist, HuffScratch *S, int gt, int group, uint8_t *g_bits, uint8_t *g_vals,
                                int *g_nvals, uint32_t *g_hcode, int n_hcode)  // n_hcode: entries of the code table (16 DC, 256 AC)
{
    // ---- ff_mjpeg_encode_huffman_close: used symbols in increasing value order, plus the dummy (256, 0) ----
    K3_STAMP(0);
    const int h0 = (int)hist[2 * gt], h1 = (int)hist[2 * gt + 1];
    int nval;
    int pos = group_excl_scan((h0 != 0) + (h1 != 0), gt, group, S->warp_tot, &nval);
    if (h0) { S->sorted[pos].a = 2 * gt; S->sorted[pos].b = h0; pos++; }
    if (h1) { S->sorted[pos].a = 2 * gt + 1; S->sorted[pos].b = h1; }
    if (gt == 0) { S->sorted[nval].a = 256; S->sorted[nval].b = 0; }
    const int size = nval + 1;
    group_sync(group);
    K3_STAMP(1);
    qsort_replay(S->sorted, size, &S->rounds, gt, group);
    K3_STAMP(2);

    // ---- ff_mjpegenc_huffman_compute_bits, max_length 16: levels 0..15 take symbols, level 16 only packages ----
    for (int k = gt; k <= size; k += kHuffGroup) {
        S->leaves[0][k] = (unsigned short)k;
        if (k < size) {
            S->prob[0][k] = S->sorted[k].b;
            S->symcnt[2 * k] = S->sorted[k].b;
            S->symcnt[2 * k + 1] = 0;
        }
    }
    int n_prev = size, cur = 0;
    for (int t = 1; t <= 16; t++) {
        group_sync(group);
        const int *pp = S->prob[cur];
        int *np = S->prob[cur ^ 1];
        const int L = t < 16 ? size : 0, npk = n_prev >> 1;
        // Ranks by binary search with a fixed number of steps (the same for every thread) and no branch inside: a step is one
        // shared-memory round trip, so a level costs log2 of them.  Symbols and packages run the SAME code (a warp whose
        // threads took two different search loops would run them one after the other): a symbol looks for the packages whose
        // sum is <= its count, a package for the symbols whose count is < its sum, i.e. <= sum - 1; both lists are arrays of
        // pairs whose sum is the key (the symbols as {count, 0}).
        const int span = 1 << (32 - __clz(max(max(L, npk), 1)));  // power of two above both list lengths
        for (int idx = gt; idx < L + npk; idx += kHuffGroup) {
            const bool is_sym = idx < L;
            const int own = is_sym ? idx : idx - L;
            const int2 mine = *reinterpret_cast<const int2 *>(is_sym ? &S->symcnt[2 * own] : &pp[2 * own]);
            const int key = mine.x + mine.y;
            const int *other = is_sym ? pp : S->symcnt;
            const int n_other = is_sym ? npk : L, bound = is_sym ? key : key - 1;
            int lo = 0;
            for (int step = span >> 1; step; step >>= 1) {
                const int c = lo + step - 1;  // candidate: items 0 .. c of the other list all in front of this one?
                const int2 pr = *reinterpret_cast<const int2 *>(&other[2 * max(min(c, n_other - 1), 0)]);
                if (c < n_other && pr.x + pr.y <= bound) lo += step;
            }
            // preceded by its own predecessors and by `lo` items of the other list
            const int p = own + lo;
            np[p] = key;
            S->leaves[t][p + 1] = (unsigned short)(is_sym ? idx + 1 : lo);
        }
        if (gt == 0) S->leaves[t][0] = 0;
        n_prev = L + npk;
        cur ^= 1;
    }
    group_sync(group);
    K3_STAMP(3);
    // ---- back-trace: how many symbols each level contributes to the first min(size-1, nitems) items ----
    if (gt == 0) {
        int p = size - 1 < n_prev ? size - 1 : n_prev;
        for (int t = 16; t >= 0; t--) {
            const int nl = p > 0 ? (int)S->leaves[t][p] : 0;
            S->nl[t] = nl;
            p = p > 0 ? 2 * (p - nl) : 0;
        }
    }
    for (int i = gt; i < 260; i += kHuffGroup) S->nbits_by_value[i] = 0;
    if (gt < 17) S->bits_cnt[gt] = 0;
    group_sync(group);
    for (int r = gt; r < size; r += kHuffGroup) {
        int nb = 0;
#pragma unroll
        for (int t = 0; t <= 16; t++) nb += S->nl[t] > r ? 1 : 0;
        S->nbits_by_value[S->sorted[r].a] = (unsigned char)nb;
    }
    group_sync(group);
    // ---- symbols with a code, in increasing value order (the dummy 256 is left out), sorted by length ----
    {
        const int b0 = S->nbits_by_value[2 * gt], b1 = S->nbits_by_value[2 * gt + 1];
        int tot;
        int p = group_excl_scan((b0 != 0) + (b1 != 0), gt, group, S->warp_tot, &tot);
        if (b0) { S->distinct[p].a = 2 * gt; S->distinct[p].b = b0; p++; }
        if (b1) { S->distinct[p].a = 2 * gt + 1; S->distinct[p].b = b1; }
        // tot == nval: every used symbol receives a code
    }
    group_sync(group);
    K3_STAMP(4);
    qsort_replay(S->distinct, nval, &S->rounds, gt, group);
    K3_STAMP(5);
    // ---- BITS / HUFFVAL, then ff_mjpeg_build_huffman_codes ----
    for (int i = gt; i < 256; i += kHuffGroup) {
        g_vals[i] = i < nval ? (uint8_t)S->distinct[i].a : 0;
        if (i < n_hcode) g_hcode[i] = 0;
        if (i < nval) atomicAdd(&S->bits_cnt[S->distinct[i].b], 1u);
    }
    group_sync(group);
    if (gt == 0) {
        int code = 0, k = 0;
        for (int i = 1; i <= 16; i++) {
            S->first_code[i] = code;
            S->first_index[i] = k;
            code = (code + (int)S->bits_cnt[i]) << 1;
            k += (int)S->bits_cnt[i];
        }
        *g_nvals = nval;
    }
    if (gt < 17) g_bits[gt] = gt ? (uint8_t)S->bits_cnt[gt] : 0;
    group_sync(group);
    for (int i = gt; i < nval; i += kHuffGroup) {
        const int len = S->distinct[i].b;
        const int code = S->first_code[len] + (i - S->first_index[len]);
        // K4a appends nb mantissa bits behind the code of a symbol whose low nibble is nb (DC: the symbol itself), so the
        // table holds the code already shifted into place and the total length: (code << nb) << 5 | (len + nb)
        const int sym = S->distinct[i].a, nb = sym & 15;
        g_hcode[sym] = (((uint32_t)code << nb) << 5) | (uint32_t)(len + nb);
    }
    K3_STAMP(6);
}

// Byte i of the picture header: SOI, COM, DQT, DHT (4 tables), SOF0, SOS (ff_mjpeg_encode_picture_header).
struct HeaderPlan {
    int off_dqt, off_dht, off_tab[4], off_sof, total;
};
__device__ __forceinline__ HeaderPlan header_plan(const int nvals[4], int comment_len)
{
    HeaderPlan h;
    h.off_dqt = 2 + 4 + comment_len + 1;
    h.off_dht = h.off_dqt + 4 + 1 + 64;
    int p = h.off_dht + 4;
    for (int t = 0; t < 4; t++) {
        h.off_tab[t] = p;
        p += 17 + nvals[t];
    }
    h.off_sof = p;
    h.total = p + 19 + 14;
    return h;
}
__device__ uint8_t header_byte(int i, const HeaderPlan &h, const FrameTab *T, const FrameLayout &L, const char *comment, int comment_len)
{
    if (i < h.off_dqt) {
        if (i < 6) {
            const int len = comment_len + 3;
            const uint8_t fixed[6] = {0xff, 0xd8, 0xff, 0xfe, (uint8_t)(len >> 8), (uint8_t)len};
            return fixed[i];
        }
        return i - 6 < comment_len ? (uint8_t)comment[i - 6] : 0;
    }
    if (i < h.off_dht) {
        const int k = i - h.off_dqt;
        if (k < 5) {
            const uint8_t fixed[5] = {0xff, 0xdb, 0, 67, 0};
            return fixed[k];
        }
        return T->dqt_zz[k - 5];
    }
    if (i < h.off_sof) {
        const int k = i - h.off_dht;
        if (k < 4) {
            const int size = h.off_sof - h.off_dht - 2;
            const uint8_t fixed[4] = {0xff, 0xc4, (uint8_t)(size >> 8), (uint8_t)size};
            return fixed[k];
        }
        int t = 3;
        while (i < h.off_tab[t]) t--;
        const int j = i - h.off_tab[t];
        if (j == 0) return (uint8_t)(((t >> 1) << 4) | (t & 1));  // class << 4 | id: DC0, DC1, AC0, AC1
        if (j <= 16) return T->bits[t][j];
        return T->vals[t][j - 17];
    }
    const int k = i - h.off_sof;
    // sampling factors (mjpegenc_common.c ff_mjpeg_init_hvsample): luma 2x2 and chroma 2 >> shift, but 4:4:4 is coded with
    // every component at h = 1, v = 2 (8x16 MCUs)
    const uint8_t hv_y = L.fmt == kFmt444 ? 0x12 : 0x22, hv_c = L.fmt == kFmt420 ? 0x11 : 0x12;
    const uint8_t tail[33] = {0xff, 0xc0, 0, 17, 8, (uint8_t)(L.h >> 8), (uint8_t)L.h, (uint8_t)(L.w >> 8), (uint8_t)L.w, 3,
                              1, hv_y, 0, 2, hv_c, 0, 3, hv_c, 0,
                              0xff, 0xda, 0, 12, 3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0};
    return tail[k];
}

// grid 4 * frames CTAs of one group each: one table per CTA.  blockIdx.x / frames picks the table, AC tables first (they
// take ~10x longer than the DC ones and decide the kernel's duration: with one CTA per FRAME the four scratch areas
// allowed two CTAs per SM, and 512 frames needed two waves of them).  The frame's CTA that finishes last writes the header.
// Frame f's output starts at out + f * out_cap; jpeg_cap (<= out_cap) is the largest JPEG allowed, and no byte at or past
// it is written.
// LIST: a list batch; the SOF segment gets the frame's own size, descs[f].L.  (The defaults keep callers that launch K3 on its
// own with the batch form's arguments -- tests/support/k3_shim.cu, tools/microbench/k3_phases.cu -- compiling unchanged.)
template <bool LIST = false>
__global__ void __launch_bounds__(kHuffGroup) huffman_kernel(FrameLayout L, FrameTab *__restrict__ tabs, FrameState *__restrict__ state,
                                                             int n_frames, uint8_t *__restrict__ out, long long out_cap, long long jpeg_cap,
                                                             const char *__restrict__ comment, int comment_len,
                                                             const FrameDesc *__restrict__ descs = nullptr)
{
    __shared__ HuffScratch scratch;
    __shared__ int s_last;
    const int tid = threadIdx.x;
    const int slot = blockIdx.x / n_frames, f = blockIdx.x - slot * n_frames;
    const int table = slot ^ 2;  // 2, 3 (AC luma, AC chroma), then 0, 1 (DC)
    FrameTab *T = tabs + f;
#ifdef H2J_K3_CLOCKS
    if (tid == 0) scratch.stamp_on = (table == 2 && f == 0);
    __syncthreads();
#endif
    // the two DC code tables (16 entries each) go right in front of the AC tables -- into the unused tail of hcode[1] -- so that
    // K4a fetches all four with ONE bulk copy
    uint32_t *hc = table < 2 ? dc_code_table(T, table) : T->hcode[table];
    build_one_table(state[f].hist[table], &scratch, tid, 0, T->bits[table], T->vals[table], &T->nvals[table], hc, table < 2 ? 16 : 256);
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&state[f].k3_done, 1u) == 3u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();  // the other three tables were written by other CTAs
    const volatile int *nv = T->nvals;
    const int nvals[4] = {nv[0], nv[1], nv[2], nv[3]};
    const HeaderPlan h = header_plan(nvals, comment_len);
    uint8_t *o = out + (long long)f * out_cap;
    for (int i = tid; i < h.total; i += kHuffGroup)
        if (i < jpeg_cap) o[i] = header_byte(i, h, T, LIST ? descs[f].L : L, comment, comment_len);
    if (tid == 0) {
        T->header_bytes = h.total;
        if (h.total > jpeg_cap) T->status = -4;
    }
}

}  // namespace h2j
