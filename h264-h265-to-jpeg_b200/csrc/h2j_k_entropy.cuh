// K4: entropy coding (mjpegenc.c record_block + ff_mjpeg_encode_picture_frame), in two kernels.
//
// K4a entropy_walk_kernel -- all the coding work, no dependency between CTAs or warps:
//   A CTA takes one K2 tile of one frame (16 MCUs: 96 consecutive blocks at 4:2:0 and 4:4:4, 128 at 4:2:2) and pulls the
//   tile image (levels and non-zero masks) and the frame's code tables into shared memory with bulk copies
//   (cp.async.bulk -> SASS UBLKCP) signalled on an mbarrier.  Each of the CTA's warps then works alone on its UNIT of 32
//   blocks in coding order (a thread finds its block's record through tile_rec_fmt):
//     1. ONE walk over the block: every lane encodes its block into a private 256-bit slot in shared memory and
//        learns its bit length on the way (a block that needs more keeps counting and is emitted directly in 2);
//        warp scan of the lengths.
//     2. the slots are merged into the warp's bit window at the scanned offsets (a couple of shifted ORs per lane).
//     3. the unit's bits, still starting at bit 0 of a word, go to a staging buffer -- at the unit's own fixed place if
//        they fit one window, else at a position reserved with an atomicAdd -- and (position, bit length) is recorded.
//   A warp window holds 8 Kibit.  A unit that needs more (> 256 bits per block on average) takes the windowed path:
//   direct emission clipped to one window of the unit's bit range at a time.
//
// K4b scan_place_kernel -- turns the staged units into the frame's bit stream (0.25 MB per 1080p frame):
//   A CTA takes a group of 256 consecutive units through an atomic ticket, scans their bit lengths, publishes the
//   group total and resolves the group's exclusive prefix with a decoupled look-back over the frame's earlier
//   groups (one 64-bit descriptor per group: [63:62] status 0 invalid / 1 group total / 2 inclusive prefix,
//   [61:0] bits).  Each warp then concatenates a run of 32 units at their global bit positions: a 32-bit word is
//   written (big-endian) by the unit that holds its last bit, the bits of the word that is still open are carried to
//   the next unit, and only a run's first unit fetches its carry from the staged unit in front.  No atomics on the
//   scan, no pre-zeroed output.  While storing, the 0xFF bytes of every word are counted into per-chunk counters for
//   K5; the frame's last word is padded with ones (put_bits / picture trailer).
#pragma once
#include <cstddef>

#include "h2j_common.cuh"

namespace h2j {

__device__ __forceinline__ unsigned long long desc_pack(unsigned status, unsigned long long len) { return ((unsigned long long)status << 62) | len; }
__device__ __forceinline__ unsigned desc_status(unsigned long long d) { return (unsigned)(d >> 62); }
__device__ __forceinline__ unsigned long long desc_len(unsigned long long d) { return d & 0x3fffffffffffffffull; }
__device__ __forceinline__ unsigned long long ld_desc(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_desc(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

#ifndef H2J_ENT_WALK
#define H2J_ENT_WALK 2
#endif
constexpr int kWalkPerTrip = H2J_ENT_WALK;                   // K4a: non-zero levels a lane takes per trip of its walk (per 2048
                                                             // frames: 1 -> 2.927 ms, 2 -> 2.758, 3 -> 2.834, 4 -> 2.907)
constexpr int kUnitBlocks = 32;                              // one warp
constexpr int kEntWarps = kEntThreads / 32;                  // units per CTA at 4:2:0 / 4:4:4 (4:2:2: four)
constexpr int kWarpWinWords = 256;                           // per-warp bit window: 8 Kibit
constexpr int kWarpWinBits = kWarpWinWords * 32;
constexpr int kWarpWinStride = kWarpWinWords + 4;            // spare words for the last partial OR
constexpr int kSlotWords = 8;                                // private slot of a block: 256 bits
constexpr int kSlotBits = kSlotWords * 32;
constexpr int kSlotStride = kSlotWords + 1;                  // odd stride: the lanes' word i never share a bank
#ifndef H2J_ENT_PREFETCH_DISTANCE
#define H2J_ENT_PREFETCH_DISTANCE 1024
#endif
constexpr int kEntPrefetchDistance = H2J_ENT_PREFETCH_DISTANCE;  // K4a: CTAs ahead whose image is requested into L2 (148 SMs x 10 CTAs are resident)
constexpr int kPlaceGroupUnits = 256;                        // K4b: units per CTA, one per thread
constexpr int kPlaceThreads = 256;
#ifndef H2J_PLACE_BATCH
#define H2J_PLACE_BATCH 4
#endif
constexpr int kPlaceBatch = H2J_PLACE_BATCH;                   // K4b: units whose staged words a warp requests before it places them

// per-unit record written by K4a: where the unit's bits were staged and how many there are
__device__ __forceinline__ unsigned long long unit_pack(unsigned pos_words, unsigned bits) { return ((unsigned long long)pos_words << 32) | bits; }
__device__ __forceinline__ unsigned unit_pos(unsigned long long r) { return (unsigned)(r >> 32); }
__device__ __forceinline__ unsigned unit_bits(unsigned long long r) { return (unsigned)r; }

// ---- bit sinks ------------------------------------------------------------------------------------
struct BitSink {  // appends MSB-first into a zeroed shared-memory word array
    unsigned int *buf;
    unsigned long long acc;
    int fill;
    int widx;
    __device__ __forceinline__ void init(unsigned int *b, unsigned pos) { buf = b; acc = 0; fill = (int)(pos & 31); widx = (int)(pos >> 5); }
    __device__ __forceinline__ void put(unsigned bits, int len)
    {
        acc = (acc << len) | bits;
        fill += len;
        if (fill >= 32) {
            atomicOr(&buf[widx++], (unsigned)(acc >> (fill - 32)));
            fill -= 32;
        }
    }
    __device__ __forceinline__ void flush() { if (fill > 0) atomicOr(&buf[widx], (unsigned)(acc << (32 - fill))); }
};

struct BitSinkClip {  // same stream, but only the bits inside [lo, hi) are kept, at position (bit - lo)
    unsigned int *buf;
    unsigned pos, lo, hi;
    __device__ __forceinline__ void init(unsigned int *b, unsigned start, unsigned lo_, unsigned hi_) { buf = b; pos = start; lo = lo_; hi = hi_; }
    __device__ __forceinline__ void put(unsigned bits, int len)
    {
        unsigned s = pos;
        const unsigned e = pos + (unsigned)len;
        pos = e;
        if (len == 0 || e <= lo || s >= hi) return;
        if (s < lo) {
            len = (int)(e - lo);
            bits &= (1u << len) - 1u;
            s = lo;
        }
        if (e > hi) {
            const int cut = (int)(e - hi);
            bits >>= cut;
            len -= cut;
        }
        const unsigned r = s - lo;
        const unsigned long long v = (unsigned long long)bits << (64 - (int)(r & 31) - len);
        atomicOr(&buf[r >> 5], (unsigned)(v >> 32));
        if ((unsigned)v) atomicOr(&buf[(r >> 5) + 1], (unsigned)v);
    }
    __device__ __forceinline__ void flush() {}
};

struct SlotSink {  // MSB-first into the lane's private slot; keeps counting (and drops the words) past its capacity
    unsigned int *slot;
    unsigned long long acc;
    int fill;
    int widx;
    __device__ __forceinline__ void init(unsigned int *s) { slot = s; acc = 0; fill = 0; widx = 0; }
    // No branch, no predicate: in a walking warp nearly every put completes a word in SOME lane, so the branch around the store
    // was taken anyway and only added its own instructions (and a reconvergence point) to every put.  len <= 27 and fill <= 31 on
    // entry, so fill + len < 64: the completed word is acc >> ((fill + len) & 31), and fill & 31 is what stays.
    __device__ __forceinline__ void put(unsigned bits, int len)
    {
        acc = (acc << len) | bits;
        const int f2 = fill + len;
        fill = f2 & 31;
        // stored whether the word is complete or not: an incomplete one is stored again when it is (or by flush()); words past
        // the slot's capacity land in the slot's spare word (kSlotStride = kSlotWords + 1)
        slot[min(widx, kSlotWords)] = (unsigned)(acc >> fill);
        widx += f2 >> 5;
    }
    __device__ __forceinline__ unsigned bits() const { return (unsigned)(widx * 32 + fill); }
    __device__ __forceinline__ void flush() { if (fill > 0 && widx < kSlotWords) slot[widx] = (unsigned)(acc << (32 - fill)); }
};

// One pass over a block.  EMIT=false: returns the bit length.  EMIT=true: writes the bits into `sink`.
// cb = the block's 66-halfword record in shared memory ([0] = DC difference, level k at [2*(k&31) + (k>>5)]).
template <bool EMIT, typename Sink>
__device__ __forceinline__ unsigned walk_block(const int16_t *cb, unsigned mask_lo, unsigned mask_hi, const uint32_t *__restrict__ hdc,
                                               const uint32_t *__restrict__ hac, Sink *sink)
{
    unsigned total = 0;
    {
        const int diff = (int)cb[0];
        const int nb = mag_bits(diff);
        const uint32_t e = hdc[nb];  // code tables come pre-shifted from K3: (code << nb) << 5 | (code length + nb)
        if (EMIT) {
            const unsigned mant = (unsigned)(diff + (diff >> 31)) & ((1u << nb) - 1u);
            sink->put((e >> 5) | mant, (int)(e & 31));
        } else total += e & 31;
    }
    int prev = 0;
    const uint32_t zrl = hac[0xf0];
    // one coded level: zero-run escapes, then (run, size) code + mantissa
    auto code_one = [&](int run, int val, int nb, uint32_t e) {
        if (run >= 16) {
            if (EMIT) {
                for (int z = run >> 4; z > 0; z--) sink->put(zrl >> 5, zrl & 31);
            } else total += (unsigned)(run >> 4) * (zrl & 31);
        }
        if (EMIT) {
            const unsigned mant = (unsigned)(val + (val >> 31)) & ((1u << nb) - 1u);
            sink->put((e >> 5) | mant, (int)(e & 31));
        } else total += e & 31;
    };
#pragma unroll
    for (int half = 0; half < 2; half++) {
        unsigned mm = half ? mask_hi : mask_lo;
        // kWalkPerTrip positions per trip: their position -> level -> size -> code look-ups are independent and overlap;
        // only the emission is in order (positions a lane has run out of are predicated off)
        while (mm) {
            unsigned b[kWalkPerTrip];
            int k[kWalkPerTrip], val[kWalkPerTrip], nb[kWalkPerTrip], run[kWalkPerTrip];
            uint32_t e[kWalkPerTrip];
#pragma unroll
            for (int i = 0; i < kWalkPerTrip; i++) {
                b[i] = mm & (0u - mm);
                mm ^= b[i];
            }
#pragma unroll
            for (int i = 0; i < kWalkPerTrip; i++) {
                const int p = (i == 0 || b[i]) ? 31 - __clz(b[i]) : k[i - 1] - half * 32;  // absent: the previous position again
                k[i] = half * 32 + p;
                val[i] = (int)cb[2 * p + half];
                nb[i] = mag_bits(val[i]);
                run[i] = k[i] - (i ? k[i - 1] : prev) - 1;
                e[i] = hac[((run[i] & 15) << 4) | nb[i]];
            }
#pragma unroll
            for (int i = 0; i < kWalkPerTrip; i++)
                if (i == 0 || b[i]) code_one(run[i], val[i], nb[i], e[i]);
            prev = k[kWalkPerTrip - 1];
        }
    }
    {
        // EOB, or zero bits of length zero: no branch around the put (2.496 -> 2.486 ms; the same for a trip's second level
        // measured slower, and the mantissa as level + (negative ? 2^nb - 1 : 0) in one three-input add too: 2.520)
        const uint32_t e = prev < 63 ? hac[0] : 0u;
        if (EMIT) sink->put(e >> 5, e & 31);
        else total += e & 31;
    }
    return total;
}

constexpr int kEntTabBytes = (2 * 16 + 2 * 256) * 4;  // DC luma/chroma (16 entries each), AC luma/chroma of FrameTab::hcode
// dynamic shared memory of a CTA: the tile image, the code tables, a window and 32 slots per warp
__host__ __device__ constexpr int ent_smem_bytes(int fmt)
{
    return fmt_roles(fmt) * kSubImageBytes + kEntTabBytes + fmt_roles(fmt) * (kWarpWinStride + kUnitBlocks * kSlotStride) * 4;
}
constexpr int kEntSmemBytes = ent_smem_bytes(kFmt420);
static_assert(offsetof(FrameTab, hcode) % 16 == 0 && sizeof(FrameTab) % 16 == 0 && (kDcCodeOff * 4) % 16 == 0, "the code tables must be bulk-copyable");

// grid (tiles_per_frame, frames); FMT = the chroma format (h2j_common.cuh): a tile is 96 blocks (three units) at 4:2:0 and
// 4:4:4, 128 blocks (four units) at 4:2:2; one thread per block, one warp per unit
// LIST: a list batch (h2j_common.cuh FrameDesc); the grid has the largest frame's tiles, the ones past this frame's return
template <int FMT, bool LIST>
__global__ void __launch_bounds__(fmt_tile_blocks(FMT)) entropy_walk_kernel(FrameLayout L_, FrameTab *__restrict__ tabs,
                                                                   const uint32_t *__restrict__ images, long long images_cap,
                                                                   unsigned long long *__restrict__ unit_info, int units_cap,
                                                                   unsigned int *__restrict__ stage_alloc,  // [frame] words handed out
                                                                   uint32_t *__restrict__ stage, long long stage_cap_words,
                                                                   const FrameDesc *__restrict__ descs)
{
    constexpr int kWarps = fmt_roles(FMT), kThreads = fmt_tile_blocks(FMT);       // units per tile = roles per tile
    constexpr int kImageWords = kWarps * kSubImageWords, kImageBytes = kImageWords * 4;
    extern __shared__ __align__(128) unsigned char ent_smem[];
    uint32_t *s_img = reinterpret_cast<uint32_t *>(ent_smem);                    // the CTA's tile image
    uint32_t *s_hdc = reinterpret_cast<uint32_t *>(ent_smem + kImageBytes);      // [2][16] DC code tables
    uint32_t *s_hac = s_hdc + 32;                                                // [2][256] AC code tables
    unsigned int *s_win_all = s_hac + 512;                                       // [warp][kWarpWinStride]
    unsigned int *s_slot_all = s_win_all + kWarps * kWarpWinStride;              // [warp][lane][kSlotStride]
    __shared__ __align__(8) unsigned long long s_bar;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int f = blockIdx.y, tile = blockIdx.x;
    const FrameLayout &L = LIST ? descs[f].L : L_;
    if (LIST && tile * kThreads >= L.n_blocks) return;
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        const uint32_t *src = images + ((long long)f * images_cap + tile) * kImageWords;
        mbar_expect_tx(&s_bar, kImageBytes + kEntTabBytes);
        bulk_g2s(s_img, src, kImageBytes, &s_bar);
        // DC luma, DC chroma, AC luma, AC chroma: contiguous (K3 puts the DC tables right in front of the AC tables), one copy
        // instead of three -- thread 0's set-up is what the CTA's other threads wait for at the barrier below (2.733 -> 2.708 ms)
        bulk_g2s(s_hdc, dc_code_table(tabs + f, 0), kEntTabBytes, &s_bar);
    }
    if (tid == 32) {
        // CTAs are dispatched in linear order, so this one asks for the image of a CTA that starts a fraction of a CTA
        // lifetime (~4 us) from now to be brought into L2; that CTA's bulk copy then finds it there.  Worth 1.3 % of the
        // kernel (any distance from 384 to 2048 CTAs measures the same, 4096 is 12 % slower): most of the wait behind
        // the mbarrier is not DRAM latency.  (Thread 32, not thread 0: everybody waits at the barrier below for thread 0 to
        // have set up the mbarrier and the copies -- 10 % of the kernel's stall samples sat there -- and the division for
        // the prefetch address was part of that wait: 2.757 -> 2.731 ms per 2048 frames.)
        const long long lin = (long long)f * gridDim.x + tile + kEntPrefetchDistance;
        if (lin < (long long)gridDim.x * gridDim.y) {
            const long long f2 = lin / gridDim.x, t2 = lin - f2 * gridDim.x;
            bulk_prefetch_l2(images + (f2 * images_cap + t2) * kImageWords, kImageBytes);
        }
    }
    static_assert((kWarps * kWarpWinStride) % 4 == 0 && (kImageBytes + kEntTabBytes) % 16 == 0, "windows are cleared 16 bytes at a time");
    for (int i = tid; i < kWarps * kWarpWinStride / 4; i += kThreads) reinterpret_cast<uint4 *>(s_win_all)[i] = make_uint4(0, 0, 0, 0);  // while the copies are on their way
    __syncthreads();  // barrier initialised, windows cleared (clearing only the words a unit needs, once its length is
                      // known, executes fewer instructions but measured 1 % slower: here it hides under the copy; the barrier
                      // right behind mbar_init, every warp clearing its own window: 2.742 ms against 2.731)

    // ---- from here on the warp is on its own ----
    const int u = tile * kWarps + warp;                     // unit index inside the frame
    const int b = u * kUnitBlocks + lane;                   // == tile * kThreads + tid
    if (u * kUnitBlocks >= L.n_blocks) return;              // trailing unit of the frame's last tile: no block at all
    const bool valid = b < L.n_blocks;
    const TileRec tr = tile_rec_fmt(FMT, tid);              // block of the tile (coding order) -> (role's sub-image, record)
    const uint32_t *rec = s_img + tr.sub * kSubImageWords + tr.idx * kBlkWords;
    // the tile starts on an MCU boundary, so the block's position in its MCU is tid % blocks per MCU
    const int cls = block_component(FMT, tid % fmt_mcu_blocks(FMT)) ? 1 : 0;
    const int16_t *cb = reinterpret_cast<const int16_t *>(rec);
    const uint32_t *hdc = s_hdc + 16 * cls, *hac = s_hac + 256 * cls;
    unsigned int *win = s_win_all + warp * kWarpWinStride;
    unsigned int *slot = s_slot_all + (warp * kUnitBlocks + lane) * kSlotStride;
    uint32_t *st = stage + (long long)f * stage_cap_words;

    mbar_wait(&s_bar, 0);  // coefficient images and code tables landed
    unsigned mask_lo = 0, mask_hi = 0;
    if (valid) {
        mask_lo = rec[kMaskLoWord];
        mask_hi = s_img[tr.sub * kSubImageWords + kSubMaskHiOff + tr.idx];
    }

    // ---- 1. the walk: bits into the private slot, length on the way ----
    unsigned len = 0;
    if (valid) {
        SlotSink ss;
        ss.init(slot);
        walk_block<true, SlotSink>(cb, mask_lo, mask_hi, hdc, hac, &ss);
        len = ss.bits();
        ss.flush();
    }
    unsigned incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned unit_len = __shfl_sync(0xffffffffu, incl, 31);
    const unsigned off = incl - len;
    const unsigned nwords = (unit_len + 31) >> 5;

    // ---- 3a. where the unit is staged.  A unit that fits one window (all but pathological content) owns the fixed place
    //      u * kWarpWinWords: nothing to reserve, nothing to wait for (the atomicAdd every unit used to make was 10 % of the
    //      kernel's stall samples although its round trip was only awaited behind the merge).  Larger units reserve their
    //      words behind the fixed places with an atomicAdd (any order). ----
    const unsigned cap_w = (unsigned)min(stage_cap_words, (long long)0xffffffffu);
    const unsigned fixed_words = (unsigned)units_cap * kWarpWinWords;
    // broadcast the position, record the unit, return how many of its words fit the buffer: all of them unless the frame
    // overflows its output cap
    auto claim = [&](unsigned pos_lane0, unsigned &pos) {
        pos = __shfl_sync(0xffffffffu, pos_lane0, 0);
        const unsigned n_fit = pos >= cap_w ? 0u : min(nwords, cap_w - pos);
        if (lane == 0) {
            unit_info[(long long)f * units_cap + u] = unit_pack(pos, unit_len);
            if (n_fit < nwords) tabs[f].status = -4;
        }
        return n_fit;
    };

    if (unit_len <= (unsigned)kWarpWinBits) {
        // ---- 2. merge the slots into the warp's window ----
        if (valid) {
            if (len <= (unsigned)kSlotBits) {
                // window word k of the block = the slot's words k - 1 and k funnelled together: one OR per window word (nw + 1 of
                // them) instead of two per slot word
                const int nw = (int)((len + 31) >> 5);
                const unsigned sh = off & 31;
                unsigned int *w = win + (off >> 5);
                unsigned prev = 0;
                for (int i = 0; i < nw; i++) {
                    const unsigned cur = slot[i];
                    const unsigned o = __funnelshift_r(cur, prev, sh);
                    if (o) atomicOr(w + i, o);
                    prev = cur;
                }
                const unsigned tail = __funnelshift_r(0u, prev, sh);  // (sh == 0: nothing left over)
                if (tail) atomicOr(w + nw, tail);
            } else {
                BitSink sink;
                sink.init(win, off);
                walk_block<true, BitSink>(cb, mask_lo, mask_hi, hdc, hac, &sink);
                sink.flush();
            }
        }
        __syncwarp();
        // ---- 3b. stage ----
        const unsigned pos = (unsigned)u * kWarpWinWords;
        if (lane == 0) unit_info[(long long)f * units_cap + u] = unit_pack(pos, unit_len);
        // (16 bytes per lane; the unit's fixed place and the window are 16-byte aligned, the words behind nwords up to the next
        // multiple of four are zeros inside the unit's own place)
        uint4 *dst4 = reinterpret_cast<uint4 *>(st + pos);
        const uint4 *src4 = reinterpret_cast<const uint4 *>(win);
        const unsigned nquads = (nwords + 3) >> 2;
        if ((unsigned)lane < nquads) dst4[lane] = src4[lane];  // (a unit of natural content: a dozen quads)
        for (unsigned i = lane + 32; i < nquads; i += 32) dst4[i] = src4[i];
    } else {
        unsigned pos;
        const unsigned n_fit = claim(lane == 0 ? fixed_words + atomicAdd(&stage_alloc[f], nwords) : 0u, pos);
        for (unsigned lo = 0; lo < unit_len; lo += kWarpWinBits) {
            const unsigned hi = min(lo + (unsigned)kWarpWinBits, unit_len);
            __syncwarp();  // previous window fully staged
            for (int i = lane; i < kWarpWinStride; i += 32) win[i] = 0;
            __syncwarp();
            if (valid && off < hi && off + len > lo) {
                BitSinkClip sink;
                sink.init(win, off, lo, hi);
                walk_block<true, BitSinkClip>(cb, mask_lo, mask_hi, hdc, hac, &sink);
            }
            __syncwarp();
            const unsigned nw = (hi - lo + 31) >> 5, w0 = lo >> 5;
            for (unsigned i = lane; i < nw; i += 32)
                if (w0 + i < n_fit) st[pos + w0 + i] = win[i];
        }
    }
}

// grid (groups_per_frame * frames), groups taken through a ticket so that every predecessor group is running.
// Bit positions are 32-bit: h2j_create bounds max_jpeg_bytes to 256 MiB.
// UPW = units a warp concatenates: 32 (256 threads, throughput form) or 8 (1024 threads: the same group spread over four
// times as many warps, for batches too small to fill the GPU with groups -- one 1080p frame is six groups, and a warp that
// walks 32 units one after the other takes ~19 us).
// LIST: a list batch (h2j_common.cuh FrameDesc); groups_per_frame is the largest frame's, and a ticket past its frame's groups
// returns at once (nobody waits for it: the look-back only reads earlier groups of the same frame)
template <int UPW, bool LIST>
__global__ void __launch_bounds__(kPlaceGroupUnits / UPW * 32) scan_place_kernel(FrameLayout L_, FrameTab *__restrict__ tabs, FrameState *__restrict__ state,
                                                                   const unsigned long long *__restrict__ unit_info, int units_cap,
                                                                   const uint32_t *__restrict__ stage, long long stage_cap_words,
                                                                   unsigned long long *__restrict__ descs, int groups_per_frame,
                                                                   unsigned int *__restrict__ ticket, uint32_t *__restrict__ scan,
                                                                   long long scan_cap_words, unsigned int *__restrict__ chunk_ff, int chunks_cap,
                                                                   const FrameDesc *__restrict__ fdescs)
{
    static_assert(kPlaceGroupUnits == kPlaceThreads, "one unit per thread in the scan (the first 256 threads)");
    static_assert(UPW == 32 || UPW == 8, "units per warp");
    __shared__ unsigned s_pos[kPlaceGroupUnits + 1];    // staging position of the unit; [0] = the unit in front of the group
    __shared__ unsigned s_len[kPlaceGroupUnits + 1];    // its bit length
    __shared__ unsigned s_excl[kPlaceGroupUnits + 1];   // exclusive bit prefix inside the frame; [n_here] = end of the group
    __shared__ unsigned s_wsum[kPlaceThreads / 32];
    __shared__ unsigned s_base;
    __shared__ unsigned s_ticket;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    const int f = (int)(s_ticket / (unsigned)groups_per_frame);
    const int g = (int)(s_ticket % (unsigned)groups_per_frame);
    const FrameLayout &L = LIST ? fdescs[f].L : L_;
    const int n_units = (L.n_blocks + kUnitBlocks - 1) / kUnitBlocks;
    const int u0 = g * kPlaceGroupUnits;
    if (LIST && u0 >= n_units) return;
    const int n_here = min(kPlaceGroupUnits, n_units - u0);  // >= 1 by construction of groups_per_frame
    const unsigned long long *info = unit_info + (long long)f * units_cap;

    // ---- lengths of the group's units, block scan ----
    const unsigned long long rec = tid < n_here ? info[u0 + tid] : 0ull;  // (threads behind the first 256 carry zeros)
    // a unit that did not fit the staging buffer gets the top bit of its position: the frame is reported, not read
    const unsigned cap_w = (unsigned)min(stage_cap_words, (long long)0x7fffffff);
    auto checked_pos = [&](unsigned long long r) {
        const unsigned pos = unit_pos(r), nw = (unit_bits(r) + 31) >> 5;
        return (pos > cap_w || nw > cap_w - pos) ? (pos | 0x80000000u) : pos;
    };
    if (tid < kPlaceGroupUnits) {
        s_pos[1 + tid] = checked_pos(rec);
        s_len[1 + tid] = unit_bits(rec);
    }
    if (tid == 0) {
        const unsigned long long rp = u0 > 0 ? info[u0 - 1] : 0ull;
        s_pos[0] = checked_pos(rp);
        s_len[0] = unit_bits(rp);
    }
    unsigned incl = unit_bits(rec);
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31 && warp < kPlaceThreads / 32) s_wsum[warp] = incl;
    __syncthreads();
    unsigned warp_off = 0, group_total = 0;
#pragma unroll
    for (int w = 0; w < kPlaceThreads / 32; w++) {
        if (w < warp) warp_off += s_wsum[w];
        group_total += s_wsum[w];
    }

    // ---- the group's exclusive prefix: decoupled look-back over the frame's earlier groups (warp 0) ----
    unsigned long long *D = descs + (long long)f * groups_per_frame;
    if (warp == 0) {
        if (lane == 0) st_desc(&D[g], desc_pack(g > 0 ? 1 : 2, group_total));
        unsigned excl = 0;
        if (g > 0) {
            int basei = g - 1;
            while (true) {
                const int idx = basei - lane;
                unsigned long long d;
                if (idx >= 0) {
                    do { d = ld_desc(&D[idx]); } while (desc_status(d) == 0);
                } else d = desc_pack(2, 0);
                const unsigned pm = __ballot_sync(0xffffffffu, desc_status(d) == 2);
                const int stop = pm ? (__ffs(pm) - 1) : 31;
                unsigned part = lane <= stop ? (unsigned)desc_len(d) : 0u;
#pragma unroll
                for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                excl += part;
                if (pm) break;
                basei -= 32;
            }
            if (lane == 0) st_desc(&D[g], desc_pack(2, excl + group_total));
        }
        if (lane == 0) { s_base = excl; s_excl[n_here] = excl + group_total; }
    }
    __syncthreads();
    if (tid < n_here) s_excl[tid] = s_base + warp_off + incl - unit_bits(rec);
    __syncthreads();

    // ---- place: bit-stream concatenation, a warp per run of 32 consecutive units.  The warp walks its units in order and
    //      carries the bits of the word that is still incomplete (c = P & 31 of them) from one unit to the next; lane l
    //      builds the unit's l-th output word from two neighbouring staged words (coalesced loads, coalesced 4-byte
    //      stores), and the lane behind the last complete word hands the new carry to everybody.  Only the first unit of a
    //      run fetches its carry from the staged unit in front.  (The first form of this step gathered per output word --
    //      bisection over the prefix table, two or three dependent scattered loads -- and was bound by their latency.) ----
    const uint32_t *st = stage + (long long)f * stage_cap_words;
    uint32_t *gs = scan + (long long)f * scan_cap_words;
    unsigned int *cff = chunk_ff + (long long)f * chunks_cap;
    const bool has_final = u0 + n_here == n_units;
    if (has_final && tid == 0) state[f].scan_bits = s_excl[n_here];
    const unsigned cap_scan = (unsigned)min(scan_cap_words, (long long)0x7fffffff);
    bool overflow = false;
    auto emit = [&](unsigned W, unsigned x) {  // x: the word's 32 stream bits, first bit in bit 31
        if (W < cap_scan) {  // (words behind the frame's capacity are dropped: the frame is reported, K5 never reads them)
            gs[W] = __byte_perm(x, 0, 0x0123);
            const unsigned nff = count_ff_bytes(x);
            if (nff) atomicAdd(&cff[W >> kChunkShift], nff);
        } else overflow = true;
    };
    const int ub = warp * UPW, ue = min(ub + UPW, n_here);
    if (ub < ue) {
        unsigned P = s_excl[ub], c = P & 31, carry = 0;
        if (c) {  // the last c bits in front of P: the tail of the unit in front (never shorter than a word)
            const unsigned plen = s_len[ub], ppos = s_pos[ub];
            if (ppos & 0x80000000u) overflow = true;  // not staged completely: the frame is reported, not read
            else {
                const uint32_t *pw = st + ppos;
                const unsigned lw = (plen - 1) >> 5, q = ((plen - 1) & 31) + 1;  // its last word and the bits used in it
                const unsigned hiw = lw ? __ldg(pw + lw - 1) : 0u;
                const unsigned tail = __funnelshift_r(__ldg(pw + lw), hiw, 32 - q);  // its last 32 bits, right aligned
                carry = tail & ((1u << c) - 1u);
            }
        }
        // A unit's first 64 staged words (256 bytes: natural content rarely has more) are loaded up front, one or two per
        // lane, for kPlaceBatch units at a time: nothing a unit needs from memory depends on the unit in front (its
        // carry-in only touches word 0), so 2 * kPlaceBatch loads per lane are in flight instead of one round trip after
        // the other.
        auto fetch = [&](int i, unsigned &a0, unsigned &a1) {
            a0 = 0; a1 = 0;
            if (i >= ue) return;
            const unsigned pos = s_pos[1 + i], nw = (s_len[1 + i] + 31) >> 5;  // staged words (the last one zero padded)
            if (pos & 0x80000000u) return;
            const uint32_t *uw = st + pos;
            if ((unsigned)lane < nw) a0 = __ldg(uw + lane);
            if ((unsigned)lane + 32 < nw) a1 = __ldg(uw + 32 + lane);
        };
        // virtual word k of a unit = the c carried bits + unit bits [32k - c, 32k - c + 32); the first n = (c + len) >> 5 of
        // them are complete output words, word n holds the (c + len) & 31 bits the unit leaves open
        auto place = [&](int i, unsigned a0, unsigned a1) {
            if (i >= ue) return;
            const unsigned pos = s_pos[1 + i], len = s_len[1 + i];
            const bool staged = !(pos & 0x80000000u);
            if (!staged) overflow = true;  // not staged completely: the frame is reported, not read
            const unsigned Wfirst = P >> 5;
            const unsigned n = (c + len) >> 5, c2 = (c + len) & 31;
            unsigned open_word;
            {
                const unsigned up = __shfl_up_sync(0xffffffffu, a0, 1);
                const unsigned prv = lane ? up : carry;
                const unsigned x = c ? (prv << (32 - c)) | (a0 >> c) : a0;
                if ((unsigned)lane < n) emit(Wfirst + lane, x);
                open_word = __shfl_sync(0xffffffffu, x, (int)(n & 31));
            }
            if (n >= 32) {
                const unsigned up = __shfl_up_sync(0xffffffffu, a1, 1), last0 = __shfl_sync(0xffffffffu, a0, 31);
                const unsigned prv = lane ? up : last0;
                const unsigned x = c ? (prv << (32 - c)) | (a1 >> c) : a1;
                if ((unsigned)lane + 32 < n) emit(Wfirst + 32 + lane, x);
                open_word = __shfl_sync(0xffffffffu, x, (int)(n & 31));
                const uint32_t *uw = st + (staged ? pos : 0u);
                const unsigned nw = staged ? (len + 31) >> 5 : 0u;
                for (unsigned k0 = 64; k0 <= n; k0 += 32) {  // long units: straight from memory
                    const unsigned k = k0 + lane;
                    unsigned xx = 0;
                    if (k <= n) {
                        const unsigned cur = k < nw ? __ldg(uw + k) : 0u;
                        const unsigned prv2 = k - 1 < nw ? __ldg(uw + k - 1) : 0u;
                        xx = c ? (prv2 << (32 - c)) | (cur >> c) : cur;
                        if (k < n) emit(Wfirst + k, xx);
                    }
                    open_word = __shfl_sync(0xffffffffu, xx, (int)(n & 31));
                }
            }
            carry = c2 ? open_word >> (32 - c2) : 0u;
            c = c2;
            P += len;
        };
        for (int i = ub; i < ue; i += kPlaceBatch) {
            unsigned a0[kPlaceBatch], a1[kPlaceBatch];
#pragma unroll
            for (int j = 0; j < kPlaceBatch; j++) fetch(i + j, a0[j], a1[j]);
#pragma unroll
            for (int j = 0; j < kPlaceBatch; j++) place(i + j, a0[j], a1[j]);
        }
        if (has_final && ue == n_here && c && lane == 0) {
            // the frame's last, partial word: 1-padding up to the byte boundary (put_bits / picture trailer), zeros after it
            const unsigned padn = (8 - (c & 7)) & 7;
            emit(P >> 5, (carry << (32 - c)) | (((1u << padn) - 1u) << (32 - c - padn)));
        }
    }
    if (overflow) tabs[f].status = -4;
}

}  // namespace h2j
