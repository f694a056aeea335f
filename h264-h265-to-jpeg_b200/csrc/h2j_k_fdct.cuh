// K2: pixels -> quantised zigzag coefficients, DC differences and symbol statistics.
//
// One thread owns one 8x8 block with all 64 values in registers.  A tile is 16 consecutive MCUs in coding order
// (it may wrap to the next MCU row); `tiles_per_cta` consecutive tiles are walked by three single-warp CTAs, one per
// role (blockIdx.x = tile group * 3 + role):
//   role 0: the four luma blocks of MCUs 0..7   (lane = mcu * 4 + n: lane order IS coding order)
//   role 1: the four luma blocks of MCUs 8..15
//   role 2: Cb of the 16 MCUs (lanes 0-15), Cr (lanes 16-31)
// A CTA is ONE warp because the warps share nothing: with three-warp CTAs the registers of a finished warp stayed
// allocated until the slowest of the three (luma and chroma blocks differ in their number of non-zero levels) reached
// the closing barrier -- 8.5 % of the stall samples -- and 128 registers x 96 threads fits five times per SM (15 warps),
// while 128 x 32 fits sixteen times.
// With this mapping every DC predictor (mjpegenc.c encode_block: the previous block of the same component) is
// the neighbouring lane's DC, so prediction is one shuffle and the warps never wait for each other.  The first
// lane of a run needs the block in front of the warp's range; its DC is recomputed from the pixels: the DC
// output of ff_fdct_sse2 is exactly the sum of the 64 samples (8 * column sums, then (8*S*16384 + 65536) >> 17
// == S), so eight lanes add one pixel row each -- no second FDCT.
//
// The tile image (h2j_common.cuh) is three sub-images, one per role.  A warp assembles its sub-image in one of its two
// shared-memory buffers and sends it with its own bulk (TMA) store.
// Pixel rows of the next tile are requested before the statistics of the current one are taken, so their latency
// is covered by work.
//
// The frame's qscale and quantiser tables are set up once per frame by the last CTA of K1 (h2j_k_planes.cuh).
#pragma once
#include "h2j_common.cuh"

namespace h2j {

constexpr int kFdctMinCtas = 16;  // resident single-warp CTAs per SM the register allocation is bounded for (16 -> 128 registers)
constexpr int kHistDummy = 257;   // s_hist: where the statistics walk counts a level that is not there (count_if)

// What a thread needs to know about the plane its block lives in: fixed for the whole kernel.
struct PlaneRef {
    const uint8_t *P;
    int pitch, pw, ph;   // row pitch in bytes, width in BYTES / height in rows the encoder reads (edges are replicated beyond)
    int step, xstep;     // block spacing per MCU in rows (16 luma, 8 chroma) and in bytes (the same, but 16 for NV12 chroma)
    int xoff, yoff;      // block offset inside the MCU (bytes / rows)
    bool can_fast;       // rows start 8-byte aligned: 64-bit loads
};
// NV12 (template parameter of the kernel): the chroma plane holds Cb/Cr PAIRS, so an MCU's two chroma blocks are the 16
// bytes [16 mx, 16 mx + 16) of eight rows; the Cb lane fetches the first eight bytes of every row, the Cr lane (16 lanes
// up) the other eight, and they trade halves before the transform (nv12_trade).
template <bool NV12> __device__ __forceinline__ PlaneRef plane_ref(const uint8_t *base, const FrameLayout &L, int n)
{
    PlaneRef r;
    if (n < 4) {
        r.P = base; r.pitch = L.y_pitch; r.pw = L.w; r.ph = L.h; r.step = 16; r.xstep = 16;
        r.xoff = (n & 1) * 8; r.yoff = (n >> 1) * 8;
    } else if (NV12) {
        r.P = base + L.u_off; r.pitch = L.c_pitch; r.pw = 2 * L.cw; r.ph = L.ch; r.step = 8; r.xstep = 16;
        r.xoff = (n - 4) * 8; r.yoff = 0;
    } else {
        r.P = base + (n == 4 ? L.u_off : L.v_off); r.pitch = L.c_pitch; r.pw = L.cw; r.ph = L.ch; r.step = 8; r.xstep = 8;
        r.xoff = 0; r.yoff = 0;
    }
    r.can_fast = L.aligned8 != 0;
    return r;
}

// Top-left sample of a thread's block in its plane plus the MCU index; advances a tile (16 MCUs) at a time without
// dividing.  mx = -1, my = 0 stands for "the MCU in front of MCU 0" (never dereferenced) and advances correctly.
struct BlockPos {
    int m, bx, by;
    __device__ __forceinline__ void init(int m_, const PlaneRef &R, int mcu_w)
    {
        m = m_;
        const int my = m_ / mcu_w, mx = m_ - my * mcu_w;  // m_ = -1: my = 0, mx = -1
        bx = mx * R.xstep + R.xoff;
        by = my * R.step + R.yoff;
    }
    __device__ __forceinline__ void advance(const PlaneRef &R, int mcu_w)
    {
        const int row_w = mcu_w * R.xstep;  // bx = mx * xstep + xoff with xoff < xstep: bx >= row_w <=> mx >= mcu_w
        m += kTileMcus;
        bx += kTileMcus * R.xstep;
        while (bx >= row_w) { bx -= row_w; by += R.step; }
    }
};

// The pixel rows a thread has in flight for its block of the coming tile.  The loads are ALWAYS issued and ALWAYS unpacked
// (blocks that do not exist, unaligned rows and rows cut by the right edge read the frame's first bytes instead and are
// then re-read bytewise): with loads and consumers under matching branches, ptxas could not tell that the registers were
// free again, and the first instruction touching them waited on a scoreboard shared with the load issued just before
// (5 % of the stall samples); flags kept across the transform were spilled to local memory (8 %).
struct BlockFetch {
    uint2 rows[8];
    uint2 prow;          // lanes that help with a predecessor DC: one row of that block
};
// C = the block is an NV12 chroma block: the vector path needs the MCU's whole 16 bytes inside the row (both lanes of a
// Cb/Cr pair take the same path, they trade halves), and sample c of the block is byte 2 * (x + c) + component.
template <bool C> __device__ __forceinline__ bool fetch_is_fast(const PlaneRef &R, int bx)
{
    return R.can_fast && (C ? bx - R.xoff + 16 : bx + 8) <= R.pw;
}
template <bool C> __device__ __forceinline__ int sample_at(const uint8_t *row, const PlaneRef &R, int bx, int c)
{
    if (C) return row[2 * min(((bx - R.xoff) >> 1) + c, (R.pw >> 1) - 1) + (R.xoff >> 3)];
    return row[min(bx + c, R.pw - 1)];
}

template <bool C, bool CQ>
__device__ __forceinline__ void fetch_issue(BlockFetch &F, const uint8_t *safe, const PlaneRef &R, const BlockPos &bp, bool valid,
                                            const PlaneRef &Q, const BlockPos &pp, bool phelp, int prow_idx)
{
    const bool pf = !CQ && phelp && fetch_is_fast<false>(Q, pp.bx);  // (NV12 chroma: the predecessor rows are read bytewise)
    const bool rf = valid && fetch_is_fast<C>(R, bp.bx);
    const uint8_t *pq = pf ? Q.P + (long long)min(pp.by + prow_idx, Q.ph - 1) * Q.pitch + pp.bx : safe;
    F.prow = ldg64(pq);
    if (!rf || bp.by + 8 <= R.ph) {  // interior: one address, then a pitch per row
        const uint8_t *p = rf ? R.P + (long long)bp.by * R.pitch + bp.bx : safe;
        const int pitch = rf ? R.pitch : 0;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            F.rows[r] = ldg64(p);
            p += pitch;
        }
    } else {
#pragma unroll
        for (int r = 0; r < 8; r++) F.rows[r] = ldg64(R.P + (long long)min(bp.by + r, R.ph - 1) * R.pitch + bp.bx);
    }
}

// NV12 chroma warp, all 32 lanes: every row arrives as four Cb/Cr pairs; the Cb lane keeps the four Cb samples and hands
// the four Cr samples to the Cr lane of its MCU (16 lanes up), which hands back the Cb samples of ITS four pairs.
__device__ __forceinline__ void nv12_trade(BlockFetch &F, bool cr_lane)
{
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const unsigned cb4 = __byte_perm(F.rows[r].x, F.rows[r].y, 0x6420), cr4 = __byte_perm(F.rows[r].x, F.rows[r].y, 0x7531);
        const unsigned keep = cr_lane ? cr4 : cb4;
        const unsigned got = __shfl_xor_sync(0xffffffffu, cr_lane ? cb4 : cr4, 16);
        F.rows[r] = cr_lane ? make_uint2(got, keep) : make_uint2(keep, got);  // Cb lane had pairs 0-3, Cr lane pairs 4-7
    }
}

// The block's 64 samples from its eight rows of eight bytes (`rows`, as fetched or with the component's bytes picked out),
// then re-read bytewise with sample(row pointer, c) where the vector rows are not the block's (`fast` false), then through
// the range LUT.
template <class Sample>
__device__ __forceinline__ void unpack_block(const uint2 (&rows)[8], bool fast, const PlaneRef &R, const BlockPos &bp, Sample sample,
                                             const uint8_t *lut, int (&v)[64])
{
#pragma unroll
    for (int r = 0; r < 8; r++) {
        // one byte permute per sample (selector 4 = a zero byte of the second operand)
        v[r * 8 + 0] = (int)__byte_perm(rows[r].x, 0u, 0x4440);
        v[r * 8 + 1] = (int)__byte_perm(rows[r].x, 0u, 0x4441);
        v[r * 8 + 2] = (int)__byte_perm(rows[r].x, 0u, 0x4442);
        v[r * 8 + 3] = (int)__byte_perm(rows[r].x, 0u, 0x4443);
        v[r * 8 + 4] = (int)__byte_perm(rows[r].y, 0u, 0x4440);
        v[r * 8 + 5] = (int)__byte_perm(rows[r].y, 0u, 0x4441);
        v[r * 8 + 6] = (int)__byte_perm(rows[r].y, 0u, 0x4442);
        v[r * 8 + 7] = (int)__byte_perm(rows[r].y, 0u, 0x4443);
    }
    if (!fast) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint8_t *row = R.P + (long long)min(bp.by + r, R.ph - 1) * R.pitch;
#pragma unroll
            for (int c = 0; c < 8; c++) v[r * 8 + c] = sample(row, c);
        }
    }
    if (lut) {
#pragma unroll
        for (int i = 0; i < 64; i++) v[i] = lut[v[i]];
    }
}

template <bool C>
__device__ __forceinline__ void fetch_consume(const BlockFetch &F, const PlaneRef &R, const BlockPos &bp, const uint8_t *lut, int (&v)[64])
{
    unpack_block(F.rows, fetch_is_fast<C>(R, bp.bx), R, bp, [&](const uint8_t *row, int c) { return sample_at<C>(row, R, bp.bx, c); }, lut, v);
}

// this lane's share (one pixel row) of the predecessor block's sample sum
template <bool CQ>
__device__ __forceinline__ int fetch_pred_rowsum(const BlockFetch &F, const PlaneRef &Q, const BlockPos &pp, bool phelp, int prow_idx,
                                                 const uint8_t *lut)
{
    int s = (int)__dp4a(F.prow.y, 0x01010101u, __dp4a(F.prow.x, 0x01010101u, 0u));
    if (!phelp) return 0;
    if (CQ || !fetch_is_fast<false>(Q, pp.bx) || lut) {
        const uint8_t *row = Q.P + (long long)min(pp.by + prow_idx, Q.ph - 1) * Q.pitch;
        s = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int p = sample_at<CQ>(row, Q, pp.bx, c);
            s += lut ? lut[p] : p;
        }
    }
    return s;
}

// ---- the per-block core of both K2 kernels (fdct_quant_kernel, fdct_quant_fmt_kernel) ----

// the frame's quantiser (set up once per frame by K1's last CTA) into shared memory, the CTA's statistics cleared
__device__ __forceinline__ void k2_setup(const FrameTab &tab, int *s_q, int *s_bq, unsigned int *s_hist, unsigned int *s_dchist, int lane)
{
    const uint2 pk = reinterpret_cast<const uint2 *>(tab.qpack)[lane];
    s_q[2 * lane] = (int)(pk.x & 0xffffu);
    s_bq[2 * lane] = (int)(pk.x >> 16);
    s_q[2 * lane + 1] = (int)(pk.y & 0xffffu);
    s_bq[2 * lane + 1] = (int)(pk.y >> 16);
#pragma unroll
    for (int i = 0; i < 8; i++) s_hist[i * 32 + lane] = 0;
    if (lane < 16) s_dchist[lane] = 0;
    __syncwarp();
}

// Transform, quantise, zigzag and pack the block's samples into its record `rec` of the sub-image `img` (h2j_common.cuh).
// Returns the quantised DC; its difference goes into the low half of word 0 later (count_block_symbols), the high half of
// word 0 is left in word0_hi.
__device__ __forceinline__ int quantise_record(int (&v)[64], const int *s_q, const int *s_bq, uint32_t *rec, uint32_t *img, int lane,
                                               unsigned &mask_lo, unsigned &mask_hi, uint32_t &word0_hi)
{
    fdct_8x8(v);
    const int dc = quant_dc(v[0]);
    // quantise without the final >> 16: the level is the upper half of the 32-bit product, so two of them
    // are packed into one record word with a single byte permute
#pragma unroll
    for (int i = 1; i < 64; i++) v[i] = quant_ac2_hi(v[i], s_q[i], s_bq[i]);
    // zigzag; word j of the record holds levels j (low half) and j + 32 (high half), so that the non-zero
    // flags of 32 levels fall out of 16 packed min(x, 1) results shifted into place (VIMNMX.U16x2)
    unsigned fa = 0, fb = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const uint32_t w = j == 0 ? __byte_perm(0u, (uint32_t)v[zz_of(32)], 0x7610) : __byte_perm((uint32_t)v[zz_of(j)], (uint32_t)v[zz_of(j + 32)], 0x7632);
        const unsigned t = __vminu2(w, 0x00010001u);
        if (j < 16) fa += t << j;
        else fb += t << (j - 16);
        if (j == 0) word0_hi = w;  // the low half becomes the DC difference
        else rec[j] = w;
    }
    mask_lo = ((fa & 0xffffu) | (fb << 16)) & ~1u;  // bit 0 is the DC position: always coded, never in the mask
    mask_hi = (fa >> 16) | (fb & 0xffff0000u);
    rec[kMaskLoWord] = mask_lo;
    img[kSubMaskHiOff + lane] = mask_hi;
    return dc;
}

// Completes the record with the DC difference to the previous block of the same component (mjpegenc.c encode_block) and
// counts the block's DC and AC symbols (ff_mjpeg_encode_coef / record_block) into the CTA's histograms.
__device__ __forceinline__ void count_block_symbols(uint32_t *rec, int diff, uint32_t word0_hi, unsigned mask_lo, unsigned mask_hi,
                                                    unsigned int *s_hist, unsigned int *s_dchist)
{
    rec[0] = (uint32_t)(diff & 0xffff) | word0_hi;
    atomicAdd(&s_dchist[mag_bits(diff)], 1u);
    // The (run, size) symbol of a non-zero level needs only its position, the position of the non-zero level below it and
    // its value, so the levels can be visited in any order.  Positions 1..31 (where nearly all of them are) are taken two
    // at a time from the low end: two independent bit-scan -> load -> size -> atomic chains per trip instead of one, half
    // the trips (three or four per trip, and two from opposite ends, measured slower: DESIGN.md section 4).
    const int16_t *lv = reinterpret_cast<const int16_t *>(rec);
    unsigned zrl = 0;  // 16-zero runs (symbol 0xF0): summed here, one update per block
    auto count = [&](int k, int below, int val) {  // val != 0
        const int run = k - below - 1;
        unsigned top;  // size - 1: the + 1 rides in the address (size <= 15, no carry into the run nibble)
        asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(abs(val)));
        zrl += (unsigned)run >> 4;
        atomicAdd(&s_hist[1 + (((run & 15) << 4) | (int)top)], 1u);
    };
    // the same for a level a lane may not have, WITHOUT a branch: in a walking warp some lane has it, so the warp ran the
    // branch's body anyway plus the branch and its reconvergence point (K2 5.458 -> 5.376 ms per 2048 frames); a lane
    // without the level counts into a word nobody reads
    auto count_if = [&](bool have, int k, int below, int val) {
        const int run = k - below - 1;
        unsigned top;
        asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(abs(val)));
        zrl += have ? (unsigned)run >> 4 : 0u;
        atomicAdd(&s_hist[have ? 1 + (((run & 15) << 4) | (int)top) : kHistDummy], 1u);
    };
    unsigned lo = mask_lo;
    const int top_lo = lo ? 31 - __clz(lo) : 0;  // highest non-zero position below 32 (0: none but the DC)
    int below = 0;
    while (lo) {
        const unsigned b0 = lo & (0u - lo);
        lo ^= b0;
        const unsigned b1 = lo & (0u - lo);
        lo ^= b1;
        const int k0 = 31 - __clz(b0), k1 = 31 - __clz(b1);  // k1 = -1: absent
        const int v0 = (int)lv[2 * k0], v1 = (int)lv[2 * max(k1, 0)];
        count(k0, below, v0);
        count_if(b1 != 0, k1, k0, v1);
        below = 31 - __clz(b0 | b1);
    }
    int prev = top_lo;
    unsigned hi = mask_hi;
    while (hi) {
        const int bp = __ffs((int)hi) - 1, k = 32 + bp;
        hi &= hi - 1;
        count(k, prev, (int)lv[2 * bp + 1]);
        prev = k;
    }
    if (prev < 63) atomicAdd(&s_hist[0], 1u);
    if (zrl) atomicAdd(&s_hist[0xf0], zrl);
}

// the CTA's statistics into the frame's histograms (class 0 luma, 1 chroma)
__device__ __forceinline__ void k2_flush(FrameState &st, int cls, const unsigned int *s_hist, const unsigned int *s_dchist, int lane)
{
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const unsigned c = s_hist[i * 32 + lane];
        if (c) atomicAdd(&st.hist[2 + cls][i * 32 + lane], c);
    }
    if (lane < 16) {
        const unsigned c = s_dchist[lane];
        if (c) atomicAdd(&st.hist[cls][lane], c);
    }
}

// LIST: a list batch (h2j_common.cuh FrameDesc): the frame's layout and address come from descs[blockIdx.y], and the grid is
// sized for the batch's largest frame (the CTAs past this frame's tiles return at the tile0 test)
template <bool NV12, bool LIST>
__global__ void __launch_bounds__(kFdctThreads, kFdctMinCtas) fdct_quant_kernel(const uint8_t *__restrict__ frames, FrameLayout L_,
                                                                     FrameState *__restrict__ state,
                                                                     const FrameTab *__restrict__ tabs,
                                                                     uint32_t *__restrict__ images,  // [frame][images_cap] tile images
                                                                     long long images_cap, int tiles_per_cta,
                                                                     const FrameDesc *__restrict__ descs)
{
    __shared__ __align__(128) uint32_t s_img[2][kSubImageWords];
    __shared__ __align__(16) int s_q[64];
    __shared__ __align__(16) int s_bq[64];
    __shared__ unsigned int s_hist[256 + 8];  // (+ kHistDummy, the word nobody reads)
    __shared__ unsigned int s_dchist[16];

    const int f = blockIdx.y;
    const int lane = threadIdx.x;
    const int group = blockIdx.x / 3, warp = blockIdx.x - group * 3;  // `warp` = the role of this single-warp CTA
    const FrameLayout &L = LIST ? descs[f].L : L_;
    const uint8_t *base = LIST ? descs[f].base : frames + (long long)f * L.frame_stride;
    const int n_tiles = (L.n_mcu + kTileMcus - 1) / kTileMcus;
    const int tile0 = group * tiles_per_cta;
    if (tile0 >= n_tiles) return;
    const int tile_end = min(tile0 + tiles_per_cta, n_tiles);

    // lane -> block of the tile
    const bool luma = warp < 2;
    const int mcu_l = luma ? warp * 8 + (lane >> 2) : (lane & 15);
    const int n = luma ? (lane & 3) : 4 + (lane >> 4);
    const int cls = luma ? 0 : 1;
    const uint8_t *lut = L.range_mode ? c_range_lut[cls] : nullptr;
    // predecessor block of the warp's first lane(s): luma -> Y3 of the MCU in front of the warp's eight;
    // chroma -> Cb (lanes 0-7 help) and Cr (lanes 8-15 help) of the MCU in front of the tile (first tile only)
    const bool phelp_lane = luma ? lane < 8 : lane < 16;
    const int mcu_first = luma ? warp * 8 : 0;
    const PlaneRef R = plane_ref<NV12>(base, L, n), Q = plane_ref<NV12>(base, L, luma ? 3 : 4 + (lane >> 3));
    const bool nvc = NV12 && !luma;  // this warp's blocks are NV12 chroma blocks (CTA-uniform)

    BlockFetch F;
    const uint8_t *safe = reinterpret_cast<const uint8_t *>(tabs);  // aligned, always readable: what skipped loads read
    BlockPos bp, pp;  // this thread's block / the predecessor block in front of the warp's range, for the tile being fetched
    bp.init(tile0 * kTileMcus + mcu_l, R, L.mcu_w);
    pp.init(tile0 * kTileMcus + mcu_first - 1, Q, L.mcu_w);
    // lanes that add a row of the predecessor block: chroma only needs it for its first tile (then the DC is carried)
    auto phelp_at = [&](int tile) { return phelp_lane && pp.m >= 0 && pp.m < L.n_mcu && (luma || tile == tile0); };
    if (nvc) fetch_issue<true, true>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_at(tile0), lane & 7);
    else fetch_issue<false, false>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_at(tile0), lane & 7);

    k2_setup(tabs[f], s_q, s_bq, s_hist, s_dchist, lane);

    int chroma_carry = 128;  // chroma warp, lanes 0 / 16: DC of the previous tile's last Cb / Cr block

    for (int tile = tile0; tile < tile_end; tile++) {
        // this warp's sub-image of the tile, in one of its two buffers; the store that used this buffer two tiles ago must
        // have read it out (lane 0 issued it, lane 0 waits)
        uint32_t *img = s_img[(tile - tile0) & 1];
        const bool valid = bp.m < L.n_mcu;
        if (lane == 0) bulk_wait_read_but_one();
        __syncwarp();

        // ---- predecessor DC for the first lane(s) of the warp, from pixel sums ----
        int psum = nvc ? fetch_pred_rowsum<true>(F, Q, pp, phelp_at(tile), lane & 7, lut) : fetch_pred_rowsum<false>(F, Q, pp, phelp_at(tile), lane & 7, lut);
        if (nvc) nv12_trade(F, lane >= 16);  // (all 32 lanes, outside `valid`: the lanes of a pair share their MCU)
        psum += __shfl_xor_sync(0xffffffffu, psum, 1);
        psum += __shfl_xor_sync(0xffffffffu, psum, 2);
        psum += __shfl_xor_sync(0xffffffffu, psum, 4);
        const int psum_cr = __shfl_sync(0xffffffffu, psum, 8);  // chroma: lanes 8-15 summed Cr
        const int pm = tile * kTileMcus + mcu_first - 1;
        int pred_first;  // meaningful in lane 0 (and lane 16 of the chroma warp)
        if (luma) pred_first = pm >= 0 ? quant_dc(psum) : 128;  // 128 = the encoder's initial last_dc (1024 >> 3)
        else if (tile == tile0) pred_first = pm >= 0 ? quant_dc(lane < 16 ? psum : psum_cr) : 128;
        else pred_first = chroma_carry;

        unsigned mask_lo = 0, mask_hi = 0;
        uint32_t word0_hi = 0;
        int dc = 0;
        uint32_t *rec = img + lane * kBlkWords;  // the lane order of every warp is its record order
        if (valid) {
            int v[64];
            if (nvc) fetch_consume<true>(F, R, bp, lut, v);
            else fetch_consume<false>(F, R, bp, lut, v);
            dc = quantise_record(v, s_q, s_bq, rec, img, lane, mask_lo, mask_hi, word0_hi);
        }

        // ---- request the next tile's pixels: nothing of this tile's 64-value block is live any more ----
        if (tile + 1 < tile_end) {
            bp.advance(R, L.mcu_w);
            pp.advance(Q, L.mcu_w);
            if (nvc) fetch_issue<true, true>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_at(tile + 1), lane & 7);
            else fetch_issue<false, false>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_at(tile + 1), lane & 7);
        }

        // ---- DC difference to the previous block of the same component (mjpegenc.c encode_block) ----
        const int up = __shfl_up_sync(0xffffffffu, dc, 1);
        const int pred = (luma ? lane == 0 : (lane & 15) == 0) ? pred_first : up;
        const int last = __shfl_sync(0xffffffffu, dc, (lane & 16) | 15);  // chroma: this tile's last Cb / Cr
        chroma_carry = last;
        if (valid) count_block_symbols(rec, dc - pred, word0_hi, mask_lo, mask_hi, s_hist, s_dchist);

        // ---- the warp's sub-image leaves with one bulk store ----
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0)
            bulk_s2g(images + ((long long)f * images_cap + tile) * kTileImageWords + warp * kSubImageWords, img, kSubImageBytes);
    }
    // the stores only have to be done READING shared memory before the CTA retires; they complete on their own and the
    // kernel boundary orders them before K4a
    if (lane == 0) bulk_wait_read_all();
    __syncwarp();
    k2_flush(state[f], cls, s_hist, s_dchist, lane);
}

}  // namespace h2j
