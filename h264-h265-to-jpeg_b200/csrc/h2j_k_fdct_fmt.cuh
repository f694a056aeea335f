// K2 for the encoder's other MCU geometries (DESIGN.md row f3): 4:2:2 and 4:4:4 frames (planar, as libavcodec's decoders
// hand them over: yuv422p / yuv444p).  Same work per block as fdct_quant_kernel -- pixel load with edge replication (+ range
// LUT), ff_fdct_sse2, quantise, zigzag, DC prediction by warp shuffle, symbol statistics, the role's sub-image of the tile
// image sent with one bulk store -- and the same helpers (h2j_k_fdct.cuh); what differs is who does what:
//   4:2:2  16x16 MCUs of Y0 Y1 Y2 Y3 Cb0 Cb1 Cr0 Cr1; four roles per 16-MCU tile: luma of MCUs 0-7 (lane = mcu * 4 + n), luma
//          of MCUs 8-15, Cb of the 16 MCUs (lane = mcu * 2 + n: top, bottom), Cr
//   4:4:4   8x16 MCUs of Y0 Y1 Cb0 Cb1 Cr0 Cr1 (every component top, bottom); three roles: Y (lane = mcu * 2 + n), Cb, Cr
// Every role holds ONE component in coding order, so a block's DC predecessor is the neighbouring lane's DC, and lane 0's
// is the component's last block of the MCU in front of the role's range, rebuilt from its pixel sum by eight helper lanes
// (the DC output of ff_fdct_sse2 is the sum of the 64 samples) -- for every tile, there is no chroma carry to keep.
// blockIdx.x = tile group * roles + role, single-warp CTAs, tiles_per_cta consecutive tiles per CTA.
// SP (semi-planar, L.nv12): chroma is ONE plane of interleaved Cb/Cr pairs (NV16 at 4:2:2, NV24 at 4:4:4), read in place.
// A chroma block's eight samples of a row are the 16 bytes of its eight pairs; every role holds one component, so each
// chroma lane fetches the whole 16 bytes and keeps its half (no lane trade as in fdct_quant_kernel's NV12 path).
#pragma once
#include "h2j_k_fdct.cuh"

namespace h2j {

// component c (0 Y, 1 Cb, 2 Cr), k-th block of that component inside the MCU (coding order)
template <int FMT, bool SP> __device__ __forceinline__ PlaneRef plane_ref_fmt(const uint8_t *base, const FrameLayout &L, int c, int k)
{
    PlaneRef r;
    if (c == 0) {
        r.P = base; r.pitch = L.y_pitch; r.pw = L.w; r.ph = L.h; r.step = 16;
        if (FMT == kFmt444) { r.xstep = 8; r.xoff = 0; r.yoff = k * 8; }          // Y top, Y bottom of an 8x16 MCU
        else { r.xstep = 16; r.xoff = (k & 1) * 8; r.yoff = (k >> 1) * 8; }       // Y0 Y1 / Y2 Y3
    } else if (SP) {  // the pair plane, positions in bytes: a block is 16 bytes wide, pw = the pairs the encoder reads
        r.P = base + L.u_off; r.pitch = L.c_pitch; r.pw = 2 * L.cw; r.ph = L.ch;
        r.step = 16; r.xstep = 16; r.xoff = 0; r.yoff = k * 8;
    } else {
        r.P = base + (c == 1 ? L.u_off : L.v_off); r.pitch = L.c_pitch; r.pw = L.cw; r.ph = L.ch;
        r.step = 16; r.xstep = 8; r.xoff = 0; r.yoff = k * 8;                      // top, bottom; chroma MCU step 8 x 16 in both formats
    }
    r.can_fast = L.aligned8 != 0;
    return r;
}

// ---- SP chroma lanes: `odd` = 0 for Cb (even bytes of the pair plane), 1 for Cr ----
// The second 8 bytes of each row of the block and of the predecessor row (the first 8 ride in BlockFetch).  Both halves
// are requested a tile ahead, as in the planar path: requesting the second halves at the top of the tile instead (16 fewer
// registers in flight across the statistics walk) left their latency exposed -- NV16 in place at 1.005x the prepass instead
// of 1.09x (DESIGN.md row (f)(4)).
struct PairHalves {
    uint2 hi[8];
    uint2 prow_hi;
};
__device__ __forceinline__ bool sp_is_fast(const PlaneRef &R, int bx) { return R.can_fast && bx + 16 <= R.pw; }
// sample c of the block at byte bx of a row, the right edge replicated: never a byte past the row's 2 * cw
__device__ __forceinline__ int sp_sample_at(const uint8_t *row, const PlaneRef &R, int bx, int c, int odd)
{
    return row[2 * min((bx >> 1) + c, (R.pw >> 1) - 1) + odd];
}

// as fetch_issue<false, false>, with the 16 bytes of each row as two 8-byte loads (the rows are 8-byte aligned), and the
// predecessor rows of the helper lanes likewise
__device__ __forceinline__ void sp_fetch_issue(BlockFetch &F, PairHalves &H, const uint8_t *safe, const PlaneRef &R, const BlockPos &bp,
                                               bool valid, const PlaneRef &Q, const BlockPos &pp, bool phelp, int prow_idx)
{
    const bool pf = phelp && sp_is_fast(Q, pp.bx);
    const uint8_t *pq = pf ? Q.P + (long long)min(pp.by + prow_idx, Q.ph - 1) * Q.pitch + pp.bx : safe;
    F.prow = ldg64(pq);
    H.prow_hi = ldg64(pq + 8);
    const bool rf = valid && sp_is_fast(R, bp.bx);
    if (!rf || bp.by + 8 <= R.ph) {
        const uint8_t *p = rf ? R.P + (long long)bp.by * R.pitch + bp.bx : safe;
        const int pitch = rf ? R.pitch : 0;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            F.rows[r] = ldg64(p);
            H.hi[r] = ldg64(p + 8);
            p += pitch;
        }
    } else {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint8_t *p = R.P + (long long)min(bp.by + r, R.ph - 1) * R.pitch + bp.bx;
            F.rows[r] = ldg64(p);
            H.hi[r] = ldg64(p + 8);
        }
    }
}

__device__ __forceinline__ void sp_fetch_consume(const BlockFetch &F, const PairHalves &H, const PlaneRef &R, const BlockPos &bp, int odd,
                                                 const uint8_t *lut, int (&v)[64])
{
    const unsigned sel = odd ? 0x7531u : 0x6420u;  // the Cr / Cb byte of four pairs
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const unsigned lo4 = __byte_perm(F.rows[r].x, F.rows[r].y, sel), hi4 = __byte_perm(H.hi[r].x, H.hi[r].y, sel);
        v[r * 8 + 0] = (int)__byte_perm(lo4, 0u, 0x4440);
        v[r * 8 + 1] = (int)__byte_perm(lo4, 0u, 0x4441);
        v[r * 8 + 2] = (int)__byte_perm(lo4, 0u, 0x4442);
        v[r * 8 + 3] = (int)__byte_perm(lo4, 0u, 0x4443);
        v[r * 8 + 4] = (int)__byte_perm(hi4, 0u, 0x4440);
        v[r * 8 + 5] = (int)__byte_perm(hi4, 0u, 0x4441);
        v[r * 8 + 6] = (int)__byte_perm(hi4, 0u, 0x4442);
        v[r * 8 + 7] = (int)__byte_perm(hi4, 0u, 0x4443);
    }
    if (!sp_is_fast(R, bp.bx)) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint8_t *row = R.P + (long long)min(bp.by + r, R.ph - 1) * R.pitch;
#pragma unroll
            for (int c = 0; c < 8; c++) v[r * 8 + c] = sp_sample_at(row, R, bp.bx, c, odd);
        }
    }
    if (lut) {
#pragma unroll
        for (int i = 0; i < 64; i++) v[i] = lut[v[i]];
    }
}

// this lane's share (one pixel row) of the predecessor block's sample sum
__device__ __forceinline__ int sp_pred_rowsum(const BlockFetch &F, const PairHalves &H, const PlaneRef &Q, const BlockPos &pp, bool phelp,
                                              int prow_idx, int odd, const uint8_t *lut)
{
    const unsigned sel = odd ? 0x7531u : 0x6420u;
    int s = (int)__dp4a(__byte_perm(H.prow_hi.x, H.prow_hi.y, sel), 0x01010101u, __dp4a(__byte_perm(F.prow.x, F.prow.y, sel), 0x01010101u, 0u));
    if (!phelp) return 0;
    if (!sp_is_fast(Q, pp.bx) || lut) {
        const uint8_t *row = Q.P + (long long)min(pp.by + prow_idx, Q.ph - 1) * Q.pitch;
        s = 0;
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int p = sp_sample_at(row, Q, pp.bx, c, odd);
            s += lut ? lut[p] : p;
        }
    }
    return s;
}

template <int FMT, bool SP>
__global__ void __launch_bounds__(kFdctThreads, H2J_FDCT_MIN_CTAS) fdct_quant_fmt_kernel(const uint8_t *__restrict__ frames, FrameLayout L,
                                                                         FrameState *__restrict__ state,
                                                                         const FrameTab *__restrict__ tabs,
                                                                         uint32_t *__restrict__ images,  // [frame][images_cap] tile images
                                                                         long long images_cap, int tiles_per_cta)
{
    constexpr int kRoles = fmt_roles(FMT);
    __shared__ __align__(128) uint32_t s_img[2][kSubImageWords];
    __shared__ __align__(16) int s_q[64];
    __shared__ __align__(16) int s_bq[64];
    __shared__ unsigned int s_hist[256 + 8];  // (+ kHistDummy)
    __shared__ unsigned int s_dchist[16];

    const int f = blockIdx.y;
    const int lane = threadIdx.x;
    const int group = blockIdx.x / kRoles, role = blockIdx.x - group * kRoles;
    const uint8_t *base = frames + (long long)f * L.frame_stride;
    const int n_tiles = (L.n_mcu + kTileMcus - 1) / kTileMcus;
    const int tile0 = group * tiles_per_cta;
    if (tile0 >= n_tiles) return;
    const int tile_end = min(tile0 + tiles_per_cta, n_tiles);

    // role -> component, blocks of it per MCU, first MCU of the tile the role covers; lane -> block
    const bool quad = FMT == kFmt422 && role < 2;  // four luma blocks per MCU, eight MCUs
    const int comp = FMT == kFmt444 ? role : (role < 2 ? 0 : role - 1);
    const int per_mcu = quad ? 4 : 2;
    const int mcu_first = quad ? role * 8 : 0;
    const int mcu_l = mcu_first + (quad ? lane >> 2 : lane >> 1);
    const int k = quad ? (lane & 3) : (lane & 1);
    const int cls = comp ? 1 : 0;
    const uint8_t *lut = L.range_mode ? c_range_lut[cls] : nullptr;
    const bool phelp_lane = lane < 8;  // add one pixel row each of the block in front of the role's range
    const PlaneRef R = plane_ref_fmt<FMT, SP>(base, L, comp, k), Q = plane_ref_fmt<FMT, SP>(base, L, comp, per_mcu - 1);
    const bool spc = SP && comp != 0;  // this role reads the pair plane (role-uniform)
    const int odd = comp - 1;          // (spc) the role's byte of a pair

    BlockFetch F;
    PairHalves H;
    const uint8_t *safe = reinterpret_cast<const uint8_t *>(tabs);  // aligned, always readable: what skipped loads read
    BlockPos bp, pp;
    bp.init(tile0 * kTileMcus + mcu_l, R, L.mcu_w);
    pp.init(tile0 * kTileMcus + mcu_first - 1, Q, L.mcu_w);
    auto phelp_now = [&]() { return phelp_lane && pp.m >= 0 && pp.m < L.n_mcu; };
    if (spc) sp_fetch_issue(F, H, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_now(), lane & 7);
    else fetch_issue<false, false>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_now(), lane & 7);

    {
        const uint2 pk = reinterpret_cast<const uint2 *>(tabs[f].qpack)[lane];
        s_q[2 * lane] = (int)(pk.x & 0xffffu);
        s_bq[2 * lane] = (int)(pk.x >> 16);
        s_q[2 * lane + 1] = (int)(pk.y & 0xffffu);
        s_bq[2 * lane + 1] = (int)(pk.y >> 16);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) s_hist[i * 32 + lane] = 0;
    if (lane < 16) s_dchist[lane] = 0;
    __syncwarp();

    for (int tile = tile0; tile < tile_end; tile++) {
        uint32_t *img = s_img[(tile - tile0) & 1];
        const bool valid = bp.m < L.n_mcu;
        if (lane == 0) bulk_wait_read_but_one();
        __syncwarp();

        // ---- predecessor DC of lane 0, from pixel sums ----
        int psum = spc ? sp_pred_rowsum(F, H, Q, pp, phelp_now(), lane & 7, odd, lut) : fetch_pred_rowsum<false>(F, Q, pp, phelp_now(), lane & 7, lut);
        psum += __shfl_xor_sync(0xffffffffu, psum, 1);
        psum += __shfl_xor_sync(0xffffffffu, psum, 2);
        psum += __shfl_xor_sync(0xffffffffu, psum, 4);
        const int pm = tile * kTileMcus + mcu_first - 1;
        const int pred_first = pm >= 0 ? quant_dc(psum) : 128;  // 128 = the encoder's initial last_dc (1024 >> 3)

        unsigned mask_lo = 0, mask_hi = 0;
        uint32_t word0_hi = 0;
        int dc = 0;
        uint32_t *rec = img + lane * kBlkWords;
        if (valid) {
            int v[64];
            if (spc) sp_fetch_consume(F, H, R, bp, odd, lut, v);
            else fetch_consume<false>(F, R, bp, lut, v);
            fdct_8x8(v);
            dc = quant_dc(v[0]);
#pragma unroll
            for (int i = 1; i < 64; i++) v[i] = quant_ac2_hi(v[i], s_q[i], s_bq[i]);
            unsigned fa = 0, fb = 0;
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const uint32_t w = j == 0 ? __byte_perm(0u, (uint32_t)v[zz_of(32)], 0x7610) : __byte_perm((uint32_t)v[zz_of(j)], (uint32_t)v[zz_of(j + 32)], 0x7632);
                const unsigned t = __vminu2(w, 0x00010001u);
                if (j < 16) fa += t << j;
                else fb += t << (j - 16);
                if (j == 0) word0_hi = w;
                else rec[j] = w;
            }
            mask_lo = ((fa & 0xffffu) | (fb << 16)) & ~1u;
            mask_hi = (fa >> 16) | (fb & 0xffff0000u);
            rec[kMaskLoWord] = mask_lo;
            img[kSubMaskHiOff + lane] = mask_hi;
        }

        // ---- request the next tile's pixels ----
        if (tile + 1 < tile_end) {
            bp.advance(R, L.mcu_w);
            pp.advance(Q, L.mcu_w);
            if (spc) sp_fetch_issue(F, H, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_now(), lane & 7);
            else fetch_issue<false, false>(F, safe, R, bp, bp.m < L.n_mcu, Q, pp, phelp_now(), lane & 7);
        }

        // ---- DC difference to the previous block of the component (mjpegenc.c record_block) ----
        const int up = __shfl_up_sync(0xffffffffu, dc, 1);
        const int pred = lane == 0 ? pred_first : up;
        if (valid) {
            const int diff = dc - pred;
            rec[0] = (uint32_t)(diff & 0xffff) | word0_hi;
            atomicAdd(&s_dchist[mag_bits(diff)], 1u);
            // ---- AC symbol statistics: as in fdct_quant_kernel, two positions per trip from the low end ----
            const int16_t *lv = reinterpret_cast<const int16_t *>(rec);
            unsigned zrl = 0;
            auto count = [&](int kk, int below, int val) {
                const int run = kk - below - 1;
                unsigned top;
                asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(abs(val)));
                zrl += (unsigned)run >> 4;
                atomicAdd(&s_hist[1 + (((run & 15) << 4) | (int)top)], 1u);
            };
            unsigned lo = mask_lo;
            const int top_lo = lo ? 31 - __clz(lo) : 0;
            int below = 0;
            while (lo) {
                const unsigned b0 = lo & (0u - lo);
                lo ^= b0;
                const unsigned b1 = lo & (0u - lo);
                lo ^= b1;
                const int k0 = 31 - __clz(b0), k1 = 31 - __clz(b1);
                const int v0 = (int)lv[2 * k0], v1 = (int)lv[2 * max(k1, 0)];
                count(k0, below, v0);
                {  // a level the lane may not have, without a branch (fdct_quant_kernel's count_if): counted into a word nobody reads
                    const int run = k1 - k0 - 1;
                    unsigned top;
                    asm("bfind.u32 %0, %1;" : "=r"(top) : "r"(abs(v1)));
                    zrl += b1 ? (unsigned)run >> 4 : 0u;
                    atomicAdd(&s_hist[b1 ? 1 + (((run & 15) << 4) | (int)top) : kHistDummy], 1u);
                }
                below = 31 - __clz(b0 | b1);
            }
            int prev = top_lo;
            unsigned hi = mask_hi;
            while (hi) {
                const int bpos = __ffs((int)hi) - 1, kk = 32 + bpos;
                hi &= hi - 1;
                count(kk, prev, (int)lv[2 * bpos + 1]);
                prev = kk;
            }
            if (prev < 63) atomicAdd(&s_hist[0], 1u);
            if (zrl) atomicAdd(&s_hist[0xf0], zrl);
        }

        // ---- the role's sub-image leaves with one bulk store ----
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0)
            bulk_s2g(images + ((long long)f * images_cap + tile) * (kRoles * kSubImageWords) + role * kSubImageWords, img, kSubImageBytes);
    }
    if (lane == 0) bulk_wait_read_all();
    __syncwarp();

#pragma unroll
    for (int i = 0; i < 8; i++) {
        const unsigned c = s_hist[i * 32 + lane];
        if (c) atomicAdd(&state[f].hist[2 + cls][i * 32 + lane], c);
    }
    if (lane < 16) {
        const unsigned c = s_dchist[lane];
        if (c) atomicAdd(&state[f].hist[cls][lane], c);
    }
}

}  // namespace h2j
