// K1 (luma variance for the rate control) and the standalone plane conversion kernel.
#pragma once
#include "h2j_common.cuh"

namespace h2j {

// ------------------------------------------------------------------------------------------------
// K1: mb_var_thread (mpegvideo_enc.c) — sum over macroblocks of ((norm1 - sum^2/256 + 628) >> 8)
// grid (mcu_h, n_frames), one thread per macroblock column, 16 independent 128-bit loads in flight.
// ------------------------------------------------------------------------------------------------
// The CTA that finishes a frame last (completion counter) turns the sum into the frame's qscale (ratecontrol.c first
// I picture) and publishes the quantiser tables (mpegvideo_enc.c encode_picture + ff_convert_matrix) for K2.
// LIST: a list batch (h2j_common.cuh FrameDesc): the grid has the largest frame's mcu_h, rows past this frame's return
template <bool LIST>
__global__ void __launch_bounds__(128) mbvar_kernel(const uint8_t *__restrict__ frames, FrameLayout L_,
                                                    FrameState *__restrict__ state, const uint8_t *__restrict__ qscale_lut,
                                                    FrameTab *__restrict__ tabs, const FrameDesc *__restrict__ descs)
{
    const int f = blockIdx.y, my = blockIdx.x;
    const FrameLayout &L = LIST ? descs[f].L : L_;
    if (LIST && my >= L.mcu_h) return;
    const uint8_t *Y = LIST ? descs[f].base : frames + (long long)f * L.frame_stride;
    int local = 0;
    for (int mx = threadIdx.x; mx < L.mb_w; mx += blockDim.x) {  // 16x16 macroblocks (= MCUs except at 4:4:4)
        unsigned sum = 0, norm = 0;
        const int x0 = mx * 16;
        if (L.aligned16 && x0 + 16 <= L.w && L.range_mode == 0) {
            uint4 v[16];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const int y = min(my * 16 + r, L.h - 1);
                v[r] = ldg128(Y + (long long)y * L.y_pitch + x0);
            }
#pragma unroll
            for (int r = 0; r < 16; r++) {
                sum = __dp4a(v[r].x, 0x01010101u, sum); norm = __dp4a(v[r].x, v[r].x, norm);
                sum = __dp4a(v[r].y, 0x01010101u, sum); norm = __dp4a(v[r].y, v[r].y, norm);
                sum = __dp4a(v[r].z, 0x01010101u, sum); norm = __dp4a(v[r].z, v[r].z, norm);
                sum = __dp4a(v[r].w, 0x01010101u, sum); norm = __dp4a(v[r].w, v[r].w, norm);
            }
        } else {
            for (int r = 0; r < 16; r++) {
                const int y = min(my * 16 + r, L.h - 1);
                const uint8_t *row = Y + (long long)y * L.y_pitch;
                for (int c = 0; c < 16; c++) {
                    unsigned p = row[min(x0 + c, L.w - 1)];
                    if (L.range_mode) p = c_range_lut[0][p];
                    sum += p;
                    norm += p * p;
                }
            }
        }
        local += (int)(norm - ((sum * sum) >> 8) + 500u + 128u) >> 8;
    }
    // block reduce
    __shared__ int warp_sums[4];
#pragma unroll
    for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = local;
    __syncthreads();
    __shared__ int s_last, s_qs;
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); i++) t += warp_sums[i];
        atomicAdd(&state[f].var_sum, (unsigned long long)t);
        __threadfence();
        const unsigned done = atomicAdd(&state[f].k1_done, 1u);
        s_last = done == (LIST ? (unsigned)L.mcu_h : gridDim.x) - 1;
        if (s_last) {
            __threadfence();
            const long long var = (long long)atomicAdd(&state[f].var_sum, 0ull);  // every CTA's share is in
            int q;
            if (L.fixed_qscale > 0) q = L.fixed_qscale;
            else {
                // predict_size(): the IEEE-exact part; the pow()/rounding tail is folded into qscale_lut by the host
                const double bits = __ddiv_rn(__dmul_rn(826.0, sqrt((double)var)), 236.0);
                int nb = (int)bits;
                nb = nb > kQscaleLutSize - 1 ? kQscaleLutSize - 1 : (nb < 0 ? 0 : nb);
                q = qscale_lut[nb];
            }
            s_qs = q;
            tabs[f].qscale = q;
            tabs[f].mb_var_sum = var;
            tabs[f].status = 0;
        }
    }
    __syncthreads();
    if (s_last && threadIdx.x < 64) {
        const int i = threadIdx.x;
        uint8_t m, mk;
        uint32_t pk, pk2;
        quant_entry(s_qs, c_mpeg1_intra[i], i, &m, &pk);
        tabs[f].qpack[i] = pk;
        tabs[f].intra[i] = m;
        quant_entry(s_qs, c_mpeg1_intra[c_zigzag[i]], c_zigzag[i], &mk, &pk2);  // DQT is stored in zigzag order
        tabs[f].dqt_zz[i] = mk;
    }
}

// ------------------------------------------------------------------------------------------------
// kernel 1 on its own: range conversion + MCU edge replication into padded planes (h2j_convert_pad).
// One thread per 16 output bytes; 128-bit loads when the source row is 16-byte aligned.
// grid (ceil(padded_w/16 / 128), padded_h, 3)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) convert_pad_kernel(const uint8_t *__restrict__ frame, FrameLayout L, int range_mode,
                                                          uint8_t *__restrict__ oy, uint8_t *__restrict__ ou, uint8_t *__restrict__ ov)
{
    __shared__ uint8_t s_lut[256];
    const int plane = blockIdx.z;
    const int pw = plane ? L.cw : L.w, ph = plane ? L.ch : L.h;
    const int padw = plane ? L.mcu_w * 8 : L.mcu_w * 16, padh = plane ? L.mcu_h * 8 : L.mcu_h * 16;
    const int pitch = plane ? L.c_pitch : L.y_pitch;
    const uint8_t *P = frame + (plane == 0 ? 0 : (plane == 1 ? L.u_off : L.v_off));
    uint8_t *O = plane == 0 ? oy : (plane == 1 ? ou : ov);
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_lut[i] = range_mode ? c_range_lut[plane ? 1 : 0][i] : (uint8_t)i;
    __syncthreads();
    const int y = blockIdx.y;
    if (y >= padh) return;
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (x0 >= padw) return;
    const uint8_t *row = P + (long long)min(y, ph - 1) * pitch;
    uint8_t px[16];
    // the 128-bit path is decided per row: L.aligned16 only speaks for the luma rows, and a chroma pitch of w/2 with
    // w = 16 (mod 32) (720, 848, 1360 ...) puts every odd chroma row 8 bytes off a 16-byte boundary
    if (x0 + 16 <= pw && ((uintptr_t)(row + x0) & 15u) == 0) {
        const uint4 v = ldg128(row + x0);
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 16; k++) px[k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
    } else {
#pragma unroll
        for (int k = 0; k < 16; k++) px[k] = row[min(x0 + k, pw - 1)];
    }
    unsigned w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 16; k++) w[k >> 2] |= (unsigned)s_lut[px[k]] << (8 * (k & 3));
    // padded chroma rows are only 8-byte aligned (padw = mcu_w * 8): two 64-bit stores
    uint2 *o2 = reinterpret_cast<uint2 *>(O + (long long)y * padw + x0);
    o2[0] = make_uint2(w[0], w[1]);
    if (x0 + 8 < padw) o2[1] = make_uint2(w[2], w[3]);
}

// ------------------------------------------------------------------------------------------------
// The copy kernels of the input stage.  Each reads the slot's FrameDesc table of m entry pairs (h2j_common.cuh): frame f as
// the pipeline reads it (planar, at the 16-byte row pitch of pitched_layout()) and the source it is made from (base nullptr:
// frame f is read in place, no copy).  grid (x, rows / kPlaneRowsPerCta, frames), sized for the largest frame that is
// copied: rows of a frame are its luma rows, then its chroma rows (kPlaneRowsPerCta rows per CTA: one row per CTA made 400 k
// CTAs of 120 busy threads for 256 frames); CTAs past their frame's extent do nothing.  A thread writes 16 bytes of a row.
// ------------------------------------------------------------------------------------------------
constexpr int kPlaneRowsPerCta = 16;

// What a copy kernel reads: the slot's uploaded table of m pairs, or with m = 1 the one pair itself, by value (a batch of
// one layout at one stride costs no upload)
struct CopyTable {
    const FrameDesc *descs;
    int m;
    FrameDesc d, s;  // m = 1
};

// frame f's pair: its own entries, or the one pair of a uniform batch with both bases moved on f frame strides
__device__ __forceinline__ void frame_pair(const CopyTable &t, int f, FrameDesc &d, FrameDesc &s)
{
    if (t.m > 1) {
        d = t.descs[f];
        s = t.descs[t.m + f];
        return;
    }
    d = t.d;
    s = t.s;
    d.base += (long long)f * d.L.frame_stride;
    if (s.base) s.base += (long long)f * s.L.frame_stride;
}

// NV12 / NV16 / NV24 (what hardware decoders produce: a luma plane and ONE plane of interleaved Cb/Cr pairs, both with a row
// pitch; the source's L.y_pitch / L.c_pitch, the pair plane at L.u_off) -> planar frames (I420 / 4:2:2 / 4:4:4 by L.fmt).
// Rows h .. h + ch - 1 split a row of pairs.  128-bit loads where the source row segment is 16-byte aligned, bytes otherwise.
__global__ void __launch_bounds__(128) nv12_to_i420_kernel(const __grid_constant__ CopyTable t)
{
    FrameDesc d, s;
    frame_pair(t, blockIdx.z, d, s);
    const FrameLayout &L = d.L;
    uint8_t *D = const_cast<uint8_t *>(d.base);
    const int pairs = (L.w + (1 << fmt_hshift(L.fmt)) - 1) >> fmt_hshift(L.fmt);  // per chroma row
    const int fch = (L.h + fmt_vshift(L.fmt)) >> fmt_vshift(L.fmt);
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    for (int row = blockIdx.y * kPlaneRowsPerCta; row < min((int)(blockIdx.y + 1) * kPlaneRowsPerCta, L.h + fch); row++)
    if (row < L.h) {
        if (x0 >= L.w) continue;
        const uint8_t *src = s.base + (long long)row * s.L.y_pitch + x0;
        uint8_t *dst = D + (long long)row * L.y_pitch + x0;
        if (x0 + 16 <= L.w && ((uintptr_t)src & 15u) == 0) *reinterpret_cast<uint4 *>(dst) = ldg128(src);
        else
            for (int i = 0; i < 16 && x0 + i < L.w; i++) dst[i] = src[i];
    } else {
        const int r = row - L.h;
        if (x0 >= 2 * pairs) continue;
        const uint8_t *src = s.base + s.L.u_off + (long long)r * s.L.c_pitch + x0;
        uint8_t *du = D + L.u_off + (long long)r * L.c_pitch + (x0 >> 1), *dv = D + L.v_off + (long long)r * L.c_pitch + (x0 >> 1);
        if (x0 + 16 <= 2 * pairs && ((uintptr_t)src & 15u) == 0) {
            const uint4 v = ldg128(src);
            const unsigned u0 = __byte_perm(v.x, v.y, 0x6420), u1 = __byte_perm(v.z, v.w, 0x6420);
            const unsigned w0 = __byte_perm(v.x, v.y, 0x7531), w1 = __byte_perm(v.z, v.w, 0x7531);
            *reinterpret_cast<uint2 *>(du) = make_uint2(u0, u1);
            *reinterpret_cast<uint2 *>(dv) = make_uint2(w0, w1);
        } else {
            for (int i = 0; i < 8 && (x0 >> 1) + i < pairs; i++) {
                du[i] = src[2 * i];
                dv[i] = src[2 * i + 1];
            }
        }
    }
}

// Planar frames whose rows do not start on 8-byte boundaries (odd widths such as 1918, an unaligned base, a caller's
// pitches or plane offsets) -> the same planes at a 16-byte row pitch, so that K1 and K2 take their vector-load paths
// (every block but the ones cut by the right edge) instead of 64 byte loads per block.  Rows h .. h + 2 ch - 1 are Cb, then
// Cr.  A thread produces 16 output bytes from five aligned source words and four funnel shifts; it reads nothing outside
// the source's extent.  A row copies the plane's width, ceil-divided by the subsampling (not the source pitch); the padding
// bytes of a row are never read by the pipeline (edges are replicated from the last real sample).
__global__ void __launch_bounds__(128) repitch_kernel(const __grid_constant__ CopyTable t)
{
    FrameDesc d, s;
    frame_pair(t, blockIdx.z, d, s);
    if (!s.base) return;
    const FrameLayout &T = s.L, &P = d.L;  // the source's layout, the copy's
    const uint8_t *sbase = s.base;
    uint8_t *dbase = const_cast<uint8_t *>(d.base);
    const int fcw = (T.w + (1 << fmt_hshift(T.fmt)) - 1) >> fmt_hshift(T.fmt), fch = (T.h + fmt_vshift(T.fmt)) >> fmt_vshift(T.fmt);
    // what may be read: the frame, or for a batch of one layout at one stride (m = 1) every frame of the caller's buffer, so
    // that only the batch's last frame ends in the bytewise path
    const uint8_t *src_begin = t.m > 1 ? sbase : t.s.base;
    const uint8_t *src_end = t.m > 1 ? sbase + s.extent : t.s.base + (long long)(gridDim.z - 1) * T.frame_stride + s.extent;
    for (int row = blockIdx.y * kPlaneRowsPerCta; row < min((int)(blockIdx.y + 1) * kPlaneRowsPerCta, T.h + 2 * fch); row++) {
    int pw, r;
    long long so, dof;
    int spitch, dpitch;
    if (row < T.h) { pw = T.w; r = row; so = 0; dof = 0; spitch = T.y_pitch; dpitch = P.y_pitch; }
    else if (row < T.h + fch) { pw = fcw; r = row - T.h; so = T.u_off; dof = P.u_off; spitch = T.c_pitch; dpitch = P.c_pitch; }
    else { pw = fcw; r = row - T.h - fch; so = T.v_off; dof = P.v_off; spitch = T.c_pitch; dpitch = P.c_pitch; }
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (x0 >= pw) continue;
    const uint8_t *sp = sbase + so + (long long)r * spitch + x0;
    uint8_t *dp = dbase + dof + (long long)r * dpitch + x0;  // 16-byte aligned, x0 + 16 <= dpitch
    const unsigned a = (unsigned)((uintptr_t)sp & 3u);
    const uint8_t *s4 = sp - a;
    if (s4 >= src_begin && s4 + 20 <= src_end) {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(s4);
        const unsigned w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2), w3 = __ldg(q + 3), w4 = a ? __ldg(q + 4) : 0u;
        const unsigned sh = a * 8;
        *reinterpret_cast<uint4 *>(dp) = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                                                    __funnelshift_r(w3, w4, sh));
    } else {
        for (int i = 0; i < 16 && x0 + i < pw; i++) dp[i] = sp[i];
    }
    }
}

// High-bit-depth frames (P010 / P016, P210 / P216, a decoder's 16-bit 4:4:4 surface, yuv420p10le ...) -> 8-bit planar frames.
// Every sample is a little-endian 16-bit word whose low `bit_depth` bits hold the value; the 8-bit sample is bits
// [bit_depth - 8, bit_depth) of the word (truncation: no rounding, no dither; bits above bit_depth never reach the picture).
// The source's L.w / L.h count samples, its pitches and offsets are in bytes.
// SP: a luma plane and one plane of interleaved Cb/Cr word pairs at L.u_off (rows h .. h + ch - 1 of the grid split one row
// of pairs), otherwise three planes (rows h .. h + 2 ch - 1: Cb, then Cr).  A thread converts 16 words of a source row: two
// 128-bit loads where that row is 16-byte aligned and holds all 16 words, 16-bit loads otherwise.  No word past a row's last
// sample is read.
template <bool SP>
__global__ void __launch_bounds__(128) depth_to_8_kernel(const __grid_constant__ CopyTable t, int shift)  // shift: bit_depth - 8
{
    FrameDesc d, s;
    frame_pair(t, blockIdx.z, d, s);
    const FrameLayout &S = s.L, &P = d.L;
    const int fcw = (P.w + (1 << fmt_hshift(P.fmt)) - 1) >> fmt_hshift(P.fmt), fch = (P.h + fmt_vshift(P.fmt)) >> fmt_vshift(P.fmt);
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;  // first word of the row this thread converts
    const uint8_t *F = s.base;
    uint8_t *D = const_cast<uint8_t *>(d.base);
    for (int row = blockIdx.y * kPlaneRowsPerCta; row < min((int)(blockIdx.y + 1) * kPlaneRowsPerCta, P.h + (SP ? 1 : 2) * fch); row++) {
        int n;  // words in the row
        const uint8_t *s;
        uint8_t *d;
        if (row < P.h) { n = P.w; s = F + (long long)row * S.y_pitch; d = D + (long long)row * P.y_pitch + x0; }
        else if (SP) { const int r = row - P.h; n = 2 * fcw; s = F + S.u_off + (long long)r * S.c_pitch; d = D + P.u_off + (long long)r * P.c_pitch + (x0 >> 1); }
        else {
            const int r = row - P.h - (row >= P.h + fch ? fch : 0);
            n = fcw;
            s = F + (row >= P.h + fch ? S.v_off : S.u_off) + (long long)r * S.c_pitch;
            d = D + (row >= P.h + fch ? P.v_off : P.u_off) + (long long)r * P.c_pitch + x0;
        }
        if (x0 >= n) continue;
        s += 2 * x0;
        unsigned t[8];  // word 2k in the low half of t[k], word 2k + 1 in the high half
        if (x0 + 16 <= n && ((uintptr_t)s & 15u) == 0) {
            const uint4 a = ldg128(s), b = ldg128(s + 16);
            t[0] = a.x; t[1] = a.y; t[2] = a.z; t[3] = a.w; t[4] = b.x; t[5] = b.y; t[6] = b.z; t[7] = b.w;
        } else {
            const unsigned short *s16 = reinterpret_cast<const unsigned short *>(s);
#pragma unroll
            for (int k = 0; k < 8; k++)
                t[k] = (x0 + 2 * k < n ? (unsigned)__ldg(s16 + 2 * k) : 0u) | (x0 + 2 * k + 1 < n ? (unsigned)__ldg(s16 + 2 * k + 1) << 16 : 0u);
        }
        // after the shift, bytes 0 and 2 of t[k] are bits [shift, shift + 8) of its two words: the high word's low bits only
        // reach bits 8..15, and nothing above bit_depth is in either byte
#pragma unroll
        for (int k = 0; k < 8; k++) t[k] >>= shift;
        const unsigned p0 = __byte_perm(t[0], t[1], 0x6420), p1 = __byte_perm(t[2], t[3], 0x6420), p2 = __byte_perm(t[4], t[5], 0x6420),
                       p3 = __byte_perm(t[6], t[7], 0x6420);
        // rows of the copy are 16-byte aligned and at least 16 bytes (8 per chroma component of a pair row) past x0
        if (SP && row >= P.h) {
            const long long cr = P.v_off - P.u_off;
            *reinterpret_cast<uint2 *>(d) = make_uint2(__byte_perm(p0, p1, 0x6420), __byte_perm(p2, p3, 0x6420));       // Cb
            *reinterpret_cast<uint2 *>(d + cr) = make_uint2(__byte_perm(p0, p1, 0x7531), __byte_perm(p2, p3, 0x7531));  // Cr
        } else {
            *reinterpret_cast<uint4 *>(d) = make_uint4(p0, p1, p2, p3);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Downscaled frames (h2j_submit_device_downscaled): every plane of the caller's frame, at its decoder size pw x ph, box-
// filtered by K (2, 4, 8) to ceil(pw/K) x ceil(ph/K): out[y][x] = (S + c/2) / c, S the sum of the c source samples of the
// box (K*K, fewer in the partial boxes at the right and bottom edges), semi-planar Cb and Cr averaged separately.  The
// result is the planar frame the pipeline reads, at pitched_layout() of the downscaled size in the slot's d_frames.
// descs[f] is that destination, descs[n + f] the source (L: its size, pitches and plane offsets; SP: the pair plane at
// u_off).  grid (x, y, frames): a warp per output row (kDownRowsPerWarp of them, one after the other), a lane per 16 output
// bytes of the row (SP chroma: 8 Cb + 8 Cr of a row of pairs), so 16 * K source bytes per source row; grid sized for the
// largest destination, CTAs past their frame's extent return.  A source row is summed into the 16 accumulators as soon as
// it is loaded (dp4a).  16-byte aligned segments take 128-bit loads (the lane cut by the row's end: the chunks inside the
// row), others aligned 32-bit words and funnel shifts; only words an end of the row cuts are read byte by byte, so no
// byte past a row's last sample is read.
// ------------------------------------------------------------------------------------------------
template <int K>
constexpr int kDownRowsPerWarp = 16 / K;  // 16 source rows per warp whatever K
constexpr int kDownWarps = 4;

// the 16 * K bytes of a source row at row + x0 as 4 * K little-endian words; bytes at or past `bytes` (the row's end) are 0
template <int K>
__device__ __forceinline__ void down_fetch(const uint8_t *__restrict__ row, int x0, int bytes, unsigned (&w)[4 * K])
{
    constexpr int kWords = 4 * K;
    const uint8_t *s = row + x0;
    const int a = (int)((uintptr_t)s & 3u);
    const uint32_t *q = reinterpret_cast<const uint32_t *>(s - a);
    // aligned word j holds bytes [x0 - a + 4j, + 4) of the row: loaded whole where it lies inside the row, byte by byte
    // where an end of the row cuts it, without the bytes outside
    auto word = [&](int j) {
        const int p = x0 - a + 4 * j;
        if (p >= 0 && p + 4 <= bytes) return __ldg(q + j);
        unsigned v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++)
            if (p + b >= 0 && p + b < bytes) v |= (unsigned)row[p + b] << (8 * b);
        return v;
    };
    if (((uintptr_t)s & 15u) == 0) {  // 16-byte chunks: whole inside the row, 0 past its end, by words where the end cuts one
#pragma unroll
        for (int i = 0; i < K; i++) {
            uint4 v = make_uint4(0, 0, 0, 0);
            if (x0 + 16 * i + 16 <= bytes) v = ldg128(s + 16 * i);
            else if (x0 + 16 * i < bytes) v = make_uint4(word(4 * i), word(4 * i + 1), word(4 * i + 2), word(4 * i + 3));
            w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
        }
        return;
    }
    unsigned prev = word(0);
#pragma unroll
    for (int i = 0; i < kWords; i++) {
        const unsigned next = (i + 1 < kWords || a) ? word(i + 1) : 0u;
        w[i] = __funnelshift_r(prev, next, a * 8);
        prev = next;
    }
}

// (S + c/2) / c of the box of output x (its first source sample k * x), rh rows high, of a row of pw samples; full boxes by a
// shift, outputs past the row's end 0
template <int K>
__device__ __forceinline__ unsigned down_avg(unsigned s, int x, int pw, int rh, bool full)
{
    constexpr int kShift = K == 2 ? 2 : (K == 4 ? 4 : 6);
    if (full) return (s + K * K / 2) >> kShift;
    const int c = min(K, pw - K * x) * rh;
    return c > 0 ? (s + (unsigned)(c >> 1)) / (unsigned)c : 0u;
}

template <int K, bool SP>
__global__ void __launch_bounds__(32 * kDownWarps, K == 2 ? 6 : 4) downscale_list_kernel(const __grid_constant__ CopyTable t)
{
    static_assert(K == 2 || K == 4 || K == 8, "box factors 2, 4, 8");
    constexpr int kWords = 4 * K;
    const int f = blockIdx.z;
    // a list (m = n): a table of one pair is frame 0's
    const FrameDesc &d = t.m > 1 ? t.descs[f] : t.d, &s = t.m > 1 ? t.descs[t.m + f] : t.s;
    const FrameLayout &D = d.L, &S = s.L;
    const int hs = fmt_hshift(S.fmt), vs = fmt_vshift(S.fmt);
    const int scw = (S.w + (1 << hs) - 1) >> hs, sch = (S.h + (1 << vs) - 1) >> vs;  // source chroma plane
    const int dch = (D.h + (1 << vs) - 1) >> vs;                                     // = ceil(sch / K) rows
    const int rows = D.h + (SP ? 1 : 2) * dch;
    const int lane = threadIdx.x & 31;
    const int x16 = blockIdx.x * 32 + lane;  // this lane's 16 output bytes of a row (SP chroma: its 8 pairs)
    const int row0 = (blockIdx.y * kDownWarps + (threadIdx.x >> 5)) * kDownRowsPerWarp<K>;
    for (int row = row0; row < min(row0 + kDownRowsPerWarp<K>, rows); row++) {
        int r, pw, ph, spitch;  // output row in its plane, source plane samples per row (SP chroma: pairs) and rows, pitch
        long long so;
        uint8_t *o;
        bool pairs = false;
        if (row < D.h) {
            r = row; pw = S.w; ph = S.h; spitch = S.y_pitch; so = 0;
            o = const_cast<uint8_t *>(d.base) + (long long)r * D.y_pitch;
        } else if (SP) {
            r = row - D.h; pw = scw; ph = sch; spitch = S.c_pitch; so = S.u_off; pairs = true;
            o = const_cast<uint8_t *>(d.base) + D.u_off + (long long)r * D.c_pitch;
        } else {
            const bool cr = row >= D.h + dch;
            r = row - D.h - (cr ? dch : 0); pw = scw; ph = sch; spitch = S.c_pitch; so = cr ? S.v_off : S.u_off;
            o = const_cast<uint8_t *>(d.base) + (cr ? D.v_off : D.u_off) + (long long)r * D.c_pitch;
        }
        const int per = pairs ? 8 : 16;  // outputs per lane and component
        const int ox = x16 * per;        // first of them
        if (K * ox >= pw) continue;
        const int bytes = pairs ? 2 * pw : pw;  // of a source row
        const int x0 = 16 * K * x16;            // first source byte of the lane's segment
        const int rh = min(K, ph - K * r);
        const uint8_t *src = s.base + so + (long long)K * r * spitch;
        unsigned acc[16];  // planar: output ox + i; SP: Cb of pair ox + i (0..7), Cr (8..15)
#pragma unroll
        for (int i = 0; i < 16; i++) acc[i] = 0;
#pragma unroll
        for (int j = 0; j < K; j++) {
            if (j >= rh) break;
            unsigned w[kWords];
            down_fetch<K>(src + (long long)j * spitch, x0, bytes, w);
            if (pairs) {  // Cb Cr Cb Cr: K / 2 words per output pair
#pragma unroll
                for (int i = 0; i < kWords; i++) {
                    acc[i / (K / 2)] = __dp4a(w[i], 0x00010001u, acc[i / (K / 2)]);
                    acc[8 + i / (K / 2)] = __dp4a(w[i], 0x01000100u, acc[8 + i / (K / 2)]);
                }
            } else if constexpr (K == 2) {  // two outputs per word
#pragma unroll
                for (int i = 0; i < kWords; i++) {
                    acc[2 * i] = __dp4a(w[i], 0x00000101u, acc[2 * i]);
                    acc[2 * i + 1] = __dp4a(w[i], 0x01010000u, acc[2 * i + 1]);
                }
            } else {  // K / 4 words per output
#pragma unroll
                for (int i = 0; i < kWords; i++) acc[i / (K / 4)] = __dp4a(w[i], 0x01010101u, acc[i / (K / 4)]);
            }
        }
        const bool full = rh == K && x0 + 16 * K <= bytes;
        unsigned p[4] = {0, 0, 0, 0};
        if (pairs) {
            unsigned q[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < 8; i++) {
                p[i >> 2] |= down_avg<K>(acc[i], ox + i, pw, rh, full) << (8 * (i & 3));
                q[i >> 2] |= down_avg<K>(acc[8 + i], ox + i, pw, rh, full) << (8 * (i & 3));
            }
            // rows of the destination are 16-byte aligned and hold at least 8 bytes from ox
            *reinterpret_cast<uint2 *>(o + ox) = make_uint2(p[0], p[1]);
            *reinterpret_cast<uint2 *>(o + (D.v_off - D.u_off) + ox) = make_uint2(q[0], q[1]);
        } else {
#pragma unroll
            for (int i = 0; i < 16; i++) p[i >> 2] |= down_avg<K>(acc[i], ox + i, pw, rh, full) << (8 * (i & 3));
            *reinterpret_cast<uint4 *>(o + ox) = make_uint4(p[0], p[1], p[2], p[3]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// RGB frames (h2j_submit_device_rgb, h2j_encode_frame_rgb) -> the planar frame C(frame) at the encoder's chroma format
// (include/h2j_b200.h): per pixel JFIF / T.871 full-range YCbCr in libjpeg's 16-bit fixed point (jccolor.c), then Cb and Cr
// box-averaged over 2x2 (4:2:0) or 2x1 (4:2:2) pixels, (S + c/2) / c over the c samples of a box inside the plane.
// descs[f] is the destination (pitched_layout() in d_frames), descs[n + f] the caller's frame: rows S.y_pitch apart from its
// base, the planar G and B planes at S.u_off / S.v_off.  K: bytes per pixel of a source row (3 or 4: packed; 1: three
// planes).  order: the __byte_perm selector that puts a packed pixel's bytes in R, G, B order (0x3210: RGB, 0x3012: BGR).
// grid (x, y, frames): a warp per destination row (4:2:0: per row pair, so that both luma rows and the chroma row they make
// come from one pass over the source), kRgbRowsPerWarp of them one after the other, and a lane per 16 pixels of a row,
// fetched with down_fetch (any alignment; nothing past a row's end is read); grid sized for the largest destination, CTAs
// past their frame return.  Stores are aligned: rows of the destination are 16-byte aligned and hold 16 bytes from x0.
// ------------------------------------------------------------------------------------------------
constexpr int kRgbRowsPerWarp = 2;

template <int K, int FMT>
__global__ void __launch_bounds__(32 * kDownWarps) rgb_to_planar_kernel(const __grid_constant__ CopyTable t, unsigned order)
{
    static_assert(K == 1 || K == 3 || K == 4, "three planes, 3- or 4-byte pixels");
    constexpr int kV = FMT == kFmt420 ? 2 : 1;             // luma rows per chroma row
    constexpr int kBoxShift = FMT == kFmt420 ? 2 : 1;      // log2 of a full box (4:4:4: none)
    const int f = blockIdx.z;
    const FrameDesc &d = t.m > 1 ? t.descs[f] : t.d, &s = t.m > 1 ? t.descs[t.m + f] : t.s;
    const FrameLayout &D = d.L, &S = s.L;
    const int w = D.w, h = D.h;
    const int x0 = (blockIdx.x * 32 + (threadIdx.x & 31)) * 16;  // the lane's first pixel
    if (x0 >= w) return;
    const bool inside = x0 + 16 <= w;
    const int g0 = (blockIdx.y * kDownWarps + (threadIdx.x >> 5)) * kRgbRowsPerWarp;
    uint8_t *const out = const_cast<uint8_t *>(d.base);
    for (int g = g0; g < min(g0 + kRgbRowsPerWarp, (h + kV - 1) / kV); g++) {
        const int rh = min(kV, h - kV * g);
        unsigned cb[16], cr[16];  // 4:4:4: pixel i; otherwise the sum over box i (i < 8)
#pragma unroll
        for (int i = 0; i < 16; i++) cb[i] = cr[i] = 0;
#pragma unroll
        for (int j = 0; j < kV; j++) {
            if (j >= rh) break;
            const int row = kV * g + j;
            const uint8_t *src = s.base + (long long)row * S.y_pitch;
            unsigned wd[K == 1 ? 12 : 4 * K];  // K = 1: the R, G, B segments one after the other
            if constexpr (K == 1) {
                unsigned r[4], gr[4], b[4];
                down_fetch<1>(src, x0, w, r);
                down_fetch<1>(src + S.u_off, x0, w, gr);
                down_fetch<1>(src + S.v_off, x0, w, b);
#pragma unroll
                for (int i = 0; i < 4; i++) { wd[i] = r[i]; wd[4 + i] = gr[i]; wd[8 + i] = b[i]; }
            } else {
                down_fetch<K>(src, K * x0, K * w, wd);
            }
            unsigned yw[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < 16; i++) {
                int R, G, B;
                if constexpr (K == 1) {
                    const int sh = 8 * (i & 3);
                    R = (wd[i >> 2] >> sh) & 255;
                    G = (wd[4 + (i >> 2)] >> sh) & 255;
                    B = (wd[8 + (i >> 2)] >> sh) & 255;
                } else {
                    // the pixel's three bytes (K = 3: bytes o .. o + 2 of words b/4 and b/4 + 1), then in R G B order
                    const int b = K * i, o = b & 3;
                    unsigned px = K == 4 ? wd[i] : __byte_perm(wd[b >> 2], wd[min((b >> 2) + 1, 4 * K - 1)], o | (o + 1) << 4 | (o + 2) << 8);
                    px = __byte_perm(px, 0, order);
                    R = px & 255;
                    G = (px >> 8) & 255;
                    B = (px >> 16) & 255;
                }
                yw[i >> 2] |= (unsigned)((19595 * R + 38470 * G + 7471 * B + 32768) >> 16) << (8 * (i & 3));
                // (128 << 16) + 32767 = 8421375: chroma rounds with ONE_HALF - 1; both always land in 0..255
                const unsigned u = (unsigned)((-11059 * R - 21709 * G + 32768 * B + 8421375) >> 16);
                const unsigned v = (unsigned)((32768 * R - 27439 * G - 5329 * B + 8421375) >> 16);
                if constexpr (FMT == kFmt444) {
                    cb[i] = u;
                    cr[i] = v;
                } else if (inside || x0 + i < w) {  // pixels past the row's end are no box's samples
                    cb[i >> 1] += u;
                    cr[i >> 1] += v;
                }
            }
            *reinterpret_cast<uint4 *>(out + (long long)row * D.y_pitch + x0) = make_uint4(yw[0], yw[1], yw[2], yw[3]);
        }
        uint8_t *const ou = out + D.u_off + (long long)g * D.c_pitch, *const ov = out + D.v_off + (long long)g * D.c_pitch;
        if constexpr (FMT == kFmt444) {
            unsigned p[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
#pragma unroll
            for (int i = 0; i < 16; i++) {
                p[i >> 2] |= cb[i] << (8 * (i & 3));
                q[i >> 2] |= cr[i] << (8 * (i & 3));
            }
            *reinterpret_cast<uint4 *>(ou + x0) = make_uint4(p[0], p[1], p[2], p[3]);
            *reinterpret_cast<uint4 *>(ov + x0) = make_uint4(q[0], q[1], q[2], q[3]);
        } else {
            const bool full = inside && rh == kV;
            unsigned p[2] = {0, 0}, q[2] = {0, 0};
#pragma unroll
            for (int i = 0; i < 8; i++) {
                unsigned a, b;
                if (full) {
                    a = (cb[i] + (1u << (kBoxShift - 1))) >> kBoxShift;
                    b = (cr[i] + (1u << (kBoxShift - 1))) >> kBoxShift;
                } else {
                    const int c = min(2, w - x0 - 2 * i) * rh;  // samples of box i inside the plane
                    a = c > 0 ? (cb[i] + (unsigned)(c >> 1)) / (unsigned)c : 0u;
                    b = c > 0 ? (cr[i] + (unsigned)(c >> 1)) / (unsigned)c : 0u;
                }
                p[i >> 2] |= a << (8 * (i & 3));
                q[i >> 2] |= b << (8 * (i & 3));
            }
            *reinterpret_cast<uint2 *>(ou + (x0 >> 1)) = make_uint2(p[0], p[1]);
            *reinterpret_cast<uint2 *>(ov + (x0 >> 1)) = make_uint2(q[0], q[1]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Resized frames (h2j_submit_device_resized): every plane of the caller's frame, at its decoder size, resized to the matching
// plane of the W x H frame by Pillow's two-pass convolution (include/h2j_b200.h): a horizontal pass over every source row
// the plane's output needs, clipped to 8 bits, then a vertical pass over those 8-bit rows, both in 22-bit fixed point with a
// 32-bit sum.  The host builds the coefficients (an axis that keeps its size gets the identity: one tap of 1 << 22, which
// gives back the sample, as Pillow's skipped pass does).  descs[f] is the destination (pitched_layout() in d_frames),
// descs[n + f] the caller's frame (SP: the pair plane at u_off, component c of pair x at byte 2x + c).
// grid (x, y, frames): a CTA owns kResizeCols output columns (a thread per column) by kResizeRows output rows of one plane
// (y: the luma bands, then Cb's, then Cr's), grid sized for the largest frame, CTAs past their frame's planes return.  It
// streams the source rows its band's vertical windows cover, in order, kResizeGroup at a time: the span of source samples the
// tile's horizontal windows cover is staged in shared memory (16-byte loads where a chunk lies inside the span, bytes at the
// cut ends: nothing outside a row's samples is read), each thread runs its column's horizontal window over it and keeps the
// 8-bit results in its own column of s_h, then adds k_v * value over the part of every output row's vertical window that
// lies in the group into that row's 32-bit sum (registers): only the taps, no test per (row, source row).  A span wider
// than the staging buffer is staged one row at a time, in pieces.
// ------------------------------------------------------------------------------------------------
constexpr int kResizeCols = 128;
constexpr int kResizeRows = 16;
constexpr int kResizeGroup = 16;          // source rows staged at once, when their spans fit
constexpr int kResizeStage = 16384;       // bytes of staged spans
constexpr int kResizeBits = 22;           // Pillow's PRECISION_BITS

// a frame's coefficient tables in the slot's arena: per output sample of an axis {first source sample, taps, first
// coefficient}, and the axis's coefficients.  Axes: luma x, luma y, chroma x, chroma y.
struct ResizeFrame {
    const int4 *win[4];
    const int *coef[4];
};

template <bool SP>
__global__ void __launch_bounds__(kResizeCols, 4) resize_list_kernel(const __grid_constant__ CopyTable t, const ResizeFrame *__restrict__ frames)
{
    __shared__ __align__(16) uint8_t s_stage[kResizeStage];
    __shared__ int4 s_win[kResizeRows];  // the band's vertical windows
    __shared__ uint8_t s_h[kResizeGroup][kResizeCols];  // the group's horizontal results, a column per thread
    const int f = blockIdx.z;
    const FrameDesc &d = t.m > 1 ? t.descs[f] : t.d, &s = t.m > 1 ? t.descs[t.m + f] : t.s;
    const FrameLayout &D = d.L, &S = s.L;
    const int hs = fmt_hshift(S.fmt), vs = fmt_vshift(S.fmt);
    const int dcw = (D.w + (1 << hs) - 1) >> hs, dch = (D.h + (1 << vs) - 1) >> vs;  // output chroma plane
    const int luma_bands = (D.h + kResizeRows - 1) / kResizeRows, chroma_bands = (dch + kResizeRows - 1) / kResizeRows;
    int band = blockIdx.y, plane = 0;
    if (band >= luma_bands) {
        band -= luma_bands;
        plane = band >= chroma_bands ? 2 : 1;
        if (plane == 2) band -= chroma_bands;
        if (band >= chroma_bands) return;
    }
    const int ow = plane ? dcw : D.w, oh = plane ? dch : D.h;
    const int c0 = blockIdx.x * kResizeCols, r0 = band * kResizeRows;
    if (c0 >= ow) return;
    const int nr = min(kResizeRows, oh - r0);
    const bool pairs = SP && plane;
    const int step = pairs ? 2 : 1, comp = pairs ? plane - 1 : 0;  // bytes per sample of a row; this component's byte
    const uint8_t *src = s.base + (plane == 0 ? 0 : plane == 1 ? S.u_off : S.v_off) + comp;
    const int spitch = plane ? S.c_pitch : S.y_pitch;
    const ResizeFrame &rf = frames[f];
    const int4 *xwin = rf.win[plane ? 2 : 0];
    const int *xk = rf.coef[plane ? 2 : 0], *yk = rf.coef[plane ? 3 : 1];
    if (threadIdx.x < kResizeRows) s_win[threadIdx.x] = threadIdx.x < nr ? rf.win[plane ? 3 : 1][r0 + threadIdx.x] : make_int4(0, 0, 0, 0);
    const int o = c0 + threadIdx.x;
    const bool active = o < ow;
    const int4 w = active ? xwin[o] : make_int4(0, 0, 0, 0);
    const int xa = xwin[c0].x;  // the tile's span of source samples: windows move right with the output sample
    const int4 wl = xwin[min(c0 + kResizeCols, ow) - 1];
    const int xb = wl.x + wl.y;
    __syncthreads();
    const int ja = s_win[0].x, jb = s_win[nr - 1].x + s_win[nr - 1].y;
    // a piece of a row's span: at most the staging buffer (with the cut of its first chunk); as many rows of pieces as fit
    const int piece = min(xb - xa, (kResizeStage - 16) / step - 1);
    const int spitch_s = (piece * step + 31) & ~15;  // staged bytes per row: whole chunks from the 16-byte boundary below
    const int group = piece < xb - xa ? 1 : min(kResizeGroup, kResizeStage / spitch_s);
    const int chunks = spitch_s >> 4;
    int acc[kResizeRows];
#pragma unroll
    for (int r = 0; r < kResizeRows; r++) acc[r] = 1 << (kResizeBits - 1);
    int h = 1 << (kResizeBits - 1);  // a row staged in pieces (group 1): its horizontal sum so far
    for (int j = ja; j < jb; j += group) {
        const int g_n = min(group, jb - j);
        for (int p0 = xa; p0 < xb; p0 += piece) {
            const int p1 = min(xb, p0 + piece);
            for (int c = threadIdx.x; c < g_n * chunks; c += kResizeCols) {
                const int g = c / chunks, k = c - g * chunks;
                const uint8_t *g0 = src + (long long)(j + g) * spitch + (long long)p0 * step, *g1 = g0 + (long long)(p1 - p0 - 1) * step + 1;
                const uint8_t *q = reinterpret_cast<const uint8_t *>((uintptr_t)g0 & ~(uintptr_t)15) + 16 * k;
                uint8_t *st = s_stage + g * spitch_s + 16 * k;
                if (q >= g0 && q + 16 <= g1) *reinterpret_cast<uint4 *>(st) = ldg128(q);
                else if (q < g1)
                    for (int b = 0; b < 16; b++)
                        if (q + b >= g0 && q + b < g1) st[b] = q[b];
            }
            __syncthreads();
            for (int g = 0; g < g_n; g++) {
                const int row = j + g;
                int sum = p0 == xa ? 1 << (kResizeBits - 1) : h;
                if (active) {
                    const int cut = (int)((uintptr_t)(src + (long long)row * spitch + (long long)p0 * step) & 15u);
                    const uint8_t *sp = s_stage + g * spitch_s + cut + (w.x - p0) * step;
                    const int *kp = xk + w.z;
                    const int t1 = min(w.y, p1 - w.x);
                    for (int tt = max(0, p0 - w.x); tt < t1; tt++) sum += (int)sp[tt * step] * __ldg(kp + tt);
                }
                if (p1 < xb) h = sum;
                else s_h[g][threadIdx.x] = (uint8_t)min(max(sum >> kResizeBits, 0), 255);
            }
            if (p1 == xb) {
#pragma unroll
                for (int r = 0; r < kResizeRows; r++) {
                    const int4 yw = s_win[r];  // (rows past the band: an empty window)
                    const int lo = max(yw.x, j), hi = min(yw.x + yw.y, j + g_n);
                    const int *kp = yk + yw.z - yw.x;
                    for (int row = lo; row < hi; row++) acc[r] += (int)s_h[row - j][threadIdx.x] * __ldg(kp + row);
                }
            }
            __syncthreads();
        }
    }
    if (!active) return;
    uint8_t *out = const_cast<uint8_t *>(d.base) + (plane == 0 ? 0 : plane == 1 ? D.u_off : D.v_off) + o;
    const int dpitch = plane ? D.c_pitch : D.y_pitch;
#pragma unroll
    for (int r = 0; r < kResizeRows; r++)
        if (r < nr) out[(long long)(r0 + r) * dpitch] = (uint8_t)min(max(acc[r] >> kResizeBits, 0), 255);
}

}  // namespace h2j
