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
__global__ void __launch_bounds__(128) mbvar_kernel(const uint8_t *__restrict__ frames, FrameLayout L,
                                                    FrameState *__restrict__ state, const uint8_t *__restrict__ qscale_lut,
                                                    FrameTab *__restrict__ tabs)
{
    const int f = blockIdx.y, my = blockIdx.x;
    const uint8_t *Y = frames + (long long)f * L.frame_stride;
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
        s_last = done == gridDim.x - 1;
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
// NV12 / NV16 / NV24 (what hardware decoders produce: a luma plane and ONE plane of interleaved Cb/Cr pairs, both with a
// row pitch) -> the tight planar frames the pipeline reads (I420 / 4:2:2 / 4:4:4 by L.fmt: c_pitch pairs per row, ch rows
// of them).  grid (x, rows, frames): rows 0..h-1 copy luma, rows h..h+ch-1 split a chroma row (kPlaneRowsPerCta rows per
// CTA: one row per CTA made 400 k CTAs of 120 busy threads for 256 frames).
// 16 bytes per thread where pitch, base and width allow, bytes otherwise.
// ------------------------------------------------------------------------------------------------
constexpr int kPlaneRowsPerCta = 16;
__global__ void __launch_bounds__(128) nv12_to_i420_kernel(const uint8_t *__restrict__ src, long long src_stride, int pitch, long long uv_off,
                                                           uint8_t *__restrict__ dst, FrameLayout L, int src_aligned16)
{
    const int f = blockIdx.z;
    const uint8_t *S = src + (long long)f * src_stride;
    uint8_t *D = dst + (long long)f * L.frame_stride;
    const int fch = (L.h + fmt_vshift(L.fmt)) >> fmt_vshift(L.fmt);
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    for (int row = blockIdx.y * kPlaneRowsPerCta; row < min((int)(blockIdx.y + 1) * kPlaneRowsPerCta, L.h + fch); row++)
    if (row < L.h) {
        if (x0 >= L.w) continue;
        const uint8_t *s = S + (long long)row * pitch + x0;
        uint8_t *d = D + (long long)row * L.y_pitch + x0;
        if (src_aligned16 && L.aligned16 && x0 + 16 <= L.w) *reinterpret_cast<uint4 *>(d) = ldg128(s);
        else
            for (int i = 0; i < 16 && x0 + i < L.w; i++) d[i] = s[i];
    } else if (row < L.h + fch) {
        const int r = row - L.h;
        if (x0 >= 2 * L.c_pitch) continue;  // c_pitch = ceil(w / 2) pairs per row
        const uint8_t *s = S + uv_off + (long long)r * pitch + x0;
        uint8_t *du = D + L.u_off + (long long)r * L.c_pitch + (x0 >> 1), *dv = D + L.v_off + (long long)r * L.c_pitch + (x0 >> 1);
        if (src_aligned16 && (uv_off & 15) == 0 && L.aligned8 && x0 + 16 <= 2 * L.c_pitch) {
            const uint4 v = ldg128(s);
            const unsigned u0 = __byte_perm(v.x, v.y, 0x6420), u1 = __byte_perm(v.z, v.w, 0x6420);
            const unsigned w0 = __byte_perm(v.x, v.y, 0x7531), w1 = __byte_perm(v.z, v.w, 0x7531);
            *reinterpret_cast<uint2 *>(du) = make_uint2(u0, u1);
            *reinterpret_cast<uint2 *>(dv) = make_uint2(w0, w1);
        } else {
            for (int i = 0; i < 8 && (x0 >> 1) + i < L.c_pitch; i++) {
                du[i] = s[2 * i];
                dv[i] = s[2 * i + 1];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Planar frames whose rows do not start on 8-byte boundaries (odd widths such as 1918, an unaligned base, a caller's
// pitches or plane offsets) -> the same planes at a 16-byte row pitch, so that K1 and K2 take their vector-load paths
// (every block but the ones cut by the right edge) instead of 64 byte loads per block.  grid (x, h + 2 * ch, frames); a
// thread produces 16 output bytes from five aligned source words and four funnel shifts.  A row copies the plane's
// width, ceil-divided by the subsampling (not the source pitch); the padding bytes of a row are never read by the pipeline
// (edges are replicated from the last real sample).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) repitch_kernel(const uint8_t *__restrict__ src, FrameLayout T,  // layout of the source
                                                      int fch,                                         // rows of a chroma plane
                                                      uint8_t *__restrict__ dst, FrameLayout P,        // pitched layout of the copy
                                                      const uint8_t *src_begin, const uint8_t *src_end)  // what may be read
{
    const int f = blockIdx.z;
    const int fcw = (T.w + (1 << fmt_hshift(T.fmt)) - 1) >> fmt_hshift(T.fmt);  // (T.c_pitch of a tight source)
    for (int row = blockIdx.y * kPlaneRowsPerCta; row < min((int)(blockIdx.y + 1) * kPlaneRowsPerCta, T.h + 2 * fch); row++) {
    int pw, r;
    long long so, dof;
    int spitch, dpitch;
    if (row < T.h) { pw = T.w; r = row; so = 0; dof = 0; spitch = T.y_pitch; dpitch = P.y_pitch; }
    else if (row < T.h + fch) { pw = fcw; r = row - T.h; so = T.u_off; dof = P.u_off; spitch = T.c_pitch; dpitch = P.c_pitch; }
    else { pw = fcw; r = row - T.h - fch; so = T.v_off; dof = P.v_off; spitch = T.c_pitch; dpitch = P.c_pitch; }
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (x0 >= pw) continue;
    const uint8_t *s = src + (long long)f * T.frame_stride + so + (long long)r * spitch + x0;
    uint8_t *d = dst + (long long)f * P.frame_stride + dof + (long long)r * dpitch + x0;  // 16-byte aligned, x0 + 16 <= dpitch
    const unsigned a = (unsigned)((uintptr_t)s & 3u);
    const uint8_t *s4 = s - a;
    if (s4 >= src_begin && s4 + 20 <= src_end) {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(s4);
        const unsigned w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2), w3 = __ldg(q + 3), w4 = a ? __ldg(q + 4) : 0u;
        const unsigned sh = a * 8;
        *reinterpret_cast<uint4 *>(d) = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                                                   __funnelshift_r(w3, w4, sh));
    } else {
        for (int i = 0; i < 16 && x0 + i < pw; i++) d[i] = s[i];
    }
    }
}

}  // namespace h2j
