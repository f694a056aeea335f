// K6: packing of a batch's JPEGs for one D2H copy.
#pragma once
#include "h2j_common.cuh"

namespace h2j {

// ------------------------------------------------------------------------------------------------
// K6: pack the JPEGs of a batch back to back (so one D2H copy moves exactly the bytes produced).
// offsets[n+1] is computed by block 0 of pack_offsets_kernel.
// ------------------------------------------------------------------------------------------------
constexpr int kPackOffsetsThreads = 256;
__global__ void __launch_bounds__(kPackOffsetsThreads) pack_offsets_kernel(const FrameTab *__restrict__ tabs, int n, long long jpeg_cap,
                                                                           unsigned long long *__restrict__ offsets, int *__restrict__ status)
{
    // one CTA: exclusive scan of the JPEG sizes, a chunk of kPackOffsetsThreads frames at a time
    __shared__ unsigned long long s_warp[kPackOffsetsThreads / 32];
    __shared__ unsigned long long s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += kPackOffsetsThreads) {
        const int i = i0 + tid;
        unsigned long long sz = 0;
        if (i < n) {
            const int st = tabs[i].status;
            status[i] = st;
            const long long b = tabs[i].jpeg_bytes;
            sz = (st != 0 || b > jpeg_cap) ? 0ull : (unsigned long long)b;
        }
        unsigned long long incl = sz;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        unsigned long long off = s_base, total = 0;
#pragma unroll
        for (int w = 0; w < kPackOffsetsThreads / 32; w++) {
            if (w < warp) off += s_warp[w];
            total += s_warp[w];
        }
        if (i < n) offsets[i] = off + incl - sz;
        __syncthreads();
        if (tid == 0) s_base += total;
        __syncthreads();
    }
    if (tid == 0) offsets[n] = s_base;
}

__global__ void __launch_bounds__(256) pack_kernel(const uint8_t *__restrict__ out, long long out_cap,
                                                   const unsigned long long *__restrict__ offsets, uint8_t *__restrict__ packed)
{
    const int f = blockIdx.y;
    const long long size = (long long)(offsets[f + 1] - offsets[f]);
    const uint8_t *src = out + (long long)f * out_cap;
    uint8_t *dst = packed + offsets[f];
    // 16 source bytes per thread; destination alignment is arbitrary, so the stores are byte wide
    for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 16; i < size; i += (long long)gridDim.x * blockDim.x * 16) {
        if (i + 16 <= size) {
            const uint4 v = *reinterpret_cast<const uint4 *>(src + i);
            const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 16; k++) dst[i + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
        } else {
            for (long long k = i; k < size; k++) dst[k] = src[k];
        }
    }
}

}  // namespace h2j
