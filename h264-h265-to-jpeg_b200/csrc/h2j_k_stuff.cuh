// K5: ff_mjpeg_escape_FF + picture trailer.  The scan of a frame is cut into chunks of 1024 words; K4 left the
// number of 0xFF bytes of every chunk in chunk_ff, so a chunk's output position is known from a short sum and
// chunks are independent: grid (ctas per frame, frames), each CTA strides over the frame's chunks.
//
// A chunk is expanded in shared memory and leaves as aligned 16-byte stores:
//   * a thread takes 16 input bytes (one 128-bit load); a block scan of the 0xFF counts gives every thread its place;
//   * each of its four words is ONE item: the word itself, or -- with a 0x00 inserted behind each 0xFF -- up to eight
//     bytes, ORed into the pre-zeroed image at its byte offset (two or three shared-memory atomics, no byte loop);
//   * the image starts at the byte offset the chunk's output has inside its 16-byte line in global memory, so image
//     quads and output quads coincide: one LDS.128 + one STG.128 per 16 bytes, bytewise only for the two ragged ends.
// The CTA that owns the last chunk appends EOI and publishes the frame's size.  Frame f's output starts at out + f * out_cap;
// jpeg_cap (<= out_cap) is the largest JPEG allowed, and no byte at or past it is written.
// (The first form of this kernel expanded byte by byte whenever ANY lane of the warp had a 0xFF -- 86 % of the warps --
// and realigned the image with funnel shifts on the way out: 39 thread instructions per byte; this one needs about 8.)
#pragma once
#include "h2j_common.cuh"

namespace h2j {

constexpr int kStuffImageWords = (2 * kChunkWords * 4 + 64) / 4;  // worst case: every byte 0xFF, plus the line offset, quad aligned
static_assert(kStuffThreads * 4 == kChunkWords, "one 128-bit load per thread and chunk");

// OR the bytes of (hi:lo) -- stream order = little-endian byte order -- into the zeroed image at byte offset q
__device__ __forceinline__ void stuff_put(unsigned int *img, unsigned q, unsigned lo, unsigned hi)
{
    const unsigned s = (q & 3u) * 8u;
    unsigned int *w = img + (q >> 2);
    const unsigned x0 = lo << s, x1 = __funnelshift_l(lo, hi, s), x2 = s ? hi >> (32u - s) : 0u;
    // the first two without a test: a test is a branch with its reconvergence point around ONE instruction, x0 is hardly ever
    // zero and x1 only when the item starts on a word boundary (ORing a zero in is harmless; w + 1 is inside the image, whose
    // size allows for w + 2); the third piece only exists behind an inserted zero
    atomicOr(w, x0);
    atomicOr(w + 1, x1);
    if (x2) atomicOr(w + 2, x2);
}

__global__ void __launch_bounds__(kStuffThreads, 8) stuff_kernel(FrameTab *__restrict__ tabs, const FrameState *__restrict__ state,
                                                              const uint32_t *__restrict__ scan, long long scan_cap_words,
                                                              const unsigned int *__restrict__ chunk_ff, int chunks_cap,
                                                              uint8_t *__restrict__ out, long long out_cap, long long jpeg_cap)
{
    __shared__ __align__(16) unsigned int s_img[kStuffImageWords];
    __shared__ unsigned s_warp[kStuffThreads / 32];
    __shared__ unsigned s_red[kStuffThreads / 32];

    const int f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    FrameTab *T = tabs + f;
    // bit positions are 32-bit: h2j_create bounds max_jpeg_bytes to 256 MiB
    const unsigned bits = (unsigned)state[f].scan_bits;
    const unsigned nbytes = (bits + 7u) >> 3;
    const unsigned nwords = (nbytes + 3u) >> 2;
    // a frame that outgrew its capacity (reported by K4b, status -4) is cut at the capacity: nothing behind it exists
    const int nchunks = min((int)((nwords + kChunkWords - 1) >> kChunkShift), chunks_cap);
    const unsigned hdr = (unsigned)T->header_bytes;
    const unsigned cap = (unsigned)min(jpeg_cap, (long long)0xffffffffu);
    const unsigned scan_cap = (unsigned)min(scan_cap_words, (long long)0xffffffffu);
    const uint32_t *gs = scan + (long long)f * scan_cap_words;
    const unsigned int *cff = chunk_ff + (long long)f * chunks_cap;
    uint8_t *o = out + (long long)f * out_cap;

    for (int c = blockIdx.x; c < nchunks; c += gridDim.x) {
        // ---- 0xFF bytes in front of this chunk ----
        unsigned part = 0;
        for (int i = tid; i < c; i += kStuffThreads) part += cff[i];
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) part += __shfl_xor_sync(0xffffffffu, part, ofs);
        if (lane == 0) s_red[warp] = part;
        // ---- this thread's 4 words ----
        const unsigned w0 = (unsigned)c * kChunkWords + tid * 4;
        uint4 q = make_uint4(0, 0, 0, 0);
        if (w0 < nwords && w0 + 4 <= scan_cap) q = *reinterpret_cast<const uint4 *>(gs + w0);
        unsigned wv[4] = {q.x, q.y, q.z, q.w};  // memory byte order == stream order: byte j is (wv[j >> 2] >> (8 * (j & 3))) & 0xff
        const int nb = w0 * 4 + 16 <= nbytes ? 16 : (nbytes > w0 * 4 ? (int)(nbytes - w0 * 4) : 0);  // valid bytes of the 16
        if (nb < 16) {  // the frame's last bytes: everything behind them counts as (and is copied as) zero
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int left = nb - 4 * k;
                if (left <= 0) wv[k] = 0;
                else if (left < 4) wv[k] &= (1u << (8 * left)) - 1u;
            }
        }
        unsigned ffm[4];  // 0x80 in every byte that is 0xFF
        unsigned cnt = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned x = ~wv[k];
            ffm[k] = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu);
            cnt += __popc(ffm[k]);
        }
        unsigned incl = cnt;
#pragma unroll
        for (int ofs = 1; ofs < 32; ofs <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, incl, ofs);
            if (lane >= ofs) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        // ---- clear the image (the previous chunk's copy-out finished behind the barrier that closes the loop body) ----
        for (int i = tid; i < kStuffImageWords / 4; i += kStuffThreads) reinterpret_cast<uint4 *>(s_img)[i] = make_uint4(0, 0, 0, 0);
        __syncthreads();
        unsigned woff = 0, chunk_total = 0, before = 0;
#pragma unroll
        for (int k = 0; k < kStuffThreads / 32; k++) {
            if (k < warp) woff += s_warp[k];
            chunk_total += s_warp[k];
            before += s_red[k];
        }
        const unsigned dst0 = hdr + (unsigned)c * (kChunkWords * 4) + before;  // the chunk's first output byte
        const unsigned a0 = (unsigned)((uintptr_t)(o + dst0) & 15u);              // ... and its offset in its 16-byte line
        // ---- expand: one item per word ----
        unsigned p = a0 + (unsigned)tid * 16 + woff + incl - cnt;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            unsigned lo = wv[k], hi = 0, y = ffm[k], ins = 0;
            while (y) {  // a 0x00 behind every 0xFF (one word in 64 has one)
                const unsigned at = ((unsigned)(__ffs((int)y) - 1) >> 3) + 1 + ins;  // byte index the zero goes to: 1..7
                y &= y - 1;
                const unsigned long long e = ((unsigned long long)hi << 32) | lo, m = (1ull << (8 * at)) - 1ull;
                const unsigned long long e2 = (e & m) | ((e & ~m) << 8);
                lo = (unsigned)e2;
                hi = (unsigned)(e2 >> 32);
                ins++;
            }
            stuff_put(s_img, p, lo, hi);
            p += 4 + ins;
        }
        __syncthreads();
        // ---- copy out: image byte a0 + i is output byte dst0 + i ----
        const unsigned chunk_bytes_in = min((unsigned)kChunkWords * 4, nbytes - (unsigned)c * (kChunkWords * 4));
        const unsigned end_i = a0 + chunk_bytes_in + chunk_total;  // image bytes [a0, end_i) are the chunk's output
        uint8_t *line0 = o + dst0 - a0;                              // 16-byte aligned
        const unsigned room = cap > dst0 - a0 ? cap - (dst0 - a0) : 0u;  // image bytes that still fit the frame's output
        for (unsigned qi = tid; qi * 16 < end_i; qi += kStuffThreads) {
            const uint4 v = reinterpret_cast<const uint4 *>(s_img)[qi];
            const unsigned b0 = qi * 16;
            if (b0 >= a0 && b0 + 16 <= end_i && b0 + 16 <= room) {
                *reinterpret_cast<uint4 *>(line0 + b0) = v;
            } else {
                const unsigned vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    const unsigned b = b0 + j;
                    if (b >= a0 && b < end_i && b < room) line0[b] = (uint8_t)(vv[j >> 2] >> (8 * (j & 3)));
                }
            }
        }
        if (c == nchunks - 1 && tid == 0) {
            const long long ff = (long long)before + chunk_total;
            const long long end = (long long)hdr + nbytes + ff;
            if (end + 2 <= jpeg_cap) { o[end] = 0xff; o[end + 1] = 0xd9; }
            else T->status = -4;
            T->scan_bits = bits;
            T->stuffed_ff = ff;
            T->jpeg_bytes = end + 2;
        }
        __syncthreads();
    }
}

}  // namespace h2j
