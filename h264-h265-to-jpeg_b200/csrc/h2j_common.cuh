// Device side of h2j_b200: the YUV -> JPEG stage of the reference (src/Encoder.cpp:104-308, i.e. libavcodec's
// mjpeg encoder as the reference configures it) as sm_100a kernels.  One launch handles a batch of frames; frames never
// interact, so the batch index is simply a grid dimension.  Every submit describes its batch by a per-frame table (FrameDesc);
// an input stage copies the frames the pipeline cannot read where they are (repitch, semi-planar split, 16-bit conversion,
// downscale: one launch), then the pipeline runs in its batch form (one layout by value, frames evenly spaced) or, for
// frames of different layouts, its list form (each CTA reads its frame's table entry).
//
//   K1  mbvar_kernel         luma 16x16 variance sums -> rate-control input              (HBM bound, 1 B/px read)
//   K2  fdct_quant_kernel    qscale + quantiser set-up, (range convert +) edge replicate + FDCT + quantise +
//                            zigzag + DC prediction + DC/AC symbol histograms           (integer issue bound, DESIGN.md)
//   K3  huffman_kernel       4 optimal (package-merge) tables, code tables, JPEG header
//   K4a entropy_walk_kernel  one walk per block into private slots, warp scan, merge, staging of 32-block units
//   K4b scan_place_kernel    unit lengths scanned (decoupled look-back over groups), units shifted into the scan, 0xFF census
//   K5  stuff_kernel         0xFF -> 0xFF00 expansion behind the header, EOI, final size
//   K6  pack_kernel          optional: JPEGs of a batch packed back to back for one D2H copy
//   convert_pad_kernel       kernel 1 on its own: range convert + MCU padding to planes (h2j_convert_pad)
//
// This header: the layout shared by host and device, constants and small helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "h2j_math.cuh"

namespace h2j {

struct FrameLayout {
    int w, h;          // luma size
    int cw, ch;        // chroma size the encoder reads: w>>1, h>>1 (mpegvideo_enc.c load_input_picture)
    int y_pitch, c_pitch;
    long long u_off, v_off, frame_stride;  // bytes from the frame base / between frames
    int mcu_w, mcu_h, n_mcu, n_blocks;
    int aligned8;      // every row of every plane starts on an 8-byte boundary -> 64-bit loads
    int aligned16;     // ... 16-byte boundary -> 128-bit loads (mbvar)
    int range_mode;
    int fixed_qscale;
    int nv12;          // chroma is ONE plane of interleaved Cb/Cr pairs at u_off, rows c_pitch apart (v_off unused)
    int fmt;           // kFmt420 (what the reference opens its encoder as), kFmt422, kFmt444: MCU geometry, see below
    int mb_w;          // 16x16 luma macroblocks per row (= mcu_w except at 4:4:4, whose MCUs are 8 wide): what K1 walks
};

// One frame of a batch.  A slot's table holds m pairs of them for n frames: entry f is frame f as the pipeline reads it,
// entry m + f the source a copy kernel makes it from (base nullptr: frame f is read in place).  m = n, or m = 1 for n frames of
// one layout at one stride: that pair stands for every frame, frame f at base + f * L.frame_stride.  The copy kernels and
// the LIST forms of K1-K4b (m = n only) read their frame's entry at blockIdx; their grids are sized for the batch's largest
// frame, and CTAs past their own frame's extent return before they touch any shared state.
struct FrameDesc {
    FrameLayout L;         // frame_stride: with m = 1, bytes between the frames' bases
    const uint8_t *base;   // the frame's first luma byte
    long long extent;      // copy sources (repitch / semi-planar split): bytes from base that may be read
};

// ---- chroma formats ------------------------------------------------------------------------------
// libavcodec's mjpeg encoder codes (mjpegenc.c ff_mjpeg_encode_mb, mjpegenc_common.c ff_mjpeg_init_hvsample)
//   4:2:0  16x16 MCUs of Y0 Y1 Y2 Y3 Cb Cr               (6 blocks; Y 2x2, chroma 1x1)      -- the reference's format
//   4:2:2  16x16 MCUs of Y0 Y1 Y2 Y3 Cb0 Cb1 Cr0 Cr1     (8 blocks; Y 2x2, chroma 1x2: top, bottom)
//   4:4:4   8x16 MCUs of Y0 Y1 Cb0 Cb1 Cr0 Cr1           (6 blocks; every component 1x2: top, bottom)
// A K2 tile is 16 consecutive MCUs whatever the format; its blocks are dealt to single-warp ROLES of 32 blocks each:
//   4:2:0  3 roles: luma of MCUs 0-7 (record = mcu * 4 + n), luma of MCUs 8-15, Cb (records 0-15) + Cr (16-31)
//   4:2:2  4 roles: luma of MCUs 0-7, luma of MCUs 8-15, Cb of the 16 MCUs (record = mcu * 2 + n), Cr
//   4:4:4  3 roles: Y of the 16 MCUs (record = mcu * 2 + n), Cb, Cr
enum { kFmt420 = 0, kFmt422 = 1, kFmt444 = 2 };
__host__ __device__ constexpr int fmt_roles(int fmt) { return fmt == kFmt422 ? 4 : 3; }
__host__ __device__ constexpr int fmt_mcu_blocks(int fmt) { return fmt == kFmt422 ? 8 : 6; }
__host__ __device__ constexpr int fmt_tile_blocks(int fmt) { return 16 * fmt_mcu_blocks(fmt); }  // 96 / 128 / 96 = roles * 32
__host__ __device__ constexpr int fmt_hshift(int fmt) { return fmt == kFmt444 ? 0 : 1; }        // chroma subsampling
__host__ __device__ constexpr int fmt_vshift(int fmt) { return fmt == kFmt420 ? 1 : 0; }
__host__ __device__ constexpr int fmt_mcu_px_w(int fmt) { return fmt == kFmt444 ? 8 : 16; }      // MCU width in luma samples

// ---- coefficient store ("tile images") -----------------------------------------------------------
// K2 works on tiles of 16 consecutive MCUs (96 blocks).  A tile leaves K2 as one contiguous image made of three
// sub-images, one per K2 warp, so that every warp can send its part on its own (no CTA barrier in K2's tile loop):
//   sub-image 0: the 32 luma blocks of MCUs 0..7  (record index = mcu * 4 + n)
//   sub-image 1: the 32 luma blocks of MCUs 8..15
//   sub-image 2: Cb of the 16 MCUs (records 0..15), Cr (records 16..31)
// A sub-image is 32 block records of 33 words each, then 32 words of high mask halves.
//   record word j (0..31)  low half: level j, high half: level j + 32 of the zigzag scan (this pairing lets K2
//                          derive the non-zero mask from packed 16-bit minima); level 0 is stored as the DC
//                          *difference* to the previous block of the same component, i.e. what gets coded
//   record word 32         non-zero mask of levels 1..31 (bit k = level k != 0, bit 0 clear).  It also makes the
//                          record stride odd in words: K2's lanes write their records without bank conflicts
//   word 1056 + r          non-zero mask of levels 32..63 of record r
// The image is assembled in shared memory and moved with bulk (TMA) copies: three stores of 4,352 bytes by K2, ONE
// load of two images by K4a.
constexpr int kTileMcus = 16;
constexpr int kTileBlocks = kTileMcus * 6;                  // 96
constexpr int kBlkWords = 33;
constexpr int kBlkHalf = kBlkWords * 2;                     // 66
constexpr int kMaskLoWord = 32;                             // inside the record
constexpr int kSubRecs = 32;
constexpr int kSubMaskHiOff = kSubRecs * kBlkWords;         // 1056
constexpr int kSubImageWords = kSubMaskHiOff + kSubRecs;    // 1088
constexpr int kSubImageBytes = kSubImageWords * 4;          // 4352 = 272 * 16
constexpr int kTileImageWords = 3 * kSubImageWords;         // 3264
constexpr int kTileImageBytes = kTileImageWords * 4;        // 13056 = 816 * 16
// block b of a tile (0..95 in coding order: Y0 Y1 Y2 Y3 Cb Cr per MCU) -> (sub-image, record)
struct TileRec { int sub, idx; };
__host__ __device__ inline TileRec tile_rec(int b)
{
    const int m = b / 6, n = b - 6 * m;
    TileRec r;
    if (n < 4) { r.sub = m >> 3; r.idx = (m & 7) * 4 + n; }
    else { r.sub = 2; r.idx = (n - 4) * 16 + m; }
    return r;
}
__host__ __device__ inline int tile_rec_word(int b) { const TileRec r = tile_rec(b); return r.sub * kSubImageWords + r.idx * kBlkWords; }
__host__ __device__ inline int tile_maskhi_word(int b) { const TileRec r = tile_rec(b); return r.sub * kSubImageWords + kSubMaskHiOff + r.idx; }
// the same for any format: block b of a tile in coding order -> (role's sub-image, record), and the block's component
__host__ __device__ inline TileRec tile_rec_fmt(int fmt, int b)
{
    if (fmt == kFmt420) return tile_rec(b);
    TileRec r;
    if (fmt == kFmt444) {
        const int m = b / 6, n = b - 6 * m;  // Y0 Y1 Cb0 Cb1 Cr0 Cr1
        r.sub = n >> 1;
        r.idx = m * 2 + (n & 1);
    } else {
        const int m = b >> 3, n = b & 7;     // Y0 Y1 Y2 Y3 Cb0 Cb1 Cr0 Cr1
        if (n < 4) { r.sub = m >> 3; r.idx = (m & 7) * 4 + n; }
        else { r.sub = 2 + ((n - 4) >> 1); r.idx = m * 2 + (n & 1); }
    }
    return r;
}
__host__ __device__ inline int block_component(int fmt, int n)  // n = position of the block in its MCU (coding order)
{
    if (fmt == kFmt420) return n < 4 ? 0 : n - 3;
    if (fmt == kFmt444) return n >> 1;
    return n < 4 ? 0 : 1 + ((n - 4) >> 1);
}
__host__ __device__ inline int fmt_tile_image_words(int fmt) { return fmt_roles(fmt) * kSubImageWords; }
constexpr int kFdctThreads = 32;                           // K2: single-warp CTAs, three roles per tile

constexpr int kEntThreads = kTileBlocks;                    // K4a: one CTA per K2 tile (two per CTA measured 3 % slower), a thread per block
constexpr int kMaxBitsPerBlock = 27 * 64;                   // DC (16+11) + 63 * (16+11); ZRLs only replace coefficients

constexpr int kHuffGroup = 128;                             // threads per table
constexpr int kHuffThreads = 4 * kHuffGroup;
constexpr int kStuffThreads = 256;
constexpr int kChunkShift = 10;                             // K5 works on chunks of 1024 scan words (4 KiB)
constexpr int kChunkWords = 1 << kChunkShift;
constexpr int kQscaleLutSize = 65536;

// Per-frame table block written by K2 (quantiser part) and K3 (Huffman part), read by K4/K5.
struct alignas(16) FrameTab {
    uint32_t qpack[64];      // raster order: q | (bias*q) << 16   (inspection)
    uint8_t dqt_zz[64];      // DQT payload (zigzag order)
    uint8_t intra[64];       // raster order (inspection)
    uint32_t hcode[4][256];  // ((code << nb) << 5) | (code length + nb), nb = symbol & 15: the mantissa bits K4a appends;
                             // classes: 0 DC luma, 1 DC chroma, 2 AC luma, 3 AC chroma
                             // The two DC tables (16 entries each) live in hcode[1][224..255] (dc_code_table), right in front of
                             // the AC tables: 16-byte aligned, K4a fetches all four with one bulk copy; hcode[0] and the rest
                             // of hcode[1] are not used
    uint8_t bits[4][17];
    uint8_t vals[4][256];
    int nvals[4];
    int qscale;
    int header_bytes;
    int status;              // h2j_status of this frame
    int pad_;
    long long mb_var_sum;
    long long scan_bits;
    long long stuffed_ff;
    long long jpeg_bytes;
};

constexpr int kDcCodeOff = 256 - 32;  // first word of the DC code tables inside hcode[1]
__host__ __device__ inline uint32_t *dc_code_table(FrameTab *T, int cls) { return T->hcode[1] + kDcCodeOff + 16 * cls; }

// Per-frame state zeroed by one memset at the start of every batch.
struct FrameState {
    unsigned long long var_sum;
    unsigned long long scan_bits;   // written by the frame's last K4b group
    unsigned int k1_done;           // K1 CTAs that have added their share of var_sum
    unsigned int k3_done;           // K3 CTAs (one per table) that have finished: the fourth writes the header
    unsigned int hist[4][256];      // DC luma, DC chroma, AC luma, AC chroma symbol counts (K2)
};

__constant__ uint8_t c_zigzag[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                     41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                     30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
// ff_mpeg1_default_intra_matrix, raster order
__constant__ uint8_t c_mpeg1_intra[64] = {8,  16, 19, 22, 26, 27, 29, 34, 16, 16, 22, 24, 27, 29, 34, 37, 19, 22, 26, 27, 29, 34,
                                          34, 38, 22, 22, 26, 27, 29, 34, 37, 40, 22, 26, 27, 29, 32, 35, 40, 48, 26, 27, 29, 32,
                                          35, 40, 48, 58, 26, 27, 29, 34, 38, 46, 56, 69, 27, 29, 35, 38, 46, 56, 69, 83};
// swscale limited->full LUTs, [0] luma, [1] chroma; filled by the host at create time from the closed form
__constant__ uint8_t c_range_lut[2][256];

// compile-time zigzag for the register-resident block
__host__ __device__ constexpr int zz_of(int k)
{
    constexpr int t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                           41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                           30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return t[k];
}

__device__ __forceinline__ uint2 ldg64(const uint8_t *p) { return __ldg(reinterpret_cast<const uint2 *>(p)); }
__device__ __forceinline__ uint4 ldg128(const uint8_t *p) { return __ldg(reinterpret_cast<const uint4 *>(p)); }

// JPEG magnitude category: number of bits of |v| (0 for v == 0)
__device__ __forceinline__ int mag_bits(int v)
{
    unsigned b;  // bfind gives 0xffffffff for 0: one add instead of the two that 32 - clz() compiles to
    asm("bfind.u32 %0, %1;" : "=r"(b) : "r"(abs(v)));
    return (int)b + 1;
}

// number of 0xFF bytes in a 32-bit word (exact zero-byte test on the complement)
__device__ __forceinline__ unsigned count_ff_bytes(unsigned v)
{
    const unsigned x = ~v;
    const unsigned y = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu);  // 0x80 in every byte of x that is zero
    return __popc(y);
}

// ---- mbarrier + bulk copy (TMA engine, 1-D) -------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// (at most the newest one may still be reading)
__device__ __forceinline__ void bulk_wait_read_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// shared -> global bulk store (TMA engine), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// ask for a range of global memory to be brought into L2 (TMA engine, fire and forget: no shared memory, nothing to wait for)
__device__ __forceinline__ void bulk_prefetch_l2(const void *src_gmem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src_gmem), "r"(bytes) : "memory");
}
// the issuing thread's bulk stores have finished READING shared memory (the source may be overwritten)
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and have completed altogether
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy writes to shared memory become visible to the async proxy (TMA) -- every writer, before the barrier
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

}  // namespace h2j
