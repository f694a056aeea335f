// C ABI of h2j_b200 (include/h2j_b200.h): host-side orchestration of the kernels in h2j_kernels.cuh.
// Pure CUDA runtime; no torch types, no CPU encode path.
#include "../../include/h2j_b200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "h2j_kernels.cuh"

// h2j_host_copy.cpp: memcpy with non-temporal stores (plain memcpy where the CPU has no AVX2)
extern "C" void h2j_stream_copy(void *dst, const void *src, size_t n);

using namespace h2j;

namespace {

thread_local std::string g_create_error;

struct KernelTiming {
    const char *name;
    int start, stop;  // indices into Slot::events; back-to-back kernels share the event between them
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_done = nullptr;
    uint8_t *d_frames = nullptr;  // staging for host submits
    uint8_t *d_pitched = nullptr; // copies of frames with unaligned rows at a 16-byte pitch (allocated on first need)
    uint32_t *d_images = nullptr;  // [max_batch][images_cap] tile images (h2j_common.cuh)
    uint8_t *d_zero = nullptr;    // FrameState[max_batch] | descs | ticket | chunk_ff — zeroed every batch
    size_t zero_bytes = 0;
    FrameState *d_state = nullptr;
    unsigned long long *d_descs = nullptr;   // K4b group descriptors
    unsigned int *d_ticket = nullptr;
    unsigned int *d_stage_alloc = nullptr;   // K4a: staging words handed out per frame
    unsigned int *d_chunk_ff = nullptr;
    uint32_t *d_stage = nullptr;             // K4a -> K4b: the units' bits, word aligned, any order
    unsigned long long *d_unit_info = nullptr;
    FrameTab *d_tabs = nullptr;
    uint32_t *d_scan = nullptr;
    uint8_t *d_out = nullptr;
    uint8_t *d_packed = nullptr;
    unsigned long long *d_offsets = nullptr;
    int *d_status = nullptr;
    unsigned long long *h_offsets = nullptr;  // pinned
    int *h_status = nullptr;                  // pinned
    long long *h_sizes = nullptr;             // pinned (jpeg_bytes per frame)
    uint8_t *h_stage = nullptr;               // pinned staging for h2j_encode_frame / convert
    size_t h_stage_bytes = 0;
    unsigned char *h_tail = nullptr;          // pinned: status .. jpeg_bytes of frame 0's FrameTab (h2j_encode_frame)
    size_t spec_bytes = 384 * 1024;           // JPEG bytes h2j_encode_frame copies back before it knows the size
    bool busy = false;
    bool own_stream = true;
    bool packed = false;      // pack_kernel already ran for the batch in flight
    int n = 0;
    FrameLayout L{};
    std::vector<KernelTiming> timings;
    std::vector<cudaEvent_t> events;
    int timings_used = 0, events_used = 0;
    bool chain = false;  // the last thing enqueued was a timed kernel: its stop event is the next kernel's start
    bool timing_failed = false;  // an event of this batch's brackets could not be created / recorded
};

}  // namespace

struct h2j_encoder {
    h2j_settings s{};
    std::string comment;
    std::string err;
    int sm_count = 0;
    size_t out_cap = 0;           // per-frame output stride: jpeg_cap rounded up to 16 bytes
    size_t jpeg_cap = 0;          // max_jpeg_bytes exactly: the largest JPEG a frame may have
    long long scan_cap_words = 0;
    long long images_cap = 0;     // K2 tile images per frame at max geometry, rounded up to whole K4 tiles
    long long blocks_cap = 0;     // images_cap * 96
    int tiles_cap = 0;            // K4 tiles per frame at max geometry
    int units_cap = 0;            // K4 units (32 blocks) per frame
    int groups_cap = 0;           // K4b groups (64 units) per frame
    long long stage_cap_words = 0;
    int chunks_cap = 0;           // K5 chunks per frame
    int stuff_ctas = 32;          // K5 CTAs per frame
    int fdct_tiles_per_cta = 16;  // upper bound of consecutive K2 tiles one CTA walks
    int force_fdct_tiles = 0;     // h2j_debug_set_knob("fdct_tiles_per_cta"): exactly this many, whatever the batch size
    int force_sp_prepass = 0;     // h2j_debug_set_knob("semiplanar_prepass"): split semi-planar frames first even when aligned
    size_t frame_bytes_cap = 0;
    uint8_t *d_qscale_lut = nullptr;
    char *d_comment = nullptr;
    std::vector<Slot> slots;
    long long launches = 0;
};

namespace {

int fail(h2j_encoder *e, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->err = buf;
    else g_create_error = buf;
    return code;
}

#define CU(e, call)                                                                                       \
    do {                                                                                                  \
        cudaError_t err__ = (call);                                                                       \
        if (err__ != cudaSuccess)                                                                         \
            return fail((e), H2J_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
    } while (0)

// ---- first-frame rate control tail, folded into a table over i_tex_bits -----------------------------
// libavcodec/ratecontrol.c (FFmpeg 6fd0116): ff_rate_estimate_qscale -> get_qscale ("tex^qComp") ->
// get_diff_limited_q (no-op for the first I picture) -> intra-only blur -> modify_qscale -> clip ->
// (int)(q + 0.5); then mpegvideo_enc.c update_qscale().  All AVCodecContext fields at their defaults, as
// reference src/Encoder.cpp leaves them (it only sets time_base = 1/25, which cancels out for picture 0).
int qscale_from_i_tex_bits(int n)
{
    const float rce_qscale = 118 * 2;                    // FF_QP2LAMBDA * 2
    const float qcompress = 0.5f, qblur = 0.5f;
    const float i_quant_factor = -0.8f, i_quant_offset = 0.0f;
    const int lmin = 2 * 118, lmax = 31 * 118;
    int qmin = (int)(lmin * std::fabs((double)i_quant_factor) + i_quant_offset + 0.5);
    int qmax = (int)(lmax * std::fabs((double)i_quant_factor) + i_quant_offset + 0.5);
    const double rate_factor = 0.001 / 0.001 * 1.0f;     // pass1_wanted_bits / pass1_rc_eq_output_sum * br_compensation
    const double tex = (double)n * (double)rce_qscale;
    double bits = std::pow(tex, (double)qcompress);
    bits *= rate_factor;
    if (bits < 0.0) bits = 0.0;
    bits += 1.0;
    double qd = rce_qscale * (double)(n + 1) / bits;     // bits2qp
    qd = -qd * i_quant_factor + i_quant_offset;
    if (qd < 1) qd = 1;
    float q = (float)qd;
    double qsum = 0.001, qcount = 0.001;                 // short-term blur (intra_only)
    qsum *= qblur;
    qcount *= qblur;
    qsum += q;
    qcount++;
    q = (float)(qsum / qcount);
    double qm = q;                                       // modify_qscale
    if (qm < qmin) qm = qmin;
    else if (qm > qmax) qm = qmax;
    q = (float)qm;
    if (q < qmin) q = (float)qmin;
    else if (q > qmax) q = (float)qmax;
    q = (float)(int)(q + 0.5);
    return lambda_to_qscale((int)q);
}

uint8_t range_lut_value(int s, bool chroma)  // libswscale lumRangeToJpeg_c / chrRangeToJpeg_c + round
{
    int v = s << 7;
    if (!chroma) { if (v > 30189) v = 30189; v = (v * 19077 - 39057361) >> 14; }
    else { if (v > 30775) v = 30775; v = (v * 4663 - 9289992) >> 12; }
    v = (v + 64) >> 7;
    return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// chroma plane of a w x h frame as the decoder hands it over: ceil-divided by the format's subsampling
int chroma_w(int w, int fmt) { return (w + (1 << fmt_hshift(fmt)) - 1) >> fmt_hshift(fmt); }
int chroma_h(int h, int fmt) { return (h + (1 << fmt_vshift(fmt)) - 1) >> fmt_vshift(fmt); }
size_t tight_frame_bytes(int w, int h, int fmt) { return (size_t)w * h + 2 * (size_t)chroma_w(w, fmt) * chroma_h(h, fmt); }

// the vector-load flags of a planar layout whose frames start at `base`
void set_alignment(FrameLayout *L, const uint8_t *base)
{
    auto al = [&](int a) {
        return ((uintptr_t)base % a) == 0 && (L->frame_stride % a) == 0 && (L->u_off % a) == 0 && (L->v_off % a) == 0 &&
               (L->y_pitch % a) == 0 && (L->c_pitch % a) == 0;
    };
    L->aligned8 = al(8) ? 1 : 0;
    L->aligned16 = ((uintptr_t)base % 16) == 0 && (L->frame_stride % 16) == 0 && (L->y_pitch % 16) == 0 ? 1 : 0;
}

int make_layout(h2j_encoder *e, const uint8_t *base, size_t frame_stride, int w, int h, FrameLayout *L)
{
    if (w < 2 || h < 2 || w > 65500 || h > 65500) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", w, h);
    if (w > e->s.max_width || h > e->s.max_height)
        return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d exceeds the configured maximum %dx%d", w, h, e->s.max_width, e->s.max_height);
    const int fmt = e->s.chroma_format;
    const int fcw = chroma_w(w, fmt), fch = chroma_h(h, fmt);
    L->fmt = fmt;
    L->w = w; L->h = h;
    L->cw = w >> fmt_hshift(fmt); L->ch = h >> fmt_vshift(fmt);  // what the encoder reads (mpegvideo_enc.c load_input_picture)
    if (L->cw < 1 || L->ch < 1) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", w, h);
    L->y_pitch = w; L->c_pitch = fcw;
    L->u_off = (long long)w * h;
    L->v_off = L->u_off + (long long)fcw * fch;
    L->frame_stride = (long long)frame_stride;
    L->mb_w = (w + 15) >> 4;
    L->mcu_w = (w + fmt_mcu_px_w(fmt) - 1) / fmt_mcu_px_w(fmt); L->mcu_h = (h + 15) >> 4;
    L->n_mcu = L->mcu_w * L->mcu_h;
    L->n_blocks = L->n_mcu * fmt_mcu_blocks(fmt);
    set_alignment(L, base);
    L->range_mode = e->s.range_mode;
    L->fixed_qscale = e->s.fixed_qscale;
    L->nv12 = 0;
    return H2J_OK;
}

// Rows that do not start on 8-byte boundaries would send every block of K1 / K2 down the bytewise path: such batches are
// copied once to a 16-byte row pitch (repitch_kernel, ~1 us per 1080p frame) and the pipeline reads the copy.
// On return sl.L describes what the pipeline reads and *pipe_src is where it reads it.
size_t pitched_frame_bytes(int w, int h, int fmt)
{
    const int fcw = chroma_w(w, fmt), fch = chroma_h(h, fmt);
    return align_up(align_up((size_t)w, 16) * h + 2 * align_up((size_t)fcw, 16) * fch, 256);
}

// the same frame at a 16-byte row pitch in a 16-byte aligned buffer
FrameLayout pitched_layout(const FrameLayout &T)
{
    FrameLayout P = T;
    const int fcw = chroma_w(T.w, T.fmt), fch = chroma_h(T.h, T.fmt);
    P.y_pitch = (int)align_up((size_t)T.w, 16);
    P.c_pitch = (int)align_up((size_t)fcw, 16);
    P.u_off = (long long)P.y_pitch * T.h;
    P.v_off = P.u_off + (long long)P.c_pitch * fch;
    P.frame_stride = (long long)pitched_frame_bytes(T.w, T.h, T.fmt);
    P.aligned8 = 1;
    P.aligned16 = 1;
    return P;
}

// sl.L describes the n frames at d_src (any planar layout); src_end is the end of the last one's last plane
int repitch_if_unaligned(h2j_encoder *e, Slot &sl, const uint8_t *d_src, const uint8_t *src_end, int n, const uint8_t **pipe_src)
{
    const int w = sl.L.w, h = sl.L.h;
    *pipe_src = d_src;
    static const bool no_repitch = getenv("H2J_NO_REPITCH") != nullptr;  // measurement knob
    if (sl.L.aligned8 || no_repitch) return H2J_OK;
    if (!sl.d_pitched) {
        const size_t bytes = pitched_frame_bytes(e->s.max_width, e->s.max_height, e->s.chroma_format) * (size_t)e->s.max_batch;
        if (cudaMalloc(&sl.d_pitched, bytes) != cudaSuccess) {  // no room for the copy: the bytewise path still works
            cudaGetLastError();
            sl.d_pitched = nullptr;
            return H2J_OK;
        }
    }
    const FrameLayout T = sl.L;
    const FrameLayout P = pitched_layout(T);
    const int fch = chroma_h(h, T.fmt);
    repitch_kernel<<<dim3((w + 128 * 16 - 1) / (128 * 16), (h + 2 * fch + kPlaneRowsPerCta - 1) / kPlaneRowsPerCta, n), 128, 0, sl.stream>>>(d_src, T, fch, sl.d_pitched, P, d_src, src_end);
    e->launches++;
    CU(e, cudaGetLastError());
    sl.L = P;
    *pipe_src = sl.d_pitched;
    return H2J_OK;
}

int prepare_input(h2j_encoder *e, Slot &sl, const uint8_t *d_src, size_t src_stride, int n, int w, int h, const uint8_t **pipe_src)
{
    int rc = make_layout(e, d_src, src_stride, w, h, &sl.L);
    if (rc) return rc;
    const uint8_t *src_end = d_src + (size_t)(n - 1) * src_stride + tight_frame_bytes(w, h, sl.L.fmt);
    return repitch_if_unaligned(e, sl, d_src, src_end, n, pipe_src);
}

struct ScopedTiming {
    Slot &sl;
    bool on;
    int idx = -1;
    // an event that cannot be created or recorded switches the brackets of this batch off (the kernels still run; the
    // failure is remembered in the slot and reported by h2j_slot_kernel_ms)
    static int record(Slot &sl)
    {
        if (sl.events_used == (int)sl.events.size()) {
            cudaEvent_t ev;
            if (cudaEventCreate(&ev) != cudaSuccess) {
                cudaGetLastError();
                sl.timing_failed = true;
                return -1;
            }
            sl.events.push_back(ev);
        }
        if (cudaEventRecord(sl.events[sl.events_used], sl.stream) != cudaSuccess) {
            cudaGetLastError();
            sl.timing_failed = true;
            return -1;
        }
        return sl.events_used++;
    }
    ScopedTiming(h2j_encoder *e, Slot &s, const char *name) : sl(s), on(e->s.profile != 0 && !s.timing_failed)
    {
        if (!on) return;
        if (sl.timings_used == (int)sl.timings.size()) sl.timings.push_back(KernelTiming{name, -1, -1});
        idx = sl.timings_used++;
        sl.timings[idx].name = name;
        sl.timings[idx].start = (sl.chain && sl.events_used > 0) ? sl.events_used - 1 : record(sl);
    }
    ~ScopedTiming()
    {
        if (!on) return;
        sl.timings[idx].stop = sl.timing_failed ? -1 : record(sl);
        sl.chain = !sl.timing_failed;
    }
};

// Enqueue the whole pipeline for `n` frames at `d_frames` on the slot's stream.
int enqueue_pack_and_sizes(h2j_encoder *e, Slot &sl, bool pack);

enum TailMode { TAIL_SIZES = 0, TAIL_PACK = 1, TAIL_SINGLE = 2 };
int enqueue_single_tail(h2j_encoder *e, Slot &sl);

int launch_pipeline(h2j_encoder *e, Slot &sl, const uint8_t *d_frames, int n, int tail)
{
    const FrameLayout &L = sl.L;
    cudaStream_t st = sl.stream;
    sl.timings_used = 0;
    sl.events_used = 0;
    sl.chain = false;
    sl.timing_failed = false;
    CU(e, cudaMemsetAsync(sl.d_zero, 0, sl.zero_bytes, st));
    {
        ScopedTiming t(e, sl, "mbvar_kernel");
        mbvar_kernel<<<dim3(L.mcu_h, n), 128, 0, st>>>(d_frames, L, sl.d_state, e->d_qscale_lut, sl.d_tabs);
        e->launches++;
    }
    const int n_tiles = (L.n_mcu + kTileMcus - 1) / kTileMcus;
    {
        ScopedTiming t(e, sl, "fdct_quant_kernel");
        // consecutive tiles per CTA: as many as keep the grid at four waves or more (amortises the per-CTA set-up
        // and histogram flush), at most 16
        int tiles_per_cta = (int)((long long)n_tiles * n * fmt_roles(L.fmt) / ((long long)e->sm_count * 16 * 4));
        tiles_per_cta = tiles_per_cta < 1 ? 1 : (tiles_per_cta > e->fdct_tiles_per_cta ? e->fdct_tiles_per_cta : tiles_per_cta);
        if (const char *env = getenv("H2J_FDCT_TILES_PER_CTA")) tiles_per_cta = atoi(env) > 0 ? atoi(env) : tiles_per_cta;  // tuning knob
        if (e->force_fdct_tiles > 0) tiles_per_cta = e->force_fdct_tiles;
        // occupancy experiment knob (DESIGN.md section 4): extra dynamic shared memory limits the CTAs resident per SM
        static const int extra_smem = getenv("H2J_K2_EXTRA_SMEM") ? atoi(getenv("H2J_K2_EXTRA_SMEM")) : 0;
        const dim3 grid(fmt_roles(L.fmt) * ((n_tiles + tiles_per_cta - 1) / tiles_per_cta), n);
        if (L.fmt == kFmt422 && L.nv12) fdct_quant_fmt_kernel<kFmt422, true><<<grid, kFdctThreads, 0, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        else if (L.fmt == kFmt422) fdct_quant_fmt_kernel<kFmt422, false><<<grid, kFdctThreads, 0, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        else if (L.fmt == kFmt444 && L.nv12) fdct_quant_fmt_kernel<kFmt444, true><<<grid, kFdctThreads, 0, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        else if (L.fmt == kFmt444) fdct_quant_fmt_kernel<kFmt444, false><<<grid, kFdctThreads, 0, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        else if (L.nv12) fdct_quant_kernel<true><<<grid, kFdctThreads, extra_smem, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        else fdct_quant_kernel<false><<<grid, kFdctThreads, extra_smem, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "huffman_kernel");
        huffman_kernel<<<4 * n, kHuffGroup, 0, st>>>(L, sl.d_tabs, sl.d_state, n, sl.d_out, (long long)e->out_cap, (long long)e->jpeg_cap,
                                                                       e->d_comment, (int)e->comment.size());
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "entropy_walk_kernel");
        const dim3 grid(n_tiles, n);
        if (L.fmt == kFmt422)
            entropy_walk_kernel<kFmt422><<<grid, fmt_tile_blocks(kFmt422), ent_smem_bytes(kFmt422), st>>>(L, sl.d_tabs, sl.d_images, e->images_cap, sl.d_unit_info, e->units_cap,
                                                                                                     sl.d_stage_alloc, sl.d_stage, e->stage_cap_words);
        else if (L.fmt == kFmt444)
            entropy_walk_kernel<kFmt444><<<grid, fmt_tile_blocks(kFmt444), ent_smem_bytes(kFmt444), st>>>(L, sl.d_tabs, sl.d_images, e->images_cap, sl.d_unit_info, e->units_cap,
                                                                                                     sl.d_stage_alloc, sl.d_stage, e->stage_cap_words);
        else
            entropy_walk_kernel<kFmt420><<<grid, fmt_tile_blocks(kFmt420), ent_smem_bytes(kFmt420), st>>>(L, sl.d_tabs, sl.d_images, e->images_cap, sl.d_unit_info, e->units_cap,
                                                                                                     sl.d_stage_alloc, sl.d_stage, e->stage_cap_words);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "scan_place_kernel");
        const int n_units = (L.n_blocks + kUnitBlocks - 1) / kUnitBlocks;
        const int groups_per_frame = (n_units + kPlaceGroupUnits - 1) / kPlaceGroupUnits;
        // fewer groups than two per SM: every group on four times as many warps
        if ((long long)groups_per_frame * n < 2LL * e->sm_count)
            scan_place_kernel<8><<<groups_per_frame * n, kPlaceGroupUnits / 8 * 32, 0, st>>>(L, sl.d_tabs, sl.d_state, sl.d_unit_info, e->units_cap, sl.d_stage,
                                                                                   e->stage_cap_words, sl.d_descs, groups_per_frame, sl.d_ticket, sl.d_scan,
                                                                                   e->scan_cap_words, sl.d_chunk_ff, e->chunks_cap);
        else
            scan_place_kernel<32><<<groups_per_frame * n, kPlaceThreads, 0, st>>>(L, sl.d_tabs, sl.d_state, sl.d_unit_info, e->units_cap, sl.d_stage,
                                                                              e->stage_cap_words, sl.d_descs, groups_per_frame, sl.d_ticket, sl.d_scan,
                                                                              e->scan_cap_words, sl.d_chunk_ff, e->chunks_cap);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "stuff_kernel");
        static const int stuff_ctas_env = getenv("H2J_STUFF_CTAS") ? atoi(getenv("H2J_STUFF_CTAS")) : 0;  // tuning knob
        stuff_kernel<<<dim3(stuff_ctas_env > 0 ? stuff_ctas_env : e->stuff_ctas, n), kStuffThreads, 0, st>>>(sl.d_tabs, sl.d_state, sl.d_scan, e->scan_cap_words, sl.d_chunk_ff,
                                                                      e->chunks_cap, sl.d_out, (long long)e->out_cap, (long long)e->jpeg_cap);
        e->launches++;
    }
    CU(e, cudaGetLastError());
    // sizes/status (and, for host consumers, the packed payload) are produced inside the same enqueue so that
    // collecting a batch costs no further kernel launches
    if (tail == TAIL_SINGLE) return enqueue_single_tail(e, sl);
    return enqueue_pack_and_sizes(e, sl, tail == TAIL_PACK);
}

// h2j_encode_frame: no offsets kernel, no packing -- the frame's status / size fields and the first spec_bytes of its JPEG
// come back with two copies enqueued behind the kernels, so one synchronisation ends the call when the guess holds.
constexpr size_t kTabTailOff = offsetof(FrameTab, status);
constexpr size_t kTabTailBytes = sizeof(FrameTab) - kTabTailOff;
int enqueue_single_tail(h2j_encoder *e, Slot &sl)
{
    cudaStream_t st = sl.stream;
    sl.packed = false;
    sl.chain = false;
    CU(e, cudaMemcpyAsync(sl.h_tail, reinterpret_cast<const unsigned char *>(sl.d_tabs) + kTabTailOff, kTabTailBytes, cudaMemcpyDeviceToHost, st));
    const size_t spec = std::min(std::min(sl.spec_bytes, e->out_cap), sl.h_stage_bytes);
    CU(e, cudaMemcpyAsync(sl.h_stage, sl.d_out, spec, cudaMemcpyDeviceToHost, st));
    CU(e, cudaEventRecord(sl.ev_done, st));
    return H2J_OK;
}

int enqueue_pack_and_sizes(h2j_encoder *e, Slot &sl, bool pack)
{
    cudaStream_t st = sl.stream;
    {
        ScopedTiming t(e, sl, "pack_offsets_kernel");
        pack_offsets_kernel<<<1, kPackOffsetsThreads, 0, st>>>(sl.d_tabs, sl.n, (long long)e->jpeg_cap, sl.d_offsets, sl.d_status);
        e->launches++;
    }
    sl.packed = pack;
    if (pack) {
        ScopedTiming t(e, sl, "pack_kernel");
        pack_kernel<<<dim3(8, sl.n), 256, 0, st>>>(sl.d_out, (long long)e->out_cap, sl.d_offsets, sl.d_packed);
        e->launches++;
    }
    sl.chain = false;
    CU(e, cudaMemcpyAsync(sl.h_offsets, sl.d_offsets, sizeof(unsigned long long) * (sl.n + 1), cudaMemcpyDeviceToHost, st));
    CU(e, cudaMemcpyAsync(sl.h_status, sl.d_status, sizeof(int) * sl.n, cudaMemcpyDeviceToHost, st));
    CU(e, cudaEventRecord(sl.ev_done, st));
    CU(e, cudaGetLastError());
    return H2J_OK;
}

// Every entry point works on the encoder's device and leaves the caller's current device as it found it.
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) err = cudaSetDevice(device);
        else prev = -1;  // nothing to restore
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard &) = delete;
    DeviceGuard &operator=(const DeviceGuard &) = delete;
};
#define ON_DEVICE(e)                        \
    DeviceGuard device_guard__((e)->s.device); \
    CU(e, device_guard__.err)

// ---- staging copies of h2j_encode_frame -----------------------------------------------------------------------
// One picture's planes go from the caller's (pageable) memory into pinned staging before they can be uploaded.  That
// memcpy is the largest part of the call (0.26 of 0.35 ms for a 1080p frame: one thread copies ~12 GB/s on the pool's
// hosts), so it is done with non-temporal stores (h2j_host_copy.cpp: the staging lines are next read by the DMA engine,
// not by this core -- no read-for-ownership, +22 %), in pieces that are uploaded as soon as they are in place.
// Measured and dropped: sharing the pieces with up to three helper threads (a process-wide pool taking pieces off an
// atomic counter, spinning briefly between pictures) -- 0.45 ms instead of 0.35 on the GPU box and no gain in a host-only
// loop either: the copy is bound by what one process gets out of memory here, and waking the helpers costs more than
// they bring.
struct CopyPiece {
    uint8_t *dst;
    const uint8_t *src;
    int rows, row_bytes, dst_pitch, src_stride;
    size_t dev_off, dev_bytes;  // where the piece goes in the slot's frame buffer
};

void copy_piece(const CopyPiece &c)
{
    if (c.src_stride == c.row_bytes && c.dst_pitch == c.row_bytes) h2j_stream_copy(c.dst, c.src, (size_t)c.rows * c.row_bytes);
    else
        for (int r = 0; r < c.rows; r++) h2j_stream_copy(c.dst + (size_t)r * c.dst_pitch, c.src + (size_t)r * c.src_stride, (size_t)c.row_bytes);
}

int check_slot(h2j_encoder *e, int slot)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    if (slot < 0 || slot >= (int)e->slots.size()) return fail(e, H2J_ERR_INVALID_ARG, "slot %d out of range (n_slots %d)", slot, (int)e->slots.size());
    return H2J_OK;
}

void free_slot(Slot &sl)
{
    if (sl.stream) cudaStreamSynchronize(sl.stream);
    cudaFree(sl.d_frames); cudaFree(sl.d_pitched); cudaFree(sl.d_images); cudaFree(sl.d_zero); cudaFree(sl.d_stage); cudaFree(sl.d_unit_info);
    cudaFree(sl.d_tabs); cudaFree(sl.d_scan); cudaFree(sl.d_out); cudaFree(sl.d_packed); cudaFree(sl.d_offsets); cudaFree(sl.d_status);
    if (sl.h_offsets) cudaFreeHost(sl.h_offsets);
    if (sl.h_status) cudaFreeHost(sl.h_status);
    if (sl.h_sizes) cudaFreeHost(sl.h_sizes);
    if (sl.h_stage) cudaFreeHost(sl.h_stage);
    if (sl.h_tail) cudaFreeHost(sl.h_tail);
    for (auto &ev : sl.events) cudaEventDestroy(ev);
    if (sl.ev_begin) cudaEventDestroy(sl.ev_begin);
    if (sl.ev_done) cudaEventDestroy(sl.ev_done);
    if (sl.stream && sl.own_stream) cudaStreamDestroy(sl.stream);
    sl = Slot{};
}

}  // namespace

extern "C" {

void h2j_default_settings(h2j_settings *s)
{
    if (!s) return;
    memset(s, 0, sizeof *s);
    s->device = 0;
    s->max_width = 1920;
    s->max_height = 1088;
    s->max_batch = 16;
    s->n_slots = 2;
    s->range_mode = H2J_RANGE_PASSTHROUGH;
    s->fixed_qscale = 0;
    s->chroma_format = H2J_CHROMA_420;
    s->max_jpeg_bytes = 0;
    s->comment = nullptr;
    s->profile = 0;
}

int h2j_abi_version(void) { return H2J_ABI_VERSION; }

int h2j_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char *h2j_status_string(int status)
{
    switch (status) {
    case H2J_OK: return "ok";
    case H2J_ERR_INVALID_ARG: return "invalid argument";
    case H2J_ERR_CUDA: return "CUDA error";
    case H2J_ERR_UNSUPPORTED: return "unsupported geometry";
    case H2J_ERR_OUTPUT_TOO_SMALL: return "output buffer too small";
    case H2J_ERR_BUSY: return "slot busy / nothing to collect";
    case H2J_ERR_NOMEM: return "out of memory";
    case H2J_ERR_BUFFER_TOO_SMALL: return "caller buffer too small (slot still collectable)";
    default: return "unknown status";
    }
}

const char *h2j_last_error(const h2j_encoder *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

long long h2j_kernel_launches(const h2j_encoder *e) { return e ? e->launches : 0; }

void *h2j_alloc_pinned(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void h2j_free_pinned(void *p) { if (p) cudaFreeHost(p); }

void h2j_destroy(h2j_encoder *e)
{
    if (!e) return;
    DeviceGuard guard(e->s.device);
    for (auto &sl : e->slots) free_slot(sl);
    cudaFree(e->d_qscale_lut);
    cudaFree(e->d_comment);
    delete e;
}

int h2j_create(const h2j_settings *s, h2j_encoder **out)
{
    if (!s || !out) return fail(nullptr, H2J_ERR_INVALID_ARG, "null settings/out");
    *out = nullptr;
    if (s->max_width < 2 || s->max_height < 2 || s->max_width > 65500 || s->max_height > 65500 || s->max_batch < 1 || s->n_slots < 1 ||
        s->n_slots > 8 || s->fixed_qscale < 0 || s->fixed_qscale > 31 || (s->range_mode != 0 && s->range_mode != 1) ||
        s->chroma_format < H2J_CHROMA_420 || s->chroma_format > H2J_CHROMA_444 ||
        s->max_jpeg_bytes > ((size_t)256 << 20))  // bit positions inside a frame's scan are 32-bit
        return fail(nullptr, H2J_ERR_INVALID_ARG, "bad settings");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(nullptr, H2J_ERR_CUDA, "no usable CUDA device (%s); h2j_b200 has no CPU path", ce == cudaSuccess ? "device count 0" : cudaGetErrorString(ce));
    if (s->device < 0 || s->device >= ndev) return fail(nullptr, H2J_ERR_INVALID_ARG, "device %d out of range (%d devices)", s->device, ndev);
    h2j_encoder *e = new h2j_encoder();
    e->s = *s;
    e->comment = s->comment ? s->comment : "Lavc58.117.101";
    e->s.comment = nullptr;
    auto bail = [&](int code) { std::string m = e->err; h2j_destroy(e); g_create_error = m; return code; };
#define CUB(call)                                                                                                   \
    do {                                                                                                            \
        cudaError_t err__ = (call);                                                                                 \
        if (err__ != cudaSuccess) {                                                                                 \
            fail(e, H2J_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__);   \
            return bail(err__ == cudaErrorMemoryAllocation ? H2J_ERR_NOMEM : H2J_ERR_CUDA);                          \
        }                                                                                                           \
    } while (0)
    DeviceGuard device_guard(s->device);
    CUB(device_guard.err);
    cudaDeviceProp prop;
    CUB(cudaGetDeviceProperties(&prop, s->device));
    e->sm_count = prop.multiProcessorCount;

    e->jpeg_cap = s->max_jpeg_bytes ? s->max_jpeg_bytes : (size_t)2 * 1024 * 1024;
    e->out_cap = align_up(e->jpeg_cap, 16);
    e->scan_cap_words = (long long)(e->out_cap / 4);
    const int fmt = s->chroma_format;
    const int mcu_w = (s->max_width + fmt_mcu_px_w(fmt) - 1) / fmt_mcu_px_w(fmt), mcu_h = (s->max_height + 15) >> 4;
    const long long n_mcu = (long long)mcu_w * mcu_h;
    e->images_cap = (n_mcu + kTileMcus - 1) / kTileMcus;
    e->blocks_cap = e->images_cap * fmt_tile_blocks(fmt);
    e->tiles_cap = (int)e->images_cap;
    e->units_cap = e->tiles_cap * fmt_roles(fmt);  // units of 32 blocks: as many per tile as roles
    e->groups_cap = (e->units_cap + kPlaceGroupUnits - 1) / kPlaceGroupUnits;
    // a fixed place of one window per unit, then the reserved area for units that need more (every unit starts on a word:
    // at most one word of slack each)
    e->stage_cap_words = ((long long)e->units_cap * kWarpWinWords + e->scan_cap_words + e->units_cap + 3) / 4 * 4;  // (frames' areas stay 16-byte aligned)
    e->chunks_cap = (int)((e->scan_cap_words + kChunkWords - 1) >> kChunkShift);
    e->frame_bytes_cap = std::max(align_up(tight_frame_bytes(s->max_width, s->max_height, s->chroma_format), 256),
                                  pitched_frame_bytes(s->max_width, s->max_height, s->chroma_format));

    // constant tables
    {
        uint8_t lut[2][256];
        for (int i = 0; i < 256; i++) { lut[0][i] = range_lut_value(i, false); lut[1][i] = range_lut_value(i, true); }
        CUB(cudaMemcpyToSymbol(c_range_lut, lut, sizeof lut));
        std::vector<uint8_t> q(kQscaleLutSize);
        for (int n = 0; n < kQscaleLutSize; n++) q[n] = (uint8_t)qscale_from_i_tex_bits(n);
        CUB(cudaMalloc(&e->d_qscale_lut, kQscaleLutSize));
        CUB(cudaMemcpy(e->d_qscale_lut, q.data(), kQscaleLutSize, cudaMemcpyHostToDevice));
        CUB(cudaMalloc(&e->d_comment, e->comment.size() + 1));
        CUB(cudaMemcpy(e->d_comment, e->comment.c_str(), e->comment.size() + 1, cudaMemcpyHostToDevice));
    }
    if (getenv("H2J_K2_EXTRA_SMEM")) CUB(cudaFuncSetAttribute(fdct_quant_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt420>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt420)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt422>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt422)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt444>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt444)));

    const int B = s->max_batch;
    e->slots.resize(s->n_slots);
    for (auto &sl : e->slots) {
        CUB(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
        CUB(cudaEventCreate(&sl.ev_begin));
        CUB(cudaEventCreate(&sl.ev_done));
        CUB(cudaMalloc(&sl.d_frames, e->frame_bytes_cap * B));
        CUB(cudaMalloc(&sl.d_images, (size_t)e->images_cap * B * fmt_tile_image_words(fmt) * 4));
        const size_t state_bytes = align_up(sizeof(FrameState) * B, 256);
        const size_t desc_bytes = align_up(sizeof(unsigned long long) * (size_t)e->groups_cap * B, 256);
        const size_t alloc_bytes = align_up(sizeof(unsigned int) * (size_t)B, 256);
        const size_t chunk_bytes = align_up(sizeof(unsigned int) * (size_t)e->chunks_cap * B, 256);
        sl.zero_bytes = state_bytes + desc_bytes + 256 + alloc_bytes + chunk_bytes;
        CUB(cudaMalloc(&sl.d_zero, sl.zero_bytes));
        sl.d_state = reinterpret_cast<FrameState *>(sl.d_zero);
        sl.d_descs = reinterpret_cast<unsigned long long *>(sl.d_zero + state_bytes);
        sl.d_ticket = reinterpret_cast<unsigned int *>(sl.d_zero + state_bytes + desc_bytes);
        sl.d_stage_alloc = reinterpret_cast<unsigned int *>(sl.d_zero + state_bytes + desc_bytes + 256);
        sl.d_chunk_ff = reinterpret_cast<unsigned int *>(sl.d_zero + state_bytes + desc_bytes + 256 + alloc_bytes);
        CUB(cudaMalloc(&sl.d_stage, (size_t)e->stage_cap_words * 4 * B));
        CUB(cudaMalloc(&sl.d_unit_info, sizeof(unsigned long long) * (size_t)e->units_cap * B));
        CUB(cudaMalloc(&sl.d_tabs, sizeof(FrameTab) * B));
        CUB(cudaMalloc(&sl.d_scan, (size_t)e->scan_cap_words * 4 * B));
        CUB(cudaMalloc(&sl.d_out, e->out_cap * B));
        CUB(cudaMalloc(&sl.d_packed, e->out_cap * B));
        CUB(cudaMalloc(&sl.d_offsets, sizeof(unsigned long long) * (B + 1)));
        CUB(cudaMalloc(&sl.d_status, sizeof(int) * B));
        CUB(cudaHostAlloc(&sl.h_offsets, sizeof(unsigned long long) * (B + 1), cudaHostAllocDefault));
        CUB(cudaHostAlloc(&sl.h_status, sizeof(int) * B, cudaHostAllocDefault));
        CUB(cudaHostAlloc(&sl.h_sizes, sizeof(long long) * B, cudaHostAllocDefault));
    }
    // single-frame staging (slot 0 only): planes in, JPEG / padded planes out
    {
        Slot &s0 = e->slots[0];
        const size_t padded = (size_t)((s->max_width + 15) >> 4) * 16 * mcu_h * 16 * 3;
        s0.h_stage_bytes = std::max(std::max(e->frame_bytes_cap, e->out_cap), padded);
        CUB(cudaHostAlloc(&s0.h_stage, s0.h_stage_bytes, cudaHostAllocDefault));
        CUB(cudaHostAlloc(&s0.h_tail, 64, cudaHostAllocDefault));
    }
#undef CUB
    *out = e;
    return H2J_OK;
}

int h2j_submit_device(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int n, int width, int height)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!d_frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    if (frame_stride < tight_frame_bytes(width, height, e->s.chroma_format)) return fail(e, H2J_ERR_INVALID_ARG, "frame_stride smaller than one frame");
    ON_DEVICE(e);
    sl.n = n;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    const uint8_t *pipe_src = nullptr;
    rc = prepare_input(e, sl, d_frames, frame_stride, n, width, height, &pipe_src);
    if (rc) return rc;
    rc = launch_pipeline(e, sl, pipe_src, n, TAIL_SIZES);
    if (rc) return rc;
    sl.busy = true;
    return H2J_OK;
}

int h2j_submit_device_semiplanar(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch, size_t uv_offset,
                                 int n, int width, int height)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!d_frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    if (width < 2 || height < 2) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", width, height);
    const int fmt = e->s.chroma_format;
    const int fcw = chroma_w(width, fmt), fch = chroma_h(height, fmt);  // pairs per row, rows of the pair plane
    if (pitch < width || pitch < 2 * fcw) return fail(e, H2J_ERR_INVALID_ARG, "pitch %d smaller than a row of %d samples", pitch, width);
    if (uv_offset < (size_t)pitch * height || frame_stride < uv_offset + (size_t)pitch * (fch - 1) + 2 * (size_t)fcw)
        return fail(e, H2J_ERR_INVALID_ARG, "uv_offset / frame_stride do not hold a semi-planar frame of %dx%d at pitch %d", width, height, pitch);
    const size_t fb = tight_frame_bytes(width, height, fmt);
    const size_t dstride = align_up(fb, 256);
    if (dstride > e->frame_bytes_cap) return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d exceeds the configured maximum", width, height);
    ON_DEVICE(e);
    rc = make_layout(e, sl.d_frames, dstride, width, height, &sl.L);
    if (rc) return rc;
    sl.n = n;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    // Rows on 8-byte boundaries (what decoders produce): the pipeline reads the frames where they are -- K1 only looks at
    // luma, K2's chroma roles fetch the pairs and keep their component in registers.  Otherwise the pairs are split into
    // the slot's planar frame buffer first (one more pass over the frame).
    static const bool force_prepass = getenv("H2J_NV12_PREPASS") != nullptr;  // measurement knob
    if (!force_prepass && !e->force_sp_prepass && (uintptr_t)d_frames % 8 == 0 && frame_stride % 8 == 0 && pitch % 8 == 0 && uv_offset % 8 == 0) {
        FrameLayout &L = sl.L;
        L.y_pitch = pitch;
        L.c_pitch = pitch;
        L.u_off = (long long)uv_offset;
        L.v_off = (long long)uv_offset;
        L.frame_stride = (long long)frame_stride;
        L.aligned8 = 1;
        L.aligned16 = ((uintptr_t)d_frames % 16 == 0 && frame_stride % 16 == 0 && pitch % 16 == 0) ? 1 : 0;
        L.nv12 = 1;
        rc = launch_pipeline(e, sl, d_frames, n, TAIL_SIZES);
        if (rc) return rc;
        sl.busy = true;
        return H2J_OK;
    }
    const int src_aligned16 = ((uintptr_t)d_frames % 16) == 0 && (frame_stride % 16) == 0 && (pitch % 16) == 0 ? 1 : 0;
    const int row_bytes = width > 2 * fcw ? width : 2 * fcw;
    nv12_to_i420_kernel<<<dim3((row_bytes + 128 * 16 - 1) / (128 * 16), (height + fch + kPlaneRowsPerCta - 1) / kPlaneRowsPerCta, n), 128, 0, sl.stream>>>(
        d_frames, (long long)frame_stride, pitch, (long long)uv_offset, sl.d_frames, sl.L, src_aligned16);
    e->launches++;
    CU(e, cudaGetLastError());
    const uint8_t *pipe_src = nullptr;
    rc = prepare_input(e, sl, sl.d_frames, dstride, n, width, height, &pipe_src);  // (odd widths: once more, to a 16-byte pitch)
    if (rc) return rc;
    rc = launch_pipeline(e, sl, pipe_src, n, TAIL_SIZES);
    if (rc) return rc;
    sl.busy = true;
    return H2J_OK;
}

int h2j_submit_device_nv12(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch, size_t uv_offset, int n,
                           int width, int height)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    if (e->slots[slot].busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!d_frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    if (width < 2 || height < 2) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", width, height);
    if (e->s.chroma_format != H2J_CHROMA_420) return fail(e, H2J_ERR_UNSUPPORTED, "NV12 is a 4:2:0 layout; this encoder was created for another chroma format");
    return h2j_submit_device_semiplanar(e, slot, d_frames, frame_stride, pitch, uv_offset, n, width, height);
}

int h2j_submit_device_pitched(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int y_pitch, int c_pitch,
                              size_t u_offset, size_t v_offset, int n, int width, int height)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!d_frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    if (width < 2 || height < 2) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", width, height);
    const int fmt = e->s.chroma_format;
    const int fcw = chroma_w(width, fmt), fch = chroma_h(height, fmt);
    if (y_pitch < width || c_pitch < fcw) return fail(e, H2J_ERR_INVALID_ARG, "pitches %d / %d smaller than rows of %d / %d samples", y_pitch, c_pitch, width, fcw);
    const size_t y_end = (size_t)y_pitch * (height - 1) + width;
    const size_t u_end = u_offset + (size_t)c_pitch * (fch - 1) + fcw, v_end = v_offset + (size_t)c_pitch * (fch - 1) + fcw;
    if (y_end > frame_stride || u_end > frame_stride || v_end > frame_stride)
        return fail(e, H2J_ERR_INVALID_ARG, "a plane of the %dx%d frame reaches past frame_stride %zu", width, height, frame_stride);
    ON_DEVICE(e);
    rc = make_layout(e, d_frames, frame_stride, width, height, &sl.L);
    if (rc) return rc;
    FrameLayout &L = sl.L;
    L.y_pitch = y_pitch;
    L.c_pitch = c_pitch;
    L.u_off = (long long)u_offset;
    L.v_off = (long long)v_offset;
    set_alignment(&L, d_frames);
    sl.n = n;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    // rows on 8-byte boundaries: the pipeline reads the frames where they are; otherwise one copy to a 16-byte pitch
    const uint8_t *pipe_src = nullptr;
    const uint8_t *src_end = d_frames + (size_t)(n - 1) * frame_stride + std::max(y_end, std::max(u_end, v_end));
    rc = repitch_if_unaligned(e, sl, d_frames, src_end, n, &pipe_src);
    if (rc) return rc;
    rc = launch_pipeline(e, sl, pipe_src, n, TAIL_SIZES);
    if (rc) return rc;
    sl.busy = true;
    return H2J_OK;
}

int h2j_submit_host(h2j_encoder *e, int slot, const uint8_t *frames, size_t frame_stride, int n, int width, int height)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    const size_t fb = tight_frame_bytes(width, height, e->s.chroma_format);
    if (frame_stride < fb) return fail(e, H2J_ERR_INVALID_ARG, "frame_stride smaller than one frame");
    ON_DEVICE(e);
    // device copy keeps frames at a 256-byte aligned stride so the vector-load paths apply
    const size_t dstride = align_up(fb, 256);
    if (dstride > e->frame_bytes_cap) return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d exceeds the configured maximum", width, height);
    rc = make_layout(e, sl.d_frames, dstride, width, height, &sl.L);
    if (rc) return rc;
    sl.n = n;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    if (frame_stride == dstride) CU(e, cudaMemcpyAsync(sl.d_frames, frames, dstride * (n - 1) + fb, cudaMemcpyHostToDevice, sl.stream));
    else CU(e, cudaMemcpy2DAsync(sl.d_frames, dstride, frames, frame_stride, fb, n, cudaMemcpyHostToDevice, sl.stream));
    const uint8_t *pipe_src = nullptr;
    rc = prepare_input(e, sl, sl.d_frames, dstride, n, width, height, &pipe_src);
    if (rc) return rc;
    rc = launch_pipeline(e, sl, pipe_src, n, TAIL_PACK);
    if (rc) return rc;
    sl.busy = true;
    return H2J_OK;
}

int h2j_slot_set_stream(h2j_encoder *e, int slot, void *cuda_stream)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    if (sl.own_stream) CU(e, cudaStreamDestroy(sl.stream));
    sl.stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    sl.own_stream = false;
    return H2J_OK;
}

int h2j_slot_wait_event(h2j_encoder *e, int slot, void *cuda_event)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    if (!cuda_event) return fail(e, H2J_ERR_INVALID_ARG, "null event");
    Slot &sl = e->slots[slot];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    ON_DEVICE(e);
    CU(e, cudaStreamWaitEvent(sl.stream, reinterpret_cast<cudaEvent_t>(cuda_event), 0));
    return H2J_OK;
}

int h2j_wait(h2j_encoder *e, int slot)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    CU(e, cudaStreamSynchronize(e->slots[slot].stream));
    return H2J_OK;
}

int h2j_collect(h2j_encoder *e, int slot, uint8_t *out, size_t out_capacity, size_t *offsets, int *status)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has nothing to collect", slot);
    if (!out || !offsets) return fail(e, H2J_ERR_INVALID_ARG, "null out/offsets");
    ON_DEVICE(e);
    if (!sl.packed) {  // submitted with h2j_submit_device: pack now
        ScopedTiming t(e, sl, "pack_kernel");
        pack_kernel<<<dim3(8, sl.n), 256, 0, sl.stream>>>(sl.d_out, (long long)e->out_cap, sl.d_offsets, sl.d_packed);
        e->launches++;
        sl.packed = true;
    }
    CU(e, cudaStreamSynchronize(sl.stream));
    const size_t total = (size_t)sl.h_offsets[sl.n];
    int worst = H2J_OK;
    for (int i = 0; i <= sl.n; i++) offsets[i] = (size_t)sl.h_offsets[i];
    for (int i = 0; i < sl.n; i++) {
        if (status) status[i] = sl.h_status[i];
        if (sl.h_status[i] != 0) worst = sl.h_status[i];
    }
    // a short caller buffer loses nothing: offsets[] now holds the sizes, the slot stays collectable
    if (total > out_capacity) return fail(e, H2J_ERR_BUFFER_TOO_SMALL, "batch needs %zu bytes, caller gave %zu (collect again with a larger buffer)", total, out_capacity);
    CU(e, cudaMemcpyAsync(out, sl.d_packed, total, cudaMemcpyDeviceToHost, sl.stream));
    CU(e, cudaEventRecord(sl.ev_done, sl.stream));
    CU(e, cudaStreamSynchronize(sl.stream));
    sl.busy = false;
    // frames that failed (status[i] != 0) have length 0 in offsets[]; the others are complete
    if (worst != H2J_OK) return fail(e, worst, "at least one frame failed: %s", h2j_status_string(worst));
    return H2J_OK;
}

int h2j_collect_device(h2j_encoder *e, int slot, const uint8_t **d_out, size_t *d_frame_capacity, size_t *sizes, int *status)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!sl.busy) return fail(e, H2J_ERR_BUSY, "slot %d has nothing to collect", slot);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    sl.busy = false;
    int worst = H2J_OK;
    for (int i = 0; i < sl.n; i++) {
        if (sizes) sizes[i] = (size_t)(sl.h_offsets[i + 1] - sl.h_offsets[i]);
        if (status) status[i] = sl.h_status[i];
        if (sl.h_status[i] != 0) worst = sl.h_status[i];
    }
    if (d_out) *d_out = sl.d_out;
    if (d_frame_capacity) *d_frame_capacity = e->out_cap;
    if (worst != H2J_OK) return fail(e, worst, "at least one frame failed: %s", h2j_status_string(worst));
    return H2J_OK;
}

int h2j_encode_frame(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int width, int height, uint8_t *out,
                     size_t out_capacity, size_t *out_size)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    if (!planes || !strides || !planes[0] || !planes[1] || !planes[2] || !out || !out_size)
        return fail(e, H2J_ERR_INVALID_ARG, "null plane/out pointer");
    if (width < 2 || height < 2 || width > e->s.max_width || height > e->s.max_height)
        return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d outside 2x2 .. %dx%d", width, height, e->s.max_width, e->s.max_height);
    Slot &sl = e->slots[0];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot 0 has a batch in flight");
    const int fcw = chroma_w(width, e->s.chroma_format), fch = chroma_h(height, e->s.chroma_format);
    if (strides[0] < width || strides[1] < fcw || strides[2] < fcw) return fail(e, H2J_ERR_INVALID_ARG, "stride smaller than the row");
    // AVFrame planes -> tight I420 in pinned memory (the only host-side touch of the pixels): copied in pieces, every
    // piece uploaded as soon as it is in place, so that the DMA of one piece runs under the memcpy of the next
    ON_DEVICE(e);
    const size_t fb = tight_frame_bytes(width, height, e->s.chroma_format);
    const size_t dstride = align_up(fb, 256);
    if (dstride > e->frame_bytes_cap) return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d exceeds the configured maximum", width, height);
    int rc = make_layout(e, sl.d_frames, dstride, width, height, &sl.L);
    if (rc) return rc;
    // rows that would not start on 8-byte boundaries (odd widths) are staged at a 16-byte pitch right here: the rows are
    // copied one by one anyway, and the kernels keep their vector loads without a second pass over the frame
    if (!sl.L.aligned8) sl.L = pitched_layout(sl.L);
    const FrameLayout &L = sl.L;
    sl.n = 1;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    {
        constexpr int kMaxPieces = 96;
        CopyPiece pieces[kMaxPieces];
        int n_pieces = 0;
        auto plane = [&](const uint8_t *src, int stride, size_t off, int pw, int pitch, int ph) {
            // pieces of ~256 KiB, but never more than a third of the table per plane
            int rows_per_piece = std::max(1, (256 * 1024) / pitch);
            rows_per_piece = std::max(rows_per_piece, (ph + kMaxPieces / 3 - 1) / (kMaxPieces / 3));
            for (int r0 = 0; r0 < ph; r0 += rows_per_piece) {
                const int r1 = std::min(ph, r0 + rows_per_piece);
                CopyPiece &c = pieces[n_pieces++];
                c.dst = sl.h_stage + off + (size_t)r0 * pitch;
                c.src = src + (size_t)r0 * stride;
                c.rows = r1 - r0;
                c.row_bytes = pw;
                c.dst_pitch = pitch;
                c.src_stride = stride;
                c.dev_off = off + (size_t)r0 * pitch;
                c.dev_bytes = (size_t)(r1 - r0 - 1) * pitch + pw;
            }
        };
        plane(planes[0], strides[0], 0, width, L.y_pitch, height);
        plane(planes[1], strides[1], (size_t)L.u_off, fcw, L.c_pitch, fch);
        plane(planes[2], strides[2], (size_t)L.v_off, fcw, L.c_pitch, fch);
        // Planes that already live in page-locked memory (h2j_alloc_pinned, cudaHostAlloc, cudaHostRegister by the caller -- a
        // decoder whose frame buffers come from such a pool) are uploaded from where they are: no staging copy, one strided
        // DMA per plane.  The host copy is three quarters of the call for pageable planes.
        auto pinned = [](const void *p) {
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
            return at.type == cudaMemoryTypeHost;
        };
        static const bool no_direct = getenv("H2J_NO_DIRECT_UPLOAD") != nullptr;  // measurement knob
        if (!no_direct && pinned(planes[0]) && pinned(planes[1]) && pinned(planes[2])) {
            CU(e, cudaMemcpy2DAsync(sl.d_frames, L.y_pitch, planes[0], strides[0], width, height, cudaMemcpyHostToDevice, sl.stream));
            CU(e, cudaMemcpy2DAsync(sl.d_frames + L.u_off, L.c_pitch, planes[1], strides[1], fcw, fch, cudaMemcpyHostToDevice, sl.stream));
            CU(e, cudaMemcpy2DAsync(sl.d_frames + L.v_off, L.c_pitch, planes[2], strides[2], fcw, fch, cudaMemcpyHostToDevice, sl.stream));
            n_pieces = 0;
        }
        cudaError_t up_err = cudaSuccess;
        auto upload = [&](int i) {
            const cudaError_t ce = cudaMemcpyAsync(sl.d_frames + pieces[i].dev_off, sl.h_stage + pieces[i].dev_off, pieces[i].dev_bytes, cudaMemcpyHostToDevice, sl.stream);
            if (ce != cudaSuccess && up_err == cudaSuccess) up_err = ce;
        };
        for (int i = 0; i < n_pieces; i++) {
            copy_piece(pieces[i]);
            upload(i);
        }
        CU(e, up_err);
    }
    rc = launch_pipeline(e, sl, sl.d_frames, 1, TAIL_SINGLE);
    if (rc) return rc;
    CU(e, cudaStreamSynchronize(sl.stream));
    int st = 0;
    long long jpeg_bytes = 0;
    memcpy(&st, sl.h_tail + (offsetof(FrameTab, status) - kTabTailOff), sizeof st);
    memcpy(&jpeg_bytes, sl.h_tail + (offsetof(FrameTab, jpeg_bytes) - kTabTailOff), sizeof jpeg_bytes);
    if (st != 0) return fail(e, st, "the frame failed: %s", h2j_status_string(st));
    if (jpeg_bytes < 0 || (size_t)jpeg_bytes > e->jpeg_cap) return fail(e, H2J_ERR_OUTPUT_TOO_SMALL, "JPEG of %lld bytes exceeds max_jpeg_bytes", jpeg_bytes);
    const size_t n_out = (size_t)jpeg_bytes;
    *out_size = n_out;
    if (n_out > out_capacity) return fail(e, H2J_ERR_OUTPUT_TOO_SMALL, "JPEG is %zu bytes, caller gave %zu", n_out, out_capacity);
    const size_t spec = std::min(std::min(sl.spec_bytes, e->out_cap), sl.h_stage_bytes);
    const size_t have = std::min(n_out, spec);
    memcpy(out, sl.h_stage, have);
    if (n_out > have) {  // the guess was short: the rest straight into the caller's buffer
        CU(e, cudaMemcpy(out + have, sl.d_out + have, n_out - have, cudaMemcpyDeviceToHost));
    }
    // next guess: a quarter above this frame, in 64 KiB steps (consecutive frames of a stream are alike)
    sl.spec_bytes = std::max<size_t>(64 * 1024, align_up(n_out + n_out / 4, 64 * 1024));
    return H2J_OK;
}

int h2j_convert_pad(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int width, int height, int range_mode,
                    uint8_t *out_y, uint8_t *out_u, uint8_t *out_v)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    if (!planes || !strides || !planes[0] || !planes[1] || !planes[2] || !out_y || !out_u || !out_v) return fail(e, H2J_ERR_INVALID_ARG, "null pointer");
    if (width < 2 || height < 2 || width > e->s.max_width || height > e->s.max_height)
        return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d outside the configured maximum", width, height);
    if (range_mode != H2J_RANGE_PASSTHROUGH && range_mode != H2J_RANGE_LIMITED_TO_FULL) return fail(e, H2J_ERR_INVALID_ARG, "bad range_mode %d", range_mode);
    Slot &sl = e->slots[0];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot 0 has a batch in flight");
    if (e->s.chroma_format != H2J_CHROMA_420) return fail(e, H2J_ERR_UNSUPPORTED, "h2j_convert_pad handles 4:2:0 frames (the reference's format) only");
    const int fcw = (width + 1) >> 1, fch = (height + 1) >> 1;
    if (strides[0] < width || strides[1] < fcw || strides[2] < fcw) return fail(e, H2J_ERR_INVALID_ARG, "stride smaller than the row");
    ON_DEVICE(e);
    uint8_t *p = sl.h_stage;
    for (int r = 0; r < height; r++) memcpy(p + (size_t)r * width, planes[0] + (size_t)r * strides[0], width);
    p += (size_t)width * height;
    for (int pl = 1; pl <= 2; pl++) {
        for (int r = 0; r < fch; r++) memcpy(p + (size_t)r * fcw, planes[pl] + (size_t)r * strides[pl], fcw);
        p += (size_t)fcw * fch;
    }
    const size_t fb = tight_frame_bytes(width, height, e->s.chroma_format);
    FrameLayout L;
    int rc = make_layout(e, sl.d_frames, align_up(fb, 256), width, height, &L);
    if (rc) return rc;
    CU(e, cudaMemcpyAsync(sl.d_frames, sl.h_stage, fb, cudaMemcpyHostToDevice, sl.stream));
    const int pw = L.mcu_w * 16, ph = L.mcu_h * 16;
    // padded planes are produced in the (otherwise idle) coefficient buffer: 136 bytes per 64 samples, always enough
    const size_t need = (size_t)pw * ph * 3 / 2;
    if (need > (size_t)e->images_cap * kTileImageBytes * e->s.max_batch) return fail(e, H2J_ERR_UNSUPPORTED, "padded planes do not fit the slot's scratch buffer");
    uint8_t *oy = reinterpret_cast<uint8_t *>(sl.d_images), *ou = oy + (size_t)pw * ph, *ov = ou + (size_t)pw * ph / 4;
    convert_pad_kernel<<<dim3((pw / 16 + 127) / 128, ph, 3), 128, 0, sl.stream>>>(sl.d_frames, L, range_mode, oy, ou, ov);
    e->launches++;
    CU(e, cudaGetLastError());
    CU(e, cudaMemcpyAsync(out_y, oy, (size_t)pw * ph, cudaMemcpyDeviceToHost, sl.stream));
    CU(e, cudaMemcpyAsync(out_u, ou, (size_t)pw * ph / 4, cudaMemcpyDeviceToHost, sl.stream));
    CU(e, cudaMemcpyAsync(out_v, ov, (size_t)pw * ph / 4, cudaMemcpyDeviceToHost, sl.stream));
    CU(e, cudaStreamSynchronize(sl.stream));
    return H2J_OK;
}

int h2j_debug_frame_info(h2j_encoder *e, int slot, int frame, h2j_frame_info *info)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!info || frame < 0 || frame >= sl.n) return fail(e, H2J_ERR_INVALID_ARG, "bad frame index %d", frame);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    FrameTab t;
    FrameState st;
    CU(e, cudaMemcpy(&t, sl.d_tabs + frame, sizeof t, cudaMemcpyDeviceToHost));
    CU(e, cudaMemcpy(&st, sl.d_state + frame, sizeof st, cudaMemcpyDeviceToHost));
    memset(info, 0, sizeof *info);
    info->qscale = t.qscale;
    info->mb_var_sum = t.mb_var_sum;
    info->mcu_w = sl.L.mcu_w;
    info->mcu_h = sl.L.mcu_h;
    info->header_bytes = t.header_bytes;
    info->scan_bits = t.scan_bits;
    info->stuffed_ff = t.stuffed_ff;
    memcpy(info->intra_matrix, t.intra, 64);
    memcpy(info->hist, st.hist, sizeof info->hist);
    memcpy(info->bits, t.bits, sizeof info->bits);
    memcpy(info->vals, t.vals, sizeof info->vals);
    memcpy(info->nvals, t.nvals, sizeof info->nvals);
    return H2J_OK;
}

int h2j_debug_coefficients(h2j_encoder *e, int slot, int frame, int16_t *out, size_t out_elems)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!out || frame < 0 || frame >= sl.n) return fail(e, H2J_ERR_INVALID_ARG, "bad frame index %d", frame);
    const size_t need = (size_t)sl.L.n_blocks * 64;
    if (out_elems < need) return fail(e, H2J_ERR_OUTPUT_TOO_SMALL, "need %zu int16 elements", need);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    // tile images -> dense blocks; halfword 0 of a record is the DC difference, so the levels are rebuilt by
    // running the encoder's predictors (one per component, reset to 128) over the blocks in coding order
    const int fmt = sl.L.fmt, tile_blocks = fmt_tile_blocks(fmt), tile_words = fmt_tile_image_words(fmt);
    const int n_tiles = (sl.L.n_mcu + kTileMcus - 1) / kTileMcus;
    std::vector<int16_t> img((size_t)n_tiles * tile_words * 2);
    CU(e, cudaMemcpy(img.data(), sl.d_images + (size_t)frame * e->images_cap * tile_words, img.size() * sizeof(int16_t),
                     cudaMemcpyDeviceToHost));
    int last_dc[3] = {128, 128, 128};
    for (int b = 0; b < sl.L.n_blocks; b++) {
        const TileRec tr = tile_rec_fmt(fmt, b % tile_blocks);
        const int16_t *rec = img.data() + ((size_t)(b / tile_blocks) * tile_words + (size_t)tr.sub * kSubImageWords + (size_t)tr.idx * kBlkWords) * 2;
        const int comp = block_component(fmt, b % fmt_mcu_blocks(fmt));
        last_dc[comp] += rec[0];
        out[(size_t)b * 64] = (int16_t)last_dc[comp];
        for (int k = 1; k < 64; k++) out[(size_t)b * 64 + k] = rec[2 * (k & 31) + (k >> 5)];
    }
    return H2J_OK;
}

int h2j_debug_read_device(h2j_encoder *e, const void *d_src, void *dst, size_t bytes)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    if (!d_src || !dst) return fail(e, H2J_ERR_INVALID_ARG, "null pointer");
    ON_DEVICE(e);
    CU(e, cudaMemcpy(dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return H2J_OK;
}

int h2j_debug_set_knob(h2j_encoder *e, const char *name, int value)
{
    if (!e || !name) return H2J_ERR_INVALID_ARG;
    if (!strcmp(name, "fdct_tiles_per_cta")) {
        if (value < 0 || value > 4096) return fail(e, H2J_ERR_INVALID_ARG, "fdct_tiles_per_cta %d out of range", value);
        e->force_fdct_tiles = value;
        return H2J_OK;
    }
    if (!strcmp(name, "semiplanar_prepass")) {
        if (value < 0 || value > 1) return fail(e, H2J_ERR_INVALID_ARG, "semiplanar_prepass %d is not 0 or 1", value);
        e->force_sp_prepass = value;
        return H2J_OK;
    }
    return fail(e, H2J_ERR_INVALID_ARG, "unknown knob %s", name);
}

int h2j_set_profile(h2j_encoder *e, int on)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    e->s.profile = on ? 1 : 0;
    return H2J_OK;
}

int h2j_slot_kernel_ms(h2j_encoder *e, int slot, const char **names, float *ms, int cap)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    if (sl.timing_failed) return fail(e, H2J_ERR_CUDA, "a timing event of the slot's last batch could not be created or recorded");
    int n = 0;
    for (int i = 0; i < sl.timings_used && n < cap; i++) {
        if (sl.timings[i].start < 0 || sl.timings[i].stop < 0) continue;
        float t = 0.f;
        CU(e, cudaEventElapsedTime(&t, sl.events[sl.timings[i].start], sl.events[sl.timings[i].stop]));
        if (names) names[n] = sl.timings[i].name;
        if (ms) ms[n] = t;
        n++;
    }
    return n;
}

int h2j_slot_total_ms(h2j_encoder *e, int slot, float *ms)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!ms) return fail(e, H2J_ERR_INVALID_ARG, "null ms");
    ON_DEVICE(e);
    CU(e, cudaEventSynchronize(sl.ev_done));
    CU(e, cudaEventElapsedTime(ms, sl.ev_begin, sl.ev_done));
    return H2J_OK;
}

}  // extern "C"
