// C ABI of h2j_b200 (include/h2j_b200.h): host-side orchestration of the kernels in h2j_kernels.cuh.
// Pure CUDA runtime; no torch types, no CPU encode path.
#include "../../include/h2j_b200.h"

#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <utility>
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
    uint8_t *d_frames = nullptr;  // staging for host submits; the input stage's split, converted and downscaled frames
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
    // the converting single-picture calls (h2j_encode_frame16, h2j_encode_frame_rgb; slot 0): the caller's picture as staged
    // on the device, before the input stage converts it, and its pinned staging; allocated on first use, grown when a call
    // needs more (reserve_convert)
    uint8_t *d_convert = nullptr;
    uint8_t *h_convert = nullptr;
    size_t convert_bytes = 0;
    // h2j_submit_device_resized: the batch's coefficient arena (ResizeFrame per frame, then the axes' windows and
    // coefficients) and its pinned mirror, allocated on first use and grown when a submit needs more; resize_used bytes of it
    // are uploaded with one copy on the slot's stream (the busy-slot rule keeps the mirror as it is while that copy is pending)
    uint8_t *d_resize = nullptr;
    uint8_t *h_resize = nullptr;
    size_t resize_bytes = 0, resize_used = 0;
    unsigned char *h_tail = nullptr;          // pinned: status .. jpeg_bytes of frame 0's FrameTab (h2j_encode_frame)
    size_t spec_bytes = 384 * 1024;           // JPEG bytes h2j_encode_frame copies back before it knows the size
    bool busy = false;
    bool own_stream = true;
    bool packed = false;      // pack_kernel already ran for the batch in flight
    int n = 0;
    // the batch (every submit), m entry pairs (h2j_common.cuh FrameDesc): descs[i] is frame i as the pipeline reads it,
    // descs[m + i] the source a copy kernel reads it from (base nullptr: no copy).  m = n, or 1 for n frames of one layout at
    // one stride.  The pinned mirror is filled by the submit and, when a kernel reads the table, uploaded with one copy on the
    // slot's stream; a busy slot refuses a submit, so it is never rewritten while that copy is pending.
    int m = 0;
    FrameDesc *d_desc = nullptr;  // [2 * max_batch]
    FrameDesc *h_desc = nullptr;  // pinned mirror
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
    int force_fdct_tiles = 0;     // h2j_debug_set_knob("fdct_tiles_per_cta"): exactly this many, whatever the batch size
    int force_sp_prepass = 0;     // h2j_debug_set_knob("semiplanar_prepass"): split semi-planar frames first even when aligned
    int planar_copy = 1;          // h2j_debug_set_knob("planar_copy"): 0 = read unaligned planar frames in place, as without d_pitched
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

// the vector-load flags of a planar layout whose frames start at `base`, `frame_stride` apart
void set_alignment(FrameLayout *L, const uint8_t *base, size_t frame_stride = 0)
{
    auto al = [&](int a) {
        return ((uintptr_t)base % a) == 0 && (frame_stride % a) == 0 && (L->u_off % a) == 0 && (L->v_off % a) == 0 &&
               (L->y_pitch % a) == 0 && (L->c_pitch % a) == 0;
    };
    L->aligned8 = al(8) ? 1 : 0;
    L->aligned16 = ((uintptr_t)base % 16) == 0 && (frame_stride % 16) == 0 && (L->y_pitch % 16) == 0 ? 1 : 0;
}

// A tight planar frame at `base`.  within_max = false: a frame the encoder does not encode at this size (the source of a
// downscaled submit)
int make_layout(h2j_encoder *e, const uint8_t *base, int w, int h, FrameLayout *L, bool within_max = true)
{
    if (w < 2 || h < 2 || w > 65500 || h > 65500) return fail(e, H2J_ERR_UNSUPPORTED, "unsupported frame size %dx%d", w, h);
    if (within_max && (w > e->s.max_width || h > e->s.max_height))
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
    L->frame_stride = 0;
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

// Rows that do not start on 8-byte boundaries would send every block of K1 / K2 down the bytewise path: such frames are
// copied once to a 16-byte row pitch (repitch_kernel, ~1 us per 1080p frame) and the pipeline reads the copy.
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
    P.aligned8 = 1;
    P.aligned16 = 1;
    return P;
}

// the h2j_frame_desc of a tight planar frame at `base`
h2j_frame_desc tight_frame(const uint8_t *base, int w, int h, int fmt)
{
    const int fcw = chroma_w(w, fmt);
    const size_t u_off = (size_t)w * h;
    return h2j_frame_desc{base, w, h, w, fcw, u_off, u_off + (size_t)fcw * chroma_h(h, fmt)};
}

bool odd(size_t v) { return (v & 1) != 0; }

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

constexpr int kFdctMaxTilesPerCta = 16;  // K2: upper bound of consecutive tiles one CTA walks (h2j_debug_set_knob may force any)
constexpr int kStuffCtas = 32;           // K5 CTAs per frame
constexpr size_t kMaxCommentBytes = 65535 - 3;  // settings.comment: a COM segment's length field counts the text, its NUL and itself

// the K2 instantiation for the layout kind (chroma format, semi-planar chroma read in place) and the batch kind
template <bool LIST>
decltype(&fdct_quant_kernel<false, false>) k2_kernel(const FrameLayout &L)
{
    return L.fmt == kFmt422 ? (L.nv12 ? fdct_quant_fmt_kernel<kFmt422, true, LIST> : fdct_quant_fmt_kernel<kFmt422, false, LIST>)
           : L.fmt == kFmt444 ? (L.nv12 ? fdct_quant_fmt_kernel<kFmt444, true, LIST> : fdct_quant_fmt_kernel<kFmt444, false, LIST>)
                              : (L.nv12 ? fdct_quant_kernel<true, LIST> : fdct_quant_kernel<false, LIST>);
}

// frame f of the slot's batch as the pipeline reads it (a table of one pair: the pair's layout, for every frame)
const FrameDesc &frame_desc(const Slot &sl, int f) { return sl.h_desc[f < sl.m ? f : 0]; }

// The batch form of the pipeline takes one layout and reads frame f at base + f * frame_stride: it runs when the frames of the
// slot's table all have the same layout and are evenly spaced (the list form costs 0.92x on uniform input).  false: a list.
bool batch_stride(const Slot &sl, long long *frame_stride)
{
    const FrameDesc *D = sl.h_desc;
    const int m = sl.m;
    const long long stride = m > 1 ? (long long)((uintptr_t)D[1].base - (uintptr_t)D[0].base) : D[0].L.frame_stride;
    for (int i = 1; i < m; i++)
        if (memcmp(&D[i].L, &D[0].L, offsetof(FrameLayout, mb_w) + sizeof(int)) != 0 ||  // (every field, not the tail padding)
            (uintptr_t)D[i].base != (uintptr_t)D[0].base + (uintptr_t)(i * stride))
            return false;
    *frame_stride = stride;
    return true;
}

// The pipeline for the slot's batch; the list form reads it from sl.d_desc (uploaded by run_batch), its grids sized for the
// largest frame
int launch_pipeline(h2j_encoder *e, Slot &sl, int n, int tail)
{
    long long stride = 0;
    const bool list = !batch_stride(sl, &stride);
    FrameLayout L = sl.h_desc[0].L;  // (list: what all frames share: chroma format, nv12)
    L.frame_stride = stride;
    const uint8_t *d_frames = list ? nullptr : sl.h_desc[0].base;
    const FrameDesc *D = list ? sl.d_desc : nullptr;
    int mcu_h = 0, n_tiles = 0, n_units = 0;
    long long total_tiles = 0;
    for (int i = 0; i < n; i++) {
        const FrameLayout &Li = frame_desc(sl, i).L;
        const int t = (Li.n_mcu + kTileMcus - 1) / kTileMcus;
        mcu_h = std::max(mcu_h, Li.mcu_h);
        n_tiles = std::max(n_tiles, t);
        n_units = std::max(n_units, (Li.n_blocks + kUnitBlocks - 1) / kUnitBlocks);
        total_tiles += t;
    }
    cudaStream_t st = sl.stream;
    sl.timings_used = 0;
    sl.events_used = 0;
    sl.chain = false;
    sl.timing_failed = false;
    CU(e, cudaMemsetAsync(sl.d_zero, 0, sl.zero_bytes, st));
    {
        ScopedTiming t(e, sl, "mbvar_kernel");
        (list ? mbvar_kernel<true> : mbvar_kernel<false>)<<<dim3(mcu_h, n), 128, 0, st>>>(d_frames, L, sl.d_state, e->d_qscale_lut, sl.d_tabs, D);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "fdct_quant_kernel");
        // consecutive tiles per CTA: as many as keep the grid at four waves or more (amortises the per-CTA set-up
        // and histogram flush), at most kFdctMaxTilesPerCta
        int tiles_per_cta = (int)(total_tiles * fmt_roles(L.fmt) / ((long long)e->sm_count * kFdctMinCtas * 4));
        tiles_per_cta = tiles_per_cta < 1 ? 1 : (tiles_per_cta > kFdctMaxTilesPerCta ? kFdctMaxTilesPerCta : tiles_per_cta);
        if (e->force_fdct_tiles > 0) tiles_per_cta = e->force_fdct_tiles;
        const dim3 grid(fmt_roles(L.fmt) * ((n_tiles + tiles_per_cta - 1) / tiles_per_cta), n);
        const auto k2 = list ? k2_kernel<true>(L) : k2_kernel<false>(L);
        k2<<<grid, kFdctThreads, 0, st>>>(d_frames, L, sl.d_state, sl.d_tabs, sl.d_images, e->images_cap, tiles_per_cta, D);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "huffman_kernel");
        (list ? huffman_kernel<true> : huffman_kernel<false>)<<<4 * n, kHuffGroup, 0, st>>>(L, sl.d_tabs, sl.d_state, n, sl.d_out, (long long)e->out_cap,
                                                                                        (long long)e->jpeg_cap, e->d_comment, (int)e->comment.size(), D);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "entropy_walk_kernel");
        const auto k4a = list ? (L.fmt == kFmt420 ? entropy_walk_kernel<kFmt420, true> : L.fmt == kFmt422 ? entropy_walk_kernel<kFmt422, true> : entropy_walk_kernel<kFmt444, true>)
                              : (L.fmt == kFmt420 ? entropy_walk_kernel<kFmt420, false> : L.fmt == kFmt422 ? entropy_walk_kernel<kFmt422, false> : entropy_walk_kernel<kFmt444, false>);
        k4a<<<dim3(n_tiles, n), fmt_tile_blocks(L.fmt), ent_smem_bytes(L.fmt), st>>>(L, sl.d_tabs, sl.d_images, e->images_cap, sl.d_unit_info, e->units_cap,
                                                                                     sl.d_stage_alloc, sl.d_stage, e->stage_cap_words, D);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "scan_place_kernel");
        const int groups_per_frame = (n_units + kPlaceGroupUnits - 1) / kPlaceGroupUnits;
        // fewer groups than two per SM: every group on four times as many warps
        if ((long long)groups_per_frame * n < 2LL * e->sm_count)
            (list ? scan_place_kernel<8, true> : scan_place_kernel<8, false>)<<<groups_per_frame * n, kPlaceGroupUnits / 8 * 32, 0, st>>>(
                L, sl.d_tabs, sl.d_state, sl.d_unit_info, e->units_cap, sl.d_stage, e->stage_cap_words, sl.d_descs, groups_per_frame, sl.d_ticket,
                sl.d_scan, e->scan_cap_words, sl.d_chunk_ff, e->chunks_cap, D);
        else
            (list ? scan_place_kernel<32, true> : scan_place_kernel<32, false>)<<<groups_per_frame * n, kPlaceThreads, 0, st>>>(
                L, sl.d_tabs, sl.d_state, sl.d_unit_info, e->units_cap, sl.d_stage, e->stage_cap_words, sl.d_descs, groups_per_frame, sl.d_ticket,
                sl.d_scan, e->scan_cap_words, sl.d_chunk_ff, e->chunks_cap, D);
        e->launches++;
    }
    {
        ScopedTiming t(e, sl, "stuff_kernel");
        stuff_kernel<<<dim3(kStuffCtas, n), kStuffThreads, 0, st>>>(sl.d_tabs, sl.d_state, sl.d_scan, e->scan_cap_words, sl.d_chunk_ff,
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

// Upload one picture's planes (the first n_planes of three: rows[i] rows of row_bytes[i] bytes, strides[i] apart in host
// memory) to dev + off[i] at pitch[i] on the slot's stream.  Pageable planes go through `stage` (pinned, laid out as on the
// device) in pieces, every piece uploaded as soon as it is in place, so that the DMA of one piece runs under the memcpy of
// the next.
int upload_planes(h2j_encoder *e, Slot &sl, const uint8_t *const planes[3], const int strides[3], const int row_bytes[3], const int rows[3],
                  const size_t off[3], const int pitch[3], uint8_t *dev, uint8_t *stage, int n_planes = 3)
{
    constexpr int kMaxPieces = 96;
    CopyPiece pieces[kMaxPieces];
    int n_pieces = 0;
    for (int p = 0; p < n_planes; p++) {
        const int ph = rows[p];
        // pieces of ~256 KiB, but never more than a third of the table per plane
        int rows_per_piece = std::max(1, (256 * 1024) / pitch[p]);
        rows_per_piece = std::max(rows_per_piece, (ph + kMaxPieces / 3 - 1) / (kMaxPieces / 3));
        for (int r0 = 0; r0 < ph; r0 += rows_per_piece) {
            const int r1 = std::min(ph, r0 + rows_per_piece);
            CopyPiece &c = pieces[n_pieces++];
            c.dst = stage + off[p] + (size_t)r0 * pitch[p];
            c.src = planes[p] + (size_t)r0 * strides[p];
            c.rows = r1 - r0;
            c.row_bytes = row_bytes[p];
            c.dst_pitch = pitch[p];
            c.src_stride = strides[p];
            c.dev_off = off[p] + (size_t)r0 * pitch[p];
            c.dev_bytes = (size_t)(r1 - r0 - 1) * pitch[p] + row_bytes[p];
        }
    }
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
    bool all_pinned = true;
    for (int p = 0; p < n_planes; p++) all_pinned = all_pinned && pinned(planes[p]);
    if (all_pinned) {
        for (int p = 0; p < n_planes; p++)
            CU(e, cudaMemcpy2DAsync(dev + off[p], pitch[p], planes[p], strides[p], row_bytes[p], rows[p], cudaMemcpyHostToDevice, sl.stream));
        n_pieces = 0;
    }
    cudaError_t up_err = cudaSuccess;
    for (int i = 0; i < n_pieces; i++) {
        copy_piece(pieces[i]);
        const cudaError_t ce = cudaMemcpyAsync(dev + pieces[i].dev_off, stage + pieces[i].dev_off, pieces[i].dev_bytes, cudaMemcpyHostToDevice, sl.stream);
        if (ce != cudaSuccess && up_err == cudaSuccess) up_err = ce;
    }
    CU(e, up_err);
    return H2J_OK;
}

// The single-picture pipeline (TAIL_SINGLE) is enqueued: wait for it and hand the JPEG over.
int finish_single(h2j_encoder *e, Slot &sl, uint8_t *out, size_t out_capacity, size_t *out_size)
{
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

void free_slot(Slot &sl)
{
    if (sl.stream) cudaStreamSynchronize(sl.stream);
    cudaFree(sl.d_frames); cudaFree(sl.d_pitched); cudaFree(sl.d_images); cudaFree(sl.d_zero); cudaFree(sl.d_stage); cudaFree(sl.d_unit_info);
    cudaFree(sl.d_tabs); cudaFree(sl.d_scan); cudaFree(sl.d_out); cudaFree(sl.d_packed); cudaFree(sl.d_offsets); cudaFree(sl.d_status);
    cudaFree(sl.d_convert);
    cudaFree(sl.d_resize);
    cudaFree(sl.d_desc);
    if (sl.h_desc) cudaFreeHost(sl.h_desc);
    if (sl.h_convert) cudaFreeHost(sl.h_convert);
    if (sl.h_resize) cudaFreeHost(sl.h_resize);
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

// The preamble of every batch submit: a slot that exists and has no batch in flight, a frames pointer, 1 .. max_batch frames.
// Every check of a submit is made before anything is enqueued or the slot's table is touched: a rejected call leaves the
// previous batch collectable and inspectable.
int check_submit(h2j_encoder *e, int slot, const void *frames, int n)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    if (e->slots[slot].busy) return fail(e, H2J_ERR_BUSY, "slot %d has a batch in flight", slot);
    if (!frames || n < 1 || n > e->s.max_batch) return fail(e, H2J_ERR_INVALID_ARG, "bad frames pointer or batch size %d (max %d)", n, e->s.max_batch);
    return H2J_OK;
}

// the preamble of a device list submit (h2j_submit_device_list, h2j_submit_device_downscaled)
int check_device_list(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n)
{
    int rc = check_submit(e, slot, frames, n);
    if (rc) return rc;
    if (layout != H2J_LAYOUT_PLANAR && layout != H2J_LAYOUT_SEMIPLANAR) return fail(e, H2J_ERR_INVALID_ARG, "bad layout %d", layout);
    return H2J_OK;
}

// Caller frame i of a device submit -> its layout where it is (semi-planar: the pair plane at u_off = v_off) and the bytes
// from its base that may be read.  bps: bytes per sample (2: 16-bit words; the layout's pitches and offsets stay in bytes).
// within_max: the frame is encoded at this size, so it must fit the encoder.
int device_frame_layout(h2j_encoder *e, int i, const h2j_frame_desc &F, bool sp, int bps, bool within_max, FrameLayout *L, long long *extent)
{
    const int fmt = e->s.chroma_format;
    if (!F.data) return fail(e, H2J_ERR_INVALID_ARG, "frame %d: null data", i);
    int rc = make_layout(e, F.data, F.width, F.height, L, within_max);
    if (rc) return rc;
    const int fcw = chroma_w(F.width, fmt), fch = chroma_h(F.height, fmt);
    const int y_row = bps * F.width, c_row = bps * (sp ? 2 * fcw : fcw);  // bytes in a luma / chroma row
    if (F.y_pitch < y_row || F.c_pitch < c_row)
        return fail(e, H2J_ERR_INVALID_ARG, "frame %d: pitches %d / %d shorter than rows of %d / %d bytes", i, F.y_pitch, F.c_pitch, y_row, c_row);
    if (sp && F.u_offset < (size_t)F.y_pitch * F.height)
        return fail(e, H2J_ERR_INVALID_ARG, "frame %d: the pair plane starts inside the luma plane", i);
    L->y_pitch = F.y_pitch;
    L->c_pitch = F.c_pitch;
    L->u_off = (long long)F.u_offset;
    L->v_off = (long long)(sp ? F.u_offset : F.v_offset);
    set_alignment(L, F.data);
    *extent = (long long)std::max((size_t)F.y_pitch * (F.height - 1) + y_row,
                                  std::max((size_t)L->u_off, (size_t)L->v_off) + (size_t)F.c_pitch * (fch - 1) + c_row);
    return H2J_OK;
}

// A batch of frames of one layout F, frame i at F.data + i * frame_stride: checked as frame 0 of a device submit, with every
// plane inside frame_stride.  Then the slot's table is one pair that describes the frames, read in place.
int describe_batch(h2j_encoder *e, Slot &sl, const h2j_frame_desc &F, size_t frame_stride, bool sp, int bps)
{
    FrameDesc d;
    int rc = device_frame_layout(e, 0, F, sp, bps, true, &d.L, &d.extent);
    if (rc) return rc;
    if ((size_t)d.extent > frame_stride)
        return fail(e, H2J_ERR_INVALID_ARG, "a plane of the %dx%d frame reaches past frame_stride %zu", F.width, F.height, frame_stride);
    set_alignment(&d.L, F.data, frame_stride);  // the vector-load flags hold for every frame of the batch
    d.L.frame_stride = (long long)frame_stride;
    d.base = F.data;
    sl.h_desc[0] = sl.h_desc[1] = d;
    return H2J_OK;
}

// What a batch's sources are
struct Input {
    bool sp = false;    // semi-planar: the Cb/Cr pairs in one plane at u_off (= v_off)
    int bit_depth = 8;  // 9 .. 16: 16-bit words, converted to 8-bit planar frames
    int factor = 1;     // 2, 4, 8: box-filtered to 1/factor
    int rgb = -1;       // an h2j_rgb_format: RGB pixels, converted to YCbCr planar frames
    int filter = -1;    // an h2j_resize_filter: resized by the coefficient tables of the slot's arena (ResizeFrame)
};

// the rgb_to_planar_kernel instantiation for an h2j_rgb_format and a chroma format
template <int K>
decltype(&rgb_to_planar_kernel<1, kFmt420>) rgb_kernel_fmt(int fmt)
{
    return fmt == kFmt422 ? rgb_to_planar_kernel<K, kFmt422> : fmt == kFmt444 ? rgb_to_planar_kernel<K, kFmt444> : rgb_to_planar_kernel<K, kFmt420>;
}
decltype(&rgb_to_planar_kernel<1, kFmt420>) rgb_kernel(int rgb, int fmt)
{
    return rgb == H2J_RGB_PLANAR ? rgb_kernel_fmt<1>(fmt) : rgb >= H2J_RGB_RGBX ? rgb_kernel_fmt<4>(fmt) : rgb_kernel_fmt<3>(fmt);
}

// The input stage of every submit, then the pipeline, for n frames described by m entry pairs (m = n, or 1: see Slot).  On
// entry sl.h_desc[m + i] is the source of frame i where it lies, and sl.h_desc[i] the frame the pipeline encodes (at its
// size: a downscaled frame's is smaller), read in place.  A frame is read
// where it is unless it has to be copied:
//   - 16-bit, downscaled and RGB frames are converted (depth_to_8_kernel, downscale_list_kernel, rgb_to_planar_kernel);
//   - a semi-planar batch is read in place when every frame's rows start on 8-byte boundaries (K1 only looks at luma, K2's
//     chroma roles fetch the pairs and keep their component in registers); otherwise, or with semiplanar_prepass, all of it
//     is split into planes (nv12_to_i420_kernel);
//   - planar frames whose rows do not all start on 8-byte boundaries are copied to a 16-byte row pitch (repitch_kernel), when
//     the slot has room for the copies; otherwise the pipeline's bytewise path reads them where they are.
// Copies are planar at pitched_layout(), the repitched ones in d_pitched, the others in the slot's frame buffer; one kernel
// makes all of them.  A table of pairs is uploaded when that kernel or the list form of the pipeline reads it; a batch of one
// layout at one stride is one pair, which the kernel takes by value.
int run_batch(h2j_encoder *e, Slot &sl, int n, int m, const Input &in, int tail)
{
    FrameDesc *D = sl.h_desc, *S = sl.h_desc + m;
    const int fmt = e->s.chroma_format;
    const bool convert = in.bit_depth > 8 || in.factor > 1 || in.rgb >= 0 || in.filter >= 0;
    bool unaligned = false;
    for (int i = 0; i < m; i++) unaligned = unaligned || !S[i].L.aligned8;
    const bool split = in.sp && (unaligned || e->force_sp_prepass);
    const size_t pitched_cap = pitched_frame_bytes(e->s.max_width, e->s.max_height, fmt);
    if (e->planar_copy && !convert && !in.sp && unaligned && !sl.d_pitched && cudaMalloc(&sl.d_pitched, pitched_cap * e->s.max_batch) != cudaSuccess) {
        cudaGetLastError();  // no room for the copies: the bytewise path still works
        sl.d_pitched = nullptr;
    }
    uint8_t *const pitched = e->planar_copy ? sl.d_pitched : nullptr;
    // the largest copy: 16-byte columns of its widest row (semi-planar: of pairs), rows of all planes (RGB: 16-pixel columns,
    // destination rows a warp makes)
    int cols = 0, rows = 0;
    for (int i = 0; i < m; i++) {
        if (!convert && !split && (in.sp || S[i].L.aligned8 || !pitched)) {
            S[i].base = nullptr;
            D[i].L.nv12 = in.sp ? 1 : 0;
            continue;
        }
        const size_t spacing = convert || in.sp ? e->frame_bytes_cap : pitched_cap;
        D[i].L = pitched_layout(D[i].L);
        D[i].L.frame_stride = (long long)spacing;
        D[i].base = (convert || in.sp ? sl.d_frames : pitched) + (size_t)i * spacing;
        const int w = D[i].L.w, h = D[i].L.h;
        if (in.filter >= 0) {  // bands of output rows of every plane
            cols = std::max(cols, (w + kResizeCols - 1) / kResizeCols);
            rows = std::max(rows, (h + kResizeRows - 1) / kResizeRows + 2 * ((chroma_h(h, fmt) + kResizeRows - 1) / kResizeRows));
            continue;
        }
        if (in.rgb >= 0) {
            cols = std::max(cols, (w + 15) / 16);
            rows = std::max(rows, fmt == kFmt420 ? (h + 1) / 2 : h);
            continue;
        }
        cols = std::max(cols, (std::max(w, (in.sp ? 2 : 1) * chroma_w(w, fmt)) + 15) / 16);
        rows = std::max(rows, h + (in.sp ? 1 : 2) * chroma_h(h, fmt));
    }
    sl.n = n;
    sl.m = m;
    long long stride;
    if (m > 1 && (rows || !batch_stride(sl, &stride)))  // (a table of one pair goes to the copy kernel by value)
        CU(e, cudaMemcpyAsync(sl.d_desc, sl.h_desc, sizeof(FrameDesc) * (rows ? 2 * m : m), cudaMemcpyHostToDevice, sl.stream));
    if (in.filter >= 0) CU(e, cudaMemcpyAsync(sl.d_resize, sl.h_resize, sl.resize_used, cudaMemcpyHostToDevice, sl.stream));
    if (rows) {
        static_assert(32 * kDownWarps == 128, "every copy kernel runs CTAs of 128 threads");
        const bool warp_rows = in.factor > 1 || in.rgb >= 0;  // a warp per row, a lane per 16 bytes or pixels of it
        const int rows_per_cta = in.rgb >= 0 ? kDownWarps * kRgbRowsPerWarp : in.factor > 1 ? kDownWarps * 16 / in.factor : kPlaneRowsPerCta;
        const dim3 grid(warp_rows ? (cols + 31) / 32 : (cols + 127) / 128, (rows + rows_per_cta - 1) / rows_per_cta, n);
        decltype(&repitch_kernel) k = in.sp ? nv12_to_i420_kernel : repitch_kernel;
        if (in.factor == 2) k = in.sp ? downscale_list_kernel<2, true> : downscale_list_kernel<2, false>;
        else if (in.factor == 4) k = in.sp ? downscale_list_kernel<4, true> : downscale_list_kernel<4, false>;
        else if (in.factor == 8) k = in.sp ? downscale_list_kernel<8, true> : downscale_list_kernel<8, false>;
        const CopyTable t{sl.d_desc, m, D[0], S[0]};
        if (in.bit_depth > 8) (in.sp ? depth_to_8_kernel<true> : depth_to_8_kernel<false>)<<<grid, 128, 0, sl.stream>>>(t, in.bit_depth - 8);
        else if (in.filter >= 0)
            (in.sp ? resize_list_kernel<true> : resize_list_kernel<false>)<<<dim3(cols, rows, n), kResizeCols, 0, sl.stream>>>(
                t, reinterpret_cast<const ResizeFrame *>(sl.d_resize));
        else if (in.rgb >= 0)
            rgb_kernel(in.rgb, fmt)<<<grid, 128, 0, sl.stream>>>(t, in.rgb == H2J_RGB_BGR24 || in.rgb == H2J_RGB_BGRX ? 0x3012u : 0x3210u);
        else k<<<grid, 128, 0, sl.stream>>>(t);
        e->launches++;
        CU(e, cudaGetLastError());
    }
    int rc = launch_pipeline(e, sl, n, tail);
    if (rc) return rc;
    if (tail != TAIL_SINGLE) sl.busy = true;
    return H2J_OK;
}

// A device buffer and its pinned mirror of a slot (the converting single-picture calls' staging, the resize arena) hold at
// least `bytes` (grown if not): H2J_ERR_NOMEM, with none held, when they cannot be had.  The device buffer is asked for
// first, so a request larger than the device pins no host memory.
int reserve_mirrored(h2j_encoder *e, uint8_t *&d, uint8_t *&h, size_t &cap, size_t bytes, const char *what)
{
    if (bytes <= cap) return H2J_OK;
    cudaFree(d);
    if (h) cudaFreeHost(h);
    d = nullptr;
    h = nullptr;
    cap = 0;
    if (cudaMalloc(&d, bytes) != cudaSuccess || cudaHostAlloc(&h, bytes, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(d);
        d = nullptr;
        h = nullptr;
        return fail(e, H2J_ERR_NOMEM, "no room for the %zu-byte %s", bytes, what);
    }
    cap = bytes;
    return H2J_OK;
}
int reserve_convert(h2j_encoder *e, Slot &sl, size_t bytes)
{
    return reserve_mirrored(e, sl.d_convert, sl.h_convert, sl.convert_bytes, bytes, "staging of a picture to convert");
}

// bytes of a row of w pixels of an h2j_rgb_format (planar: of each plane); 0 for a bad format
int rgb_row_bytes(int format, int w)
{
    switch (format) {
    case H2J_RGB_RGB24: case H2J_RGB_BGR24: return 3 * w;
    case H2J_RGB_RGBX: case H2J_RGB_BGRX: return 4 * w;
    case H2J_RGB_PLANAR: return w;
    default: return 0;
    }
}

// Caller RGB frame i (h2j_submit_device_rgb) -> tab[i], the planar frame the pipeline encodes (range_mode 0: the YCbCr of
// an RGB frame is full range by construction), and tab[n + i], the frame where it is (rows y_pitch apart, planar G and B
// planes at u_off / v_off, extent: the bytes from its base that may be read)
int rgb_frame_layout(h2j_encoder *e, int i, int n, int format, const h2j_frame_desc &F, FrameDesc *tab)
{
    if (!F.data) return fail(e, H2J_ERR_INVALID_ARG, "frame %d: null data", i);
    FrameDesc &d = tab[i], &s = tab[n + i];
    int rc = make_layout(e, nullptr, F.width, F.height, &d.L);
    if (rc) return rc;
    d.L.range_mode = 0;
    const int row = rgb_row_bytes(format, F.width);
    if (F.y_pitch < row) return fail(e, H2J_ERR_INVALID_ARG, "frame %d: pitch %d shorter than a row of %d bytes", i, F.y_pitch, row);
    const size_t plane = (size_t)F.y_pitch * F.height;
    const bool planar = format == H2J_RGB_PLANAR;
    if (planar && (F.u_offset < plane || F.v_offset < plane))
        return fail(e, H2J_ERR_INVALID_ARG, "frame %d: the G or B plane starts inside the R plane", i);
    s = d;
    s.L.y_pitch = s.L.c_pitch = F.y_pitch;
    s.L.u_off = planar ? (long long)F.u_offset : 0;
    s.L.v_off = planar ? (long long)F.v_offset : 0;
    s.base = F.data;
    s.extent = (long long)((planar ? std::max(F.u_offset, F.v_offset) : 0) + (size_t)F.y_pitch * (F.height - 1) + row);
    return H2J_OK;
}

// ---- h2j_submit_device_resized: Pillow's coefficients (libImaging/Resample.c precompute_coeffs, normalize_coeffs_8bpc) ----
// Built on the host in double, with Pillow's operations in Pillow's order.  This file's host code is compiled by g++ without
// -march, which emits no FMA on x86-64: a contracted multiply-add (as nvcc makes of device code) would change the weights.
double resize_filter(int filter, double x)
{
    if (filter == H2J_FILTER_BOX) return x > -0.5 && x <= 0.5 ? 1.0 : 0.0;
    if (x < 0.0) x = -x;
    if (filter == H2J_FILTER_BILINEAR) return x < 1.0 ? 1.0 - x : 0.0;
    const double a = -0.5;
    if (x < 1.0) return ((a + 2.0) * x - (a + 3.0)) * x * x + 1;
    if (x < 2.0) return (((x - 5) * x + 8) * x - 4) * a;
    return 0.0;
}

// One axis, in to out samples: win[o] = {first source sample, taps, first coefficient in coef} for every output o, and the
// taps' coefficients in 22-bit fixed point.  in == out: the identity (Pillow skips the pass; one tap of 1 << 22 gives the
// sample back).  win null: only counts.  Returns the number of coefficients.
long long resize_axis(int filter, int in, int out, int4 *win, int *coef)
{
    const double scale = (double)in / out;
    const double fs = scale < 1.0 ? 1.0 : scale;
    const double support = (filter == H2J_FILTER_BOX ? 0.5 : filter == H2J_FILTER_BILINEAR ? 1.0 : 2.0) * fs;
    std::vector<double> w;
    long long k = 0;
    for (int o = 0; o < out; o++) {
        if (in == out) {
            if (win) {
                win[o] = make_int4(o, 1, o, 0);
                coef[o] = 1 << kResizeBits;
            }
            k++;
            continue;
        }
        const double center = (o + 0.5) * scale;
        const double ss = 1.0 / fs;
        int xmin = (int)(center - support + 0.5);
        if (xmin < 0) xmin = 0;
        int xmax = (int)(center + support + 0.5);
        if (xmax > in) xmax = in;
        const int n = xmax - xmin;
        if (win) {
            w.resize(n);
            double ww = 0.0;
            for (int x = 0; x < n; x++) {
                w[x] = resize_filter(filter, (x + xmin - center + 0.5) * ss);
                ww += w[x];
            }
            for (int x = 0; x < n; x++) {
                if (ww != 0.0) w[x] /= ww;
                coef[k + x] = w[x] < 0 ? (int)(-0.5 + w[x] * (1 << kResizeBits)) : (int)(0.5 + w[x] * (1 << kResizeBits));
            }
            win[o] = make_int4(xmin, n, (int)k, 0);
        }
        k += n;
    }
    return k;
}

// The arena of a resized batch: a ResizeFrame per frame, then per distinct (in, out) axis its windows, then its
// coefficients.  axes[f * 4 + a] is frame f's axis a (luma x, luma y, chroma x, chroma y) as {in, out}.
struct ResizeAxis {
    int in, out;
    size_t win_off, coef_off;  // bytes into the arena
};
int build_resize_arena(h2j_encoder *e, Slot &sl, int n, int filter, const std::vector<std::pair<int, int>> &axes)
{
    std::vector<ResizeAxis> uniq;
    std::vector<int> which(axes.size());
    std::map<std::pair<int, int>, int> seen;
    size_t bytes = align_up(sizeof(ResizeFrame) * n, 16);
    for (size_t a = 0; a < axes.size(); a++) {
        auto it = seen.find(axes[a]);
        if (it == seen.end()) {
            it = seen.emplace(axes[a], (int)uniq.size()).first;
            uniq.push_back(ResizeAxis{axes[a].first, axes[a].second, 0, 0});
        }
        which[a] = it->second;
    }
    for (ResizeAxis &x : uniq) {
        x.win_off = bytes;
        x.coef_off = bytes + sizeof(int4) * x.out;
        bytes = align_up(x.coef_off + sizeof(int) * resize_axis(filter, x.in, x.out, nullptr, nullptr), 16);
    }
    int rc = reserve_mirrored(e, sl.d_resize, sl.h_resize, sl.resize_bytes, bytes, "coefficient tables of a resized batch");
    if (rc) return rc;
    sl.resize_used = bytes;
    for (const ResizeAxis &x : uniq)
        resize_axis(filter, x.in, x.out, reinterpret_cast<int4 *>(sl.h_resize + x.win_off), reinterpret_cast<int *>(sl.h_resize + x.coef_off));
    ResizeFrame *rf = reinterpret_cast<ResizeFrame *>(sl.h_resize);
    for (int f = 0; f < n; f++)
        for (int a = 0; a < 4; a++) {
            const ResizeAxis &x = uniq[which[(size_t)f * 4 + a]];
            rf[f].win[a] = reinterpret_cast<const int4 *>(sl.d_resize + x.win_off);
            rf[f].coef[a] = reinterpret_cast<const int *>(sl.d_resize + x.coef_off);
        }
    return H2J_OK;
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
    if (s->comment && strlen(s->comment) > kMaxCommentBytes)
        return fail(nullptr, H2J_ERR_INVALID_ARG, "comment of %zu bytes: at most %zu fit a COM segment", strlen(s->comment), kMaxCommentBytes);
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
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt420, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt420)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt422, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt422)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt444, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt444)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt420, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt420)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt422, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt422)));
    CUB(cudaFuncSetAttribute(entropy_walk_kernel<kFmt444, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ent_smem_bytes(kFmt444)));

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
        CUB(cudaMalloc(&sl.d_desc, sizeof(FrameDesc) * 2 * B));
        CUB(cudaHostAlloc(&sl.h_desc, sizeof(FrameDesc) * 2 * B, cudaHostAllocDefault));
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
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    rc = describe_batch(e, sl, tight_frame(d_frames, width, height, e->s.chroma_format), frame_stride, false, 1);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, 1, Input{}, TAIL_SIZES);
}

int h2j_submit_device_semiplanar(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch, size_t uv_offset,
                                 int n, int width, int height)
{
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    rc = describe_batch(e, sl, h2j_frame_desc{d_frames, width, height, pitch, pitch, uv_offset, uv_offset}, frame_stride, true, 1);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, 1, Input{true}, TAIL_SIZES);
}

int h2j_submit_device_nv12(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch, size_t uv_offset, int n,
                           int width, int height)
{
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    if (e->s.chroma_format != H2J_CHROMA_420) return fail(e, H2J_ERR_UNSUPPORTED, "NV12 is a 4:2:0 layout; this encoder was created for another chroma format");
    return h2j_submit_device_semiplanar(e, slot, d_frames, frame_stride, pitch, uv_offset, n, width, height);
}

int h2j_submit_device_pitched(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int y_pitch, int c_pitch,
                              size_t u_offset, size_t v_offset, int n, int width, int height)
{
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    rc = describe_batch(e, sl, h2j_frame_desc{d_frames, width, height, y_pitch, c_pitch, u_offset, v_offset}, frame_stride, false, 1);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, 1, Input{}, TAIL_SIZES);
}

int h2j_submit_device_semiplanar16(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch, size_t uv_offset,
                                   int bit_depth, int n, int width, int height)
{
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    if (bit_depth < 9 || bit_depth > 16) return fail(e, H2J_ERR_INVALID_ARG, "bit_depth %d outside 9..16", bit_depth);
    if (odd((uintptr_t)d_frames) || odd(frame_stride) || odd((size_t)pitch) || odd(uv_offset))
        return fail(e, H2J_ERR_INVALID_ARG, "16-bit samples need even pointers, strides, pitches and offsets");
    Slot &sl = e->slots[slot];
    rc = describe_batch(e, sl, h2j_frame_desc{d_frames, width, height, pitch, pitch, uv_offset, uv_offset}, frame_stride, true, 2);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, 1, Input{true, bit_depth}, TAIL_SIZES);
}

int h2j_submit_device_pitched16(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int y_pitch, int c_pitch,
                                size_t u_offset, size_t v_offset, int bit_depth, int n, int width, int height)
{
    int rc = check_submit(e, slot, d_frames, n);
    if (rc) return rc;
    if (bit_depth < 9 || bit_depth > 16) return fail(e, H2J_ERR_INVALID_ARG, "bit_depth %d outside 9..16", bit_depth);
    if (odd((uintptr_t)d_frames) || odd(frame_stride) || odd((size_t)y_pitch) || odd((size_t)c_pitch) || odd(u_offset) || odd(v_offset))
        return fail(e, H2J_ERR_INVALID_ARG, "16-bit samples need even pointers, strides, pitches and offsets");
    Slot &sl = e->slots[slot];
    rc = describe_batch(e, sl, h2j_frame_desc{d_frames, width, height, y_pitch, c_pitch, u_offset, v_offset}, frame_stride, false, 2);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, 1, Input{false, bit_depth}, TAIL_SIZES);
}

int h2j_submit_host(h2j_encoder *e, int slot, const uint8_t *frames, size_t frame_stride, int n, int width, int height)
{
    int rc = check_submit(e, slot, frames, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    const size_t fb = tight_frame_bytes(width, height, e->s.chroma_format);
    if (frame_stride < fb) return fail(e, H2J_ERR_INVALID_ARG, "frame_stride smaller than one frame");
    // device copy keeps frames at a 256-byte aligned stride so the vector-load paths apply
    const size_t dstride = align_up(fb, 256);
    if (dstride > e->frame_bytes_cap) return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d exceeds the configured maximum", width, height);
    rc = describe_batch(e, sl, tight_frame(sl.d_frames, width, height, e->s.chroma_format), dstride, false, 1);
    if (rc) return rc;
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    if (frame_stride == dstride) CU(e, cudaMemcpyAsync(sl.d_frames, frames, dstride * (n - 1) + fb, cudaMemcpyHostToDevice, sl.stream));
    else CU(e, cudaMemcpy2DAsync(sl.d_frames, dstride, frames, frame_stride, fb, n, cudaMemcpyHostToDevice, sl.stream));
    return run_batch(e, sl, n, 1, Input{}, TAIL_PACK);
}

int h2j_submit_device_list(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n)
{
    int rc = check_device_list(e, slot, layout, frames, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    const bool sp = layout == H2J_LAYOUT_SEMIPLANAR;
    std::vector<FrameDesc> tab(n);  // (every frame is checked before the slot's table is touched)
    for (int i = 0; i < n; i++) {
        rc = device_frame_layout(e, i, frames[i], sp, 1, true, &tab[i].L, &tab[i].extent);
        if (rc) return rc;
        tab[i].base = frames[i].data;
    }
    for (int i = 0; i < n; i++) sl.h_desc[i] = sl.h_desc[n + i] = tab[i];
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, n, Input{sp}, TAIL_SIZES);
}

int h2j_submit_device_downscaled(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n, int factor)
{
    int rc = check_device_list(e, slot, layout, frames, n);
    if (rc) return rc;
    if (factor != 2 && factor != 4 && factor != 8) return fail(e, H2J_ERR_INVALID_ARG, "factor %d is not 2, 4 or 8", factor);
    Slot &sl = e->slots[slot];
    const bool sp = layout == H2J_LAYOUT_SEMIPLANAR;
    // tab[i]: the downscaled frame the pipeline encodes, tab[n + i]: the caller's frame.  Only the downscaled size is held to
    // the encoder's maximum.
    std::vector<FrameDesc> tab(2 * (size_t)n);
    for (int i = 0; i < n; i++) {
        const h2j_frame_desc &F = frames[i];
        FrameDesc &src = tab[n + i];
        rc = device_frame_layout(e, i, F, sp, 1, false, &src.L, &src.extent);
        if (rc) return rc;
        src.base = F.data;
        const int w = (F.width + factor - 1) / factor, h = (F.height + factor - 1) / factor;
        if (w < 2 || h < 2)
            return fail(e, H2J_ERR_UNSUPPORTED, "frame %d: %dx%d at 1/%d is %dx%d, smaller than 2x2", i, F.width, F.height, factor, w, h);
        rc = make_layout(e, nullptr, w, h, &tab[i].L);
        if (rc) return rc;
    }
    memcpy(sl.h_desc, tab.data(), sizeof(FrameDesc) * 2 * n);
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    return run_batch(e, sl, n, n, Input{sp, 8, factor}, TAIL_SIZES);
}

int h2j_submit_device_resized(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n, const int *out_widths,
                              const int *out_heights, int filter)
{
    int rc = check_device_list(e, slot, layout, frames, n);
    if (rc) return rc;
    if (!out_widths || !out_heights) return fail(e, H2J_ERR_INVALID_ARG, "null out_widths / out_heights");
    if (filter != H2J_FILTER_BOX && filter != H2J_FILTER_BILINEAR && filter != H2J_FILTER_BICUBIC)
        return fail(e, H2J_ERR_INVALID_ARG, "bad resize filter %d", filter);
    Slot &sl = e->slots[slot];
    const bool sp = layout == H2J_LAYOUT_SEMIPLANAR;
    const int fmt = e->s.chroma_format;
    // tab[i]: the resized frame the pipeline encodes, tab[n + i]: the caller's frame.  Only the output size is held to the
    // encoder's maximum.
    std::vector<FrameDesc> tab(2 * (size_t)n);
    std::vector<std::pair<int, int>> axes(4 * (size_t)n);
    for (int i = 0; i < n; i++) {
        const h2j_frame_desc &F = frames[i];
        FrameDesc &src = tab[n + i];
        rc = device_frame_layout(e, i, F, sp, 1, false, &src.L, &src.extent);
        if (rc) return rc;
        src.base = F.data;
        const int w = out_widths[i], h = out_heights[i];
        rc = make_layout(e, nullptr, w, h, &tab[i].L);
        if (rc) return rc;
        axes[4 * i] = {F.width, w};
        axes[4 * i + 1] = {F.height, h};
        axes[4 * i + 2] = {chroma_w(F.width, fmt), chroma_w(w, fmt)};
        axes[4 * i + 3] = {chroma_h(F.height, fmt), chroma_h(h, fmt)};
    }
    ON_DEVICE(e);
    rc = build_resize_arena(e, sl, n, filter, axes);
    if (rc) return rc;
    memcpy(sl.h_desc, tab.data(), sizeof(FrameDesc) * 2 * n);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    Input in;
    in.sp = sp;
    in.filter = filter;
    return run_batch(e, sl, n, n, in, TAIL_SIZES);
}

int h2j_submit_device_rgb(h2j_encoder *e, int slot, int format, const h2j_frame_desc *frames, int n)
{
    int rc = check_submit(e, slot, frames, n);
    if (rc) return rc;
    if (!rgb_row_bytes(format, 2)) return fail(e, H2J_ERR_INVALID_ARG, "bad RGB format %d", format);
    Slot &sl = e->slots[slot];
    std::vector<FrameDesc> tab(2 * (size_t)n);  // (every frame is checked before the slot's table is touched)
    for (int i = 0; i < n; i++) {
        rc = rgb_frame_layout(e, i, n, format, frames[i], tab.data());
        if (rc) return rc;
    }
    memcpy(sl.h_desc, tab.data(), sizeof(FrameDesc) * 2 * n);
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    Input in;
    in.rgb = format;
    return run_batch(e, sl, n, n, in, TAIL_SIZES);
}

int h2j_submit_host_list(h2j_encoder *e, int slot, const uint8_t *const *frames, const int *widths, const int *heights, int n)
{
    int rc = check_submit(e, slot, widths && heights ? frames : nullptr, n);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    const int fmt = e->s.chroma_format;
    std::vector<FrameDesc> tab(n);  // (every frame is checked before the slot's table is touched)
    for (int i = 0; i < n; i++) {
        if (!frames[i]) return fail(e, H2J_ERR_INVALID_ARG, "frame %d: null pointer", i);
        // frame i goes to its own place of the slot's frame buffer, sized for a tight frame at the maximum geometry
        uint8_t *dev = sl.d_frames + (size_t)i * e->frame_bytes_cap;
        rc = make_layout(e, dev, widths[i], heights[i], &tab[i].L);
        if (rc) return rc;
        tab[i].base = dev;
        tab[i].extent = (long long)tight_frame_bytes(widths[i], heights[i], fmt);
    }
    for (int i = 0; i < n; i++) sl.h_desc[i] = sl.h_desc[n + i] = tab[i];
    ON_DEVICE(e);
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    for (int i = 0; i < n; i++)
        CU(e, cudaMemcpyAsync(sl.d_frames + (size_t)i * e->frame_bytes_cap, frames[i], tight_frame_bytes(widths[i], heights[i], fmt),
                              cudaMemcpyHostToDevice, sl.stream));
    return run_batch(e, sl, n, n, Input{}, TAIL_PACK);
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
    FrameLayout L;
    int rc = make_layout(e, sl.d_frames, width, height, &L);
    if (rc) return rc;
    // rows that would not start on 8-byte boundaries (odd widths) are staged at a 16-byte pitch right here: the rows are
    // copied one by one anyway, and the kernels keep their vector loads without a second pass over the frame
    if (!L.aligned8) L = pitched_layout(L);
    sl.h_desc[0] = sl.h_desc[1] = FrameDesc{L, sl.d_frames, 0};
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    {
        const int row_bytes[3] = {width, fcw, fcw}, rows[3] = {height, fch, fch}, pitch[3] = {L.y_pitch, L.c_pitch, L.c_pitch};
        const size_t off[3] = {0, (size_t)L.u_off, (size_t)L.v_off};
        rc = upload_planes(e, sl, planes, strides, row_bytes, rows, off, pitch, sl.d_frames, sl.h_stage);
        if (rc) return rc;
    }
    rc = run_batch(e, sl, 1, 1, Input{}, TAIL_SINGLE);
    if (rc) return rc;
    return finish_single(e, sl, out, out_capacity, out_size);
}

int h2j_encode_frame16(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int bit_depth, int width, int height,
                       uint8_t *out, size_t out_capacity, size_t *out_size)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    if (!planes || !strides || !planes[0] || !planes[1] || !planes[2] || !out || !out_size)
        return fail(e, H2J_ERR_INVALID_ARG, "null plane/out pointer");
    if (bit_depth < 9 || bit_depth > 16) return fail(e, H2J_ERR_INVALID_ARG, "bit_depth %d outside 9..16", bit_depth);
    if (width < 2 || height < 2 || width > e->s.max_width || height > e->s.max_height)
        return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d outside 2x2 .. %dx%d", width, height, e->s.max_width, e->s.max_height);
    Slot &sl = e->slots[0];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot 0 has a batch in flight");
    const int fmt = e->s.chroma_format;
    const int fcw = chroma_w(width, fmt), fch = chroma_h(height, fmt);
    for (int p = 0; p < 3; p++)
        if (odd((uintptr_t)planes[p]) || odd((size_t)strides[p])) return fail(e, H2J_ERR_INVALID_ARG, "plane %d: odd pointer or stride", p);
    if (strides[0] < 2 * width || strides[1] < 2 * fcw || strides[2] < 2 * fcw) return fail(e, H2J_ERR_INVALID_ARG, "stride smaller than the row");
    ON_DEVICE(e);
    // the 16-bit planes go to the device at 16-byte aligned row pitches, so that the conversion reads them with vector loads
    const int yp = (int)align_up((size_t)2 * width, 16), cp = (int)align_up((size_t)2 * fcw, 16);
    {
        const int mcw = chroma_w(e->s.max_width, fmt), mch = chroma_h(e->s.max_height, fmt);
        const int rc = reserve_convert(e, sl, align_up((size_t)2 * e->s.max_width, 16) * e->s.max_height + 2 * align_up((size_t)2 * mcw, 16) * mch);
        if (rc) return rc;
    }
    // a batch of one frame: the planes as staged on the device, converted by the input stage
    const h2j_frame_desc F{sl.d_convert, width, height, yp, cp, (size_t)yp * height, (size_t)yp * height + (size_t)cp * fch};
    int rc = describe_batch(e, sl, F, (size_t)yp * height + 2 * (size_t)cp * fch, false, 2);
    if (rc) return rc;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    const int row_bytes[3] = {2 * width, 2 * fcw, 2 * fcw}, rows[3] = {height, fch, fch}, pitch[3] = {yp, cp, cp};
    const size_t off[3] = {0, F.u_offset, F.v_offset};
    rc = upload_planes(e, sl, planes, strides, row_bytes, rows, off, pitch, sl.d_convert, sl.h_convert);
    if (rc) return rc;
    rc = run_batch(e, sl, 1, 1, Input{false, bit_depth}, TAIL_SINGLE);
    if (rc) return rc;
    return finish_single(e, sl, out, out_capacity, out_size);
}

int h2j_encode_frame_rgb(h2j_encoder *e, int format, const uint8_t *const planes[3], const int strides[3], int width, int height,
                         uint8_t *out, size_t out_capacity, size_t *out_size)
{
    if (!e) return H2J_ERR_INVALID_ARG;
    const bool planar = format == H2J_RGB_PLANAR;
    if (!planes || !strides || !planes[0] || (planar && (!planes[1] || !planes[2])) || !out || !out_size)
        return fail(e, H2J_ERR_INVALID_ARG, "null plane/out pointer");
    const int row = rgb_row_bytes(format, width);
    if (!row) return fail(e, H2J_ERR_INVALID_ARG, "bad RGB format %d", format);
    if (width < 2 || height < 2 || width > e->s.max_width || height > e->s.max_height)
        return fail(e, H2J_ERR_UNSUPPORTED, "frame %dx%d outside 2x2 .. %dx%d", width, height, e->s.max_width, e->s.max_height);
    Slot &sl = e->slots[0];
    if (sl.busy) return fail(e, H2J_ERR_BUSY, "slot 0 has a batch in flight");
    for (int p = 0; p < (planar ? 3 : 1); p++)
        if (strides[p] < row) return fail(e, H2J_ERR_INVALID_ARG, "stride %d of plane %d smaller than a row of %d bytes", strides[p], p, row);
    ON_DEVICE(e);
    // the picture goes to the device at a 16-byte aligned row pitch, so that the conversion reads it with vector loads
    const int pitch = (int)align_up((size_t)row, 16);
    {
        const size_t max_pitch = align_up((size_t)rgb_row_bytes(format, e->s.max_width), 16);
        const int rc = reserve_convert(e, sl, max_pitch * e->s.max_height * (planar ? 3 : 1));
        if (rc) return rc;
    }
    // a batch of one frame: the picture as staged on the device, converted by the input stage
    const size_t plane = (size_t)pitch * height;
    const h2j_frame_desc F{sl.d_convert, width, height, pitch, pitch, planar ? plane : 0, planar ? 2 * plane : 0};
    int rc = rgb_frame_layout(e, 0, 1, format, F, sl.h_desc);
    if (rc) return rc;
    CU(e, cudaEventRecord(sl.ev_begin, sl.stream));
    const int row_bytes[3] = {row, row, row}, rows[3] = {height, height, height}, pitches[3] = {pitch, pitch, pitch};
    const size_t off[3] = {0, plane, 2 * plane};
    rc = upload_planes(e, sl, planes, strides, row_bytes, rows, off, pitches, sl.d_convert, sl.h_convert, planar ? 3 : 1);
    if (rc) return rc;
    Input in;
    in.rgb = format;
    rc = run_batch(e, sl, 1, 1, in, TAIL_SINGLE);
    if (rc) return rc;
    return finish_single(e, sl, out, out_capacity, out_size);
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
    int rc = make_layout(e, sl.d_frames, width, height, &L);
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
    const FrameLayout &L = frame_desc(sl, frame).L;
    info->mcu_w = L.mcu_w;
    info->mcu_h = L.mcu_h;
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
    const FrameLayout &L = frame_desc(sl, frame).L;
    const size_t need = (size_t)L.n_blocks * 64;
    if (out_elems < need) return fail(e, H2J_ERR_OUTPUT_TOO_SMALL, "need %zu int16 elements", need);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    // tile images -> dense blocks; halfword 0 of a record is the DC difference, so the levels are rebuilt by
    // running the encoder's predictors (one per component, reset to 128) over the blocks in coding order
    const int fmt = L.fmt, tile_blocks = fmt_tile_blocks(fmt), tile_words = fmt_tile_image_words(fmt);
    const int n_tiles = (L.n_mcu + kTileMcus - 1) / kTileMcus;
    std::vector<int16_t> img((size_t)n_tiles * tile_words * 2);
    CU(e, cudaMemcpy(img.data(), sl.d_images + (size_t)frame * e->images_cap * tile_words, img.size() * sizeof(int16_t),
                     cudaMemcpyDeviceToHost));
    int last_dc[3] = {128, 128, 128};
    for (int b = 0; b < L.n_blocks; b++) {
        const TileRec tr = tile_rec_fmt(fmt, b % tile_blocks);
        const int16_t *rec = img.data() + ((size_t)(b / tile_blocks) * tile_words + (size_t)tr.sub * kSubImageWords + (size_t)tr.idx * kBlkWords) * 2;
        const int comp = block_component(fmt, b % fmt_mcu_blocks(fmt));
        last_dc[comp] += rec[0];
        out[(size_t)b * 64] = (int16_t)last_dc[comp];
        for (int k = 1; k < 64; k++) out[(size_t)b * 64 + k] = rec[2 * (k & 31) + (k >> 5)];
    }
    return H2J_OK;
}

int h2j_debug_frame_planes(h2j_encoder *e, int slot, int frame, uint8_t *y, uint8_t *u, uint8_t *v)
{
    int rc = check_slot(e, slot);
    if (rc) return rc;
    Slot &sl = e->slots[slot];
    if (!y || !u || !v || frame < 0 || frame >= sl.n) return fail(e, H2J_ERR_INVALID_ARG, "null plane or bad frame index %d", frame);
    FrameDesc d = frame_desc(sl, frame);
    if (sl.m == 1) d.base += (long long)frame * d.L.frame_stride;  // a batch of one layout at one stride
    const FrameLayout &L = d.L;
    const int cw = chroma_w(L.w, L.fmt), ch = chroma_h(L.h, L.fmt);
    ON_DEVICE(e);
    CU(e, cudaStreamSynchronize(sl.stream));
    CU(e, cudaMemcpy2D(y, L.w, d.base, L.y_pitch, L.w, L.h, cudaMemcpyDeviceToHost));
    if (!L.nv12) {
        CU(e, cudaMemcpy2D(u, cw, d.base + L.u_off, L.c_pitch, cw, ch, cudaMemcpyDeviceToHost));
        CU(e, cudaMemcpy2D(v, cw, d.base + L.v_off, L.c_pitch, cw, ch, cudaMemcpyDeviceToHost));
        return H2J_OK;
    }
    // semi-planar, read in place: the rows of pairs, split here
    std::vector<uint8_t> pairs((size_t)2 * cw * ch);
    CU(e, cudaMemcpy2D(pairs.data(), 2 * cw, d.base + L.u_off, L.c_pitch, 2 * cw, ch, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < (size_t)cw * ch; i++) {
        u[i] = pairs[2 * i];
        v[i] = pairs[2 * i + 1];
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
    if (!strcmp(name, "planar_copy")) {
        if (value < 0 || value > 1) return fail(e, H2J_ERR_INVALID_ARG, "planar_copy %d is not 0 or 1", value);
        e->planar_copy = value;
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
