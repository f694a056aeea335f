/*
 * h2j_b200 — B200-native (sm_100a) JPEG encoder for the YUV -> JPEG stage of
 * BornToDeath/h264-h265-to-jpeg, behind a plain C ABI.
 *
 * What it replaces in the reference (file:line in /root/reference):
 *   src/Encoder.cpp:104-308  Encoder::yuv2Jpeg(AVFrame*)  — avcodec "mjpeg" encoder opened with
 *                            pix_fmt YUVJ420P (:162), time_base 1/25 (:201), defaults otherwise,
 *                            avcodec_send_frame (:250) / avcodec_receive_packet (:259), raw "mjpeg" muxer
 *                            write (:278), bytes gathered through writeCallback (:27) into a 2 MiB buffer
 *                            (src/Common.h:16 HEAP_SIZE) and saved with saveJpegtoFile (:338).
 *   src/Decoder.cpp:349      the only call site: Encoder(outputFilePath).yuv2Jpeg(frame).
 * Everything in front of it (src/Decoder.cpp libavformat/libavcodec H.264/H.265 decode) and the public
 * surface (export_inc/IDecoder.h, src/jni/...) stay the reference's own code.
 *
 * The bytes produced are identical to what the reference writes for the same decoded planes: same
 * quantised coefficients, same optimal Huffman tables, same header, same stuffing (see DESIGN.md).
 *
 * All entry points return 0 (H2J_OK) or a negative h2j_status.  No CPU fallback exists: if no CUDA
 * device is usable h2j_create fails with H2J_ERR_CUDA.
 *
 * Threading: an h2j_encoder is not internally synchronised.  Use it from one thread at a time (or one encoder
 * per thread); different encoders are independent.  Work of different slots of one encoder overlaps on the GPU.
 * Every entry point selects the encoder's device for the duration of the call and restores the caller's current device.
 */
#ifndef H2J_B200_H
#define H2J_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define H2J_ABI_VERSION 3

typedef enum h2j_status {
    H2J_OK = 0,
    H2J_ERR_INVALID_ARG = -1,     /* null pointer, non-positive size, batch larger than configured ... */
    H2J_ERR_CUDA = -2,            /* a CUDA runtime call failed; see h2j_last_error() */
    H2J_ERR_UNSUPPORTED = -3,     /* geometry outside max_width/max_height, width or height < 2 or > 65500 */
    H2J_ERR_OUTPUT_TOO_SMALL = -4,/* a JPEG did not fit max_jpeg_bytes / the caller's buffer */
    H2J_ERR_BUSY = -5,            /* slot already has a batch in flight, or nothing to collect */
    H2J_ERR_NOMEM = -6,
    H2J_ERR_BUFFER_TOO_SMALL = -7 /* h2j_collect: the CALLER's buffer is shorter than the batch; offsets[] holds the
                                     sizes, the slot stays collectable -- call again with a larger buffer */
} h2j_status;

/* How the planes are interpreted before encoding. */
typedef enum h2j_range_mode {
    /* Planes go to the encoder as they are.  This is what reference src/Encoder.cpp does: it never calls
     * sws_scale; a yuv420p AVFrame is handed to an encoder opened as yuvj420p (Encoder.cpp:162, :250). */
    H2J_RANGE_PASSTHROUGH = 0,
    /* yuv420p (limited) -> yuvj420p (full) first, bit-exact with libswscale 5.8.100's unscaled
     * lumRangeToJpeg/chrRangeToJpeg path (what a sws_scale call in front of the encoder would produce). */
    H2J_RANGE_LIMITED_TO_FULL = 1
} h2j_range_mode;

/* Chroma format of the frames an encoder takes.  The reference opens libavcodec's mjpeg encoder as yuvj420p and nothing
 * else (src/Encoder.cpp:162): H2J_CHROMA_420 is the drop-in.  The other two are the same encoder at its other MCU
 * geometries (yuvj422p: 16x16 MCUs of 4 Y + 2 Cb + 2 Cr blocks; yuvj444p: 8x16 MCUs of 2 Y + 2 Cb + 2 Cr), byte-identical
 * to what that libavcodec writes for planar 4:2:2 / 4:4:4 frames. */
typedef enum h2j_chroma_format {
    H2J_CHROMA_420 = 0, /* planes: Y w x h, U and V ceil(w/2) x ceil(h/2) */
    H2J_CHROMA_422 = 1, /* U and V ceil(w/2) x h */
    H2J_CHROMA_444 = 2  /* U and V w x h */
} h2j_chroma_format;

typedef struct h2j_settings {
    int device;            /* CUDA device ordinal */
    int max_width;         /* largest frame the encoder will be asked for */
    int max_height;
    int max_batch;         /* frames per submitted batch (>= 1) */
    int n_slots;           /* batches that may be in flight at once, each on its own stream (1..8) */
    int range_mode;        /* h2j_range_mode */
    int fixed_qscale;      /* 0: the reference's first-frame rate control decides (default);
                              1..31: force it (AV_CODEC_FLAG_QSCALE equivalent; not used by the reference) */
    size_t max_jpeg_bytes; /* largest JPEG a frame may have, exactly (a larger one fails with H2J_ERR_OUTPUT_TOO_SMALL);
                              0 = 2 MiB, the reference's HEAP_SIZE; at most 256 MiB */
    const char *comment;   /* COM segment payload; NULL = "Lavc58.117.101", the LIBAVCODEC_IDENT of the
                              ffmpeg build the reference links on x86-64 (lib/ffmpeg/x86_64_shared) */
    int profile;           /* non-zero: bracket every kernel with CUDA events (see h2j_slot_kernel_ms) */
    int chroma_format;     /* h2j_chroma_format of every frame this encoder is given (default H2J_CHROMA_420) */
} h2j_settings;

typedef struct h2j_encoder h2j_encoder;

/* Fill a settings struct with defaults (1080p, batch 16, 2 slots, reference behaviour). */
void h2j_default_settings(h2j_settings *s);

int h2j_create(const h2j_settings *s, h2j_encoder **out);
void h2j_destroy(h2j_encoder *e);
const char *h2j_last_error(const h2j_encoder *e); /* e may be NULL: error of the last failed h2j_create */
const char *h2j_status_string(int status);
int h2j_abi_version(void);
/* CUDA devices this process can use (0 when there is none or the driver cannot be initialised). */
int h2j_device_count(void);

/*
 * One frame, host planes in, JPEG bytes out, synchronous — the drop-in for
 * Encoder::yuv2Jpeg() (reference src/Encoder.cpp:104).  planes/strides follow AVFrame.data/.linesize for
 * an 8-bit 4:2:0 planar frame: plane 0 is width x height, planes 1/2 are ceil(width/2) x ceil(height/2) (for an encoder
 * created with another chroma_format: ceil(width/2) x height at 4:2:2, width x height at 4:4:4).
 * Uses slot 0; the planes are staged through pinned memory and copied asynchronously.  Planes that are page-locked already
 * (allocated with h2j_alloc_pinned / cudaHostAlloc or registered with cudaHostRegister) are uploaded from where they are,
 * without the staging copy (which is most of the call's time for pageable planes).
 */
int h2j_encode_frame(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int width, int height,
                     uint8_t *out, size_t out_capacity, size_t *out_size);

/*
 * Batches.  Frames are same-sized, tightly packed planar: Y (w*h), U (cw*ch), V (cw*ch) with cw = ceil(w/2), ch = ceil(h/2)
 * for 4:2:0 (I420; cw x h for 4:2:2, w x h for 4:4:4: settings.chroma_format); consecutive frames are frame_stride bytes apart.
 *
 * h2j_submit_host:   frames live in HOST memory (pinned for full PCIe speed); the copy to the device, the
 *                    kernels and nothing else are enqueued on the slot's stream.  Returns immediately.
 * h2j_submit_device: frames already live in device memory on the encoder's device.
 * h2j_collect:       waits for the slot, copies the JPEGs back packed one after another into `out`
 *                    (offsets[i] .. offsets[i+1]) and frees the slot.  offsets has n+1 entries.  A frame that failed
 *                    (status[i] != 0, e.g. its JPEG outgrew max_jpeg_bytes) has length 0; the others are complete and the
 *                    call returns the failed frames' status.  If `out` itself is too short for the batch the call returns
 *                    H2J_ERR_BUFFER_TOO_SMALL with offsets[] filled in and the slot still collectable.
 * h2j_collect_device:waits for the slot and only reports where the JPEGs are on the device: frame i is
 *                    at (*d_out) + i * (*d_frame_capacity), sizes[i] bytes long (sizes is a host array);
 *                    *d_frame_capacity is max_jpeg_bytes rounded up to a multiple of 16.
 *                    The memory stays valid until the slot is submitted to again.
 * status[i] (optional, may be NULL) receives a per-frame h2j_status.
 *
 * Stream ordering of device inputs: the kernels of a slot run on the slot's own (non-blocking) stream, or on the stream
 * given with h2j_slot_set_stream.  h2j_submit_device and the other h2j_submit_device_* read the caller's device memory on THAT
 * stream; nothing orders them behind work of other streams.  A caller whose frames are produced on another stream (a
 * decoder's, torch's current stream) must, before submitting, either synchronise that stream, or make the slot use it
 * (h2j_slot_set_stream), or record an event behind the producer and hand it to h2j_slot_wait_event.  The same holds
 * for reusing the input memory: it may be overwritten once the slot has been collected (or h2j_wait returned).
 */
int h2j_submit_host(h2j_encoder *e, int slot, const uint8_t *frames, size_t frame_stride, int n, int width,
                    int height);
int h2j_submit_device(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int n, int width,
                      int height);
/* h2j_submit_device_nv12: the batch is NV12 in device memory, as hardware decoders (NVDEC) leave it: per frame a luma
 * plane of `height` rows and, `uv_offset` bytes behind the frame's start, a plane of ceil(height/2) rows of interleaved
 * Cb/Cr pairs; both planes have rows `pitch` bytes apart, frames are `frame_stride` bytes apart.  With the pointer, the
 * stride, the pitch and uv_offset multiples of 8 the frames are read where they are (the chroma pairs are split in
 * registers); otherwise the pairs are first split into the slot's own I420 frame buffer by one extra kernel.  The JPEGs are
 * the ones the reference writes for the equivalent yuv420p frame (the reference itself has no NV12 input: its decoder is
 * libavcodec's software decoder, src/Decoder.cpp:183, :324-342).  Collect with h2j_collect / h2j_collect_device. */
int h2j_submit_device_nv12(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch,
                           size_t uv_offset, int n, int width, int height);
/* Semi-planar frames in device memory, by the encoder's chroma_format: NV12 (4:2:0), NV16 (4:2:2), NV24 (4:4:4).
 * Per frame: a luma plane of `height` rows; `uv_offset` bytes behind the frame's start, a plane of interleaved Cb/Cr pairs
 * with ceil(width/2) pairs x ceil(height/2) rows (NV12), ceil(width/2) x height (NV16) or width x height (NV24).
 * Both planes have rows `pitch` bytes apart; frames are `frame_stride` bytes apart.
 * JPEGs: those of the equivalent planar frame.
 * With the pointer, the stride, the pitch and uv_offset multiples of 8 the frames are read where they are; otherwise the
 * pairs are first split into the slot's own planar frame buffer by one extra kernel.  At 4:2:0 this is
 * h2j_submit_device_nv12.  H2J_ERR_INVALID_ARG: a pitch shorter than a luma row or a row of pairs, a pair plane that
 * starts inside the luma plane, or a plane that reaches past frame_stride. */
int h2j_submit_device_semiplanar(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch,
                                 size_t uv_offset, int n, int width, int height);
/* Planar frames in device memory at any layout: luma rows `y_pitch` apart at the frame's start; Cb and Cr planes at
 * `u_offset` / `v_offset` (any order, e.g. YV12's V before U), rows `c_pitch` apart.
 * Plane sizes as for h2j_submit_device.
 * A hardware decoder's 4:4:4 surface is y_pitch = c_pitch = pitch, u_offset = pitch * surface_height, v_offset =
 * 2 * pitch * surface_height.  With the pointer, the stride, both pitches and both offsets multiples of 8 the frames are
 * read where they are; otherwise one extra kernel copies them to a 16-byte pitch first.  H2J_ERR_INVALID_ARG: a pitch
 * shorter than its plane's row, or a plane that reaches past frame_stride. */
int h2j_submit_device_pitched(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int y_pitch,
                              int c_pitch, size_t u_offset, size_t v_offset, int n, int width, int height);
int h2j_collect(h2j_encoder *e, int slot, uint8_t *out, size_t out_capacity, size_t *offsets, int *status);
int h2j_collect_device(h2j_encoder *e, int slot, const uint8_t **d_out, size_t *d_frame_capacity, size_t *sizes,
                       int *status);
/* Make the slot enqueue on a caller-owned CUDA stream (a cudaStream_t, e.g. torch.cuda.Stream().cuda_stream)
 * instead of its own, so the caller can bracket the work with its own events.  The slot must be idle. */
int h2j_slot_set_stream(h2j_encoder *e, int slot, void *cuda_stream);
/* Make everything submitted to the (idle) slot from now on wait, on the device, for a CUDA event (a cudaEvent_t recorded
 * by the caller behind the work that produces the next batch's input).  No host synchronisation. */
int h2j_slot_wait_event(h2j_encoder *e, int slot, void *cuda_event);
/* Block until the slot's stream is idle without collecting (timing helper). */
int h2j_wait(h2j_encoder *e, int slot);

/* Pinned host memory helpers so callers in any language can get full-speed copies. */
void *h2j_alloc_pinned(size_t bytes);
void h2j_free_pinned(void *p);
/* memcpy for filling pinned staging that the GPU reads next: non-temporal stores where the CPU has AVX2 (no
 * read-for-ownership of the destination, the caller's cache keeps its contents), plain memcpy otherwise. */
void h2j_stream_copy(void *dst, const void *src, size_t n);

/*
 * Standalone plane conversion (kernel 1 on its own): yuv420p limited -> yuvj420p full, with the encoder's
 * edge replication to whole 16x16 MCUs.  Host in, host out.  out planes are padded:
 * luma (mcu_w*16) x (mcu_h*16), chroma (mcu_w*8) x (mcu_h*8); pass range_mode to choose the mapping.
 */
int h2j_convert_pad(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int width, int height,
                    int range_mode, uint8_t *out_y, uint8_t *out_u, uint8_t *out_v);

/* ---- inspection (parity tests read the intermediate products through these) ---------------------- */
typedef struct h2j_frame_info {
    int qscale;              /* what the rate control chose */
    int64_t mb_var_sum;      /* its input */
    int mcu_w, mcu_h;
    int header_bytes;        /* SOI .. end of SOS */
    int64_t scan_bits;       /* entropy-coded bits before padding/stuffing */
    int64_t stuffed_ff;      /* number of 0x00 bytes inserted */
    uint8_t intra_matrix[64];/* raster order */
    uint32_t hist[4][256];   /* DC luma, DC chroma, AC luma, AC chroma symbol counts */
    uint8_t bits[4][17];     /* DHT BITS (index 1..16) */
    uint8_t vals[4][256];    /* DHT HUFFVAL */
    int nvals[4];
} h2j_frame_info;

/* Valid after h2j_wait/h2j_collect* on the slot and before the next submit to it. */
int h2j_debug_frame_info(h2j_encoder *e, int slot, int frame, h2j_frame_info *info);
/* Quantised levels of one frame: mcu_w*mcu_h*6 blocks in MCU order (Y0 Y1 Y2 Y3 Cb Cr), 64 int16 each in
 * zigzag order (index 0 = quantised DC level, not the difference). */
int h2j_debug_coefficients(h2j_encoder *e, int slot, int frame, int16_t *out, size_t out_elems);

/* Synchronous copy of `bytes` bytes of device memory on the encoder's device (e.g. a JPEG reported by h2j_collect_device)
 * to host memory: lets callers without a CUDA binding of their own look at device-resident results. */
int h2j_debug_read_device(h2j_encoder *e, const void *d_src, void *dst, size_t bytes);
/* Launch-shape overrides for tests that must reach code paths a small batch would not take on its own.  Results never
 * depend on a knob.  "fdct_tiles_per_cta": consecutive 16-MCU tiles one CTA of the FDCT kernel walks (0 = automatic:
 * 1 for small batches, up to 16 for large ones).  "semiplanar_prepass": 1 = h2j_submit_device_semiplanar /
 * h2j_submit_device_nv12 split the pairs into planes first even where the frames could be read in place (0 = by
 * alignment). */
int h2j_debug_set_knob(h2j_encoder *e, const char *name, int value);

/* With settings.profile != 0: milliseconds each kernel of the slot's last batch took, measured with CUDA
 * events on the stream the kernels were launched on.  names/ms have `cap` entries; returns the count. */
int h2j_slot_kernel_ms(h2j_encoder *e, int slot, const char **names, float *ms, int cap);
/* Switch the per-kernel event brackets of batches submitted from now on (settings.profile at run time): a bracket
 * costs a few microseconds of idle GPU per kernel boundary, so throughput runs take them on a sample of their batches. */
int h2j_set_profile(h2j_encoder *e, int on);
/* Milliseconds between the first and the last event of the slot's last batch (includes copies). */
int h2j_slot_total_ms(h2j_encoder *e, int slot, float *ms);
/* Number of kernel launches issued by this encoder so far. */
long long h2j_kernel_launches(const h2j_encoder *e);

#ifdef __cplusplus
}
#endif
#endif /* H2J_B200_H */
