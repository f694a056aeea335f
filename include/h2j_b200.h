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

/* Bumped when an existing entry point or struct changes.  Additions (the semi-planar, pitched, 16-bit and list submits)
 * leave it as it is: a caller built against an older header keeps working unchanged. */
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
                              ffmpeg build the reference links on x86-64 (lib/ffmpeg/x86_64_shared); at most
                              65,532 bytes, the most a COM segment's 16-bit length (text + NUL + the field's own two
                              bytes) can hold -- a longer one fails with H2J_ERR_INVALID_ARG */
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

/*
 * High-bit-depth frames (H.265 Main10 / Main12 and the like).  Every sample is a little-endian 16-bit word that holds a
 * `bit_depth`-bit value (9..16) in its low bits.  MSB-aligned formats -- P010 / P016, P210 / P216 and a hardware decoder's
 * 16-bit 4:4:4 surface -- are bit_depth 16.  The 8-bit sample the encoder uses is
 *     (word & ((1 << bit_depth) - 1)) >> (bit_depth - 8)
 * i.e. truncation: bits above bit_depth are ignored, there is no rounding and no dither.  The JPEG is byte-identical to
 * the one this encoder writes for the 8-bit planar frame of those samples, with the same range_mode and fixed_qscale
 * (H2J_RANGE_LIMITED_TO_FULL maps 10-bit limited range, 64..940 -> 16..235, exactly as 8-bit).  No colour-space or transfer
 * conversion is done: BT.2020 / PQ content is encoded as it stands, as the reference ignores colour metadata.
 * All pitches, strides and offsets are in BYTES (as AVFrame.linesize); pointers, pitches, strides and offsets must be even.
 * Each device submit converts the batch into the slot's own 8-bit frame buffer with one extra kernel, then runs the
 * usual pipeline; collect with h2j_collect / h2j_collect_device.
 *
 * h2j_submit_device_semiplanar16: as h2j_submit_device_semiplanar with 16-bit words: P010 / P016 (4:2:0), P210 / P216
 *   (4:2:2) or the 4:4:4 equivalent, by the encoder's chroma_format.  A row of pairs is 2 * pair count words.
 * h2j_submit_device_pitched16: as h2j_submit_device_pitched with 16-bit words (a decoder's 16-bit 4:4:4 surface,
 *   yuv420p10le frames in device memory ...).
 * h2j_encode_frame16: as h2j_encode_frame with 16-bit planes (libavcodec's yuv420p10le / yuv420p12le are bit_depth 10 /
 *   12).  Its device buffer and pinned staging are allocated on its first call (H2J_ERR_NOMEM if that fails; the encoder
 *   stays usable) and freed by h2j_destroy.
 * H2J_ERR_INVALID_ARG: bit_depth outside 9..16, an odd pointer / pitch / stride / offset, a pitch or stride shorter than
 * two bytes per sample of its row (semi-planar: 2 * max(width, 2 * pairs per row)), a pair plane that starts inside the
 * luma plane, or a plane that reaches past frame_stride.  H2J_ERR_UNSUPPORTED: a size above the encoder's maximum.
 */
int h2j_submit_device_semiplanar16(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int pitch,
                                   size_t uv_offset, int bit_depth, int n, int width, int height);
int h2j_submit_device_pitched16(h2j_encoder *e, int slot, const uint8_t *d_frames, size_t frame_stride, int y_pitch,
                                int c_pitch, size_t u_offset, size_t v_offset, int bit_depth, int n, int width, int height);
int h2j_encode_frame16(h2j_encoder *e, const uint8_t *const planes[3], const int strides[3], int bit_depth, int width,
                       int height, uint8_t *out, size_t out_capacity, size_t *out_size);

/*
 * Lists of frames, each at its own address and of its own size (at most max_width x max_height): frames of several
 * streams at different resolutions in one batch, or a decoder's surfaces where they are, without gathering them into one
 * strided buffer first.  One layout kind per call; chroma format, range_mode and fixed_qscale are the encoder's.  Frame i's
 * JPEG is byte-identical to the one h2j_submit_device writes for that frame alone.  Collect with h2j_collect /
 * h2j_collect_device as for the other submits.  The device frames are read on the slot's stream, under the stream-ordering
 * rule above.
 * h2j_submit_device_list: n device frames.  H2J_LAYOUT_PLANAR: luma rows y_pitch apart from data, Cb and Cr planes at
 *   u_offset / v_offset with rows c_pitch apart; frames whose rows are not all on 8-byte boundaries are copied to a 16-byte
 *   pitch (one extra kernel for all of them), the others are read where they are.  H2J_LAYOUT_SEMIPLANAR: NV12 / NV16 /
 *   NV24 by the encoder's chroma format, the pair plane at u_offset with rows c_pitch apart (v_offset unused); read in
 *   place when every frame's pointer, pitches and offset are multiples of 8, otherwise the whole batch is split into
 *   planes first by one extra kernel.
 * h2j_submit_host_list: n tight planar frames in host memory (the layout of h2j_submit_host); frame i is uploaded with
 *   one copy.
 * H2J_ERR_INVALID_ARG: a null pointer, n < 1 or n > max_batch, a pitch shorter than its plane's row (semi-planar chroma:
 * 2 * pairs per row), or a pair plane that starts inside the luma plane.  H2J_ERR_UNSUPPORTED: a frame outside 2..65500 or
 * above the encoder's maximum.  H2J_ERR_BUSY: the slot has a batch in flight.
 */
typedef enum h2j_layout { H2J_LAYOUT_PLANAR = 0, H2J_LAYOUT_SEMIPLANAR = 1 } h2j_layout;

typedef struct h2j_frame_desc {
    const uint8_t *data;   /* device address of the frame's first luma byte */
    int width, height;
    int y_pitch;           /* bytes between luma rows */
    int c_pitch;           /* bytes between chroma rows (semi-planar: rows of Cb/Cr pairs) */
    size_t u_offset;       /* bytes from data to the Cb plane (semi-planar: to the pair plane) */
    size_t v_offset;       /* bytes from data to the Cr plane (semi-planar: unused) */
} h2j_frame_desc;

int h2j_submit_device_list(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n);
int h2j_submit_host_list(h2j_encoder *e, int slot, const uint8_t *const *frames, const int *widths, const int *heights, int n);

/*
 * Downscaled device frames: thumbnails and previews of decoder surfaces, encoded without a full-size pass.  `layout` and
 * `frames` are those of h2j_submit_device_list (planar at any pitches and plane offsets, or NV12 / NV16 / NV24 by the
 * encoder's chroma format; any alignment; each frame of its own size).  `factor` is 2, 4 or 8.  Frame i's JPEG is
 * byte-identical to the one h2j_submit_device writes, with the same encoder settings, for the planar frame D_k(frame i):
 *   every plane, at its decoder size pw x ph (chroma ceil-divided as for the other submits), becomes a plane of
 *   ceil(pw/k) x ceil(ph/k) samples, out[y][x] = (S + c/2) / c in integers (rounded half up), where S is the sum of the
 *   c source samples P[j][i] with k*x <= i < min(k*x + k, pw) and k*y <= j < min(k*y + k, ph) -- c = k*k except in the
 *   partial boxes at the right and bottom edges.  Semi-planar Cb and Cr are averaged separately.
 * The downscaled frame is ceil(w/k) x ceil(h/k), and its chroma planes are exactly that frame's chroma size
 * (ceil(ceil(w/2)/k) == ceil(ceil(w/k)/2)).  Range conversion (range_mode) applies to the downscaled samples.
 * Sources may be up to 65500 on a side whatever max_width / max_height; only the downscaled frame must fit the encoder (an
 * encoder created for 480x272 takes 1920x1080 sources at factor 4).  One kernel writes the downscaled frames into the slot's
 * own frame buffer, then the usual pipeline runs on them.  Collect with h2j_collect / h2j_collect_device; the inspection
 * calls answer for the downscaled frames; the device frames are read on the slot's stream, under the stream-ordering
 * rule above.
 * H2J_ERR_INVALID_ARG: as h2j_submit_device_list, or a factor other than 2, 4, 8.  H2J_ERR_UNSUPPORTED: a source outside
 * 2..65500, or a downscaled frame smaller than 2 on a side or larger than the encoder's maximum.  H2J_ERR_BUSY: the slot has
 * a batch in flight.  Every frame is checked before anything is enqueued: a rejected call leaves the previous batch as it was.
 */
int h2j_submit_device_downscaled(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n, int factor);

/*
 * Resized device frames: thumbnails, previews and model inputs at any size (2/3, 1/6, a fixed 224x224, "longest side 512",
 * an upscale to a fixed grid), with Pillow's BOX, BILINEAR or BICUBIC filter.  `layout` and `frames` are those of
 * h2j_submit_device_list; frame i is encoded at out_widths[i] x out_heights[i] (W x H).  Frame i's JPEG is byte-identical to
 * the one h2j_submit_device writes, with the same encoder settings, for the planar frame R(frame i):
 *   every plane, at its decoder size (luma w x h, Cb and Cr at the encoder's chroma size of w x h; semi-planar Cb and Cr
 *   separately), is resized as a Pillow "L" image to the matching plane of the W x H frame (luma W x H, chroma the
 *   encoder's chroma size of W x H): PIL.Image.resize((pw_out, ph_out), filter) of Pillow's libImaging/Resample.c.  Per
 *   axis, in to out samples: scale = in / out, fs = max(scale, 1), support = s_f * fs (s_f 0.5, 1, 2); output o has the
 *   window xmin = max((int)(center - support + 0.5), 0) .. min((int)(center + support + 0.5), in), center = (o + 0.5) *
 *   scale, weights f((x - center + 0.5) / fs) normalised by their sum, in double, and rounded to 22-bit fixed point
 *   ((int)(w * 2^22 +- 0.5)).  The horizontal pass runs first, on every source row, and its result is clipped to 0..255;
 *   the vertical pass runs on those 8-bit rows; each sums (2^21 + sum of sample * coefficient) in 32 bits and keeps
 *   clamp(sum >> 22, 0, 255).  An axis whose size does not change has no pass, so W x H = w x h encodes the frame as
 *   h2j_submit_device_list does.
 * The resized samples are pinned bit for bit against Pillow itself (tests/test_resize_model.py); the JPEG is the existing
 * encoder's.  BOX at an integer factor is NOT D_k above: Pillow rounds between its passes and its edge weights are not
 * exact.  range_mode applies to the resized samples.  Sources may be 2..65500 on a side whatever max_width / max_height; only
 * W x H must fit the encoder.  The coefficient tables are built on the host and kept in a per-slot buffer allocated on
 * first use and grown when a submit needs more; one kernel writes the resized frames into the slot's own frame buffer,
 * then the usual pipeline runs (frames of one size run its batch form).  Collect with h2j_collect / h2j_collect_device; the
 * inspection calls answer for the resized frames; the device frames are read on the slot's stream, under the
 * stream-ordering rule above.
 * H2J_ERR_INVALID_ARG: as h2j_submit_device_list, null out_widths / out_heights, or a bad filter.  H2J_ERR_UNSUPPORTED: a
 * source outside 2..65500, or an output size outside 2..65500 or above the encoder's maximum.  H2J_ERR_NOMEM: no room for
 * the coefficient tables (the encoder stays usable).  H2J_ERR_BUSY: the slot has a batch in flight.  Every frame is checked
 * before anything is enqueued: a rejected call leaves the previous batch as it was.
 */
typedef enum h2j_resize_filter { H2J_FILTER_BOX = 0, H2J_FILTER_BILINEAR = 1, H2J_FILTER_BICUBIC = 2 } h2j_resize_filter;

int h2j_submit_device_resized(h2j_encoder *e, int slot, int layout, const h2j_frame_desc *frames, int n, const int *out_widths,
                              const int *out_heights, int filter);

/*
 * RGB frames: torch tensors ((3, H, W) planar as torchvision.io.encode_jpeg takes them, or (H, W, 3)), model outputs and
 * annotated frames, rendered RGBA8 surfaces, a hardware decoder's BGRA post-processing output, OpenCV / numpy images.
 * Frame i's JPEG is byte-identical to the one h2j_submit_device writes, with the same fixed_qscale and chroma_format, for
 * the planar frame C(frame i) built in two steps:
 *   1. per pixel, JFIF / ITU-T T.871 full-range YCbCr in libjpeg's integer form (jccolor.c: 16 fraction bits,
 *      FIX(x) = (int)(x * 65536 + 0.5), chroma rounded with ONE_HALF - 1):
 *        Y  = ( 19595 R + 38470 G +  7471 B + 32768)              >> 16
 *        Cb = (-11059 R - 21709 G + 32768 B + (128 << 16) + 32767) >> 16
 *        Cr = ( 32768 R - 27439 G -  5329 B + (128 << 16) + 32767) >> 16
 *      Every result lies in 0..255 (no clamp), and it is within 1 of the float T.871 formula rounded half up.  T.871 is the
 *      only matrix: the JPEG carries component ids 1, 2, 3 and no JFIF or Adobe marker, which every decoder reads as T.871
 *      YCbCr, so no other matrix would decode back to the caller's colours.
 *   2. at 4:2:0 / 4:2:2, the 8-bit Cb and Cr planes are box-averaged over 2x2 / 2x1 pixels to the encoder's usual chroma
 *      sizes (ceil(w/2) x ceil(h/2), ceil(w/2) x h; 4:4:4: w x h, no averaging): out = (S + c/2) / c in integers (rounded
 *      half up), S the sum of the c samples of the box that lie inside the plane (fewer than the box's at the right and
 *      bottom edges), as for D_k above.
 * range_mode does not apply: the YCbCr of an RGB frame is full range by construction, and an encoder created with
 * H2J_RANGE_LIMITED_TO_FULL writes the same RGB JPEGs as one created with H2J_RANGE_PASSTHROUGH.  Alpha / X bytes never
 * reach the picture.
 *
 * h2j_submit_device_rgb: n device frames, each of its own size (at most max_width x max_height) at its own address, with
 *   any alignment, described by h2j_frame_desc: packed formats use data, width, height and y_pitch (bytes between rows);
 *   H2J_RGB_PLANAR has the R plane at data, G at data + u_offset and B at data + v_offset, every plane's rows y_pitch
 *   apart.  Other fields are ignored.  One kernel converts the frames into the slot's own frame buffer, then the usual
 *   pipeline runs (frames of one size run its batch form, others its list form).  Collect with h2j_collect /
 *   h2j_collect_device; the device frames are read on the slot's stream, under the stream-ordering rule above.
 * h2j_encode_frame_rgb: one picture from host memory, synchronously on slot 0, as h2j_encode_frame: packed formats take
 *   planes[0] / strides[0] only, H2J_RGB_PLANAR the R, G and B planes with their own strides.  The picture is staged on
 *   the device at a 16-byte aligned pitch in a buffer h2j_encode_frame16 shares, allocated on first use and grown when a
 *   call needs more (H2J_ERR_NOMEM if that fails; the encoder stays usable), freed by h2j_destroy.
 * H2J_ERR_INVALID_ARG: as h2j_submit_device_list, a bad format, a null data pointer, a pitch or stride shorter than a row
 * (3w, 4w or w bytes), or a planar G or B plane that starts inside the R plane (offset < y_pitch * height).
 * H2J_ERR_UNSUPPORTED: a size outside 2..65500 or above the encoder's maximum.  H2J_ERR_BUSY: the slot has a batch in
 * flight.  Every frame is checked before anything is enqueued: a rejected call leaves the previous batch as it was.
 */
typedef enum h2j_rgb_format {
    H2J_RGB_RGB24 = 0,   /* R G B, 3 bytes per pixel (numpy / torch HWC) */
    H2J_RGB_BGR24 = 1,   /* B G R (OpenCV) */
    H2J_RGB_RGBX = 2,    /* R G B + one ignored byte (RGBA8) */
    H2J_RGB_BGRX = 3,    /* B G R + one ignored byte (BGRA8) */
    H2J_RGB_PLANAR = 4   /* three planes R, G, B (torch CHW) */
} h2j_rgb_format;

int h2j_submit_device_rgb(h2j_encoder *e, int slot, int format, const h2j_frame_desc *frames, int n);
int h2j_encode_frame_rgb(h2j_encoder *e, int format, const uint8_t *const planes[3], const int strides[3], int width,
                         int height, uint8_t *out, size_t out_capacity, size_t *out_size);

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
/* Frame `frame` of the slot's last batch as the pipeline read it (before range_mode's mapping), copied to tight host
 * planes: Y width x height, U and V at the frame's chroma size (ceil-divided by the chroma format's subsampling).  A frame
 * the input stage wrote (RGB, 16-bit, downscaled, split or repitched) is read from the slot's buffer; a frame read in place
 * from the caller's memory, which must still hold it (semi-planar pairs are split on the host).  Same validity as above:
 * JPEG byte equality can hide a one-off sample behind quantisation, these planes cannot. */
int h2j_debug_frame_planes(h2j_encoder *e, int slot, int frame, uint8_t *y, uint8_t *u, uint8_t *v);

/* Synchronous copy of `bytes` bytes of device memory on the encoder's device (e.g. a JPEG reported by h2j_collect_device)
 * to host memory: lets callers without a CUDA binding of their own look at device-resident results. */
int h2j_debug_read_device(h2j_encoder *e, const void *d_src, void *dst, size_t bytes);
/* Launch-shape overrides for tests that must reach code paths a small batch would not take on its own.  Results never
 * depend on a knob.  "fdct_tiles_per_cta": consecutive 16-MCU tiles one CTA of the FDCT kernel walks (0 = automatic:
 * 1 for small batches, up to 16 for large ones).  "semiplanar_prepass": 1 = h2j_submit_device_semiplanar /
 * h2j_submit_device_nv12 split the pairs into planes first even where the frames could be read in place (0 = by
 * alignment).  "planar_copy": 0 = planar frames whose rows do not all start on 8-byte boundaries are read in place by the
 * kernels' bytewise path, as when the slot has no room for their 16-byte-pitch copies (1 = copied first, the default). */
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
