// Host-side mirror of the reference's encoder class (reference src/Encoder.h:29-85) over the h2j_b200 C ABI.
//
// This header takes the place of the reference's src/Encoder.h -- it carries that file's include guard, so a
// translation unit that has seen this one skips the reference's -- and Encoder.cpp takes the place of
// src/Encoder.cpp.  Same class name, same constructor, same yuv2Jpeg(AVFrame*) -> bool contract and the same
// observable behaviour: on success the JPEG is written to outputFilePath with fopen(..., "wb+") (reference
// src/Encoder.cpp:338-361), on any failure a line goes to LOG() and false is returned.  The bytes written are
// identical to the reference's.  src/Decoder.cpp (the only caller, Decoder.cpp:349), export_inc/IDecoder.h and
// src/jni stay untouched.
//
// The libavcodec/libavformat machinery the reference's Encoder drove (AVIOContext, AVFormatContext, mjpeg
// AVCodecContext ...) is gone: the planes go to the GPU through pinned staging and asynchronous copies.
#ifndef H265TOJPEG_ENCODER_H
#define H265TOJPEG_ENCODER_H

#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <memory>

// The reference's src/Encoder.h is where src/Decoder.cpp gets src/Common.h from (DEBUG, HEAP_SIZE, STACK_SIZE, LOG):
// inside the reference tree this header passes it on the same way; built alone it supplies the few names itself.
#if defined(__has_include)
#if __has_include("Common.h")
#include "Common.h"
#define H2J_HAVE_REFERENCE_COMMON_H 1
#endif
#endif
#ifndef H2J_HAVE_REFERENCE_COMMON_H
#ifndef DEBUG
#define DEBUG 0
#endif
/* 堆缓冲大小 / 栈缓冲大小 of the reference (src/Common.h:16,19) */
#ifndef HEAP_SIZE
#define HEAP_SIZE (1024 * 1024 * 2)
#endif
#ifndef STACK_SIZE
#define STACK_SIZE (1024)
#endif
extern void LOG(const char *format, ...);  // reference src/Decoder.cpp:20 (host/log_default.cpp when built alone)
#endif

struct AVFrame;  // libavutil/frame.h — only needed by Encoder.cpp, and only when built with H2J_WITH_LIBAV

// What yuv2Jpeg needs from an AVFrame, for callers (and tests) that have no libavutil headers.
struct H2JFrameView {
    const uint8_t *data[3];
    int linesize[3];
    int width, height;
    int format;  // AVPixelFormat (libavutil 56): 0 = AV_PIX_FMT_YUV420P, 12 = AV_PIX_FMT_YUVJ420P, and the 16-bit little-endian
                 // 64 = AV_PIX_FMT_YUV420P10LE, 125 = AV_PIX_FMT_YUV420P12LE (linesize in bytes, as AVFrame's), which are
                 // encoded from their 8-bit truncation (h2j_encode_frame16 in include/h2j_b200.h)
};

class Encoder {
public:
    explicit Encoder(const char *outputFilePath);
    ~Encoder();

    // reference src/Encoder.cpp:104
    bool yuv2Jpeg(AVFrame *pFrame);
    // same, from plain pointers
    bool yuv2Jpeg(const H2JFrameView &frame);

    // Bytes of the last JPEG produced (the reference keeps them in Output::jpeg_data, src/Common.h:65).
    const uint8_t *jpegData() const { return jpeg_.get(); }
    size_t jpegSize() const { return jpegSize_; }

private:
    void release();
    bool saveJpegtoFile(const char *filePath);

    const char *outputFilePath;
    std::unique_ptr<uint8_t[]> jpeg_;
    size_t jpegSize_ = 0;
    size_t jpegCap_ = 0;
};

// ---- process-wide knobs (optional; the defaults reproduce the reference's behaviour) -------------------------------
// cuda_device >= 0: every picture goes to that device.  cuda_device = -1 (the default): all visible devices may be
// used -- a device is brought up only when the ones already running are busy, so a single-threaded caller stays on
// one GPU and a threaded service (one IDecoder per thread, as the reference's getInstance() hands them out,
// src/Decoder.cpp:39-44) or a batch scope spreads over the box.  range_mode: H2J_RANGE_* of include/h2j_b200.h (the
// reference converts nothing).  Waits for queued work, then drops the GPU state; call it before the first yuv2Jpeg.
extern "C" void h2j_host_configure(int cuda_device, int range_mode);

// Batch scope for services that convert many pictures (the reference has no such call: a loop over
// IDecoder::H265ToJpeg is what it offers, main.cpp:37-65).  Between begin and end, yuv2Jpeg() -- and therefore the
// unchanged IDecoder::H265ToJpeg() that calls it (reference src/Decoder.cpp:349) -- only copies the decoded planes into
// pinned staging and returns true; it may be called from any number of threads.  Pictures of any sizes, in any order, are
// encoded `max_frames` at a time (each gets pinned room for its own size; a picture that no longer fits the batch's room
// closes it early): a full batch goes to a GPU worker thread (one per device in use, two batches in flight
// per device so that the upload of one runs under the kernels of the other), which also writes the JPEG files, while
// the callers already fill the next batch.  h2j_host_batch_end() drains everything and returns the number of files
// written (-1 outside a scope); *failed receives the number of pictures that could not be encoded or saved.
// High-bit-depth pictures (yuv420p10le / yuv420p12le) are not queued: inside a scope they take the synchronous path, so
// their file exists when yuv2Jpeg returns, and they do not count in h2j_host_batch_end's result.
extern "C" int h2j_host_batch_begin(int max_frames);
extern "C" int h2j_host_batch_end(int *failed);
// Devices that currently hold GPU state for this process (inspection).
extern "C" int h2j_host_devices_in_use(void);
// Batches the scope has handed to a GPU since h2j_host_batch_begin (inspection).
extern "C" int h2j_host_batches_submitted(void);

#endif  // H265TOJPEG_ENCODER_H
