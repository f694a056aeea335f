// See Encoder.h.  Mirrors reference src/Encoder.cpp's control flow and error behaviour; the encode itself is
// the C ABI (include/h2j_b200.h), which runs the CUDA kernels.  There is no CPU encode here: if the GPU library
// cannot be used, yuv2Jpeg logs and returns false.
//
// Process-wide state (`Hub`):
//   * one DeviceCtx per CUDA device in use.  It owns a small synchronous encoder (the yuv2Jpeg call shape: one
//     picture, host planes in, file out) and, once a batch scope has used the device, a batch encoder with two slots
//     and the worker thread that drives it;
//   * a pool of Jobs: pinned input staging for one batch + pinned output for its JPEGs, allocated once and reused.
// The reference builds a fresh libavcodec context per picture (src/Decoder.cpp:349 constructs an Encoder per call); a
// CUDA context and its buffers are far too expensive for that, so Encoder objects are thin and share the Hub.
#include "Encoder.h"

#include <algorithm>
#include <cerrno>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/h2j_b200.h"

#ifdef H2J_WITH_LIBAV
extern "C" {
#include "libavutil/frame.h"
}
#endif

namespace {

constexpr int kSlotsPerDevice = 2;  // batches in flight per device: the upload of one runs under the kernels of the other

// What libavcodec's HEVC decoder produces for Main10 / Main12 4:2:0: 16-bit little-endian words holding 10 / 12-bit values.
#ifdef H2J_WITH_LIBAV
constexpr int kFmtYuv420p10le = AV_PIX_FMT_YUV420P10LE, kFmtYuv420p12le = AV_PIX_FMT_YUV420P12LE;
static_assert(AV_PIX_FMT_YUV420P == 0 && AV_PIX_FMT_YUVJ420P == 12 && kFmtYuv420p10le == 64 && kFmtYuv420p12le == 125,
              "H2JFrameView callers pass the AVPixelFormat numbers of libavutil 56");
#else
constexpr int kFmtYuv420p10le = 64, kFmtYuv420p12le = 125;  // AV_PIX_FMT_YUV420P10LE / AV_PIX_FMT_YUV420P12LE (libavutil 56)
#endif

size_t i420_bytes(int w, int h) { return (size_t)w * h + 2 * (size_t)((w + 1) >> 1) * ((h + 1) >> 1); }

// reference src/Encoder.cpp:338-361 saveJpegtoFile: same open mode, same log lines, same false on error
bool save_jpeg(const char *filePath, const uint8_t *data, size_t n)
{
    if (filePath == nullptr || strlen(filePath) == 0) {
        LOG("Jpeg 文件路径为空，请核查！");
        return false;
    }
    FILE *fp_write = fopen(filePath, "wb+");
    if (!fp_write) {
        LOG("%s line=%d | Open file error! filePath=%s, errno=%d", __PRETTY_FUNCTION__, __LINE__, filePath, errno);
        return false;
    }
    const size_t ret = fwrite(data, 1, n, fp_write);
    if (ret == 0) {
        LOG("%s line=%d | fwrite error! Jpeg 文件路径：%s", __PRETTY_FUNCTION__, __LINE__, filePath);
        fclose(fp_write);
        return false;
    }
    LOG("保存 Jpeg 数据到文件: %s", filePath);
    fclose(fp_write);
    return true;
}

void copy_planes(uint8_t *p, const H2JFrameView &f)
{
    const int cw = (f.width + 1) >> 1, ch = (f.height + 1) >> 1;
    // (h2j_stream_copy: non-temporal stores -- the staging lines are read next by the GPU's DMA engine, not by this core)
    if (f.linesize[0] == f.width) h2j_stream_copy(p, f.data[0], (size_t)f.width * f.height);
    else
        for (int r = 0; r < f.height; r++) h2j_stream_copy(p + (size_t)r * f.width, f.data[0] + (size_t)r * f.linesize[0], f.width);
    p += (size_t)f.width * f.height;
    for (int pl = 1; pl <= 2; pl++) {
        if (f.linesize[pl] == cw) h2j_stream_copy(p, f.data[pl], (size_t)cw * ch);
        else
            for (int r = 0; r < ch; r++) h2j_stream_copy(p + (size_t)r * cw, f.data[pl] + (size_t)r * f.linesize[pl], cw);
        p += (size_t)cw * ch;
    }
}

// One batch on its way: pinned staging for up to `cap_frames` pictures of any sizes, each tight at its own offset, their
// output paths, pinned output.
struct Job {
    uint8_t *in = nullptr;
    size_t in_bytes = 0;
    size_t used = 0;           // bytes of `in` reserved by pictures so far
    std::vector<size_t> at;    // where picture k starts in `in`
    std::vector<int> ws, hs;   // its size
    uint8_t *out = nullptr;
    size_t out_bytes = 0;
    int cap_frames = 0;
    int reserved = 0;  // pictures that have a place in this job
    int filled = 0;    // ... and whose planes have been copied in
    bool sealed = false;
    bool busy = false;  // filling, queued or running
    std::vector<std::string> paths;
};

struct EncoderBox {  // an h2j_encoder and what it was created for
    h2j_encoder *enc = nullptr;
    int max_w = 0, max_h = 0, max_batch = 0;
    size_t cap = 0;  // per-picture output capacity
};

struct DeviceCtx {
    int device = 0;
    std::mutex sync_mu;  // the synchronous path of this device: one picture at a time
    EncoderBox sync_box;
    // batch path: the encoder is touched by the device's worker thread only; queue and counters are guarded by Hub::mu
    EncoderBox batch_box;
    bool batch_box_stale = false;  // h2j_host_configure changed the settings: rebuild before the next batch
    std::deque<Job *> queue;
    int inflight = 0;  // jobs queued or running here
    bool worker_started = false;
};

struct Hub {
    std::mutex mu;
    std::condition_variable cv_jobs;    // a job became free
    std::condition_variable cv_queue;   // a device queue got a job
    int only_device = -1;               // h2j_host_configure
    int range_mode = H2J_RANGE_PASSTHROUGH;
    int n_visible = -1;                 // CUDA devices (asked once)
    std::vector<std::unique_ptr<DeviceCtx>> devices;  // index = position in the allowed list, created on first use
    unsigned turn = 0;
    // batch scope
    bool batching = false;
    int batch_frames = 0;
    size_t room = 0;           // pinned bytes per picture a new job gets: the largest picture of the scope so far
    int batches = 0;           // jobs handed to a GPU since h2j_host_batch_begin
    std::vector<std::unique_ptr<Job>> jobs;
    Job *filling = nullptr;
    int written = 0, failed = 0;
};

Hub &hub()
{
    static Hub *h = new Hub();  // never destroyed: worker threads and CUDA state must not be torn down from a static destructor
    return *h;
}

int allowed_devices(Hub &H)
{
    if (H.only_device >= 0) return 1;
    if (H.n_visible < 0) H.n_visible = h2j_device_count();
    return H.n_visible > 0 ? H.n_visible : 1;
}

// (H.mu held) the idx-th allowed device, created on first use
DeviceCtx &device_at(Hub &H, int idx)
{
    while ((int)H.devices.size() <= idx) {
        H.devices.emplace_back(new DeviceCtx());
        H.devices.back()->device = H.only_device >= 0 ? H.only_device : (int)H.devices.size() - 1;
    }
    return *H.devices[idx];
}

void drop_box(EncoderBox &b)
{
    if (b.enc) h2j_destroy(b.enc);
    b = EncoderBox{};
}

bool ensure_box(EncoderBox &b, int device, int range_mode, int w, int h, int batch, int n_slots)
{
    if (b.enc && w <= b.max_w && h <= b.max_h && batch <= b.max_batch) return true;
    if (b.enc) {  // grow, never shrink
        if (w < b.max_w) w = b.max_w;
        if (h < b.max_h) h = b.max_h;
        if (batch < b.max_batch) batch = b.max_batch;
        drop_box(b);
    }
    h2j_settings st;
    h2j_default_settings(&st);
    st.device = device;
    st.max_width = w > 1920 ? w : 1920;
    st.max_height = h > 1088 ? h : 1088;
    st.max_batch = batch;
    st.n_slots = n_slots;
    st.range_mode = range_mode;
    // the reference sizes its packet as width*height*3 (src/Encoder.cpp:241) and its copy buffer as HEAP_SIZE
    size_t cap = (size_t)st.max_width * st.max_height * 3;
    if (cap < HEAP_SIZE) cap = HEAP_SIZE;
    st.max_jpeg_bytes = cap;
    const int rc = h2j_create(&st, &b.enc);
    if (rc != H2J_OK) {
        LOG("h2j_create failed, rc=%d (%s), error=%s", rc, h2j_status_string(rc), h2j_last_error(nullptr));
        b = EncoderBox{};
        return false;
    }
    b.max_w = st.max_width;
    b.max_h = st.max_height;
    b.max_batch = batch;
    b.cap = cap;
    return true;
}

// ---- batch path ------------------------------------------------------------------------------------------------

// (worker thread, no lock held) wait for the slot, fetch the JPEGs into the job's pinned output, write the files
void finish_job(Hub &H, DeviceCtx &D, int slot, Job *j, bool submitted)
{
    const int n = j->reserved;
    std::vector<size_t> offs(n + 1, 0);
    std::vector<int> st(n, 0);
    bool ok = submitted;
    if (ok) {
        int rc = h2j_collect(D.batch_box.enc, slot, j->out, j->out_bytes, offs.data(), st.data());
        if (rc == H2J_ERR_BUFFER_TOO_SMALL) {  // more than 4 bits per pixel: the slot is still collectable, offs[n] is the size
            h2j_free_pinned(j->out);
            j->out_bytes = offs[n];
            j->out = static_cast<uint8_t *>(h2j_alloc_pinned(j->out_bytes));
            rc = j->out ? h2j_collect(D.batch_box.enc, slot, j->out, j->out_bytes, offs.data(), st.data()) : H2J_ERR_NOMEM;
            if (!j->out) j->out_bytes = 0;
        }
        if (rc != H2J_OK && rc != H2J_ERR_OUTPUT_TOO_SMALL) {  // (too small: the per-picture status says which)
            LOG("h2j batch of %d frames failed, rc=%d (%s), error=%s", n, rc, h2j_status_string(rc), h2j_last_error(D.batch_box.enc));
            ok = false;
        }
    }
    int written = 0, failed = 0;
    for (int k = 0; k < n; k++) {
        if (ok && st[k] == H2J_OK && save_jpeg(j->paths[k].c_str(), j->out + offs[k], offs[k + 1] - offs[k])) written++;
        else {
            if (ok && st[k] != H2J_OK) LOG("frame for %s failed: %s", j->paths[k].c_str(), h2j_status_string(st[k]));
            failed++;
        }
    }
    std::lock_guard<std::mutex> lock(H.mu);
    H.written += written;
    H.failed += failed;
    j->busy = false;
    D.inflight--;
    H.cv_jobs.notify_all();
}

void worker_main(Hub *Hp, DeviceCtx *Dp)
{
    Hub &H = *Hp;
    DeviceCtx &D = *Dp;
    struct Running { int slot; Job *job; bool submitted; };
    std::deque<Running> running;  // oldest first
    int next_slot = 0;
    auto finish_oldest = [&] {
        finish_job(H, D, running.front().slot, running.front().job, running.front().submitted);
        running.pop_front();
    };
    for (;;) {
        Job *j = nullptr;
        bool stale = false;
        {
            std::unique_lock<std::mutex> lock(H.mu);
            if (running.empty()) H.cv_queue.wait(lock, [&] { return !D.queue.empty(); });
            if (!D.queue.empty() && (int)running.size() < kSlotsPerDevice) {
                j = D.queue.front();
                D.queue.pop_front();
                stale = D.batch_box_stale;
                D.batch_box_stale = false;
            }
        }
        if (j) {
            int jw = 0, jh = 0;  // the encoder is sized for the job's largest picture
            for (int k = 0; k < j->reserved; k++) {
                jw = std::max(jw, j->ws[k]);
                jh = std::max(jh, j->hs[k]);
            }
            // a geometry or batch size the encoder was not built for (or new settings): everything in flight leaves first
            const bool fits = !stale && D.batch_box.enc && jw <= D.batch_box.max_w && jh <= D.batch_box.max_h && j->cap_frames <= D.batch_box.max_batch;
            if (!fits)
                while (!running.empty()) finish_oldest();
            if (stale) drop_box(D.batch_box);
            bool ok = ensure_box(D.batch_box, D.device, H.range_mode, jw, jh, j->cap_frames, kSlotsPerDevice);
            // pinned room for the batch's JPEGs: 4 bits per pixel to start with (camera pictures at the reference's settings
            // come to about 1 bit); a batch that needs more is collected again into a buffer of exactly its size (finish_job)
            size_t out_guess = 0;
            for (int k = 0; k < j->reserved; k++) out_guess += std::min((size_t)j->ws[k] * j->hs[k] / 2 + 65536, D.batch_box.cap);
            if (ok && j->out_bytes < out_guess) {
                if (j->out) h2j_free_pinned(j->out);
                j->out_bytes = out_guess;
                j->out = static_cast<uint8_t *>(h2j_alloc_pinned(j->out_bytes));
                if (!j->out) {
                    LOG("%s line=%d | pinned allocation of %zu bytes failed", __PRETTY_FUNCTION__, __LINE__, j->out_bytes);
                    j->out_bytes = 0;
                    ok = false;
                }
            }
            const int slot = next_slot;
            if (ok) {
                std::vector<const uint8_t *> pics(j->reserved);
                for (int k = 0; k < j->reserved; k++) pics[k] = j->in + j->at[k];
                const int rc = h2j_submit_host_list(D.batch_box.enc, slot, pics.data(), j->ws.data(), j->hs.data(), j->reserved);
                if (rc != H2J_OK) {
                    LOG("h2j_submit_host of %d frames failed, rc=%d (%s), error=%s", j->reserved, rc, h2j_status_string(rc), h2j_last_error(D.batch_box.enc));
                    ok = false;
                } else next_slot = (next_slot + 1) % kSlotsPerDevice;
            }
            running.push_back(Running{slot, j, ok});
            // another batch is already waiting and a slot is free: it is enqueued behind this one before anything is collected
            bool more;
            {
                std::lock_guard<std::mutex> lock(H.mu);
                more = !D.queue.empty() && (int)running.size() < kSlotsPerDevice;
            }
            if (more) continue;
        }
        if (!running.empty()) finish_oldest();
    }
}

// (H.mu held) hand a complete job to a device: the least loaded of the devices already running, a new device when all
// of those have their two batches in flight and the configuration allows another one
void route_job(Hub &H, Job *j)
{
    const int n_allowed = allowed_devices(H);
    int best = -1;
    for (int i = 0; i < (int)H.devices.size() && i < n_allowed; i++)
        if (H.devices[i]->worker_started && (best < 0 || H.devices[i]->inflight < H.devices[best]->inflight)) best = i;
    if (best < 0 || H.devices[best]->inflight >= kSlotsPerDevice) {
        for (int i = 0; i < n_allowed; i++) {
            DeviceCtx &D = device_at(H, i);
            if (!D.worker_started) {
                D.worker_started = true;
                std::thread(worker_main, &H, &D).detach();
                best = i;
                break;
            }
        }
    }
    DeviceCtx &D = *H.devices[best];
    H.batches++;
    D.queue.push_back(j);
    D.inflight++;
    H.cv_queue.notify_all();
}

// (H.mu held) nobody will add to the job any more; it leaves as soon as every reserved picture has been copied in
void seal_job(Hub &H, Job *j)
{
    j->sealed = true;
    if (H.filling == j) H.filling = nullptr;
    if (j->filled == j->reserved) {
        if (j->reserved > 0) route_job(H, j);
        else {
            j->busy = false;
            H.cv_jobs.notify_all();
        }
    }
}

// (lock held) give a job that is being filled room for `cap_frames` pictures of H.room bytes.  Only while no copy into it is
// in progress (filled == reserved): the pictures already in are moved over.
bool grow_job(Hub &H, Job *j)
{
    const size_t bytes = H.room * (size_t)j->cap_frames;
    if (j->filled != j->reserved || bytes <= j->in_bytes) return false;
    uint8_t *p = static_cast<uint8_t *>(h2j_alloc_pinned(bytes));
    if (!p) return false;
    if (j->used) memcpy(p, j->in, j->used);
    h2j_free_pinned(j->in);
    j->in = p;
    j->in_bytes = bytes;
    return true;
}

// (lock held on entry and exit) a job with room for a w x h picture: the one being filled (pictures of any sizes share a
// job), or a free one (re-cut if it was made for smaller pictures), or a new one while fewer than two per device plus one
// exist; otherwise wait for one
Job *job_for(Hub &H, std::unique_lock<std::mutex> &lock, int w, int h, size_t need)
{
    if (need > H.room) H.room = need;
    for (;;) {
        if (H.filling) {
            Job *j = H.filling;
            if (j->used + need <= j->in_bytes || grow_job(H, j)) return j;
            seal_job(H, j);  // no pinned room left for this picture: it goes as it is
        }
        Job *free_job = nullptr;
        for (auto &jp : H.jobs)
            if (!jp->busy) {
                free_job = jp.get();
                break;
            }
        const size_t max_jobs = (size_t)kSlotsPerDevice * allowed_devices(H) + 1;
        if (!free_job && H.jobs.size() < max_jobs) {
            H.jobs.emplace_back(new Job());
            free_job = H.jobs.back().get();
        }
        if (!free_job) {
            H.cv_jobs.wait(lock);
            continue;
        }
        Job *j = free_job;
        j->busy = true;
        if (j->in_bytes < H.room * (size_t)H.batch_frames) {
            if (j->in) h2j_free_pinned(j->in);
            j->in_bytes = H.room * (size_t)H.batch_frames;
            j->in = static_cast<uint8_t *>(h2j_alloc_pinned(j->in_bytes));
            if (!j->in) {
                LOG("%s line=%d | pinned allocation of %zu bytes failed", __PRETTY_FUNCTION__, __LINE__, j->in_bytes);
                j->in_bytes = 0;
                j->busy = false;
                return nullptr;
            }
        }
        j->used = 0;
        j->at.clear();
        j->ws.clear();
        j->hs.clear();
        j->cap_frames = H.batch_frames;
        j->reserved = j->filled = 0;
        j->sealed = false;
        j->paths.clear();
        H.filling = j;
        return j;
    }
}

// A picture arrives inside a batch scope: reserve a place, copy the planes (the only host-side touch of the pixels,
// outside the lock so that callers on several threads copy side by side), hand the batch over when it is complete.
bool enqueue_frame(Hub &H, const H2JFrameView &f, const char *path)
{
    std::unique_lock<std::mutex> lock(H.mu);
    if (!H.batching) return false;
    const size_t need = (i420_bytes(f.width, f.height) + 255) / 256 * 256;
    Job *j = job_for(H, lock, f.width, f.height, need);
    if (!j) return false;
    j->reserved++;
    const size_t at = j->used;
    j->used += need;
    j->at.push_back(at);
    j->ws.push_back(f.width);
    j->hs.push_back(f.height);
    j->paths.emplace_back(path);
    if (j->reserved == j->cap_frames) {  // full: the next picture opens another job
        j->sealed = true;
        H.filling = nullptr;
    }
    lock.unlock();
    copy_planes(j->in + at, f);
    lock.lock();
    j->filled++;
    if (j->sealed && j->filled == j->reserved) route_job(H, j);
    return true;
}

// (lock held) every job idle
void drain(Hub &H, std::unique_lock<std::mutex> &lock)
{
    if (H.filling) seal_job(H, H.filling);
    H.cv_jobs.wait(lock, [&] {
        for (auto &jp : H.jobs)
            if (jp->busy) return false;
        return true;
    });
}

}  // namespace

extern "C" int h2j_host_batch_begin(int max_frames)
{
    Hub &H = hub();
    std::lock_guard<std::mutex> lock(H.mu);
    if (H.batching || max_frames < 1) return -1;
    H.batching = true;
    H.batch_frames = max_frames;
    H.written = H.failed = 0;
    H.room = 0;
    H.batches = 0;
    return 0;
}

extern "C" int h2j_host_batch_end(int *failed)
{
    Hub &H = hub();
    std::unique_lock<std::mutex> lock(H.mu);
    if (!H.batching) return -1;
    drain(H, lock);
    H.batching = false;
    if (failed) *failed = H.failed;
    return H.written;
}

extern "C" void h2j_host_configure(int cuda_device, int range_mode)
{
    Hub &H = hub();
    std::unique_lock<std::mutex> lock(H.mu);
    drain(H, lock);
    // the workers sit idle on their empty queues: their encoders are rebuilt by them before the next batch
    for (size_t i = 0; i < H.devices.size(); i++) {
        DeviceCtx &d = *H.devices[i];
        std::lock_guard<std::mutex> sl(d.sync_mu);
        drop_box(d.sync_box);
        d.batch_box_stale = true;
        d.device = cuda_device >= 0 ? cuda_device : (int)i;
    }
    H.only_device = cuda_device >= 0 ? cuda_device : -1;
    H.range_mode = range_mode;
}

extern "C" int h2j_host_batches_submitted(void)
{
    Hub &H = hub();
    std::lock_guard<std::mutex> lock(H.mu);
    return H.batches;
}

extern "C" int h2j_host_devices_in_use(void)
{
    Hub &H = hub();
    std::lock_guard<std::mutex> lock(H.mu);
    int n = 0;
    for (auto &d : H.devices) n += (d->sync_box.enc || (d->batch_box.enc && !d->batch_box_stale)) ? 1 : 0;
    return n;
}

Encoder::Encoder(const char *const outputFilePath) { this->outputFilePath = outputFilePath; }

Encoder::~Encoder() { release(); }

void Encoder::release()
{
    if (outputFilePath) outputFilePath = nullptr;
}

#ifdef H2J_WITH_LIBAV
bool Encoder::yuv2Jpeg(AVFrame *pFrame)
{
    if (!pFrame) {
        LOG("%s line=%d | null frame", __PRETTY_FUNCTION__, __LINE__);
        release();
        return false;
    }
    H2JFrameView v;
    for (int i = 0; i < 3; i++) {
        v.data[i] = pFrame->data[i];
        v.linesize[i] = pFrame->linesize[i];
    }
    v.width = pFrame->width;
    v.height = pFrame->height;
    v.format = pFrame->format;
    return yuv2Jpeg(v);
}
#else
bool Encoder::yuv2Jpeg(AVFrame *)
{
    LOG("%s | built without libavutil headers (H2J_WITH_LIBAV); use yuv2Jpeg(const H2JFrameView&)", __PRETTY_FUNCTION__);
    release();
    return false;
}
#endif

bool Encoder::yuv2Jpeg(const H2JFrameView &f)
{
    // The reference feeds whatever the decoder produced to an encoder opened as YUVJ420P (src/Encoder.cpp:162);
    // anything but 8-bit 4:2:0 planar would be read as garbage there.  Here 10 / 12-bit 4:2:0 (Main10 / Main12 streams) is
    // encoded from its 8-bit truncation (include/h2j_b200.h, h2j_encode_frame16); everything else is refused.
    const int bit_depth = f.format == kFmtYuv420p10le ? 10 : (f.format == kFmtYuv420p12le ? 12 : 8);
    if (bit_depth == 8 && f.format != 0 /* AV_PIX_FMT_YUV420P */ && f.format != 12 /* AV_PIX_FMT_YUVJ420P */) {
        LOG("%s line=%d | unsupported pixel format %d (need yuv420p / yuvj420p / yuv420p10le / yuv420p12le)", __PRETTY_FUNCTION__, __LINE__,
            f.format);
        release();
        return false;
    }
    if (!f.data[0] || !f.data[1] || !f.data[2] || f.width < 2 || f.height < 2) {
        LOG("%s line=%d | bad frame: %dx%d", __PRETTY_FUNCTION__, __LINE__, f.width, f.height);
        release();
        return false;
    }
    Hub &H = hub();
    DeviceCtx *D = nullptr;
    std::unique_lock<std::mutex> dev_lock;
    int range_mode;
    {
        std::unique_lock<std::mutex> lock(H.mu);
        if (H.batching && bit_depth == 8) {  // (high-bit-depth pictures take the synchronous path below)
            // batch scope: the picture is queued; it is encoded and its file written when its batch is complete or the scope ends
            if (this->outputFilePath == nullptr || strlen(this->outputFilePath) == 0) {
                LOG("Jpeg 文件路径为空，请核查！");
                return false;
            }
            lock.unlock();
            const bool queued = enqueue_frame(H, f, this->outputFilePath);
            release();
            return queued;
        }
        // synchronous path: a device nobody is encoding on; all of them busy -> the next device comes up; none left -> this
        // thread waits its turn on one of them
        const int n_allowed = allowed_devices(H);
        for (int i = 0; i < n_allowed && !D; i++) {
            DeviceCtx &C = device_at(H, i);
            std::unique_lock<std::mutex> tl(C.sync_mu, std::try_to_lock);
            if (tl.owns_lock()) {
                D = &C;
                dev_lock = std::move(tl);
            }
        }
        if (!D) D = &device_at(H, (int)(H.turn++ % (unsigned)n_allowed));
        range_mode = H.range_mode;
    }
    if (!dev_lock.owns_lock()) dev_lock = std::unique_lock<std::mutex>(D->sync_mu);
    if (!ensure_box(D->sync_box, D->device, range_mode, f.width, f.height, 1, 1)) {
        release();
        return false;
    }
    if (jpegCap_ < D->sync_box.cap) {
        jpeg_.reset(new (std::nothrow) uint8_t[D->sync_box.cap]);
        jpegCap_ = jpeg_ ? D->sync_box.cap : 0;
    }
    if (!jpeg_) {
        LOG("%s line=%d | malloc failed.", __PRETTY_FUNCTION__, __LINE__);
        release();
        return false;
    }
    const uint8_t *planes[3] = {f.data[0], f.data[1], f.data[2]};
    const int strides[3] = {f.linesize[0], f.linesize[1], f.linesize[2]};
    jpegSize_ = 0;
    const int rc = bit_depth == 8 ? h2j_encode_frame(D->sync_box.enc, planes, strides, f.width, f.height, jpeg_.get(), jpegCap_, &jpegSize_)
                                  : h2j_encode_frame16(D->sync_box.enc, planes, strides, bit_depth, f.width, f.height, jpeg_.get(), jpegCap_, &jpegSize_);
    if (rc != H2J_OK) {
        LOG("h2j_encode_frame%s failed, rc=%d (%s), error=%s", bit_depth == 8 ? "" : "16", rc, h2j_status_string(rc), h2j_last_error(D->sync_box.enc));
        release();
        return false;
    }
    dev_lock.unlock();  // the file is written outside the device's lock: the next picture is already encoding
    const bool isOk = saveJpegtoFile(this->outputFilePath);
    if (!isOk) {
        LOG("%s line=%d | 保存 Jpeg 文件出错！Jpeg 文件路径：%s", __PRETTY_FUNCTION__, __LINE__, this->outputFilePath);
        return false;
    }
    release();
    return true;
}

bool Encoder::saveJpegtoFile(const char *const filePath) { return save_jpeg(filePath, jpeg_.get(), jpegSize_); }
