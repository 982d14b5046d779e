// server.cc — in-process multi-model, multi-GPU dispatcher behind the reference's perform() call shape.
//
// The reference shares ONE detector object per model spec across all sessions (server/server.py:295,311-312: the
// `detectors` dict handed to every RTSPService) and serves every payload with one blocking
// `detector.perform(data, threshold)` (server/server.py:232) from a single select loop (:156-163), so all streams of a
// model queue behind batch-1 latency on one device.  Here every (device, model) pair is a LANE: a replica of the model on
// that device (its own streams, execution state and captured graphs), a worker thread, and a queue of micro-batches.
// A stream is pinned to a device (stream_id mod devices: per-stream ordering, no cross-GPU traffic — frames are
// independent, SURVEY 8e), its blocking fd_server_perform() call copies the frame straight into the open batch's pinned
// buffer (the copies of concurrent callers run in parallel, in the callers' threads) and sleeps until the batch's
// records are back.  The worker keeps two batches in flight per lane through fd_submit / fd_collect, so the
// host->device copy and the entropy of forming the next batch overlap the conv stack of the previous one, and — like
// fastdet_b200/service.py — never waits for more requests while the device has work: whatever has arrived when a slot
// frees up is the next batch.
// JPEG payloads (fd_server_perform_jpeg, the reference's own request) ride JPEG batches: each caller parses its payload and
// entropy-decodes it straight into its place in the batch's pinned buffer, again in parallel in the callers' threads; the
// worker submits the batch to the device half of fd_submit_jpeg (IDCT + colour on the device, then the forward pass).  The
// threshold is per frame in a JPEG batch, so requests with different thresholds share it; an RGB batch keeps one threshold.
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/fastdet_b200.h"
#include "jpeg.h"
#include "options.h"

void* fd_internal_pinned_alloc(int device, size_t bytes);  // capi.cu
void fd_internal_pinned_free(int device, void* p);
int fd_internal_submit_jpeg(fd_model* m, int slot, const uint8_t* pinned, int n, int cap, size_t stride, const double* thresholds,
                            int max_det);

namespace {

using Clock = std::chrono::steady_clock;

thread_local char g_serr[512] = "";

struct Backend {  // what a lane drives: the two-slot submit / collect pair of one model replica
    int w = 0, h = 0, device = 0;
    virtual ~Backend() {}
    virtual int submit(int slot, const uint8_t* frames, int n, double thr, int max_det) = 0;
    // a JPEG batch laid out as fd_internal_submit_jpeg takes it; frame f at threshold thr[f]
    virtual int submit_jpeg(int slot, const uint8_t* pinned, int n, int cap, size_t stride, const double* thr, int max_det) = 0;
    virtual int collect(int slot, fd_det* out, int32_t* counts) = 0;
    virtual uint8_t* alloc_pinned(size_t bytes) = 0;
    virtual void free_pinned(uint8_t* p) = 0;
};

struct ModelBackend : Backend {
    fd_model* m = nullptr;
    ~ModelBackend() override { fd_model_destroy(m); }
    int submit(int slot, const uint8_t* frames, int n, double thr, int max_det) override {
        return fd_submit(m, slot, frames, n, w, h, 0, 0, thr, max_det);
    }
    int submit_jpeg(int slot, const uint8_t* pinned, int n, int cap, size_t stride, const double* thr, int max_det) override {
        return fd_internal_submit_jpeg(m, slot, pinned, n, cap, stride, thr, max_det);
    }
    int collect(int slot, fd_det* out, int32_t* counts) override { return fd_collect(m, slot, out, counts, nullptr); }
    // (under the device's set-up lock: a pinned allocation must not run into another lane's graph capture, capi.cu)
    uint8_t* alloc_pinned(size_t bytes) override { return static_cast<uint8_t*>(fd_internal_pinned_alloc(device, bytes)); }
    void free_pinned(uint8_t* p) override { fd_internal_pinned_free(device, p); }
};

// Host-only stand-in (tests of the routing / batching logic on machines without a GPU): "detects" one box per frame
// that records where and how the frame was served: klass = first byte of the frame, box = batch size it rode in,
// conf = device, x = model index, y = slot.  JPEG frames (decoded by the real host half): klass = the first quantised
// luma DC coefficient, w = the frame's threshold.
struct FakeBackend : Backend {
    int model = 0, latency_us = 0;
    struct Held { std::vector<int> first; std::vector<double> thr; int n = 0, slot = 0; } held[FD_MAX_SLOTS];
    int submit(int slot, const uint8_t* frames, int n, double, int) override {
        held[slot].first.resize(n);
        held[slot].thr.assign(n, 0.0);
        for (int i = 0; i < n; ++i) held[slot].first[i] = frames[static_cast<size_t>(i) * w * h * 3];
        held[slot].n = n;
        held[slot].slot = slot;
        return FD_OK;
    }
    int submit_jpeg(int slot, const uint8_t* pinned, int n, int cap, size_t stride, const double* thr, int) override {
        held[slot].first.resize(n);
        held[slot].thr.assign(thr, thr + n);
        for (int i = 0; i < n; ++i)
            held[slot].first[i] = *reinterpret_cast<const int16_t*>(pinned + fd::jpeg_head_bytes(cap) + static_cast<size_t>(i) * stride);
        held[slot].n = n;
        held[slot].slot = slot;
        return FD_OK;
    }
    int collect(int slot, fd_det* out, int32_t* counts) override {
        if (latency_us) std::this_thread::sleep_for(std::chrono::microseconds(latency_us));
        for (int i = 0; i < held[slot].n; ++i) {
            counts[i] = 1;
            fd_det& d = out[static_cast<size_t>(i) * max_det];
            memset(&d, 0, sizeof(d));
            d.klass = held[slot].first[i]; d.box = held[slot].n; d.conf = device; d.x = model; d.y = slot; d.w = held[slot].thr[i];
        }
        return FD_OK;
    }
    uint8_t* alloc_pinned(size_t bytes) override { return new uint8_t[bytes]; }
    void free_pinned(uint8_t* p) override { delete[] p; }
    int max_det = 1;
};

struct Batch {
    enum Kind { RGB, JPEG } kind = RGB;
    uint8_t* pinned = nullptr;  // RGB: frames [cap][h][w][3]; JPEG: [JpegFrameDev x cap], then coefficients at Lane::jpeg_stride
    int cap = 0;                // frames the pinned buffer holds
    int n = 0;                  // frames claimed by callers
    std::atomic<int> ready{0};  // frames copied (RGB) or entropy-decoded (JPEG) in
    double threshold = 0.0;     // RGB: the batch's threshold
    std::vector<double> thr;    // JPEG: [cap] each frame's threshold
    Clock::time_point t_first;
    std::vector<fd_det> dets;
    std::vector<int32_t> counts;
    int rc = FD_OK;
    std::string err;
    bool done = false;
    int waiting = 0;  // callers that have not picked up their result yet
    int slot = -1;
};

struct Lane {
    std::unique_ptr<Backend> be;
    int max_batch = 64, max_det = 256;
    double max_delay_s = 0.0;
    size_t frame_bytes = 0;
    size_t jpeg_stride = 0;  // coefficient bytes per frame of a JPEG batch (a network-sized 4:4:4 frame)
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    Batch* open = nullptr;
    std::deque<Batch*> closed, inflight;
    std::vector<Batch*> pool, all;
    int max_inflight = FD_MAX_SLOTS;  // batches in flight (option server_inflight)
    int cur_cap = 8;  // pinned frames per new batch: doubles (up to max_batch) whenever a batch fills up, so a lane's pinned
                      // footprint follows its load instead of being max_batch x 0.5 MB per batch from the start
    bool stop = false;
    std::thread worker;
    int64_t batches = 0, frames = 0;

    size_t pinned_bytes(Batch::Kind kind, int cap) const {
        return kind == Batch::RGB ? frame_bytes * cap : fd::jpeg_head_bytes(cap) + jpeg_stride * cap;
    }

    Batch* fresh(Batch::Kind kind) {  // mu held; nullptr when pinned memory cannot be had
        Batch* b = nullptr;
        for (size_t i = 0; i < pool.size(); ++i)
            if (pool[i]->kind == kind && pool[i]->cap >= cur_cap) { b = pool[i]; pool.erase(pool.begin() + i); break; }
        if (!b) {
            if (!pool.empty()) {  // recycle an object whose buffer has become too small
                b = pool.back(); pool.pop_back();
                be->free_pinned(b->pinned);
                b->pinned = nullptr; b->cap = 0;
            } else {
                b = new Batch();
                all.push_back(b);
            }
            b->kind = kind;
            b->pinned = be->alloc_pinned(pinned_bytes(kind, cur_cap));
            if (!b->pinned) { pool.push_back(b); return nullptr; }
            b->cap = cur_cap;
            b->dets.resize(static_cast<size_t>(b->cap) * max_det);
            b->counts.resize(b->cap);
            b->thr.resize(b->cap);
        }
        b->n = 0; b->ready.store(0); b->rc = FD_OK; b->err.clear(); b->done = false; b->waiting = 0; b->slot = -1;
        return b;
    }

    void run() {
        std::unique_lock<std::mutex> lk(mu);
        bool slot_busy[FD_MAX_SLOTS] = {false, false};
        for (;;) {
            if (static_cast<int>(inflight.size()) < max_inflight) {
                Batch* b = nullptr;
                if (!closed.empty()) { b = closed.front(); closed.pop_front(); }
                else if (open && open->n > 0) {
                    // nothing in flight: a short wait lets concurrent callers share the batch; with work in flight the
                    // device is the clock — whatever has arrived when a slot is free goes
                    if (inflight.empty() && max_delay_s > 0.0 && !stop) {
                        const double age = std::chrono::duration<double>(Clock::now() - open->t_first).count();
                        if (age < max_delay_s && open->n < open->cap) {
                            cv_work.wait_for(lk, std::chrono::duration<double>(max_delay_s - age));
                            continue;
                        }
                    }
                    b = open;
                    open = nullptr;
                }
                if (b) {
                    int slot = slot_busy[0] ? 1 : 0;
                    slot_busy[slot] = true;
                    b->slot = slot;
                    const int n = b->n;
                    lk.unlock();
                    // a caller is still copying its frame in (RGB: microseconds) or entropy-decoding it (JPEG: a millisecond or more)
                    while (b->ready.load(std::memory_order_acquire) < n) {
                        if (b->kind == Batch::JPEG) std::this_thread::sleep_for(std::chrono::microseconds(20));
                        else std::this_thread::yield();
                    }
                    const int rc = b->kind == Batch::JPEG ? be->submit_jpeg(slot, b->pinned, n, b->cap, jpeg_stride, b->thr.data(), max_det)
                                                          : be->submit(slot, b->pinned, n, b->threshold, max_det);
                    std::string err = rc ? fd_last_error() : "";
                    lk.lock();
                    ++batches; frames += n;
                    if (rc) {
                        slot_busy[slot] = false;
                        b->rc = rc; b->err = err; b->done = true;
                        cv_done.notify_all();
                    } else {
                        inflight.push_back(b);
                    }
                    continue;
                }
            }
            if (!inflight.empty()) {
                Batch* b = inflight.front();
                inflight.pop_front();
                lk.unlock();
                const int rc = be->collect(b->slot, b->dets.data(), b->counts.data());
                std::string err = rc ? fd_last_error() : "";
                lk.lock();
                slot_busy[b->slot] = false;
                b->rc = rc; b->err = err; b->done = true;
                cv_done.notify_all();
                continue;
            }
            if (stop) return;
            cv_work.wait(lk);
        }
    }

    // A caller's place in the open batch of `kind`: the open batch is closed first when it is full or of the other kind, or
    // (RGB, whose batches hold one threshold) has another threshold.  Returns nullptr when pinned memory cannot be had.
    Batch* claim(Batch::Kind kind, double threshold, int* idx) {
        std::unique_lock<std::mutex> lk(mu);
        if (open && (open->n >= open->cap || open->kind != kind || (kind == Batch::RGB && open->threshold != threshold))) {
            closed.push_back(open);
            open = nullptr;
        }
        if (!open) {
            open = fresh(kind);
            if (!open) return nullptr;
            open->threshold = threshold;
            open->t_first = Clock::now();
        }
        Batch* b = open;
        *idx = b->n++;
        ++b->waiting;
        b->thr[*idx] = threshold;
        if (b->n >= b->cap) {  // full: it goes as it is, and the next batches get more room
            if (b->cap < max_batch) cur_cap = std::min(max_batch, 2 * b->cap);
            closed.push_back(b);
            open = nullptr;
        }
        lk.unlock();
        cv_work.notify_one();
        return b;
    }

    // Sleeps until the batch is back, then copies frame idx's records out (none when out is null) and lets go of the batch.
    int await(Batch* b, int idx, fd_det* out, int out_max, int32_t* count) {
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return b->done; });
        const int rc = b->rc;
        if (rc == FD_OK && out) {
            const int c = std::min<int>(b->counts[idx], out_max);
            *count = c;
            memcpy(out, b->dets.data() + static_cast<size_t>(idx) * max_det, sizeof(fd_det) * static_cast<size_t>(c));
        } else if (rc != FD_OK) {
            snprintf(g_serr, sizeof(g_serr), "%s", b->err.c_str());
        }
        if (--b->waiting == 0) pool.push_back(b);
        return rc;
    }
};

int sfail(int code, const char* msg) {
    snprintf(g_serr, sizeof(g_serr), "%s", msg);
    return code;
}

}  // namespace

struct fd_server {
    int n_models = 0, n_devices = 0, max_det = 256;
    std::vector<std::unique_ptr<Lane>> lanes;  // [device][model]
    std::vector<int> net_w, net_h;
    std::atomic<bool> closing{false};
    Lane& lane(int dev_slot, int model) { return *lanes[static_cast<size_t>(dev_slot) * n_models + model]; }
};

namespace {

void start_lanes(fd_server* s) {
    for (auto& l : s->lanes) l->worker = std::thread([p = l.get()] { p->run(); });
}

}  // namespace

extern "C" {

const char* fd_server_last_error(void) { return g_serr[0] ? g_serr : fd_last_error(); }

int fd_server_create(const fd_server_model* models, int n_models, const int32_t* devices, int n_devices, int max_batch, int max_det,
                     double max_delay_ms, fd_server** out) {
    if (!models || !devices || !out || n_models < 1 || n_models > FD_SERVER_MAX_MODELS || n_devices < 1 || n_devices > FD_SERVER_MAX_DEVICES ||
        max_batch < 1 || max_det < 1)
        return sfail(FD_ERR_ARG, "fd_server_create: bad argument");
    g_serr[0] = 0;
    *out = nullptr;
    std::unique_ptr<fd_server> s(new fd_server());
    s->n_models = n_models; s->n_devices = n_devices; s->max_det = max_det;
    for (int m = 0; m < n_models; ++m) { s->net_w.push_back(models[m].net_w); s->net_h.push_back(models[m].net_h); }
    for (int d = 0; d < n_devices; ++d)
        for (int m = 0; m < n_models; ++m) {
            std::unique_ptr<ModelBackend> be(new ModelBackend());
            be->w = models[m].net_w; be->h = models[m].net_h; be->device = devices[d];
            if (int rc = fd_model_create(models[m].onnx_bytes, models[m].len, models[m].num_classes, models[m].net_w, models[m].net_h, devices[d], &be->m))
                return rc;  // fd_last_error() holds the reason; lanes built so far are destroyed with `s`
            std::unique_ptr<Lane> l(new Lane());
            l->max_batch = max_batch; l->max_det = max_det; l->max_delay_s = max_delay_ms * 1e-3; l->cur_cap = std::min(8, max_batch);
            l->max_inflight = std::max(1, std::min<int>(FD_MAX_SLOTS, fd::options().server_inflight));
            l->frame_bytes = static_cast<size_t>(be->w) * be->h * 3;
            l->jpeg_stride = fd::jpeg_frame_stride(be->w, be->h);
            l->be = std::move(be);
            s->lanes.push_back(std::move(l));
        }
    start_lanes(s.get());
    *out = s.release();
    return FD_OK;
}

int fd_server_create_fake(int n_models, int n_devices, int net_w, int net_h, int max_batch, double max_delay_ms, int latency_us, fd_server** out) {
    if (!out || n_models < 1 || n_models > FD_SERVER_MAX_MODELS || n_devices < 1 || n_devices > FD_SERVER_MAX_DEVICES || max_batch < 1)
        return sfail(FD_ERR_ARG, "fd_server_create_fake: bad argument");
    std::unique_ptr<fd_server> s(new fd_server());
    s->n_models = n_models; s->n_devices = n_devices; s->max_det = 1;
    for (int m = 0; m < n_models; ++m) { s->net_w.push_back(net_w); s->net_h.push_back(net_h); }
    for (int d = 0; d < n_devices; ++d)
        for (int m = 0; m < n_models; ++m) {
            std::unique_ptr<FakeBackend> be(new FakeBackend());
            be->w = net_w; be->h = net_h; be->device = d; be->model = m; be->latency_us = latency_us;
            std::unique_ptr<Lane> l(new Lane());
            l->max_batch = max_batch; l->max_det = 1; l->max_delay_s = max_delay_ms * 1e-3; l->cur_cap = std::min(8, max_batch);
            l->max_inflight = std::max(1, std::min<int>(FD_MAX_SLOTS, fd::options().server_inflight));
            l->frame_bytes = static_cast<size_t>(net_w) * net_h * 3;
            l->jpeg_stride = fd::jpeg_frame_stride(net_w, net_h);
            l->be = std::move(be);
            s->lanes.push_back(std::move(l));
        }
    start_lanes(s.get());
    *out = s.release();
    return FD_OK;
}

void fd_server_destroy(fd_server* s) {
    if (!s) return;
    s->closing.store(true);
    for (auto& l : s->lanes) {
        { std::lock_guard<std::mutex> g(l->mu); l->stop = true; }
        l->cv_work.notify_all();
    }
    for (auto& l : s->lanes)
        if (l->worker.joinable()) l->worker.join();
    for (auto& l : s->lanes) {
        for (Batch* b : l->all) { if (b->pinned) l->be->free_pinned(b->pinned); delete b; }
        l->be.reset();
    }
    delete s;
}

int fd_server_perform(fd_server* s, int stream_id, int model, const uint8_t* frame, int src_w, int src_h, double threshold, fd_det* out,
                      int max_det, int32_t* count) {
    if (!s || !frame || !out || !count || stream_id < 0 || model < 0 || model >= s->n_models || max_det < 1)
        return sfail(FD_ERR_ARG, "fd_server_perform: bad argument");
    if (src_w != s->net_w[model] || src_h != s->net_h[model]) return sfail(FD_ERR_SIZE, "invalid image size");  // reference detector.py:132
    if (s->closing.load()) return sfail(FD_ERR_ARG, "fd_server_perform: server is shutting down");
    Lane& L = s->lane(stream_id % s->n_devices, model);
    int idx;
    Batch* b = L.claim(Batch::RGB, threshold, &idx);
    if (!b) return sfail(FD_ERR_CUDA, "fd_server_perform: pinned host memory for a micro-batch could not be allocated");
    memcpy(b->pinned + static_cast<size_t>(idx) * L.frame_bytes, frame, L.frame_bytes);  // in the caller's thread: concurrent callers copy in parallel
    b->ready.fetch_add(1, std::memory_order_release);
    return L.await(b, idx, out, max_det, count);
}

int fd_server_perform_jpeg(fd_server* s, int stream_id, int model, const uint8_t* data, size_t len, double threshold, fd_det* out,
                           int max_det, int32_t* count, int32_t* status) {
    int32_t st_local = 0;
    int32_t& st = status ? *status : st_local;
    st = FD_JPEG_OK;
    if (!s || !data || !out || !count || stream_id < 0 || model < 0 || model >= s->n_models || max_det < 1)
        return sfail(FD_ERR_ARG, "fd_server_perform_jpeg: bad argument");
    std::unique_ptr<fd::JpegInfo> J(new fd::JpegInfo());
    char why[160] = "";
    st = fd::jpeg_parse(data, len, J.get(), why, sizeof(why));
    if (st != fd::JPEG_OK) {
        snprintf(g_serr, sizeof(g_serr), "%s (status %d)", why, st);
        return FD_ERR_JPEG;
    }
    if (J->width != s->net_w[model] || J->height != s->net_h[model]) {  // reference detector.py:132
        st = FD_JPEG_SIZE;
        return sfail(FD_ERR_SIZE, "invalid image size");
    }
    if (s->closing.load()) return sfail(FD_ERR_ARG, "fd_server_perform_jpeg: server is shutting down");
    Lane& L = s->lane(stream_id % s->n_devices, model);
    if (fd::jpeg_coef_count(*J) * sizeof(int16_t) > L.jpeg_stride) {  // (the sampling factors jpeg_parse takes always fit)
        st = FD_JPEG_UNSUPPORTED;
        return sfail(FD_ERR_JPEG, "fd_server_perform_jpeg: coefficients exceed the batch's per-frame stride");
    }
    int idx;
    Batch* b = L.claim(Batch::JPEG, threshold, &idx);
    if (!b) return sfail(FD_ERR_CUDA, "fd_server_perform_jpeg: pinned host memory for a micro-batch could not be allocated");
    // in the caller's thread: concurrent callers entropy-decode in parallel.  The descriptor comes from the header alone, so a
    // frame whose entropy data is damaged still rides the batch (its caller gets no records)
    const size_t off = static_cast<size_t>(idx) * L.jpeg_stride;
    const int dst = fd::jpeg_decode_coefficients(data, len, *J, reinterpret_cast<int16_t*>(b->pinned + fd::jpeg_head_bytes(b->cap) + off),
                                                 why, sizeof(why));
    fd::jpeg_frame_desc(*J, off / sizeof(int16_t), reinterpret_cast<fd::JpegFrameDev*>(b->pinned) + idx);
    b->ready.fetch_add(1, std::memory_order_release);
    const int rc = L.await(b, idx, dst == fd::JPEG_OK ? out : nullptr, max_det, count);
    if (rc == FD_OK && dst != fd::JPEG_OK) {
        st = dst;
        snprintf(g_serr, sizeof(g_serr), "%s (status %d)", why, dst);
        return FD_ERR_JPEG;
    }
    return rc;
}

// Builds every lane's execution state (buffers, tensor maps, captured graphs) for the batch-size buckets up to `up_to`
// frames, so that no request ever pays for it (0.1 - 0.8 s per bucket).  Call before serving; lanes are warmed in parallel.
int fd_server_warm(fd_server* s, int up_to) {
    if (!s || up_to < 1) return sfail(FD_ERR_ARG, "fd_server_warm: bad argument");
    std::vector<std::thread> th;
    std::vector<int> rcs(s->lanes.size(), FD_OK);
    std::vector<std::string> errs(s->lanes.size());
    for (size_t li = 0; li < s->lanes.size(); ++li)
        th.emplace_back([&, li] {
            Lane& L = *s->lanes[li];
            const int top = std::min(up_to, L.max_batch);
            uint8_t* buf = L.be->alloc_pinned(L.frame_bytes * top);
            if (!buf) { rcs[li] = FD_ERR_CUDA; errs[li] = "pinned allocation failed"; return; }
            memset(buf, 128, L.frame_bytes * top);
            std::vector<fd_det> dets(static_cast<size_t>(top) * L.max_det);
            std::vector<int32_t> counts(top);
            for (int b = 1;; b *= 2) {
                const int n = std::min(b, top);
                int rc = L.be->submit(0, buf, n, 0.5, L.max_det);
                if (!rc) rc = L.be->collect(0, dets.data(), counts.data());
                if (rc) { rcs[li] = rc; errs[li] = fd_last_error(); break; }
                if (n == top) break;
            }
            L.be->free_pinned(buf);
        });
    for (auto& t : th) t.join();
    for (size_t li = 0; li < rcs.size(); ++li)
        if (rcs[li]) { snprintf(g_serr, sizeof(g_serr), "lane %zu: %s", li, errs[li].c_str()); return rcs[li]; }
    return FD_OK;
}

int fd_server_lane_stats(fd_server* s, int device_slot, int model, int64_t* batches, int64_t* frames) {
    if (!s || device_slot < 0 || device_slot >= s->n_devices || model < 0 || model >= s->n_models) return sfail(FD_ERR_ARG, "fd_server_lane_stats: bad argument");
    Lane& L = s->lane(device_slot, model);
    std::lock_guard<std::mutex> g(L.mu);
    if (batches) *batches = L.batches;
    if (frames) *frames = L.frames;
    return FD_OK;
}

// Closed-loop load: n_streams caller threads, stream i -> model stream_model[i], each sending its next frame as soon as the
// previous result is back (BASELINE config 5: "emitting frames as fast as results return"), for `seconds` after a warm-up.
int fd_server_closed_loop(fd_server* s, int n_streams, const int32_t* stream_model, const uint8_t* frames, int n_frames, int src_w,
                          int src_h, double threshold, double warmup_seconds, double seconds, fd_serve_stats* st) {
    if (!s || !stream_model || !frames || !st || n_streams < 1 || n_frames < 1 || seconds <= 0) return sfail(FD_ERR_ARG, "fd_server_closed_loop: bad argument");
    memset(st, 0, sizeof(*st));
    const size_t frame_bytes = static_cast<size_t>(src_w) * src_h * 3;
    std::vector<std::vector<float>> lat(n_streams);
    std::vector<int> rcs(n_streams, 0);
    std::vector<std::string> errs(n_streams);
    std::vector<int64_t> dets_seen(n_streams, 0);
    int64_t b0 = 0, f0 = 0, b1 = 0, f1 = 0;
    std::atomic<int> phase{0};  // 0 warm-up, 1 measuring, 2 stop
    std::vector<std::thread> th;
    const int max_det = s->max_det;
    for (int i = 0; i < n_streams; ++i)
        th.emplace_back([&, i] {
            std::vector<fd_det> out(max_det);
            int32_t count = 0;
            lat[i].reserve(1 << 16);
            for (int64_t it = 0; phase.load(std::memory_order_relaxed) < 2; ++it) {
                const uint8_t* f = frames + static_cast<size_t>((i * 7 + it) % n_frames) * frame_bytes;
                const auto t0 = Clock::now();
                const int rc = fd_server_perform(s, i, stream_model[i], f, src_w, src_h, threshold, out.data(), max_det, &count);
                const auto t1 = Clock::now();
                if (rc) { rcs[i] = rc; errs[i] = fd_server_last_error(); return; }
                if (phase.load(std::memory_order_relaxed) == 1) {
                    lat[i].push_back(std::chrono::duration<float, std::milli>(t1 - t0).count());
                    dets_seen[i] += count;
                }
            }
        });
    std::this_thread::sleep_for(std::chrono::duration<double>(warmup_seconds));
    for (int d = 0; d < s->n_devices; ++d)
        for (int m = 0; m < s->n_models; ++m) { int64_t b, f; fd_server_lane_stats(s, d, m, &b, &f); b0 += b; f0 += f; }
    const auto t_start = Clock::now();
    phase.store(1);
    std::this_thread::sleep_for(std::chrono::duration<double>(seconds));
    phase.store(2);
    const double elapsed = std::chrono::duration<double>(Clock::now() - t_start).count();
    for (int d = 0; d < s->n_devices; ++d)
        for (int m = 0; m < s->n_models; ++m) { int64_t b, f; fd_server_lane_stats(s, d, m, &b, &f); b1 += b; f1 += f; }
    for (auto& t : th) t.join();
    for (int i = 0; i < n_streams; ++i)
        if (rcs[i]) { snprintf(g_serr, sizeof(g_serr), "stream %d: %s", i, errs[i].c_str()); return rcs[i]; }
    std::vector<float> all;
    for (int i = 0; i < n_streams; ++i) {
        all.insert(all.end(), lat[i].begin(), lat[i].end());
        st->frames_per_device[i % s->n_devices] += static_cast<int64_t>(lat[i].size());
        st->frames_per_model[stream_model[i]] += static_cast<int64_t>(lat[i].size());
        st->detections += dets_seen[i];
    }
    if (all.empty()) return sfail(FD_ERR_ARG, "fd_server_closed_loop: no request completed inside the measured window");
    std::sort(all.begin(), all.end());
    auto pct = [&](double p) { return static_cast<double>(all[std::min(all.size() - 1, static_cast<size_t>(p * all.size()))]); };
    double sum = 0;
    for (float v : all) sum += v;
    st->seconds = elapsed;
    st->frames = static_cast<int64_t>(all.size());
    st->frames_per_second = all.size() / elapsed;
    st->latency_ms_p50 = pct(0.50); st->latency_ms_p90 = pct(0.90); st->latency_ms_p99 = pct(0.99);
    st->latency_ms_mean = sum / all.size(); st->latency_ms_max = all.back();
    st->batches = b1 - b0;
    st->mean_batch = (b1 > b0) ? static_cast<double>(f1 - f0) / (b1 - b0) : 0.0;
    st->streams = n_streams;
    return FD_OK;
}

}  // extern "C"
