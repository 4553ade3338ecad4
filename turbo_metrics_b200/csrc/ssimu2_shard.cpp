// ssimu2_shard.cpp -- frame-sharded scoring across the GPUs of one box, behind the C ABI (include/ssimu2_b200.h,
// "ssimu2_shard_*").
//
// The reference drives ONE GPU from one thread: device 0 is hard-coded in init_cuda
// (crates/turbo-metrics/src/lib.rs:438-456) and the frame loop is crates/turbo-metrics/src/lib.rs:362-433.
// SSIMULACRA2 pairs are independent (crates/ssimulacra2-cuda/README.md:26-27), so the multi-GPU form needs no collective:
// one ssimu2 handle per device, each driven by its own host thread inside this library; the caller keeps a
// single-threaded submit / fetch loop and sees one ordered score stream.  Pair g (global ticket) goes to worker
// (g / batch) % n, so whole launch groups stay on one GPU and consecutive groups rotate over the GPUs.
// Only the public C API of the scorer is used here: no CUDA calls, no torch, no NCCL.
#include "../../include/ssimu2_b200.h"
#include "frame_layout.h"

#include <atomic>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

namespace {

constexpr uint64_t kShardResultCap = 1u << 16;   // global tickets kept in the result ring

struct Job {
    ssimu2_frame ref, dis;
    size_t frame_bytes;    // host frames: bytes to copy (of the reference frame when dis_bytes != 0); 0 = device frames
    size_t dis_bytes;      // host frames of ssimu2_shard_submit_host_sized: bytes of the distorted frame
    void* stream;          // device frames: producer stream on that device
    uint64_t global;       // global ticket
};

struct Worker {
    int32_t device = 0;
    ssimu2_t* h = nullptr;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::deque<Job> queue;
    bool stop = false, flush = false;
    uint64_t want = 0;               // fetch everything below this LOCAL ticket even if its batch is partial
    uint64_t submitted = 0, fetched = 0;   // local tickets
    std::vector<uint64_t> global_of;       // ring: local ticket -> global ticket
    int create_rc = 0;
    bool ready = false;
};

}  // namespace

struct ssimu2_shard {
    ssimu2_config cfg{};
    ssimu2_source dis{};             // the distorted frames' description (has_dis: ssimu2_shard_create_mixed)
    bool has_dis = false;
    uint32_t batch = 0;
    std::vector<Worker*> workers;
    uint64_t next_global = 0;
    std::vector<double> results;
    std::vector<uint8_t> done;
    std::mutex res_mu;
    std::condition_variable res_cv;
    std::atomic<int> error{0};
};

namespace {

void publish(ssimu2_shard* s, const Worker& w, uint64_t local0, uint32_t n, const double* sc)
{
    std::lock_guard<std::mutex> lk(s->res_mu);
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t g = w.global_of[(local0 + i) % w.global_of.size()];
        s->results[g % kShardResultCap] = sc[i];
        s->done[g % kShardResultCap] = 1;
    }
    s->res_cv.notify_all();
}

void fail(ssimu2_shard* s, int rc)
{
    int zero = 0;
    s->error.compare_exchange_strong(zero, rc);
    std::lock_guard<std::mutex> lk(s->res_mu);
    s->res_cv.notify_all();
}

void worker_main(ssimu2_shard* s, Worker* w)
{
    {
        ssimu2_config c = s->cfg;
        c.device = w->device;
        const int rc = ssimu2_create_mixed(&w->h, &c, s->has_dis ? &s->dis : nullptr);
        std::lock_guard<std::mutex> lk(w->mu);
        w->create_rc = rc;
        w->ready = true;
        w->cv.notify_all();
        if (rc) return;
    }
    const uint32_t batch = s->batch;
    const uint64_t ring = s->cfg.ring ? s->cfg.ring : 3;
    std::vector<double> sc(batch);
    std::unique_lock<std::mutex> lk(w->mu);
    for (;;) {
        // what can be done now?
        const uint64_t outstanding = w->submitted - w->fetched;
        const uint64_t full_ready = (w->submitted / batch) * batch;          // local tickets below this sit in complete batches
        const bool can_fetch_full = w->fetched < full_ready;
        const bool must_fetch = w->fetched < w->submitted && (w->flush || w->want > w->fetched);
        if (!w->queue.empty() && outstanding < (uint64_t)batch * ring) {
            // submit ahead while the ring has room
            Job j = w->queue.front();
            w->queue.pop_front();
            w->global_of[w->submitted % w->global_of.size()] = j.global;
            w->submitted++;
            lk.unlock();
            const int rc = j.dis_bytes     ? ssimu2_submit_host_sized(w->h, 1, &j.ref, j.frame_bytes, &j.dis, j.dis_bytes, nullptr)
                           : j.frame_bytes ? ssimu2_submit_host(w->h, &j.ref, &j.dis, j.frame_bytes, nullptr)
                                           : ssimu2_submit(w->h, &j.ref, &j.dis, j.stream, nullptr);
            if (rc) fail(s, rc);
            lk.lock();
            continue;
        }
        if (can_fetch_full || must_fetch) {
            const uint64_t upto = can_fetch_full ? w->fetched + batch - (w->fetched % batch) : w->submitted;
            const uint64_t first = w->fetched;
            const uint32_t n = (uint32_t)((upto < w->submitted ? upto : w->submitted) - first);
            lk.unlock();
            const int rc = ssimu2_get_scores(w->h, first, n, sc.data());
            if (rc) fail(s, rc); else publish(s, *w, first, n, sc.data());
            lk.lock();
            w->fetched = first + n;
            if (w->fetched == w->submitted && w->queue.empty()) w->flush = false;
            continue;
        }
        if (w->stop) break;
        w->cv.wait(lk);
    }
    lk.unlock();
    ssimu2_destroy(w->h);
    w->h = nullptr;
}

// worker index and local ticket of a global ticket
inline void route(const ssimu2_shard* s, uint64_t g, uint32_t* wi, uint64_t* local)
{
    const uint64_t b = g / s->batch, n = s->workers.size();
    *wi = (uint32_t)(b % n);
    *local = (b / n) * s->batch + g % s->batch;
}

int submit_common(ssimu2_shard* s, uint32_t n, const ssimu2_frame* refs, const ssimu2_frame* diss, size_t frame_bytes,
                  size_t dis_bytes, void* const* streams, uint64_t* first_ticket)
{
    if (!s || (n && (!refs || !diss))) return SSIMU2_E_INVALID;
    if (int e = s->error.load()) return e;
    // every frame is checked here, before any is queued: a frame the worker rejected later would fail the whole shard
    const bool host = frame_bytes != 0;
    const int ref_fmt = s->cfg.format, dis_fmt = s->has_dis ? s->dis.format : s->cfg.format;
    // distorted frames at their own size (ssimu2_source.width / height; 0 = the reference's)
    const uint32_t dis_w = s->has_dis && s->dis.width ? s->dis.width : s->cfg.width;
    const uint32_t dis_h = s->has_dis && s->dis.height ? s->dis.height : s->cfg.height;
    for (uint32_t i = 0; i < n; i++)
        if (!frame_layout_ok(ref_fmt, s->cfg.width, s->cfg.height, &refs[i], host, frame_bytes) ||
            !frame_layout_ok(dis_fmt, dis_w, dis_h, &diss[i], host, dis_bytes ? dis_bytes : frame_bytes))
            return SSIMU2_E_INVALID;
    if (first_ticket) *first_ticket = s->next_global;
    uint32_t i = 0;
    while (i < n) {
        uint32_t wi;
        uint64_t local;
        route(s, s->next_global, &wi, &local);
        Worker* w = s->workers[wi];
        // everything up to the end of this batch goes to the same worker: one lock, one wake-up
        const uint32_t room = s->batch - (uint32_t)(s->next_global % s->batch);
        const uint32_t m = n - i < room ? n - i : room;
        {
            std::lock_guard<std::mutex> lk(s->res_mu);
            for (uint32_t k = 0; k < m; k++) s->done[(s->next_global + k) % kShardResultCap] = 0;
        }
        {
            std::lock_guard<std::mutex> lk(w->mu);
            for (uint32_t k = 0; k < m; k++)
                w->queue.push_back(Job{refs[i + k], diss[i + k], frame_bytes, dis_bytes, streams ? streams[wi] : nullptr, s->next_global + k});
            w->cv.notify_one();
        }
        s->next_global += m;
        i += m;
    }
    return SSIMU2_OK;
}

}  // namespace

extern "C" {

int ssimu2_shard_create(ssimu2_shard_t** out, const ssimu2_config* cfg, const int32_t* devices, uint32_t n_devices)
{
    return ssimu2_shard_create_mixed(out, cfg, nullptr, devices, n_devices);
}

int ssimu2_shard_create_mixed(ssimu2_shard_t** out, const ssimu2_config* cfg, const ssimu2_source* dis, const int32_t* devices,
                              uint32_t n_devices)
{
    if (!out || !cfg || !devices || n_devices == 0 || n_devices > 64) return SSIMU2_E_INVALID;
    *out = nullptr;
    ssimu2_shard* s = new (std::nothrow) ssimu2_shard();
    if (!s) return SSIMU2_E_NOMEM;
    s->cfg = *cfg;
    if (dis) {
        s->dis = *dis;
        s->has_dis = true;
    }
    s->batch = cfg->batch ? cfg->batch : 8;
    if (s->batch > 1024) s->batch = 1024;
    s->cfg.batch = s->batch;
    try {
        s->results.assign(kShardResultCap, 0.0);
        s->done.assign(kShardResultCap, 0);
        for (uint32_t i = 0; i < n_devices; i++) {
            Worker* w = new Worker();
            w->device = devices[i];
            w->global_of.assign(kShardResultCap, 0);
            s->workers.push_back(w);
        }
        for (Worker* w : s->workers) w->th = std::thread(worker_main, s, w);
    } catch (...) {
        ssimu2_shard_destroy(s);
        return SSIMU2_E_NOMEM;
    }
    int rc = 0;
    for (Worker* w : s->workers) {
        std::unique_lock<std::mutex> lk(w->mu);
        w->cv.wait(lk, [&] { return w->ready; });
        if (w->create_rc && !rc) rc = w->create_rc;
    }
    if (rc) {
        ssimu2_shard_destroy(s);
        return rc;
    }
    *out = s;
    return SSIMU2_OK;
}

int ssimu2_shard_destroy(ssimu2_shard_t* s)
{
    if (!s) return SSIMU2_OK;
    for (Worker* w : s->workers) {
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->stop = true;
            w->flush = true;
            w->cv.notify_all();
        }
        if (w->th.joinable()) w->th.join();
        delete w;
    }
    delete s;
    return SSIMU2_OK;
}

int ssimu2_shard_submit_host(ssimu2_shard_t* s, uint32_t n, const ssimu2_frame* refs, const ssimu2_frame* diss, size_t frame_bytes,
                             uint64_t* first_ticket)
{
    if (frame_bytes == 0) return SSIMU2_E_INVALID;
    return submit_common(s, n, refs, diss, frame_bytes, 0, nullptr, first_ticket);
}

int ssimu2_shard_submit_host_sized(ssimu2_shard_t* s, uint32_t n, const ssimu2_frame* refs, size_t ref_bytes, const ssimu2_frame* diss,
                                   size_t dis_bytes, uint64_t* first_ticket)
{
    if (ref_bytes == 0 || dis_bytes == 0) return SSIMU2_E_INVALID;
    return submit_common(s, n, refs, diss, ref_bytes, dis_bytes, nullptr, first_ticket);
}

int ssimu2_shard_submit_device(ssimu2_shard_t* s, uint32_t n, const ssimu2_frame* refs, const ssimu2_frame* diss, void* const* streams,
                               uint64_t* first_ticket)
{
    return submit_common(s, n, refs, diss, 0, 0, streams, first_ticket);
}

int ssimu2_shard_device_of(const ssimu2_shard_t* s, uint64_t ticket, int32_t* device)
{
    if (!s || !device) return SSIMU2_E_INVALID;
    uint32_t wi;
    uint64_t local;
    route(s, ticket, &wi, &local);
    *device = s->workers[wi]->device;
    return SSIMU2_OK;
}

int ssimu2_shard_flush(ssimu2_shard_t* s)
{
    if (!s) return SSIMU2_E_INVALID;
    for (Worker* w : s->workers) {
        std::lock_guard<std::mutex> lk(w->mu);
        w->flush = true;
        w->cv.notify_one();
    }
    return SSIMU2_OK;
}

int ssimu2_shard_get_scores(ssimu2_shard_t* s, uint64_t first_ticket, uint32_t n, double* scores)
{
    if (!s || (n && !scores)) return SSIMU2_E_INVALID;
    if (first_ticket + n > s->next_global || s->next_global - first_ticket > kShardResultCap) return SSIMU2_E_TICKET;
    // tell every worker how far it has to fetch, even through a partial batch
    for (uint32_t i = 0; i < n;) {
        uint32_t wi;
        uint64_t local;
        route(s, first_ticket + i, &wi, &local);
        const uint32_t room = s->batch - (uint32_t)((first_ticket + i) % s->batch);
        const uint32_t m = n - i < room ? n - i : room;
        Worker* w = s->workers[wi];
        {
            std::lock_guard<std::mutex> lk(w->mu);
            if (w->want < local + m) w->want = local + m;
            w->cv.notify_one();
        }
        i += m;
    }
    std::unique_lock<std::mutex> lk(s->res_mu);
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t g = first_ticket + i;
        s->res_cv.wait(lk, [&] { return s->done[g % kShardResultCap] || s->error.load(); });
        if (int e = s->error.load()) return e;
        scores[i] = s->results[g % kShardResultCap];
    }
    return SSIMU2_OK;
}

}  // extern "C"
