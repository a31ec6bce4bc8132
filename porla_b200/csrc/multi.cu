// In-call multi-GPU partition, pipelined host-buffer MSM and the pageable-memory copy pool.  See multi.h / staging.h.
#include "multi.h"

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/porla_multiexp.h"

namespace porla {

// ---------------------------------------------------------------------------- pageable-memory copy pool
bool host_pointer_is_pinned(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();   // unregistered host memory reports an error on old drivers: not sticky, clear it
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

namespace {

// bytes per pinned slot (PORLA_COPY_CHUNK_KB to tune)
static const size_t kRingChunk = [] {
    const char* e = getenv("PORLA_COPY_CHUNK_KB");
    const size_t kb = e && atoi(e) >= 64 ? (size_t)atoi(e) : 1024;
    return kb << 10;
}();
constexpr int kRingSlots = 3;                  // slots per copy thread
constexpr size_t kRingThreshold = 4u << 20;    // smaller pageable copies go through the driver's own staging (a hand-off to the
                                               // copy threads costs ~0.1 ms: measured on the 1 MiB audit aggregation call)

std::atomic<uint64_t> g_ring_bytes{0};

struct CopyJob {
    int dev;
    uint8_t* dst;
    const uint8_t* src;
    size_t bytes;
    cudaStream_t stream;
    std::atomic<size_t> next{0};     // next chunk to hand out
    size_t nchunks;
    std::mutex mu;
    std::condition_variable cv;
    size_t done = 0;
};

class CopyPool {
  public:
    static CopyPool& get() {
        static CopyPool* p = new CopyPool();   // leaked on purpose: threads may outlive static destruction order
        return *p;
    }
    // Blocks until every chunk of the job has been copied into the ring and its DMA has been issued on job.stream.
    void run(int dev, void* dst, const void* src, size_t bytes, cudaStream_t stream) {
        auto job = std::make_shared<CopyJob>();
        job->dev = dev;
        job->dst = (uint8_t*)dst;
        job->src = (const uint8_t*)src;
        job->bytes = bytes;
        job->stream = stream;
        job->nchunks = (bytes + kRingChunk - 1) / kRingChunk;
        {
            std::lock_guard<std::mutex> g(mu_);
            start_threads_locked();
            jobs_.push_back(job);
        }
        cv_.notify_all();
        std::unique_lock<std::mutex> lk(job->mu);
        job->cv.wait(lk, [&] { return job->done == job->nchunks; });
        g_ring_bytes.fetch_add(bytes, std::memory_order_relaxed);
    }
    int threads() const { return nthreads_; }

  private:
    struct Slot {
        uint8_t* buf = nullptr;
        cudaEvent_t pending = nullptr;          // DMA out of this slot that must finish before it is overwritten
        cudaEvent_t ev[kMaxDevices] = {};       // one event per device (an event belongs to a device)
    };
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::shared_ptr<CopyJob>> jobs_;
    std::vector<std::thread> workers_;
    int nthreads_ = 0;

    CopyPool() {
        const char* e = getenv("PORLA_COPY_THREADS");
        int hw = (int)std::thread::hardware_concurrency();
        // measured on the GPU box (16 vCPUs, tools/h2d_probe.py): 4 threads 29 GB/s, 8 threads 22 GB/s, 16 threads 18 GB/s -- the copy
        // into the ring, the DMA out of it and the source reads share the host's memory bandwidth
        nthreads_ = e && atoi(e) > 0 ? atoi(e) : (hw >= 8 ? 4 : (hw >= 4 ? 2 : 1));
        if (nthreads_ > 32) nthreads_ = 32;
    }
    void start_threads_locked() {
        if (!workers_.empty()) return;
        for (int i = 0; i < nthreads_; i++) workers_.emplace_back([this] { loop(); });
        for (auto& t : workers_) t.detach();
    }
    void loop() {
        Slot slots[kRingSlots];
        int turn = 0;
        for (;;) {
            std::shared_ptr<CopyJob> job;
            size_t k = 0;
            {
                std::unique_lock<std::mutex> lk(mu_);
                for (;;) {
                    while (!jobs_.empty() && jobs_.front()->next.load() >= jobs_.front()->nchunks) jobs_.pop_front();
                    if (!jobs_.empty()) {
                        job = jobs_.front();
                        k = job->next.fetch_add(1);
                        if (k < job->nchunks) break;
                        continue;
                    }
                    cv_.wait(lk);
                }
            }
            const size_t off = k * kRingChunk;
            const size_t len = job->bytes - off < kRingChunk ? job->bytes - off : kRingChunk;
            Slot& s = slots[turn];
            turn = (turn + 1) % kRingSlots;
            PORLA_CUDA(cudaSetDevice(job->dev));
            if (!s.buf) PORLA_CUDA(cudaHostAlloc(&s.buf, kRingChunk, cudaHostAllocPortable));
            if (s.pending) PORLA_CUDA(cudaEventSynchronize(s.pending));
            memcpy(s.buf, job->src + off, len);
            PORLA_CUDA(cudaMemcpyAsync(job->dst + off, s.buf, len, cudaMemcpyHostToDevice, job->stream));
            if (!s.ev[job->dev]) PORLA_CUDA(cudaEventCreateWithFlags(&s.ev[job->dev], cudaEventDisableTiming));
            PORLA_CUDA(cudaEventRecord(s.ev[job->dev], job->stream));
            s.pending = s.ev[job->dev];
            {
                std::lock_guard<std::mutex> g(job->mu);
                job->done++;
            }
            job->cv.notify_all();
        }
    }
};

}  // namespace

uint64_t h2d_ring_bytes() { return g_ring_bytes.load(); }

void h2d_copy(void* d_dst, const void* h_src, size_t bytes, cudaStream_t stream) {
    if (!bytes) return;
    static const bool ring_off = getenv("PORLA_NO_COPY_RING") != nullptr;
    if (bytes < kRingThreshold || ring_off || host_pointer_is_pinned(h_src)) {
        PORLA_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, stream));
        return;
    }
    CopyPool::get().run(current_device(), d_dst, h_src, bytes, stream);
}

// ---------------------------------------------------------------------------- one worker thread per device
namespace {

struct DevWorker {
    int dev = 0;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    const std::function<void(int)>* fn = nullptr;
    int part = 0;
    bool busy = false;
    Staging stage;
};

int visible_devices() {
    const int c = device_count();
    return c > kMaxDevices ? kMaxDevices : c;
}
int slot_device(int slot) { return slot % visible_devices(); }

std::mutex g_multi_mu;                       // one fan-out at a time
DevWorker* g_workers[kMaxDevices] = {};      // leaked on purpose: the detached threads outlive static destruction
thread_local DevWorker* t_worker = nullptr;

void worker_main(DevWorker* w) {
    DeviceScope scope(w->dev);   // for the life of the thread
    t_worker = w;
    w->stage.init();
    std::unique_lock<std::mutex> lk(w->mu);
    for (;;) {
        w->cv.wait(lk, [&] { return w->busy; });
        const std::function<void(int)>* fn = w->fn;
        const int part = w->part;
        lk.unlock();
        (*fn)(part);
        lk.lock();
        w->busy = false;
        w->cv.notify_all();
    }
}

// Worker `slot` drives device slot % visible: with fewer devices than parts (PORLA_OVERSUBSCRIBE_DEVICES=1, a test
// setting) several workers share a device, each with its own stream and staging; the per-device engine mutex
// serialises their kernels' scratch.
DevWorker* get_worker(int slot) {
    if (!g_workers[slot]) {
        DevWorker* w = new DevWorker();
        g_workers[slot] = w;
        w->dev = slot_device(slot);
        w->th = std::thread(worker_main, w);
        w->th.detach();
    }
    return g_workers[slot];
}

}  // namespace

Staging& worker_staging() {
    if (!t_worker) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: worker_staging() outside a device worker\n");
        abort();
    }
    return t_worker->stage;
}

int part_device(int part) { return slot_device(part); }

void run_on_devices(int ndev, const std::function<void(int)>& fn) {
    if (ndev < 1 || ndev > kMaxDevices) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: run_on_devices: %d parts\n", ndev);
        abort();
    }
    std::lock_guard<std::mutex> g(g_multi_mu);
    for (int p = 0; p < ndev; p++) {
        DevWorker* w = get_worker(p);
        std::lock_guard<std::mutex> lk(w->mu);
        w->fn = &fn;
        w->part = p;
        w->busy = true;
        w->cv.notify_all();
    }
    for (int p = 0; p < ndev; p++) {
        DevWorker* w = g_workers[p];
        std::unique_lock<std::mutex> lk(w->mu);
        w->cv.wait(lk, [&] { return !w->busy; });
    }
}

int fanout_devices(int64_t n) {
    static const int limit = [] {
        const char* e = getenv("PORLA_DEVICES");
        const int count = device_count() > kMaxDevices ? kMaxDevices : device_count();
        if (e && atoi(e) >= 1) {
            const int cap = getenv("PORLA_OVERSUBSCRIBE_DEVICES") ? kMaxDevices : count;
            return atoi(e) < cap ? atoi(e) : cap;
        }
        return device_pinned_by_env() ? 1 : count;    // one process per GPU: stay on the process's own device
    }();
    static const int64_t min_per_dev = [] {
        const char* e = getenv("PORLA_FANOUT_MIN");
        return e && atoll(e) > 0 ? (int64_t)atoll(e) : (int64_t)1 << 16;
    }();
    if (limit <= 1) return 1;
    int d = limit;
    while (d > 1 && n / d < min_per_dev) d >>= 1;
    return d;
}

// ---------------------------------------------------------------------------- pipelined host-buffer MSM (one device)
// The terms of a large call cross PCIe in several parts; every part is imported, recoded, sorted and accumulated INTO ONE
// shared bucket array as soon as it has arrived (MsmOptions::part_mode), while the next part is being copied; the buckets
// are reduced once, after the last part.  Only the first part's copy is exposed, and a slow source (pageable memory through
// the pinned ring: ~29 GB/s on the GPU box against ~54 GB/s for pinned buffers, tools/h2d_probe.py) hides behind the
// kernels of the previous part as long as a part's copy is not longer than its kernels.  Round 1 ran two independent
// MSMs (25 % + 75 % of the terms) and added their window sums: 4.79 ms at 2^20 with pinned buffers, 6.98 ms with pageable ones.
// Every part pays one extra mixed addition per non-empty bucket (it continues from the stored sum) and ~15 launches, so a
// part should hold at least 2^18 terms and bring at least ~8 pairs to each bucket.  Measured (one B200, pinned buffers,
// tools/e2e_stages.py), whole call: 2^20 -- 1 part 5.54 ms, 2 parts 4.90, 4 parts 4.85, 8 parts 5.36; 2^22 -- 19.4 / 16.1 /
// 15.0 (4 parts); 2^24 -- 73.1 / 59.1 / 52.5 (4 parts).
static int stream_parts_for(int64_t n, const MsmPlan& plan) {
    const char* e = getenv("PORLA_STREAM_PARTS");     // (read per call: the tests force small MSMs through the streamed path)
    const int forced = e ? atoi(e) : 0;
    if (forced >= 1 && forced <= 8) return n >= forced ? forced : 1;
    if (n < (1 << 19) || getenv("PORLA_NO_SPLIT")) return 1;
    const int64_t per_bucket = (n * (plan.glv ? 2 : 1)) >> (plan.c - 1);
    int64_t p = per_bucket / 8;
    if (p > (n >> 18)) p = n >> 18;
    return p < 1 ? 1 : (p > 8 ? 8 : (int)p);
}

// End of part h of n terms in `nparts` streamed parts: the first part is half a regular part (its copy is the exposed one),
// the last part takes what that leaves.
static int64_t part_end(int64_t n, int h, int nparts) {
    return h == nparts - 1 ? n : (n * (2 * h + 1)) / (2 * nparts);
}

static int part_mode(int h, int nparts) {
    return nparts == 1 ? kPartWhole : (h == 0 ? kPartFirst : (h == nparts - 1 ? kPartLast : kPartMiddle));
}

// Options of an MSM that hands its plan.nwin window sums to the caller: the window layout is forced to `plan`, so that all
// parts of one MSM fill the same buckets and all devices produce window sums that add up.
static MsmOptions window_sums_options(const MsmPlan& plan, int scalar_fmt, int out_fmt, void* d_window_sums) {
    MsmOptions opt;
    opt.scalar_be = scalar_fmt == PORLA_SCALAR_BE32;
    opt.out_fmt = out_fmt;
    opt.shared_points = 1;
    opt.window_bits = plan.c;
    opt.glv = plan.glv;
    opt.no_fixed_base = 1;
    opt.no_small = 1;
    opt.d_window_sums = d_window_sums;
    return opt;
}

void msm_host_pipelined(Staging& sg, int curve, const uint8_t* scalars, const uint8_t* points, int64_t n, int scalar_fmt,
                        int point_fmt, const MsmPlan& plan, uint8_t* h_ws) {
    const int nparts = stream_parts_for(n, plan);
    const size_t ws_bytes = (size_t)plan.nwin * 128;
    // staging layout: scalars | raw points | table + endomorphism image (2 * 64 B per point) | flags | window sums | buckets
    StageLayout lay;
    const size_t sc_off = lay.add((size_t)n * 32), pt_off = lay.add((size_t)n * 64), tab_off = lay.add((size_t)n * 128),
                 fl_off = lay.add((size_t)n), ws_off = lay.add(ws_bytes), bk_off = lay.add(nparts > 1 ? msm_bucket_bytes(plan) : 0);
    uint8_t* d = sg.dev(lay.size);
    cudaStream_t st = sg.stream, cs = sg.copy_stream;
    MsmOptions opt = window_sums_options(plan, scalar_fmt, point_fmt, d + ws_off);
    if (nparts > 1) opt.d_buckets = d + bk_off;
    int64_t first = 0;
    for (int h = 0; h < nparts; h++) {
        const int64_t last = part_end(n, h, nparts);
        const size_t a = (size_t)first, m = (size_t)(last - first);
        h2d_copy(d + sc_off + a * 32, scalars + a * 32, m * 32, cs);
        h2d_copy(d + pt_off + a * 64, points + a * 64, m * 64, cs);
        PORLA_CUDA(cudaEventRecord(sg.ev[h], cs));
        PORLA_CUDA(cudaStreamWaitEvent(st, sg.ev[h], 0));
        PointTable tab;
        table_import_into(curve, d + pt_off + a * 64, point_fmt, (uint32_t)m, d + tab_off + a * 128, d + fl_off + a, &tab, st);
        opt.part_mode = part_mode(h, nparts);
        msm_device(curve, tab, d + sc_off + a * 32, (uint32_t)m, 1, opt, nullptr, nullptr, st);
        first = last;
    }
    uint8_t* hbuf = sg.pinned(ws_bytes);
    PORLA_CUDA(cudaMemcpyAsync(hbuf, d + ws_off, ws_bytes, cudaMemcpyDeviceToHost, st));
    PORLA_CUDA(cudaStreamSynchronize(st));
    memcpy(h_ws, hbuf, ws_bytes);
}

// ---------------------------------------------------------------------------- fan-out over the devices of the box
static void device_ranges(int64_t n, int ndev, int64_t* first, int64_t* count) {
    // contiguous ranges, the last device takes the remainder (Client.hpp:753-754)
    const int64_t each = n / ndev;
    for (int p = 0; p < ndev; p++) {
        first[p] = each * p;
        count[p] = p == ndev - 1 ? n - each * p : each;
    }
}

void msm_host_fanout(int curve, const uint8_t* scalars, const uint8_t* points, int64_t n, int scalar_fmt, int point_fmt,
                     int ndev, uint8_t* out64) {
    int64_t first[kMaxDevices], count[kMaxDevices];
    device_ranges(n, ndev, first, count);
    const MsmPlan plan = msm_plan(curve, (uint32_t)count[ndev - 1], 1, 0);
    const size_t ws_bytes = (size_t)plan.nwin * 128;
    std::vector<uint8_t> ws((size_t)ndev * ws_bytes);
    run_on_devices(ndev, [&](int p) {
        msm_host_pipelined(worker_staging(), curve, scalars + (size_t)first[p] * 32, points + (size_t)first[p] * 64, count[p],
                           scalar_fmt, point_fmt, plan, ws.data() + (size_t)p * ws_bytes);
    });
    // one set of window sums per device: add window by window, Horner, normalise
    finalize_host_parts(curve, ws.data(), ndev, plan.nwin, plan.c, point_fmt, out64);
}

}  // namespace porla

// ============================================================================ C-ABI: tables sharded over devices
using namespace porla;

struct porla_mtable {
    int curve = 0;
    int ndev = 0;
    int64_t n = 0;
    int devices[kMaxDevices] = {};
    int64_t first[kMaxDevices] = {}, count[kMaxDevices] = {};
    PointTable part[kMaxDevices];
    uint8_t* d_scalars[kMaxDevices] = {};     // per-device scratch for host-scalar calls (count * 32 B)
    uint8_t* d_ws[kMaxDevices] = {};          // per-device window sums
};

extern "C" {

int porla_device_count(void) { return device_count(); }

porla_mtable* porla_mtable_create(int curve, const void* h_points, int64_t n, int point_fmt, int ndev) {
    device_init();
    const int visible = device_count() > kMaxDevices ? kMaxDevices : device_count();
    if (ndev <= 0) ndev = visible;
    const bool oversubscribe = getenv("PORLA_OVERSUBSCRIBE_DEVICES") != nullptr;   // tests on a box with fewer GPUs
    if ((ndev > visible && !oversubscribe) || ndev > kMaxDevices || n < 0 || n >= ((int64_t)1 << 31) * ndev) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: porla_mtable_create: %d devices requested, %d visible (n = %lld)\n", ndev,
                visible, (long long)n);
        abort();
    }
    porla_mtable* mt = new porla_mtable();
    mt->curve = curve;
    mt->ndev = ndev;
    mt->n = n;
    device_ranges(n, ndev, mt->first, mt->count);
    for (int p = 0; p < ndev; p++) mt->devices[p] = part_device(p);
    const uint8_t* pts = (const uint8_t*)h_points;
    run_on_devices(ndev, [&](int p) {
        Staging& sg = worker_staging();
        const size_t m = (size_t)mt->count[p];
        uint8_t* d_tmp = nullptr;
        PORLA_CUDA(cudaMalloc(&d_tmp, (m ? m : 1) * 64));
        h2d_copy(d_tmp, pts + (size_t)mt->first[p] * 64, m * 64, sg.stream);
        table_import_device(curve, d_tmp, point_fmt, (uint32_t)m, &mt->part[p], sg.stream);
        PORLA_CUDA(cudaFree(d_tmp));
        PORLA_CUDA(cudaMalloc(&mt->d_scalars[p], (m ? m : 1) * 32));
        PORLA_CUDA(cudaMalloc(&mt->d_ws[p], 256 * 128));
    });
    return mt;
}

int porla_mtable_devices(const porla_mtable* mt) { return mt->ndev; }
int64_t porla_mtable_len(const porla_mtable* mt) { return mt->n; }

void porla_mtable_range(const porla_mtable* mt, int part, int* device, int64_t* first, int64_t* count) {
    if (part < 0 || part >= mt->ndev) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: porla_mtable_range: part %d of %d\n", part, mt->ndev);
        abort();
    }
    *device = mt->devices[part];
    *first = mt->first[part];
    *count = mt->count[part];
}

// Shared body: scalars either in host memory (one array of n, copied range by range) or already resident
// (d_scalars_per_part[p] on device p).
static void mtable_msm(const porla_mtable* mt, const uint8_t* h_scalars, void* const* d_scalars_per_part, int scalar_fmt,
                       int out_fmt, uint8_t* out64) {
    if (mt->n == 0) {
        memset(out64, 0, 64);
        return;
    }
    int64_t largest = 0;
    for (int p = 0; p < mt->ndev; p++) largest = mt->count[p] > largest ? mt->count[p] : largest;
    const MsmPlan plan = msm_plan(mt->curve, (uint32_t)largest, 1, 0);
    const size_t ws_bytes = (size_t)plan.nwin * 128;
    std::vector<uint8_t> ws((size_t)mt->ndev * ws_bytes);
    run_on_devices(mt->ndev, [&](int p) {
        Staging& sg = worker_staging();
        const size_t m = (size_t)mt->count[p];
        const uint8_t* d_sc;
        const int nparts = d_scalars_per_part ? 1 : stream_parts_for((int64_t)m, plan);
        MsmOptions opt = window_sums_options(plan, scalar_fmt, out_fmt, mt->d_ws[p]);
        if (d_scalars_per_part) {
            d_sc = (const uint8_t*)d_scalars_per_part[p];
        } else if (nparts > 1) {
            // host scalars of a large range: streamed like msm_host_pipelined -- the scalars of part h+1 cross PCIe while
            // part h (a view of the resident table) is accumulated into the shared bucket set
            opt.d_buckets = sg.dev(msm_bucket_bytes(plan));
            size_t a = 0;
            for (int h = 0; h < nparts; h++) {
                const size_t last = (size_t)part_end((int64_t)m, h, nparts);
                const size_t len = last - a;
                h2d_copy(mt->d_scalars[p] + a * 32, h_scalars + ((size_t)mt->first[p] + a) * 32, len * 32, sg.copy_stream);
                PORLA_CUDA(cudaEventRecord(sg.ev[h], sg.copy_stream));
                PORLA_CUDA(cudaStreamWaitEvent(sg.stream, sg.ev[h], 0));
                // entries [a, a + len) of this device's range (a sharded part has no fixed-base expansion)
                const PointTable view = table_window(mt->part[p], (int64_t)a, (int64_t)len);
                opt.part_mode = part_mode(h, nparts);
                msm_device(mt->curve, view, mt->d_scalars[p] + a * 32, (uint32_t)len, 1, opt, nullptr, nullptr, sg.stream);
                a = last;
            }
            d_sc = nullptr;
        } else {
            h2d_copy(mt->d_scalars[p], h_scalars + (size_t)mt->first[p] * 32, m * 32, sg.stream);
            d_sc = mt->d_scalars[p];
        }
        if (m && d_sc)
            msm_device(mt->curve, mt->part[p], d_sc, (uint32_t)m, 1, opt, nullptr, nullptr, sg.stream);
        else if (!m) PORLA_CUDA(cudaMemsetAsync(mt->d_ws[p], 0, ws_bytes, sg.stream));
        uint8_t* h = sg.pinned(ws_bytes);
        PORLA_CUDA(cudaMemcpyAsync(h, mt->d_ws[p], ws_bytes, cudaMemcpyDeviceToHost, sg.stream));
        PORLA_CUDA(cudaStreamSynchronize(sg.stream));
        memcpy(ws.data() + (size_t)p * ws_bytes, h, ws_bytes);
    });
    finalize_host_parts(mt->curve, ws.data(), mt->ndev, plan.nwin, plan.c, out_fmt, out64);
}

void porla_mtable_msm_host_scalars(const porla_mtable* mt, const void* h_scalars, int scalar_fmt, int out_fmt, void* out64) {
    mtable_msm(mt, (const uint8_t*)h_scalars, nullptr, scalar_fmt, out_fmt, (uint8_t*)out64);
}

void porla_mtable_msm_resident(const porla_mtable* mt, void* const* d_scalars_per_part, int scalar_fmt, int out_fmt, void* out64) {
    mtable_msm(mt, nullptr, d_scalars_per_part, scalar_fmt, out_fmt, (uint8_t*)out64);
}

void* porla_mtable_scalars_upload(const porla_mtable* mt, int part, const void* h_scalars_of_part) {
    if (part < 0 || part >= mt->ndev) return nullptr;
    void* d = nullptr;
    DeviceScope scope(mt->devices[part]);
    const size_t bytes = (size_t)(mt->count[part] ? mt->count[part] : 1) * 32;
    PORLA_CUDA(cudaMalloc(&d, bytes));
    PORLA_CUDA(cudaMemcpy(d, h_scalars_of_part, (size_t)mt->count[part] * 32, cudaMemcpyHostToDevice));
    return d;
}

void porla_mtable_scalars_free(const porla_mtable* mt, int part, void* d_scalars) {
    if (part < 0 || part >= mt->ndev || !d_scalars) return;
    DeviceScope scope(mt->devices[part]);
    PORLA_CUDA(cudaFree(d_scalars));
}

void porla_mtable_destroy(porla_mtable* mt) {
    if (!mt) return;
    run_on_devices(mt->ndev, [&](int p) {
        table_free(&mt->part[p]);
        if (mt->d_scalars[p]) PORLA_CUDA(cudaFree(mt->d_scalars[p]));
        if (mt->d_ws[p]) PORLA_CUDA(cudaFree(mt->d_ws[p]));
    });
    delete mt;
}

void porla_msm_host_devices(int curve, const void* scalars, const void* points, int64_t n, int scalar_fmt, int point_fmt, int ndev,
                            void* out64) {
    device_init();
    const int visible = device_count() > kMaxDevices ? kMaxDevices : device_count();
    if (ndev <= 0) ndev = visible;
    if (n < 0 || n >= ((int64_t)1 << 31) * ndev || ndev > kMaxDevices || (ndev > visible && !getenv("PORLA_OVERSUBSCRIBE_DEVICES"))) {
        fprintf(stderr, "[libmultiexp/porla_b200] FATAL: porla_msm_host_devices: n = %lld over %d devices (%d visible)\n", (long long)n,
                ndev, visible);
        abort();
    }
    if (n == 0) {
        memset(out64, 0, 64);
        return;
    }
    if (n < ndev) ndev = (int)n;
    msm_host_fanout(curve, (const uint8_t*)scalars, (const uint8_t*)points, n, scalar_fmt, point_fmt, ndev, (uint8_t*)out64);
}

uint64_t porla_debug_copy_ring_bytes(void) { return h2d_ring_bytes(); }

// Host-to-device copy rate of the library's own copy path (GB/s): `bytes` from a host buffer the caller provides (pinned or
// pageable) into a scratch device buffer, `reps` times, stream-synchronised.  Development aid for the copy pool.
double porla_debug_h2d_rate(const void* h_src, uint64_t bytes, int reps) {
    device_init();
    static void* d = nullptr;
    static uint64_t cap = 0;
    static cudaStream_t st = nullptr;
    if (!st) PORLA_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    if (bytes > cap) {
        if (d) PORLA_CUDA(cudaFree(d));
        PORLA_CUDA(cudaMalloc(&d, bytes));
        cap = bytes;
    }
    h2d_copy(d, h_src, bytes, st);
    PORLA_CUDA(cudaStreamSynchronize(st));
    const auto t0 = std::chrono::steady_clock::now();
    for (int r = 0; r < reps; r++) {
        h2d_copy(d, h_src, bytes, st);
        PORLA_CUDA(cudaStreamSynchronize(st));
    }
    const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return (double)bytes * reps / sec / 1e9;
}

}  // extern "C"
