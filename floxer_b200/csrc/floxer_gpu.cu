// floxer_gpu.cu -- C ABI (include/floxer_gpu.h) and host-side batch queue of the B200 PEX verification path.
//
// Host responsibilities (the work of parallelization.cpp:193-293 and verification.cpp:8-245 of the
// reference, re-organised for a GPU): turn align calls into DP passes, pick a (words-per-lane, ring size)
// configuration per pass, bucket passes by configuration and length, launch the engine, and drive the
// leaf -> root walk of every anchor level-synchronously ("waves").  The inner tree levels of a batch run
// on the device from a handful of records per read (run_levels_on_device; the host only enqueues kernels
// and waits once), the root level -- windows that coincide share one score pass and one traceback
// (run_root_passes) -- from the host.  Up to 32 batches are in flight at a time (worker groups), each
// split over one or more host workers with their own CUDA streams and buffers.
// No CPU fallback exists: every alignment result comes from dp_kernels.cuh.
#include "../../include/floxer_gpu.h"
#include "bgzf_kernels.cuh"
#include "dp_kernels.cuh"
#include "read_kernels.cuh"
#include "record_kernels.cuh"
#include "root_kernels.cuh"
#include "seed_kernels.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <functional>
#include <ctime>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

using namespace fxg;

// ------------------------------------------------------------------------------------------------ utilities

namespace {

// Device memory comes from the device's stream-ordered pool (cudaMallocAsync), on a stream of its own per device:
// cudaMalloc / cudaFree synchronise the whole device, and with batches of changing sizes in flight a buffer that has to
// grow would stall every other batch for the length of the kernels that happen to run (measured: steps of 600 ms among
// steps of 10 ms).  The allocation is waited for on the host, so the memory may be used on any stream afterwards; a
// buffer is only ever replaced by its owner between two of its uses, when nothing reads it any more.
inline cudaStream_t alloc_stream() {
    static std::mutex mu;
    static cudaStream_t streams[64] = {nullptr};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!streams[dev]) {
        if (cudaStreamCreateWithFlags(&streams[dev], cudaStreamNonBlocking) != cudaSuccess) { streams[dev] = nullptr; return nullptr; }
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;                    // freed memory stays with the pool instead of going back to the driver
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    return streams[dev];
}
// time spent allocating (device and page-locked memory), for fxg_counters: in the steady state it must not grow
std::atomic<uint64_t> g_alloc_ns{0}, g_alloc_calls{0};
struct AllocTimer {
    const char* what; size_t bytes;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    AllocTimer(const char* w, size_t b) : what(w), bytes(b) {}
    ~AllocTimer() {
        uint64_t const ns = uint64_t(std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count());
        g_alloc_ns += ns; g_alloc_calls++;
        static bool const trace = std::getenv("FXG_TRACE_BATCHES") != nullptr;
        if (trace && ns > 2000000) fprintf(stderr, "[fxg] alloc %s %.1f MB took %.1f ms\n", what, double(bytes) / 1048576.0, double(ns) * 1e-6);
    }
};
inline cudaError_t device_alloc(void** p, size_t bytes) {
    AllocTimer timer("device", bytes);
    cudaStream_t const s = alloc_stream();
    if (!s) return cudaMalloc(p, bytes);
    cudaError_t e = cudaMallocAsync(p, bytes, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    return e;
}
inline void device_free(void* p) {
    cudaStream_t const s = alloc_stream();
    if (!s || cudaFreeAsync(p, s) != cudaSuccess) cudaFree(p);
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    // (a buffer that serves merged batches is sized for the largest one the queue forms the first time it has to grow:
    //  `scale` = that batch's size over this one's)
    cudaError_t ensure_scaled(size_t bytes, double scale) {
        if (bytes <= cap) return cudaSuccess;
        size_t const big = std::min(size_t(double(bytes) * std::min(std::max(scale, 1.0), 16.0)), std::max(bytes, size_t(2) << 30));
        if (big > bytes && ensure(big) == cudaSuccess) return cudaSuccess;
        (void)cudaGetLastError();
        return ensure(bytes);
    }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { device_free(p); p = nullptr; }
        size_t const want = std::max(bytes + bytes / 4 + 256, 2 * cap);      // grows geometrically: few replacements on the way to the steady state
        cap = 0;
        cudaError_t e = device_alloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = device_alloc(&p, bytes);
            if (e != cudaSuccess) { p = nullptr; return e; }
            cap = bytes;
            return e;
        }
        cap = want;
        return e;
    }
    // grows the buffer keeping its first `keep` bytes
    cudaError_t ensure_preserving(size_t bytes, size_t keep, cudaStream_t stream) {
        if (bytes <= cap) return cudaSuccess;
        void* np = nullptr;
        size_t const want = std::max(bytes + bytes / 2 + 256, 2 * cap);
        cudaError_t e = device_alloc(&np, want);
        if (e != cudaSuccess) return e;
        if (p && keep) {
            e = cudaMemcpyAsync(np, p, keep, cudaMemcpyDeviceToDevice, stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
            if (e != cudaSuccess) { device_free(np); return e; }
        }
        if (p) device_free(p);
        p = np; cap = want;
        return cudaSuccess;
    }
    void release() { if (p) device_free(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinnedBuf {                       // page-locked host staging memory
    void* p = nullptr;
    size_t cap = 0;
    const char* tag = "page-locked";     // what it holds (FXG_TRACE_BATCHES names slow allocations)
    cudaError_t ensure_scaled(size_t bytes, double scale) {
        if (bytes <= cap) return cudaSuccess;
        size_t const big = std::min(size_t(double(bytes) * std::min(std::max(scale, 1.0), 16.0)), std::max(bytes, size_t(96) << 20));   // (page-locking is slow: tens of ms per 100 MB)
        if (big > bytes && ensure(big) == cudaSuccess) return cudaSuccess;
        (void)cudaGetLastError();
        return ensure(bytes);
    }
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        size_t const want = std::max(bytes + bytes / 2 + 4096, 2 * cap);
        AllocTimer timer(tag, want);
        if (p) { cudaFreeHost(p); p = nullptr; }
        cap = 0;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = want;
        return e;
    }
    cudaError_t exactly(size_t bytes) {           // a fresh buffer of exactly this size
        AllocTimer timer(tag, bytes);
        release();
        cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocDefault);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = bytes;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct RefStore {
    DevBuf packed;                       // 4 bits per base, every reference starts at a multiple of 32 bases
    std::vector<uint64_t> base, len;
    DevBuf d_base, d_len;                // the same two tables on the device (level kernels)
    uint64_t total = 0;
    uint64_t version = 0;                // counts the successful fxg_set_references calls (staged batches hold store positions)
};

// one staged pool of query bytes with its Peq planes (+ optional inline reference pool)
struct Pool {
    DevBuf bytes, peq, inline_packed, bad_rank;   // bad_rank: one word the Peq builder sets when it meets a rank above 5
    uint64_t len = 0, plane_words = 0, inline_len = 0;
    void release() { bytes.release(); peq.release(); inline_packed.release(); bad_rank.release(); }
};

struct Pass {                            // one DP pass of the engine
    uint64_t ref_base;                   // position in the packed store / inline pool
    uint64_t query_base;                 // position in the pool
    uint32_t n, m;
    int32_t dlo, dhi;
    uint32_t flags;
};

constexpr int kWidths[6] = {1, 2, 4, 8, 16, 32};

struct Config { uint8_t widx; uint8_t G; uint32_t nb; uint64_t word_steps; };

struct ConfigCacheEntry { uint32_t n, m; int32_t dlo, dhi; Config cfg; bool ok; bool valid; bool traced; };

// Everything one host worker needs to run passes on its own stream.
struct WorkerGroup;
struct Worker {
    int id = 0;
    WorkerGroup* group = nullptr;
    cudaStream_t stream = nullptr;
    static constexpr int kSide = 3;      // the launches of one wave are independent: the smaller ones run beside the largest
    cudaStream_t side[kSide] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[kSide] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_b0 = nullptr, ev_b1 = nullptr;
    cudaEvent_t ev_sleep = nullptr;
    // Waits for everything queued on `s` so far.  cudaStreamSynchronize spins (measured: 94 ms of CPU per batch, 13 cores'
    // worth, taken from the other workers and the other ranks of the host); a blocking event alone adds its wake-up
    // latency to every wave (a batch took 14.8 instead of 11.5 ms when every tree level was a wait).  So: poll for a short
    // while, handing the core over between polls, then sleep on the event.  (Since the tree levels run on the device a part
    // waits five times per batch and the polling time hardly matters: 150 us cost 1 ms of CPU per batch for nothing.)
    int spin_us = 20;
    cudaError_t wait_for(cudaStream_t s) {
        cudaError_t e = cudaEventRecord(ev_sleep, s);
        if (e != cudaSuccess) return e;
        auto const t0 = std::chrono::steady_clock::now();
        while ((e = cudaEventQuery(ev_sleep)) == cudaErrorNotReady) {
            if (std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(spin_us)) return cudaEventSynchronize(ev_sleep);
            std::this_thread::yield();
        }
        return e;
    }
    // n independent launches side by side: fork(main, n) before the first, fan_stream(main, q) for launch q -- `main` for
    // the first, a side stream that waits for the fork for the others -- and join(main, n) after the last
    cudaError_t fork(cudaStream_t main, int n) { return n > 1 ? cudaEventRecord(ev_fork, main) : cudaSuccess; }
    cudaError_t fan_stream(cudaStream_t main, int q, cudaStream_t& s) {
        if (q == 0) { s = main; return cudaSuccess; }
        s = side[(q - 1) % kSide];
        return q <= kSide ? cudaStreamWaitEvent(s, ev_fork, 0) : cudaSuccess;
    }
    cudaError_t join(cudaStream_t main, int n) {
        cudaError_t e = cudaSuccess;
        for (int q = 0; q < std::min(n - 1, kSide) && e == cudaSuccess; ++q)
            if ((e = cudaEventRecord(ev_join[q], side[q])) == cudaSuccess) e = cudaStreamWaitEvent(main, ev_join[q], 0);
        return e;
    }
    // tracebacks are long chains of dependent steps: the root alignments of a wave are cut into chunks, each chunk's
    // tracebacks run on a stream of their own beside the score passes (and tracebacks) of the other chunks
    static constexpr int kWalkSlots = 4;
    DevBuf d_tasks, d_results, d_ck[kWalkSlots], d_wtasks, d_wresults, d_cigars, d_rtasks, d_rresults, d_lv, d_roots, d_root, d_cub, d_hits;
    cudaStream_t walk_stream[kWalkSlots] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_walk_done[kWalkSlots] = {nullptr, nullptr, nullptr, nullptr}, ev_w0 = nullptr, ev_w1[kWalkSlots] = {nullptr, nullptr, nullptr, nullptr};
    PinnedBuf h_tasks, h_results, h_wtasks, h_wresults, h_rtasks, h_rresults, h_lv, h_lv_back, h_roots, h_root_back, h_hits;
    Worker() {
        h_tasks.tag = "page-locked tasks"; h_results.tag = "page-locked results"; h_wtasks.tag = "page-locked traceback tasks";
        h_wresults.tag = "page-locked traceback results"; h_rtasks.tag = "page-locked range tasks"; h_rresults.tag = "page-locked range results";
        h_lv.tag = "page-locked level records"; h_lv_back.tag = "page-locked level counters"; h_roots.tag = "page-locked root entries";
        h_root_back.tag = "page-locked root counters"; h_hits.tag = "page-locked alignment records";
    }
    fxg_counters ctr{};
    std::string err;
    std::vector<ConfigCacheEntry> cfg_cache = std::vector<ConfigCacheEntry>(8192);
    std::vector<uint64_t> keys, keys_tmp;
    std::vector<Config> cfgs;
    uint64_t cig_used = 0;               // ops of d_cigars filled by the current run
    // (measured: handing the device buffers back to the memory pool after every batch and taking them again costs 2.5 ms
    //  per allocation when batch sizes vary -- the pool splits and grows -- so a worker keeps its buffers)
    void release_device() {
        for (DevBuf* b : {&d_tasks, &d_results, &d_wtasks, &d_wresults, &d_cigars, &d_rtasks, &d_rresults, &d_lv, &d_roots, &d_root, &d_cub, &d_hits}) b->release();
        for (int q = 0; q < kWalkSlots; ++q) d_ck[q].release();
    }
    void release() {
        for (DevBuf* b : {&d_tasks, &d_results, &d_wtasks, &d_wresults, &d_cigars, &d_rtasks, &d_rresults, &d_lv, &d_roots, &d_root, &d_cub, &d_hits}) b->release();
        if (ev_w0) { cudaEventDestroy(ev_w0); ev_w0 = nullptr; }
        if (ev_b0) { cudaEventDestroy(ev_b0); ev_b0 = nullptr; }
        if (ev_b1) { cudaEventDestroy(ev_b1); ev_b1 = nullptr; }
        if (ev_sleep) { cudaEventDestroy(ev_sleep); ev_sleep = nullptr; }
        for (int q = 0; q < kWalkSlots; ++q) {
            d_ck[q].release();
            if (ev_walk_done[q]) cudaEventDestroy(ev_walk_done[q]);
            if (ev_w1[q]) cudaEventDestroy(ev_w1[q]);
            if (walk_stream[q]) cudaStreamDestroy(walk_stream[q]);
            ev_walk_done[q] = ev_w1[q] = nullptr; walk_stream[q] = nullptr;
        }
        for (PinnedBuf* b : {&h_tasks, &h_results, &h_wtasks, &h_wresults, &h_rtasks, &h_rresults, &h_lv, &h_lv_back, &h_roots, &h_root_back, &h_hits}) b->release();
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (ev_fork) cudaEventDestroy(ev_fork);
        for (int i = 0; i < kSide; ++i) {
            if (ev_join[i]) cudaEventDestroy(ev_join[i]);
            if (side[i]) cudaStreamDestroy(side[i]);
            ev_join[i] = nullptr; side[i] = nullptr;
        }
        if (stream) cudaStreamDestroy(stream);
        ev0 = ev1 = ev_fork = nullptr; stream = nullptr;
    }
};

// The workers that serve one *_run call.  A context has several groups, so that several batches can be in flight: the
// host-side preparation and the latency-bound tracebacks of one batch hide behind the score passes of the others.
// The first group owns more workers than a group uses when the context is busy: a batch that runs alone is split over
// all of them, which shortens its latency, while with many batches in flight fewer, larger launches per batch are the
// better deal.
struct WorkerGroup {
    std::vector<std::unique_ptr<Worker>> workers;
    size_t use_workers = 0;              // decided when the group is acquired
    cudaEvent_t ev_run0 = nullptr, ev_run1 = nullptr, ev_merged = nullptr;
    Pool merged;                         // the Peq planes of a batch merged from several jobs (build_merged_pool)
    bool busy = false;
};

inline double thread_cpu_ms() {
    timespec ts{};
    clock_gettime(CLOCK_THREAD_CPUTIME_ID, &ts);
    return double(ts.tv_sec) * 1e3 + double(ts.tv_nsec) * 1e-6;
}

// host-side phase timing, printed when FXG_PROFILE is set (development aid; worker 0 only)
struct HostProf {
    bool on = std::getenv("FXG_PROFILE") != nullptr;
    double acc[16] = {0}, acc_cpu[16] = {0};     // wall and thread-CPU milliseconds per phase
    const char* names[16] = {"setup", "admission", "build_passes", "plan", "sort", "tasks+h2d", "launch", "root prep", "sync+d2h", "finish",
                             "root chunk", "root sync", "walk issue", "emit", "barrier", "cigars d2h"};
    std::chrono::steady_clock::time_point t0;
    double c0 = 0;
    void start(Worker const& w) { if (on && w.id == 0) { t0 = std::chrono::steady_clock::now(); c0 = thread_cpu_ms(); } }
    void lap(Worker const& w, int i) {
        if (!on || w.id != 0) return;
        auto t1 = std::chrono::steady_clock::now();
        double const c1 = thread_cpu_ms();
        acc[i] += std::chrono::duration<double, std::milli>(t1 - t0).count();
        acc_cpu[i] += c1 - c0;
        t0 = t1; c0 = c1;
    }
    void report() {
        if (!on) return;
        for (int i = 0; i < 16; ++i) if (names[i][0]) fprintf(stderr, "[fxg] %-14s %8.3f ms  (%.3f ms of CPU)\n", names[i], acc[i], acc_cpu[i]);
        for (double& a : acc) a = 0;
        for (double& a : acc_cpu) a = 0;
    }
};
HostProf g_prof;

struct ClassDef { uint8_t widx, G; uint32_t max_words; };   // a (block width, ring size) configuration of the engine and its widest Eq table

// The device-resident records of a job (prepare_job / run_device_walks).
struct Prepared {
    bool ok = false;                     // the device-side walk can take the job
    DevBuf dev; PinnedBuf staging;       // nodes | leaves | reads | anchors, carved at the offsets below
    size_t o_nodes = 0, o_leaves = 0, o_reads = 0, o_anchors = 0, used = 0;   // (64 spare bytes follow the records in `staging`)
    uint32_t n_nodes = 0, n_leaves = 0, n_walks = 0, n_reads = 0;
    uint32_t max_depth = 0;
    uint32_t level_mask[256] = {0};      // classes that occur per tree depth
    std::vector<ReadRec> hreads;         // the ReadRecs on the host (bases relative to the job)
    cudaEvent_t ready = nullptr;         // the upload has finished
};

struct Ticket;

}  // namespace

std::atomic<uint64_t> g_ctx_serial{0};

struct fxg_ctx {
    uint64_t serial = ++g_ctx_serial;     // never reused, unlike the context's address
    int device = 0;
    std::string err;
    RefStore refs;
    bool have_refs = false;
    fxg_counters ctr{};
    int num_sms = 0;
    size_t smem_limit = 0;
    static constexpr int kMaxGroups = 32;
    int n_groups = 6;                     // batches that can be in flight (FXG_GROUPS, read by fxg_create)
    WorkerGroup groups[kMaxGroups];
    cudaStream_t stage_stream = nullptr; // uploads of references / query pools, Peq construction
    DevBuf d_tmp;
    uint64_t trace_budget = 0;
    int workers_busy = 4;                        // workers a group uses when more than a quarter of the groups are busy
    bool device_levels = true;                   // FXG_DEVICE_LEVELS=0 runs the inner tree levels from the host (development knob)
    bool share_root_passes = true;               // FXG_SHARE_ROOTS=0 scores every root window on its own (development knob)
    bool infer_inner = true;                     // FXG_INFER_INNER=0 computes every inner window (development knob)
    bool device_roots = true;                    // FXG_DEVICE_ROOTS=0 runs the root level from the host (development knob)
    bool force_wide = false;                     // FXG_FORCE_WIDE=1 sends every pass to the multi-warp kernel (development knob: tests)
    int root_chunks = 1, root_chunk_min = 512;   // FXG_ROOT_CHUNKS / FXG_ROOT_CHUNK_MIN (development knobs, read by fxg_create)
    std::vector<Pool> spare_pools;       // device buffers of freed batches / jobs, reused by the next stage call
    std::vector<PinnedBuf> spare_pinned; // page-locked cigar pools of freed batches / jobs (cudaHostAlloc costs milliseconds)
    std::vector<DevBuf> spare_dev;       // record buffers of freed jobs ...
    std::vector<PinnedBuf> spare_staging;// ... and the page-locked memory they were uploaded from
    std::mutex mu;
    // the queue of fxg_verify_run / fxg_verify_reads calls: a caller that finds a free worker group takes every compatible
    // job that is waiting with it and runs them as one batch (submit_and_wait)
    std::vector<Ticket*> pending;
    std::condition_variable cv;
    uint64_t merge_max_walks = uint64_t(1) << 20;   // FXG_MERGE_WALKS: anchors of a merged batch at most (a single job may be larger)
    int merge_max_jobs = 16;                        // FXG_MERGE_JOBS (1 = never merge)
    int merged_parts = 1;                           // FXG_MERGED_PARTS: host workers (and launch sets) of a merged batch
    int merge_wait_us = 300;                        // FXG_MERGE_WAIT_US: how long a job waits for company while other batches run
    double alloc_ms0 = 0; uint64_t alloc_calls0 = 0;    // allocation time / calls at the last fxg_reset_counters
    std::mutex class_mu;
    ClassDef classes[kMaxLevelClasses];
    int n_classes = 0;
    int seeders_reading = 0;             // fxg_gpu_seeder_create / fxg_seed_reads calls that read the packed store without mu
};

struct fxg_batch {
    std::vector<fxg_align_task> tasks;
    // the tasks' DP passes, made when the batch is staged (fxg_align_batch_run is device work): score passes and passes whose
    // CIGAR is wanted, each with the task it belongs to; a task without a pass has its result already
    std::vector<Pass> passes, root_passes;
    std::vector<uint32_t> owner, root_owner, root_k;
    uint64_t passes_refs_version = ~uint64_t(0);     // the reference store the passes' positions refer to
    Pool pool;
    std::vector<fxg_align_result> results;
    PinnedBuf cigars;                    // the device writes the cigars of a run straight into this pool
    size_t cigars_len = 0;
    bool ran = false;
};

namespace {

enum : uint8_t { W_WAITING = 0, W_WALKING = 1, W_DONE = 2 };

struct Span { uint64_t offset, length, extra; };

struct Walk {                 // one query_verifier::verify() call
    uint32_t read, anchor;    // anchor = index into the job's anchor array
    uint32_t group;           // verified_intervals set it shares (read, orientation, reference)
    uint8_t orient, state;
    bool hit;
    const fxg_pex_node* node; // node to align next
    uint64_t r_start, r_end;  // root window
    uint64_t t_start, t_end;  // root window trimmed by the extra length (root_was_already_verified)
    Span root_span;
    bool have_root_span;
    uint32_t n_inner; uint64_t sum_inner, cells_inner;   // its inner-node alignments so far (verification.cpp:238-242)
    uint64_t start_in_reference; uint32_t num_errors; uint64_t cigar_offset; uint32_t cigar_len;
    uint32_t ref_id, member;  // reference of its anchor; member job of its read
    uint32_t rm, rk;          // the root node's piece length and errors ...
    uint64_t rqbase;          // ... and where that piece begins in the pool, in the walk's orientation
};

struct Group { uint32_t first, count; };   // members are consecutive entries of group_members

}  // namespace

struct fxg_job {
    fxg_verify_config cfg{};
    // the batch: either the job's own copies (fxg_verify_stage) or the caller's arrays, borrowed for the duration of
    // the one call that uses them (fxg_verify_reads)
    std::vector<fxg_read> reads;
    std::vector<fxg_pex_node> nodes;
    std::vector<fxg_anchor> anchors;
    const fxg_read* reads_p = nullptr; const fxg_pex_node* nodes_p = nullptr; const fxg_anchor* anchors_p = nullptr;
    size_t n_reads = 0, n_nodes = 0, n_anchors = 0;
    bool borrowed = false;
    uint64_t pool_len = 0;
    Pool pool;                           // forward pool followed by the reverse-complement pool
    std::vector<uint32_t> read_walk_begin;   // per read (+1 sentinel): index of its first walk (= anchor) in job order
    Prepared prep;
    cudaEvent_t pool_ready = nullptr;    // (fxg_verify_reads) the query pools and their Peq planes are in place
    // results
    std::vector<fxg_alignment> alignments;
    PinnedBuf cigars;                    // page-locked; every worker's cigars arrive here directly from the device
    size_t cigars_len = 0;
    std::vector<uint32_t> cigars_copy;   // a job that ran merged with others copies its cigars out of the batch's pool
    bool use_copy = false;
    fxg_stats stats{};
    bool ran = false;
};

namespace {

// The text of the calling thread's last failed call (fxg_last_error): calls run concurrently on one context, so the
// message is kept per thread, not per context.
thread_local std::string tls_last_error;

int fail(std::string& err, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    err = buf;
    tls_last_error = buf;
    return code;
}

#define CUDA_TRY(errstr, expr)                                                                          \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) return fail(errstr, FXG_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

void add_counters(fxg_counters& a, fxg_counters const& b) {
    a.kernel_launches += b.kernel_launches; a.dp_tasks += b.dp_tasks; a.dp_word_steps += b.dp_word_steps;
    a.dp_cells_full += b.dp_cells_full; a.trace_bytes += b.trace_bytes; a.h2d_bytes += b.h2d_bytes; a.d2h_bytes += b.d2h_bytes;
    a.root_launch_ms += b.root_launch_ms; a.root_launch_word_steps += b.root_launch_word_steps; a.shared_tracebacks += b.shared_tracebacks; a.inferred_inner += b.inferred_inner;
    a.shared_score_passes += b.shared_score_passes; a.rescored_roots += b.rescored_roots; a.batches += b.batches; a.batch_jobs += b.batch_jobs; a.root_launches += b.root_launches;
    a.trace_word_steps += b.trace_word_steps; a.dp_kernel_ms += b.dp_kernel_ms; a.trace_kernel_ms += b.trace_kernel_ms; a.waves += b.waves; a.run_ms += b.run_ms;
}

// brackets a *_run call with events on the stream of the group's first worker (the first kernels are launched there)
struct RunTimer {
    WorkerGroup& g; fxg_counters& ctr;
    RunTimer(WorkerGroup& group, fxg_counters& counters) : g(group), ctr(counters) { cudaEventRecord(g.ev_run0, g.workers[0]->stream); }
    ~RunTimer() {
        if (cudaEventRecord(g.ev_run1, g.workers[0]->stream) != cudaSuccess || cudaEventSynchronize(g.ev_run1) != cudaSuccess) return;
        float ms = 0;
        if (cudaEventElapsedTime(&ms, g.ev_run0, g.ev_run1) == cudaSuccess) ctr.run_ms += ms;
    }
};

// a free worker group, waiting for one if both are busy; call with c->mu held through `lock`
WorkerGroup& acquire_group(fxg_ctx* c, std::unique_lock<std::mutex>& lock) {
    for (;;) {
        int busy = 0;
        for (int i = 0; i < c->n_groups; ++i) busy += c->groups[i].busy;
        for (int i = 0; i < c->n_groups; ++i) if (!c->groups[i].busy) {
            WorkerGroup& g = c->groups[i];
            g.busy = true;
            g.use_workers = busy == 0 ? g.workers.size() : std::min(g.workers.size(), size_t(c->workers_busy));
            return g;
        }
        c->cv.wait(lock);
    }
}
void release_group(fxg_ctx* c, WorkerGroup& g) { g.busy = false; c->cv.notify_all(); }

int env_int(const char* name, int dflt, int lo, int hi) {
    if (const char* e = std::getenv(name)) { int const v = std::atoi(e); if (v >= lo && v <= hi) return v; }
    return dflt;
}

// ------------------------------------------------------------------------------------------------ kernel dispatch

template <int W, bool CKPT>
cudaError_t launch_one(DpLaunch const& L, uint32_t grid, size_t smem, cudaStream_t s) {
    dp_kernel<W, CKPT><<<grid, 32, smem, s>>>(L);
    return cudaGetLastError();
}

cudaError_t launch_dp(int widx, bool checkpoints, DpLaunch const& L, uint32_t grid, size_t smem, cudaStream_t s) {
    if (widx < 0) {                                  // the multi-warp kernel for bands no ring of one warp holds
        if (checkpoints) dp_wide_kernel<true><<<grid, kWideThreads, smem, s>>>(L);
        else dp_wide_kernel<false><<<grid, kWideThreads, smem, s>>>(L);
        return cudaGetLastError();
    }
    switch (widx * 2 + (checkpoints ? 1 : 0)) {
        case 0: return launch_one<1, false>(L, grid, smem, s);
        case 1: return launch_one<1, true>(L, grid, smem, s);
        case 2: return launch_one<2, false>(L, grid, smem, s);
        case 3: return launch_one<2, true>(L, grid, smem, s);
        case 4: return launch_one<4, false>(L, grid, smem, s);
        case 5: return launch_one<4, true>(L, grid, smem, s);
        case 6: return launch_one<8, false>(L, grid, smem, s);
        case 7: return launch_one<8, true>(L, grid, smem, s);
        case 8: return launch_one<16, false>(L, grid, smem, s);
        case 9: return launch_one<16, true>(L, grid, smem, s);
        case 10: return launch_one<32, false>(L, grid, smem, s);
        case 11: return launch_one<32, true>(L, grid, smem, s);
    }
    return cudaErrorInvalidValue;
}

template <int W>
cudaError_t launch_walk_one(Walk2Launch const& L, cudaStream_t s) {
    size_t const smem = walk2_smem_bytes(W);
    walk2_kernel<W><<<(L.n_tasks + walk2_per_cta(W) - 1) / walk2_per_cta(W), walk2_threads(), smem, s>>>(L);
    return cudaGetLastError();
}

cudaError_t launch_walk(int widx, Walk2Launch const& L, cudaStream_t s) {
    switch (widx) {
        case 0: return launch_walk_one<1>(L, s);
        case 1: return launch_walk_one<2>(L, s);
        case 2: return launch_walk_one<4>(L, s);
        case 3: return launch_walk_one<8>(L, s);
        case 4: return launch_walk_one<16>(L, s);
        case 5: return launch_walk_one<32>(L, s);
    }
    return cudaErrorInvalidValue;
}

template <int W>
cudaError_t set_smem_attr(size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(dp_kernel<W, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(dp_kernel<W, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
    if (e == cudaSuccess && walk2_smem_bytes(W) <= bytes) e = cudaFuncSetAttribute(walk2_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(walk2_smem_bytes(W)));
    return e;
}

cudaError_t set_all_smem_attrs(size_t bytes) {
    cudaError_t e;
#define FXG_SET(W) if ((e = set_smem_attr<W>(bytes)) != cudaSuccess) return e;
    FXG_SET(1) FXG_SET(2) FXG_SET(4) FXG_SET(8) FXG_SET(16) FXG_SET(32)
#undef FXG_SET
    if (wide_smem_bytes() <= bytes) {
        if ((e = cudaFuncSetAttribute(dp_wide_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(wide_smem_bytes()))) != cudaSuccess) return e;
        if ((e = cudaFuncSetAttribute(dp_wide_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(wide_smem_bytes()))) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ------------------------------------------------------------------------------------------------ configuration choice

inline uint32_t peq_stride_for(uint32_t words) { return (words + 3u) & ~3u; }   // rows stay 16-byte aligned for LDS.128

// shared memory of an engine launch with ring size G and Eq tables of `words` words: a window buffer and a table per
// task of the warp, or the multi-warp kernel's (G = kWideG)
inline size_t engine_smem_bytes(uint32_t G, uint32_t words) {
    return G == kWideG ? wide_smem_bytes() : size_t(32 / G) * (kWinBytes + size_t(kNumSymbols) * peq_stride_for(words) * 4);
}

// word-steps the engine issues for a pass: block b is active for columns cs(b)..ce(b)
uint64_t word_steps_of(Pass const& p, uint32_t W, uint32_t nb) {
    uint32_t const rows = 32 * W;
    int64_t const pad = int64_t(nb) * rows - p.m;
    uint64_t ws = 0;
    for (uint32_t b = 0; b < nb; ++b) {
        int64_t lo = int64_t(rows) * b + 1 + p.dlo - pad, hi = int64_t(rows) * (b + 1) + p.dhi - pad;
        if (lo < 1) lo = 1;
        if (hi > p.n) hi = p.n;
        if (hi >= lo) ws += uint64_t(hi - lo + 1) * W;
    }
    return ws;
}

// Picks words-per-lane W and ring size G for one pass.  A lane takes its next block (G blocks further down) only after
// its current one has ended: with R = 32 W rows per block, block b works during the steps (R + 1) b + 1 + dlo ..
// (R + 1) b + R + dhi, so
//   (R + 1) G >= R + B - 1,  B = number of diagonals in the band,  i.e.  G >= 2 + (B - 3) / (R + 1).
// (The block below a block that has ended substitutes the "+1 per column" bound itself -- run_steps, `Upper` -- so the
// lane above need not stay idle for it; that requirement cost one more lane per ring in round 1.)
// FXG_LATENCY_WEIGHT > 0 makes the chooser prefer narrower blocks (development knob; measured with 0.3 on config 2: a batch
// running alone 7.4 -> 6.9 ms, 16 batches in flight unchanged, a machine-filling launch 0.61 -> 0.48 of the issue peak)
double g_latency_weight = [] { const char* e = std::getenv("FXG_LATENCY_WEIGHT"); return e ? std::atof(e) : 0.0; }();

inline int64_t ring_lanes_needed(int64_t B, uint32_t W) { return B > 4 ? 2 + (B - 3) / (32 * int64_t(W) + 1) : 3; }
// the widest band a ring of G lanes takes (inverse of ring_lanes_needed)
inline int64_t ring_band_limit(uint32_t G, uint32_t W) { return 2 + (int64_t(G) - 1) * (32 * int64_t(W) + 1); }

bool choose_config(Pass const& p, size_t smem_limit, bool force_wide, Config& out, bool traced = false) {
    uint32_t const nw = (p.m + 31) / 32;
    int64_t const B = int64_t(p.dhi) - int64_t(p.dlo) + 1;
    double best_cost = 1e300;
    bool found = false;
    for (int wi = 0; wi < 6 && !force_wide; ++wi) {
        uint32_t const W = uint32_t(kWidths[wi]);
        uint32_t const nb = (nw + W - 1) / W;
        uint32_t G;
        if (nb == 1) G = 1;
        else {
            int64_t const need = ring_lanes_needed(B, W);
            int64_t const g = std::max<int64_t>(std::min<int64_t>(need, nb), 2);
            if (g > 32) continue;
            G = uint32_t(g);
        }
        uint32_t const tpw = 32 / G;
        G = 32 / tpw;                        // the lanes a smaller ring would leave idle cost nothing, and fewer classes mean fuller launches
        size_t const smem = engine_smem_bytes(G, nb * W);
        if (smem > smem_limit) continue;
        // The engine is bound by the ALU pipe: a warp step issues about 10 W + 6 instructions there, two cycles each on one
        // of the SM's four schedulers, whatever the number of lanes that do useful work.  Wide blocks need many registers
        // (fewer warps to hide the shuffle latency behind); many tables per SM cost occupancy as well.
        double const resident = std::min<double>(32.0, std::floor(double(227 * 1024) / double(smem + 1024)));
        double const reg_eff = W <= 8 ? 1.0 : (W == 16 ? 0.85 : 0.7);
        double const occ_eff = std::min(1.0, resident / 12.0);
        uint64_t const steps = uint64_t(p.n) + nb - 1;
        double cost = double(steps) * (10.0 * W + 6.0) * 2.0 / 4.0 / (reg_eff * occ_eff) / tpw;      // SM cycles per task
        // every block start / end interrupts the warp for a few hundred issue slots; the rings of a warp mostly, but not
        // always, have the same shape and then share these interruptions
        cost += 2.0 * nb * 100.0 / std::sqrt(double(tpw));
        // a task is also a chain of `steps` dependent steps, each as long as the dependent instructions of one column
        cost += g_latency_weight * double(steps) * (30.0 + 12.0 * W);
        // A pass whose CIGAR is wanted is followed by its traceback (walk2_kernel<W>): the tiles (block x 32 steps) the path
        // crosses are recomputed by a group of W lanes, 32 + W single-word steps of ~25 instructions each.  Counted as if
        // every pass were traced: where few are (repeat-rich references) the pass itself is long and this term is small.
        // Measured on config 2 (profiles/r02_config2_issue_share_final.txt): pass + traceback 133 k + 36 k ALU-pipe warp
        // instructions per read at W = 4 against 125 k + 60 k at W = 8.
        if (traced) cost += (double(p.n) / 32.0 + nb) * (32.0 + W) * 25.0 * 0.5 * (double(W) / 32.0);
        if (cost < best_cost) { best_cost = cost; out = Config{uint8_t(wi), uint8_t(G), nb, 0}; found = true; }
    }
    if (!found) {
        // no ring of one warp holds this band: the multi-warp kernel (dp_wide_kernel), one block of 1 024 rows per thread
        uint32_t const nb = (nw + 31) / 32;
        if (nb <= kWideThreads && engine_smem_bytes(kWideG, nb * 32) <= smem_limit) { out = Config{5, uint8_t(kWideG), nb, 0}; found = true; }
    }
    if (found) out.word_steps = word_steps_of(p, uint32_t(kWidths[out.widx]), out.nb);
    return found;
}

// the same (m, n, band) recurs for every anchor of a read at one tree level: memoise
bool cached_config(std::vector<ConfigCacheEntry>& cache, Pass const& p, size_t smem_limit, bool force_wide, Config& out, bool traced = false) {
    uint64_t h = (uint64_t(p.n) * 0x9E3779B97F4A7C15ull) ^ (uint64_t(p.m) * 0xC2B2AE3D27D4EB4Full) ^ (uint64_t(uint32_t(p.dlo)) << 21) ^ uint64_t(uint32_t(p.dhi));
    h ^= h >> 29;
    ConfigCacheEntry& e = cache[(h + (traced ? 1 : 0)) & (cache.size() - 1)];
    if (e.valid && e.traced == traced && e.n == p.n && e.m == p.m && e.dlo == p.dlo && e.dhi == p.dhi) { out = e.cfg; return e.ok; }
    e.valid = true; e.traced = traced; e.n = p.n; e.m = p.m; e.dlo = p.dlo; e.dhi = p.dhi;
    e.ok = choose_config(p, smem_limit, force_wide, e.cfg, traced);
    out = e.cfg;
    return e.ok;
}

// Host loops over a million independent alignments (fxg_align_batch: the verification-only microbenchmark of config 5)
// are cut into contiguous chunks for up to 8 threads; the loops of a verification batch stay on the caller's thread.
size_t parallel_threads(size_t n, size_t min_chunk) {
    size_t const hw = std::max<size_t>(1, std::thread::hardware_concurrency() / 2);
    return std::max<size_t>(1, std::min<size_t>({size_t(8), hw, n / std::max<size_t>(min_chunk, 1)}));
}
template <class F> void parallel_chunks(size_t T, size_t n, F&& f) {         // f(thread, lo, hi); the caller's thread takes the first chunk
    if (T <= 1) { f(size_t(0), size_t(0), n); return; }
    std::vector<std::thread> th;
    th.reserve(T - 1);
    for (size_t t = 1; t < T; ++t) th.emplace_back([&f, t, T, n] { f(t, n * t / T, n * (t + 1) / T); });
    f(size_t(0), size_t(0), n / T);
    for (std::thread& x : th) x.join();
}

// LSD radix sort of 64-bit keys on bits [lo_bit, hi_bit): per-thread histograms, then every thread scatters its own chunk
// to where the chunks before it leave off (stable)
void radix_sort(std::vector<uint64_t>& keys, std::vector<uint64_t>& tmp, int lo_bit, int hi_bit) {
    size_t const N = keys.size();
    tmp.resize(N);
    size_t const T = parallel_threads(N, size_t(1) << 16);
    std::vector<uint32_t> hist(T * 2048);
    for (int shift = lo_bit; shift < hi_bit; shift += 11) {
        std::fill(hist.begin(), hist.end(), 0u);
        const uint64_t* const src = keys.data();
        uint64_t* const dst = tmp.data();
        parallel_chunks(T, N, [&](size_t t, size_t lo, size_t hi) {
            uint32_t* const h = hist.data() + t * 2048;
            for (size_t i = lo; i < hi; ++i) h[(src[i] >> shift) & 2047u]++;
        });
        uint32_t running = 0;
        for (size_t d = 0; d < 2048; ++d)
            for (size_t t = 0; t < T; ++t) { uint32_t const n = hist[t * 2048 + d]; hist[t * 2048 + d] = running; running += n; }
        parallel_chunks(T, N, [&](size_t t, size_t lo, size_t hi) {
            uint32_t* const h = hist.data() + t * 2048;
            for (size_t i = lo; i < hi; ++i) dst[h[(src[i] >> shift) & 2047u]++] = src[i];
        });
        keys.swap(tmp);
    }
}

std::vector<ConfigCacheEntry>& thread_config_cache(const fxg_ctx* c);

// ------------------------------------------------------------------------------------------------ running passes

// One engine launch over the tasks of class K: n_tasks of them, counted on the host, or -- n_tasks_dev set -- as many as
// the device has counted there for class `cls` of class_active, n_tasks being an upper bound.  ck: the checkpoint buffer
// of a launch that leaves checkpoint records, else nullptr.
struct EngineLaunch { DpLaunch L; int widx; uint32_t grid; size_t smem; };      // widx -1: dp_wide_kernel
int engine_launch(fxg_ctx* c, Worker& w, Pool const& pool, ClassDef const& K, const DpTask* tasks, DpResult* results, uint32_t* ck, uint32_t n_tasks,
                  const uint32_t* n_tasks_dev, const uint32_t* class_active, uint32_t cls, EngineLaunch& X) {
    bool const wide = K.G == kWideG;
    uint32_t const tpw = wide ? 1u : 32u / K.G;
    DpLaunch& L = X.L;
    L = DpLaunch{};
    L.tasks = tasks; L.n_tasks = n_tasks; L.n_tasks_dev = n_tasks_dev; L.class_active = class_active; L.cls = cls;
    L.group = K.G; L.win_stride = kWinBytes; L.two = 2;
    L.peq_stride = peq_stride_for(K.max_words);
    L.ref_packed = c->refs.packed.as<uint32_t>(); L.ref_chunks = c->refs.total / 32 + 1;
    // (read only for tasks flagged kFlagInlineRef: fxg_align_batch's against inline references; the device builds none)
    L.inline_packed = pool.inline_packed.as<uint32_t>(); L.inline_chunks = pool.inline_len / 32 + 1;
    L.peq_table = pool.peq.as<uint32_t>(); L.peq_plane_words = pool.plane_words;
    L.results = results; L.trace = ck;
    X.widx = wide ? -1 : int(K.widx);
    X.smem = engine_smem_bytes(K.G, K.max_words);
    if (X.smem > c->smem_limit) return fail(w.err, FXG_ERR_INVALID_ARGUMENT, "internal: launch needs %zu bytes of shared memory", X.smem);
    if (n_tasks_dev)        // (no more CTAs than a few waves of the machine: the CTAs take the task groups in turn)
        X.grid = uint32_t(std::min<size_t>((size_t(n_tasks) + tpw - 1) / tpw, size_t(c->num_sms) * (wide ? 2 : 32)));
    else
        X.grid = wide ? uint32_t(std::min<size_t>(n_tasks, size_t(c->num_sms) * 2)) : (n_tasks + tpw - 1) / tpw;
    return FXG_OK;
}

// The tracebacks of n_tasks alignments whose score passes left their checkpoint records in ck; they write to the
// worker's cigar buffer and traceback results.
Walk2Launch walk_launch(fxg_ctx* c, Worker& w, Pool const& pool, const uint32_t* ck, const Walk2Task* tasks, uint32_t n_tasks) {
    Walk2Launch WL{};
    WL.tasks = tasks; WL.n_tasks = n_tasks; WL.ck = ck;
    // (read only for tasks flagged kFlagInlineRef: fxg_align_batch's against inline references; the device builds none)
    WL.ref_packed = c->refs.packed.as<uint32_t>(); WL.inline_packed = pool.inline_packed.as<uint32_t>();
    WL.peq_table = pool.peq.as<uint32_t>(); WL.peq_plane_words = pool.plane_words;
    WL.cigars = w.d_cigars.as<uint32_t>(); WL.results = w.d_wresults.as<WalkResult>(); WL.two = 2;
    return WL;
}

// Runs `passes` on the worker's streams: plain score passes, or (ck_bases != nullptr) score passes that leave checkpoint
// records at those offsets of the worker's checkpoint buffer.
// results points to pinned memory owned by the worker and stays valid until its next call.
int run_passes(fxg_ctx* c, Worker& w, Pool const& pool, std::vector<Pass> const& passes, const uint64_t* ck_bases, uint32_t* ck_buffer,
               const DpResult** results, std::function<int()> const* after_launch = nullptr) {
    size_t const N = passes.size();
    *results = nullptr;
    if (N == 0) return FXG_OK;
    bool const trace = ck_bases != nullptr;

    g_prof.start(w);
    // sort key: configuration (descending cost class), then steps descending, then the pass index
    w.cfgs.resize(N);
    w.keys.resize(N);
    size_t const T = parallel_threads(N, size_t(1) << 16);
    {
        std::vector<size_t> bad(T, SIZE_MAX);
        parallel_chunks(T, N, [&](size_t t, size_t lo, size_t hi) {
            std::vector<ConfigCacheEntry>& cache = t == 0 ? w.cfg_cache : thread_config_cache(c);
            for (size_t i = lo; i < hi; ++i) {
                Config& cf = w.cfgs[i];
                if (!cached_config(cache, passes[i], c->smem_limit, c->force_wide, cf, trace)) { bad[t] = i; return; }
                uint64_t const steps = std::min<uint64_t>(uint64_t(passes[i].n) + cf.nb - 1, (1u << 19) - 1);
                uint64_t const cls = cf.G == kWideG ? 0 : uint64_t(5 - cf.widx) * 32 + (32 - cf.G) + 1;         // 0 = the multi-warp kernel, 1 = W 32, G 32
                w.keys[i] = (cls << 51) | ((((1ull << 19) - 1) - steps) << 32) | uint64_t(i);
            }
        });
        for (size_t t = 0; t < T; ++t)
            if (bad[t] != SIZE_MAX)
                return fail(w.err, FXG_ERR_INVALID_ARGUMENT, "alignment of query length %u against window %u with band %d..%d exceeds the supported size",
                            passes[bad[t]].m, passes[bad[t]].n, passes[bad[t]].dlo, passes[bad[t]].dhi);
    }
    g_prof.lap(w, 3);
    radix_sort(w.keys, w.keys_tmp, 32, 64);
    g_prof.lap(w, 4);

    CUDA_TRY(w.err, w.h_tasks.ensure(N * sizeof(DpTask)));
    CUDA_TRY(w.err, w.h_results.ensure(N * sizeof(DpResult)));
    CUDA_TRY(w.err, w.d_tasks.ensure(N * sizeof(DpTask)));
    CUDA_TRY(w.err, w.d_results.ensure(N * sizeof(DpResult)));
    DpTask* tasks = w.h_tasks.as<DpTask>();
    {
        std::vector<uint64_t> sums(2 * T, 0);
        parallel_chunks(T, N, [&](size_t th, size_t lo, size_t hi) {
            uint64_t ws = 0, cells = 0;
            for (size_t i = lo; i < hi; ++i) {
                uint32_t const idx = uint32_t(w.keys[i]);
                Pass const& p = passes[idx];
                DpTask& t = tasks[i];
                t.ref_base = p.ref_base; t.query_base = p.query_base;
                t.trace_base = trace ? ck_bases[idx] : 0;
                t.n = p.n; t.m = p.m; t.dlo = p.dlo; t.dhi = p.dhi; t.flags = p.flags; t.out = idx;
                ws += w.cfgs[idx].word_steps;
                cells += uint64_t(p.m) * p.n;
            }
            sums[2 * th] = ws; sums[2 * th + 1] = cells;
        });
        for (size_t th = 0; th < T; ++th) { w.ctr.dp_word_steps += sums[2 * th]; w.ctr.dp_cells_full += sums[2 * th + 1]; }
    }
    w.ctr.dp_tasks += N;
    CUDA_TRY(w.err, cudaMemcpyAsync(w.d_tasks.p, tasks, N * sizeof(DpTask), cudaMemcpyHostToDevice, w.stream));
    w.ctr.h2d_bytes += N * sizeof(DpTask);
    g_prof.lap(w, 5);

    CUDA_TRY(w.err, cudaEventRecord(w.ev0, w.stream));
    struct Launch { EngineLaunch E; uint64_t work, word_steps; };
    std::vector<Launch> launches;
    size_t i = 0;
    while (i < N) {
        // one launch: same (W, G)
        Config const& c0 = w.cfgs[uint32_t(w.keys[i])];
        int const widx = c0.widx; uint32_t const G = c0.G;
        uint32_t const W = uint32_t(kWidths[widx]);
        uint32_t const tpw = G == kWideG ? 1 : 32 / G;
        size_t j = i;
        uint32_t max_words = 0;
        uint64_t work = 0, ws = 0;
        while (j < N) {
            uint32_t const idx = uint32_t(w.keys[j]);
            Config const& cj = w.cfgs[idx];
            if (cj.widx != widx || cj.G != G) break;
            max_words = std::max(max_words, cj.nb * W);
            work += (uint64_t(passes[idx].n) + cj.nb) * (10 * W + 6);
            ws += cj.word_steps;
            ++j;
        }
        Launch X{};
        int const rc = engine_launch(c, w, pool, ClassDef{uint8_t(widx), uint8_t(G), max_words}, w.d_tasks.as<DpTask>() + i, w.d_results.as<DpResult>(),
                                     ck_buffer, uint32_t(j - i), nullptr, nullptr, 0, X.E);
        if (rc != FXG_OK) return rc;
        X.work = work / tpw; X.word_steps = ws;
        launches.push_back(X);
        i = j;
    }
    // largest first on the worker's own stream, the rest spread over the side streams so that they fill the machine together
    std::sort(launches.begin(), launches.end(), [](Launch const& a, Launch const& b) { return a.work > b.work; });
    int const n_launch = int(launches.size());
    CUDA_TRY(w.err, w.fork(w.stream, n_launch));
    for (int q = 0; q < n_launch; ++q) {
        EngineLaunch const& X = launches[q].E;
        cudaStream_t st;
        CUDA_TRY(w.err, w.fan_stream(w.stream, q, st));
        if (q == 0 && trace) CUDA_TRY(w.err, cudaEventRecord(w.ev_b0, w.stream));
        CUDA_TRY(w.err, launch_dp(X.widx, trace, X.L, X.grid, X.smem, st));
        if (q == 0 && trace) CUDA_TRY(w.err, cudaEventRecord(w.ev_b1, w.stream));
        w.ctr.kernel_launches++;
    }
    CUDA_TRY(w.err, w.join(w.stream, n_launch));
    CUDA_TRY(w.err, cudaEventRecord(w.ev1, w.stream));
    g_prof.lap(w, 6);
    CUDA_TRY(w.err, cudaMemcpyAsync(w.h_results.p, w.d_results.p, N * sizeof(DpResult), cudaMemcpyDeviceToHost, w.stream));
    w.ctr.d2h_bytes += N * sizeof(DpResult);
    if (after_launch) {                              // more work of the caller's that needs the engine's results on the device only
        int const rc = (*after_launch)();
        if (rc != FXG_OK) return rc;
    }
    CUDA_TRY(w.err, w.wait_for(w.stream));
    float ms = 0;
    CUDA_TRY(w.err, cudaEventElapsedTime(&ms, w.ev0, w.ev1));
    w.ctr.dp_kernel_ms += ms;
    if (g_prof.on && std::getenv("FXG_TRACE_WAVES")) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, w.group->ev_run0, w.ev0); cudaEventElapsedTime(&b, w.group->ev_run0, w.ev1);
        fprintf(stderr, "[fxg] timeline worker %d %s %zu passes: device %.3f .. %.3f ms\n", w.id, trace ? "root" : "wave", N, a, b);
    }
    if (trace) {
        // the largest launch of a root wave is the engine's dominant launch: timed on its own for the roofline
        CUDA_TRY(w.err, cudaEventElapsedTime(&ms, w.ev_b0, w.ev_b1));
        w.ctr.root_launch_ms += ms; w.ctr.root_launch_word_steps += launches[0].word_steps; w.ctr.root_launches++;
    }
    g_prof.lap(w, trace ? 11 : 8);
    *results = w.h_results.as<DpResult>();
    for (size_t q = 0; q < N; ++q)
        if ((*results)[q].score == kPoisonScore) return fail(w.err, FXG_ERR_CUDA, "internal: the DP engine lost track of its window buffer");
    return FXG_OK;
}

// ops reserved for the cigar of an alignment with s errors: at most s error runs and s + 1 match runs
inline uint64_t cigar_cap_for(uint32_t s) { return uint64_t(2) * s + 3; }

// result of a root alignment whose CIGAR is wanted
struct RootOut {
    int32_t score; uint32_t end_col;     // as DpResult
    uint32_t begin_col;                  // column where the traceback reached row 0
    uint64_t cigar_offset;               // first op, counted in the worker's cigar buffer (w.d_cigars)
    uint32_t cigar_len;
};

// Score passes with checkpoints + tracebacks for `passes` (alignment.cpp:147-180): pass i is accepted when its score is
// at most max_errors[i]; accepted passes get their CIGAR, written by the device into a slot of cigar_cap_for(score) ops
// of the worker's cigar buffer (slots follow each other from w.cig_used on).  Works in chunks bounded by `budget_bytes`
// of checkpoint records.
//
// Shared score passes.  The anchors of one true locus lead to root windows of the same query piece that nearly coincide
// (they differ by the indels between the seeds).  Such windows are scored by ONE pass over their union U: for a member
// window B inside U, row m of B's own matrix is >= row m of U's at every column of B (B allows fewer start positions),
// with equality wherever some optimal alignment of U's cell starts inside B.  So with (L, e) = the minimum of U's row m
// over B's columns and the rightmost column attaining it (range_min_kernel):
//   * L > k: B holds no alignment with <= k errors either;
//   * L <= k and e - m - L >= (start of B - start of U): every alignment of cost L ending at e spans at most m + L
//     columns, hence starts inside B; B's matrix then agrees with U's on every cell such an alignment touches, B's
//     minimum is L, no column right of e attains it, and the traceback takes the same decisions (the argument of the
//     shared tracebacks below, DESIGN.md section 5) -- B's result is read off U's pass, shifted by the windows' distance;
//   * otherwise B is scored again on its own.
int run_root_passes(fxg_ctx* c, Worker& w, Pool const& pool, std::vector<Pass> const& passes, std::vector<uint32_t> const& max_errors,
                    uint64_t budget_bytes, std::vector<RootOut>& outs) {
    size_t const N = passes.size();
    outs.assign(N, RootOut{kNoScore, 0, 0, 0, 0});
    if (N == 0) return FXG_OK;
    g_prof.start(w);
    // kWalkSlots checkpoint buffers: the tracebacks of a chunk read one while the score passes of the next chunks fill the others
    uint64_t budget_words = std::max<uint64_t>(budget_bytes / Worker::kWalkSlots, uint64_t(64) << 20) / 4;

    // ---- units: the passes that are actually run, each serving one or more member windows ----
    struct Unit { Pass p; uint32_t k; uint32_t first, count; Config cfg; uint64_t words; };
    std::vector<Unit> units;
    std::vector<uint32_t> unit_members;
    auto finish_unit = [&](Unit& u) -> int {
        if (!cached_config(w.cfg_cache, u.p, c->smem_limit, c->force_wide, u.cfg, true))
            return fail(w.err, FXG_ERR_INVALID_ARGUMENT, "alignment of query length %u against window %u with band %d..%d exceeds the supported size",
                        u.p.m, u.p.n, u.p.dlo, u.p.dhi);
        uint32_t const W = uint32_t(kWidths[u.cfg.widx]);
        uint64_t const per_block = ck_records_per_block(int64_t(u.p.dhi) - int64_t(u.p.dlo) + 1, 32 * W);
        u.words = (uint64_t(u.cfg.nb) * per_block * ck_record_words(W) + 3) & ~uint64_t(3);
        return FXG_OK;
    };
    auto add_single = [&](uint32_t q) -> int {
        Unit u{passes[q], max_errors[q], uint32_t(unit_members.size()), 1, Config{}, 0};
        unit_members.push_back(q);
        int const rc = finish_unit(u);
        if (rc == FXG_OK) units.push_back(u);
        return rc;
    };
    // (sized up front: members scored again are appended while units are referenced, and a million growing push_backs
    //  cost more than the passes of a batch of small alignments)
    units.reserve(2 * N); unit_members.reserve(2 * N);
    {
        std::vector<uint32_t> order(N);
        for (size_t i = 0; i < N; ++i) order[i] = uint32_t(i);
        if (c->share_root_passes) {
            // windows of one query piece are to follow each other by position.  The passes of a read and strand arrive
            // together (walk order), so runs of equal (query piece, length) are sorted one by one -- a piece that shows up
            // in two separate runs merely shares less
            size_t r0 = 0;
            while (r0 < N) {
                size_t r1 = r0 + 1;
                while (r1 < N && passes[r1].query_base == passes[r0].query_base && passes[r1].m == passes[r0].m) ++r1;
                if (r1 - r0 > 1)
                    std::sort(order.begin() + long(r0), order.begin() + long(r1), [&](uint32_t a, uint32_t b) {
                        return passes[a].ref_base != passes[b].ref_base ? passes[a].ref_base < passes[b].ref_base : a < b;
                    });
                r0 = r1;
            }
        }
        // cost of a pass ~ columns x (diagonals of the band + one block of rows)
        auto cost = [](uint64_t n, uint64_t m, uint64_t k) { return double(n) * double(int64_t(n) - int64_t(m) + 2 * int64_t(k) + 256); };
        size_t i = 0;
        while (i < N) {
            uint32_t const q0 = order[i];
            Pass const& P0 = passes[q0];
            uint64_t const k0 = max_errors[q0];
            uint64_t u_start = P0.ref_base, u_end = P0.ref_base + P0.n;
            size_t j = i + 1;
            if (c->share_root_passes && P0.flags == 0) {
                while (j < N) {
                    Pass const& B = passes[order[j]];
                    if (B.query_base != P0.query_base || B.m != P0.m || B.flags != 0 || max_errors[order[j]] != k0 || B.ref_base > u_end) break;
                    uint64_t const new_end = std::max(u_end, B.ref_base + B.n);
                    if (cost(new_end - u_start, P0.m, k0) > cost(u_end - u_start, P0.m, k0) + 0.75 * cost(B.n, B.m, k0)) break;
                    u_end = new_end;
                    ++j;
                }
            }
            if (j - i == 1) {
                int const rc = add_single(q0);
                if (rc != FXG_OK) return rc;
            } else {
                Unit u{};
                u.k = uint32_t(k0); u.first = uint32_t(unit_members.size()); u.count = uint32_t(j - i);
                // the union as a window of its own: same band rule as score_pass_for
                u.p = P0; u.p.n = uint32_t(u_end - u_start);
                u.p.dlo = -int32_t(k0); u.p.dhi = int32_t(int64_t(u.p.n) - int64_t(u.p.m) + int64_t(k0));
                Config probe;
                if (cached_config(w.cfg_cache, u.p, c->smem_limit, c->force_wide, probe, true)) {
                    for (size_t q = i; q < j; ++q) unit_members.push_back(order[q]);
                    int const rc = finish_unit(u);
                    if (rc != FXG_OK) return rc;
                    units.push_back(u);
                } else {
                    // the union's band is wider than the engine takes although each member's may not be: every member on its own
                    for (size_t q = i; q < j; ++q) { int const rc = add_single(order[q]); if (rc != FXG_OK) return rc; }
                }
            }
            i = j;
        }
    }
    uint64_t total_words = 0, max_words = 0, cigar_bound = 0;
    for (Unit const& u : units) { total_words += u.words; max_words = std::max(max_words, u.words); }
    for (size_t i = 0; i < N; ++i) {
        cigar_bound += cigar_cap_for(max_errors[i]);
        // a member that has to be scored again on its own must fit the budget as well
        Config cf;
        if (cached_config(w.cfg_cache, passes[i], c->smem_limit, c->force_wide, cf, true)) {
            uint32_t const W = uint32_t(kWidths[cf.widx]);
            max_words = std::max(max_words, (uint64_t(cf.nb) * ck_records_per_block(int64_t(passes[i].dhi) - int64_t(passes[i].dlo) + 1, 32 * W) * ck_record_words(W) + 3) & ~uint64_t(3));
        }
    }
    if (max_words > budget_words) budget_words = max_words;
    // optionally cut a large batch into chunks whose tracebacks run beside the next chunk's score passes (measured on
    // config 2: no gain -- a traceback is one long chain of dependent steps, so the last chunk's tail stays, and the
    // tracebacks' shared memory takes occupancy from the score passes -- hence one chunk unless memory forces more)
    int const n_chunks = c->root_chunks, chunk_min = c->root_chunk_min;
    if (units.size() >= size_t(chunk_min) && n_chunks > 1)
        budget_words = std::min(budget_words, std::max<uint64_t>(total_words / uint64_t(n_chunks) + 1, max_words));
    // no reallocation while tracebacks are in flight: everything they write to is sized up front
    CUDA_TRY(w.err, w.d_cigars.ensure_preserving((w.cig_used + cigar_bound) * 4, w.cig_used * 4, w.stream));
    CUDA_TRY(w.err, w.h_wtasks.ensure(N * sizeof(Walk2Task)));
    CUDA_TRY(w.err, w.h_wresults.ensure(N * sizeof(WalkResult)));
    CUDA_TRY(w.err, w.d_wtasks.ensure(N * sizeof(Walk2Task)));
    CUDA_TRY(w.err, w.d_wresults.ensure(N * sizeof(WalkResult)));
    Walk2Task* const wt = w.h_wtasks.as<Walk2Task>();
    WalkResult* const wr = w.h_wresults.as<WalkResult>();

    g_prof.lap(w, 7);
    std::vector<Pass> chunk; std::vector<uint64_t> ck_base;
    std::vector<uint32_t> hit_pass;          // accepted members in traceback order (index into passes) ...
    std::vector<uint64_t> hit_shift;         // ... and how far their window starts behind the window of the pass that was traced
    std::vector<uint8_t> hit_widx;
    struct Accepted { uint32_t member, unit_in_chunk; uint32_t end_col_u; uint32_t score; };
    std::vector<Accepted> accepted;
    constexpr uint32_t kOwnTraceback = 0xfffffffeu, kNotAccepted = 0xffffffffu;
    std::vector<uint32_t> dup_of(N, kNotAccepted);   // member whose traceback this one shares, or one of the two marks
    struct DupKey {
        uint64_t query_base, end_abs; uint32_t m, score, flags;
        bool operator==(DupKey const& o) const { return query_base == o.query_base && end_abs == o.end_abs && m == o.m && score == o.score && flags == o.flags; }
    };
    struct DupHash {
        size_t operator()(DupKey const& k) const {
            uint64_t h = k.query_base * 0x9E3779B97F4A7C15ull ^ (k.end_abs + 0x7F4A7C15ull) * 0xC2B2AE3D27D4EB4Full ^ (uint64_t(k.m) << 32 | k.score) ^ k.flags;
            return size_t(h ^ (h >> 31));
        }
    };
    std::unordered_map<DupKey, uint32_t, DupHash> dup_key;
    dup_key.reserve(N);
    hit_pass.reserve(N); hit_shift.reserve(N); hit_widx.reserve(N); accepted.reserve(N);
    std::vector<std::pair<uint64_t, uint32_t>> unit_seen;           // (end column << 32 | score, member) of the pass at hand
    uint64_t cig_at = w.cig_used;
    size_t H = 0;                            // tracebacks issued so far
    size_t i = 0;
    int k = 0;
    bool walk_timed = false;
    while (i < units.size()) {
        size_t j = i; uint64_t used = 0;
        chunk.clear(); ck_base.clear();
        size_t n_shared = 0;                 // members of this chunk that read their result off a shared pass
        while (j < units.size() && (j == i || used + units[j].words <= budget_words)) {
            chunk.push_back(units[j].p); ck_base.push_back(used); used += units[j].words;
            if (units[j].count > 1) n_shared += units[j].count;
            ++j;
        }
        size_t const M = j - i;
        int const slot = k % Worker::kWalkSlots;
        DevBuf& ckb = w.d_ck[slot];
        cudaStream_t const ws = w.walk_stream[slot];
        if (k >= Worker::kWalkSlots) CUDA_TRY(w.err, cudaEventSynchronize(w.ev_walk_done[slot]));       // the tracebacks that read this buffer
        CUDA_TRY(w.err, ckb.ensure(used * 4));
        g_prof.lap(w, 10);
        // ---- the members of shared passes: minimum of the last row over their own columns, right behind the passes ----
        const DpResult* mres = nullptr;
        if (n_shared) {
            CUDA_TRY(w.err, w.h_rtasks.ensure(n_shared * sizeof(RangeMinTask)));
            CUDA_TRY(w.err, w.d_rtasks.ensure(n_shared * sizeof(RangeMinTask)));
            CUDA_TRY(w.err, w.h_rresults.ensure(n_shared * sizeof(DpResult)));
            CUDA_TRY(w.err, w.d_rresults.ensure(n_shared * sizeof(DpResult)));
            RangeMinTask* rt = w.h_rtasks.as<RangeMinTask>();
            size_t r = 0;
            for (size_t u = 0; u < M; ++u) {
                Unit const& U = units[i + u];
                if (U.count < 2) continue;
                for (uint32_t q = 0; q < U.count; ++q) {
                    Pass const& B = passes[unit_members[U.first + q]];
                    RangeMinTask& t = rt[r];
                    t.ck_base = ck_base[u]; t.n = U.p.n; t.m = U.p.m; t.dlo = U.p.dlo; t.dhi = U.p.dhi; t.W = uint32_t(kWidths[U.cfg.widx]);
                    t.col_from = uint32_t(B.ref_base - U.p.ref_base) + 1; t.col_to = uint32_t(B.ref_base - U.p.ref_base) + B.n;
                    t.unit = uint32_t(u); t.out = uint32_t(r); t.reserved = 0;
                    ++r;
                }
            }
            CUDA_TRY(w.err, cudaMemcpyAsync(w.d_rtasks.p, rt, n_shared * sizeof(RangeMinTask), cudaMemcpyHostToDevice, w.stream));
            w.ctr.h2d_bytes += n_shared * sizeof(RangeMinTask);
        }
        std::function<int()> const range_minima = [&]() -> int {
            if (!n_shared) return FXG_OK;
            range_min_kernel<<<uint32_t((n_shared + 63) / 64), 64, 0, w.stream>>>(w.d_rtasks.as<RangeMinTask>(), uint32_t(n_shared), ckb.as<uint32_t>(),
                                                                                 w.d_results.as<DpResult>(), w.d_rresults.as<DpResult>());
            CUDA_TRY(w.err, cudaGetLastError());
            CUDA_TRY(w.err, cudaMemcpyAsync(w.h_rresults.p, w.d_rresults.p, n_shared * sizeof(DpResult), cudaMemcpyDeviceToHost, w.stream));
            w.ctr.kernel_launches++;
            w.ctr.d2h_bytes += n_shared * sizeof(DpResult);
            return FXG_OK;
        };
        const DpResult* res = nullptr;
        int rc = run_passes(c, w, pool, chunk, ck_base.data(), ckb.as<uint32_t>(), &res, &range_minima);      // one wait for both
        if (rc != FXG_OK) return rc;
        w.ctr.trace_bytes += used * 4;
        g_prof.start(w);
        if (n_shared) mres = w.h_rresults.as<DpResult>();
        // ---- tracebacks of the accepted ones on their own stream, one launch per block width ----
        // Alignments of the same query piece that end at the same reference position with the same score -- the usual case:
        // every true anchor of a read leads to the same locus -- have the same traceback, provided every optimal alignment
        // ending there starts inside each of their windows: an alignment of cost s ending at column e spans at least
        // m - s columns... and at most m + s, so its first column is >= e - m - s (in store coordinates); windows that
        // begin at or before that bound contain every such alignment, the DP values along them agree, and so does every
        // "left / up / diagonal" decision (DESIGN.md, section 5).  One member of such a group is traced back, the others
        // share its begin position and its cigar.
        size_t const H0 = H;
        accepted.clear();
        {
            size_t r = 0;
            for (size_t u = 0; u < M; ++u) {
                Unit const& U = units[i + u];
                unit_seen.clear();
                for (uint32_t q = 0; q < U.count; ++q) {
                    uint32_t const mem = unit_members[U.first + q];
                    Pass const& B = passes[mem];
                    DpResult const R = U.count > 1 ? mres[r++] : res[u];
                    uint64_t const shift = B.ref_base - U.p.ref_base;
                    outs[mem].score = R.score; outs[mem].end_col = uint32_t(R.end_col - shift);
                    dup_of[mem] = kNotAccepted;
                    if (R.score > int32_t(max_errors[mem])) { if (U.count > 1) w.ctr.shared_score_passes++; continue; }
                    // (store coordinates: the alignment's first base is at or after end - m - score)
                    bool const safe = int64_t(R.end_col) - int64_t(B.m) - int64_t(R.score) >= int64_t(shift);
                    if (U.count > 1) {
                        if (!safe) {                             // scored again on its own, in a later chunk
                            outs[mem] = RootOut{kNoScore, 0, 0, 0, 0};
                            rc = add_single(mem);
                            if (rc != FXG_OK) return rc;
                            w.ctr.rescored_roots++;
                            continue;
                        }
                        w.ctr.shared_score_passes++;
                    }
                    dup_of[mem] = kOwnTraceback;
                    if (safe) {
                        if (U.count > 1) {
                            // the members of a shared pass are one query piece: (end, score) identifies the alignment, and
                            // a pass sees a handful of different ones at most -- a short list instead of the hash table
                            uint64_t const ident = (uint64_t(R.end_col) << 32) | uint32_t(R.score);
                            size_t h = 0;
                            while (h < unit_seen.size() && unit_seen[h].first != ident) ++h;
                            if (h < unit_seen.size()) { dup_of[mem] = unit_seen[h].second; continue; }   // shares the traceback of an earlier member
                            unit_seen.emplace_back(ident, mem);
                        } else {
                            DupKey const key{B.query_base, U.p.ref_base + R.end_col, B.m, uint32_t(R.score), B.flags};
                            auto const ins = dup_key.emplace(key, mem);
                            if (!ins.second) { dup_of[mem] = ins.first->second; continue; }  // shares the traceback of an earlier pass
                        }
                    }
                    accepted.push_back(Accepted{mem, uint32_t(u), R.end_col, uint32_t(R.score)});
                }
            }
        }
        for (int wi = 0; wi < 6; ++wi) {
            for (Accepted const& a : accepted) {
                Unit const& U = units[i + a.unit_in_chunk];
                if (U.cfg.widx != wi) continue;
                Walk2Task& t = wt[H];
                t.ck_base = ck_base[a.unit_in_chunk]; t.ref_base = U.p.ref_base; t.query_base = U.p.query_base;
                t.cigar_cap = uint32_t(cigar_cap_for(a.score)); t.cigar_base = cig_at; cig_at += t.cigar_cap;
                t.n = U.p.n; t.m = U.p.m; t.dlo = U.p.dlo; t.dhi = U.p.dhi; t.end_col = a.end_col_u; t.score = a.score;
                t.flags = U.p.flags; t.out = uint32_t(H); t.reserved = 0;
                hit_pass.push_back(a.member); hit_shift.push_back(passes[a.member].ref_base - U.p.ref_base); hit_widx.push_back(uint8_t(wi));
                ++H;
            }
        }
        if (H > H0) {
            CUDA_TRY(w.err, cudaMemcpyAsync(w.d_wtasks.as<Walk2Task>() + H0, wt + H0, (H - H0) * sizeof(Walk2Task), cudaMemcpyHostToDevice, ws));
            w.ctr.h2d_bytes += (H - H0) * sizeof(Walk2Task);
            if (!walk_timed) { CUDA_TRY(w.err, cudaEventRecord(w.ev_w0, ws)); walk_timed = true; }
            // every traceback is one long chain of dependent steps, so launches of different block widths must not queue
            // behind each other: the first runs on the chunk's stream, the others fork onto side streams and join it again
            int n_launch = 0;
            for (size_t h = H0; h < H; ++h) n_launch += h == H0 || hit_widx[h] != hit_widx[h - 1];
            CUDA_TRY(w.err, w.fork(ws, n_launch));
            size_t h0 = H0;
            for (int q = 0; q < n_launch; ++q) {
                int const widx = hit_widx[h0];
                size_t h1 = h0;
                while (h1 < H && hit_widx[h1] == widx) ++h1;
                cudaStream_t st;
                CUDA_TRY(w.err, w.fan_stream(ws, q, st));
                CUDA_TRY(w.err, launch_walk(widx, walk_launch(c, w, pool, ckb.as<uint32_t>(), w.d_wtasks.as<Walk2Task>() + h0, uint32_t(h1 - h0)), st));
                w.ctr.kernel_launches++;
                h0 = h1;
            }
            CUDA_TRY(w.err, w.join(ws, n_launch));
            CUDA_TRY(w.err, cudaMemcpyAsync(wr + H0, w.d_wresults.as<WalkResult>() + H0, (H - H0) * sizeof(WalkResult), cudaMemcpyDeviceToHost, ws));
            w.ctr.d2h_bytes += (H - H0) * sizeof(WalkResult);
        }
        CUDA_TRY(w.err, cudaEventRecord(w.ev_walk_done[slot], ws));
        CUDA_TRY(w.err, cudaEventRecord(w.ev_w1[slot], ws));
        i = j; ++k;
        g_prof.lap(w, 12);
    }
    for (int q = 0; q < std::min(k, int(Worker::kWalkSlots)); ++q) CUDA_TRY(w.err, w.wait_for(w.walk_stream[q]));
    if (walk_timed) {
        // first traceback launch to last traceback done (they run beside score passes)
        float best = 0;
        for (int q = 0; q < std::min(k, int(Worker::kWalkSlots)); ++q) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, w.ev_w0, w.ev_w1[q]) == cudaSuccess) best = std::max(best, ms);
        }
        w.ctr.trace_kernel_ms += best;
    }
    for (size_t h = 0; h < H; ++h) {
        if (wr[h].cigar_len == 0xffffffffu || wr[h].begin_col < hit_shift[h])
            return fail(w.err, FXG_ERR_CUDA, "internal: the traceback of an alignment disagrees with its score pass (query length %u, window %u, "
                        "band %d..%d, end column %u, score %u, begin column %u, window shift %llu, %s)", wt[h].m, wt[h].n, wt[h].dlo, wt[h].dhi, wt[h].end_col,
                        wt[h].score, wr[h].begin_col, (unsigned long long)hit_shift[h], wr[h].cigar_len == 0xffffffffu ? "path cost differs" : "begins before its window");
        RootOut& o = outs[hit_pass[h]];
        o.begin_col = uint32_t(wr[h].begin_col - hit_shift[h]); o.cigar_len = wr[h].cigar_len;     // seen from the member's own window
        o.cigar_offset = wt[h].cigar_base + wt[h].cigar_cap - wr[h].cigar_len;
    }
    for (size_t q = 0; q < N; ++q) {
        if (dup_of[q] >= kOwnTraceback) continue;
        RootOut const& rep = outs[dup_of[q]];
        RootOut& o = outs[q];
        // same alignment, seen from this pass' window: its begin column moves by the distance between the windows' starts
        o.begin_col = uint32_t(passes[dup_of[q]].ref_base + rep.begin_col - passes[q].ref_base);
        o.cigar_offset = rep.cigar_offset; o.cigar_len = rep.cigar_len;
        w.ctr.shared_tracebacks++;
    }
    w.cig_used = cig_at;
    g_prof.lap(w, 12);
    return FXG_OK;
}

// copies the worker's cigars (w.d_cigars[0 .. w.cig_used)) to `dst` (page-locked)
int fetch_cigars(Worker& w, uint32_t* dst) {
    if (!w.cig_used) return FXG_OK;
    CUDA_TRY(w.err, cudaMemcpyAsync(dst, w.d_cigars.p, w.cig_used * 4, cudaMemcpyDeviceToHost, w.stream));
    CUDA_TRY(w.err, w.wait_for(w.stream));
    w.ctr.d2h_bytes += w.cig_used * 4;
    return FXG_OK;
}

// Trace planes may take up to about half of what is free on the device (at most 64 GiB), shared by the parts of a
// run.  cudaMemGetInfo costs milliseconds, so the figure is refreshed only when the resident set changes.
void refresh_trace_budget(fxg_ctx* c) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) free_b = size_t(8) << 30;
    uint64_t held = 0;
    for (WorkerGroup const& g : c->groups) for (auto const& w : g.workers) for (DevBuf const& b : w->d_ck) held += b.cap;
    c->trace_budget = std::min<uint64_t>((uint64_t(free_b) + held) / 2, uint64_t(64) << 30);
}
uint64_t trace_budget_bytes(fxg_ctx* c, size_t n_parts) {
    if (c->trace_budget == 0) refresh_trace_budget(c);
    return c->trace_budget / (std::max<size_t>(n_parts, 1) * size_t(c->n_groups));
}

// ------------------------------------------------------------------------------------------------ pools

// cudaMalloc / cudaFree synchronise the device and cost milliseconds: staged pools are recycled instead
Pool take_pool(fxg_ctx* c) {
    Pool p;
    if (!c->spare_pools.empty()) { p = c->spare_pools.back(); c->spare_pools.pop_back(); }
    p.len = p.plane_words = p.inline_len = 0;
    return p;
}
void give_pool(fxg_ctx* c, Pool& p) {
    if (c->spare_pools.size() < 96) c->spare_pools.push_back(p); else p.release();   // one per caller whose job waits or is being staged
    p = Pool{};
}

PinnedBuf take_pinned(fxg_ctx* c) {
    PinnedBuf b;
    if (!c->spare_pinned.empty()) {          // the largest one: the next run most likely needs as much as the last
        size_t best = 0;
        for (size_t i = 1; i < c->spare_pinned.size(); ++i) if (c->spare_pinned[i].cap > c->spare_pinned[best].cap) best = i;
        b = c->spare_pinned[best];
        c->spare_pinned.erase(c->spare_pinned.begin() + long(best));
    }
    return b;
}
void give_pinned(fxg_ctx* c, PinnedBuf& b) {
    if (b.p && c->spare_pinned.size() < size_t(2 * c->n_groups + 72)) c->spare_pinned.push_back(b); else b.release();   // (one per caller and batch in flight)
    b = PinnedBuf{};
}
// the smallest spare pool that holds `bytes`, else the largest (it will grow)
PinnedBuf take_pinned_fit(fxg_ctx* c, size_t bytes) {
    PinnedBuf b;
    if (c->spare_pinned.empty()) return b;
    size_t best = SIZE_MAX, largest = 0;
    for (size_t i = 0; i < c->spare_pinned.size(); ++i) {
        if (c->spare_pinned[i].cap >= bytes && (best == SIZE_MAX || c->spare_pinned[i].cap < c->spare_pinned[best].cap)) best = i;
        if (c->spare_pinned[i].cap > c->spare_pinned[largest].cap) largest = i;
    }
    size_t const pick = best != SIZE_MAX ? best : largest;
    b = c->spare_pinned[pick];
    c->spare_pinned.erase(c->spare_pinned.begin() + long(pick));
    return b;
}
PinnedBuf take_staging(fxg_ctx* c) {
    PinnedBuf b;
    if (!c->spare_staging.empty()) { b = c->spare_staging.back(); c->spare_staging.pop_back(); }
    return b;
}
void give_staging(fxg_ctx* c, PinnedBuf& b) {
    if (b.p && c->spare_staging.size() < 96) c->spare_staging.push_back(b); else b.release();
    b = PinnedBuf{};
}

int check_ranks(std::string& err, const uint8_t* p, size_t n, const char* what) {
    // any byte above FXG_MAX_RANK?  eight bytes at a time: (b & 0x7f) + 0x7a has its top bit set iff (b & 0x7f) >= 6
    uint64_t bad = 0;
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
        uint64_t x;
        std::memcpy(&x, p + i, 8);
        bad |= (((x & 0x7f7f7f7f7f7f7f7full) + 0x7a7a7a7a7a7a7a7aull) | x) & 0x8080808080808080ull;
    }
    for (; i < n; ++i) bad |= p[i] > FXG_MAX_RANK;
    if (bad) return fail(err, FXG_ERR_INVALID_ARGUMENT, "%s contains a rank above %d (allowed 0..%d)", what, FXG_MAX_RANK, FXG_MAX_RANK);
    return FXG_OK;
}

int upload_packed(fxg_ctx* c, const uint8_t* ranks, uint64_t len, DevBuf& dst, uint64_t word_offset) {
    // pack on the device: upload bytes to a temporary, 8 bases per output word
    if (len == 0) return FXG_OK;
    cudaStream_t const st = c->stage_stream;
    CUDA_TRY(c->err, c->d_tmp.ensure(len));
    CUDA_TRY(c->err, cudaMemcpyAsync(c->d_tmp.p, ranks, len, cudaMemcpyHostToDevice, st));
    c->ctr.h2d_bytes += len;
    uint64_t const n_words = (len + 7) / 8;
    uint32_t const grid = uint32_t(std::min<uint64_t>((n_words + 255) / 256, uint64_t(c->num_sms) * 16));
    pack_nibbles_kernel<<<grid, 256, 0, st>>>(c->d_tmp.as<uint8_t>(), len, dst.as<uint32_t>() + word_offset);
    CUDA_TRY(c->err, cudaGetLastError());
    c->ctr.kernel_launches++;
    CUDA_TRY(c->err, cudaStreamSynchronize(st));
    return FXG_OK;
}

// uploads up to two byte ranges back to back (forward / reverse pools) and builds the Peq planes; errors and
// accounting go to the caller's objects (fxg_verify_reads runs this beside the workers).  kind = cudaMemcpyDeviceToDevice:
// the ranges are in device memory already (fxg_map_fastq's parsed pools) and are not counted as uploads.
int stage_pool(fxg_ctx* c, Pool& pool, const uint8_t* a, size_t a_len, const uint8_t* b, size_t b_len, std::string& err, fxg_counters& ctr,
               bool check_ranks_on_device = false, cudaMemcpyKind kind = cudaMemcpyHostToDevice) {
    cudaStream_t const st = c->stage_stream;
    pool.len = a_len + b_len;
    pool.plane_words = (pool.len + 31) / 32 + kPeqFrontPadWords + kPeqBackPadWords;
    CUDA_TRY(err, pool.bytes.ensure(pool.len + 64));
    CUDA_TRY(err, pool.peq.ensure(pool.plane_words * kNumSymbols * 4));
    CUDA_TRY(err, pool.bad_rank.ensure(4));
    if (a_len) CUDA_TRY(err, cudaMemcpyAsync(pool.bytes.p, a, a_len, kind, st));
    if (b_len) CUDA_TRY(err, cudaMemcpyAsync(pool.bytes.as<uint8_t>() + a_len, b, b_len, kind, st));
    if (kind == cudaMemcpyHostToDevice) ctr.h2d_bytes += pool.len;
    CUDA_TRY(err, cudaMemsetAsync(pool.peq.p, 0, pool.plane_words * kNumSymbols * 4, st));
    CUDA_TRY(err, cudaMemsetAsync(pool.bad_rank.p, 0, 4, st));
    if (pool.len) {
        uint64_t const n_words = (pool.len + 31) / 32;
        uint32_t const grid = uint32_t(std::min<uint64_t>((n_words + 7) / 8, uint64_t(c->num_sms) * 16));
        build_peq_kernel<<<grid, 256, 0, st>>>(pool.bytes.as<uint8_t>(), pool.len, pool.peq.as<uint32_t>(), pool.plane_words,
                                               check_ranks_on_device ? pool.bad_rank.as<uint32_t>() : nullptr);
        CUDA_TRY(err, cudaGetLastError());
        ctr.kernel_launches++;
    }
    return FXG_OK;
}

// ------------------------------------------------------------------------------------------------ align semantics

// band of a score pass: every alignment with <= k errors of a query of length m inside a window of length n
// stays on diagonals j - i in [-k, n - m + k]
inline bool score_pass_for(uint64_t ref_base, uint64_t query_base, uint32_t n, uint32_t m, uint32_t k, uint32_t flags, Pass& p) {
    if (m == 0) return false;
    if (int64_t(m) - int64_t(n) > int64_t(k)) return false;          // more insertions needed than errors allowed
    p.ref_base = ref_base; p.query_base = query_base; p.n = n; p.m = m;
    int64_t const lo = -int64_t(k), hi = int64_t(n) - int64_t(m) + int64_t(k);
    p.dlo = int32_t(lo); p.dhi = int32_t(hi); p.flags = flags;
    return true;
}

// math::floating_point_error_aware_ceil, include/math.hpp:22-27
inline uint64_t ceil_eps(double v) { return uint64_t(std::ceil(v - 0.000000001) + 0.000000001); }

// verification::internal::compute_reference_span_start_and_length, src/lib/verification.cpp:157-184
inline Span compute_span(uint64_t anchor_pos, fxg_pex_node const& node, uint64_t leaf_from, uint64_t ref_len, double ratio) {
    uint64_t const base = (node.query_index_to - node.query_index_from + 1) + 2 * node.num_errors + 1;
    uint64_t const extra = ratio == 0.0 ? 0 : ceil_eps(double(base) * ratio);
    int64_t const s = int64_t(anchor_pos) - int64_t(leaf_from - node.query_index_from) - int64_t(node.num_errors) - int64_t(extra);
    Span r;
    r.offset = s >= 0 ? uint64_t(s) : 0;
    r.length = std::min<uint64_t>(base + 2 * extra, ref_len - r.offset);
    r.extra = extra;
    return r;
}

// half_open_interval::trim_from_both_sides, src/lib/intervals.cpp:48-58
inline void trim(uint64_t& start, uint64_t& end, uint64_t amount) {
    uint64_t const e = amount > end ? 0 : end - amount;
    uint64_t const ne = std::max(start + 1, e);
    uint64_t const ns = std::min(ne - 1, start + amount);
    start = ns; end = ne;
}

// ------------------------------------------------------------------------------------------------ verify, one part

// One Walk per anchor of reads [read_lo, read_hi) in the reference's order (read, forward package, reverse package);
// anchors of one (read, orientation, reference) share a verified_intervals set (parallelization.cpp:224-226).
void build_walks(fxg_ctx* c, fxg_job const* J, uint32_t read_lo, uint32_t read_hi, std::vector<Walk>& walks,
                 std::vector<Group>& groups, std::vector<uint32_t>& group_members) {
    bool const direct = J->cfg.verification_kind == FXG_KIND_DIRECT_FULL;
    bool const ivopt = J->cfg.interval_optimization != 0;
    double const ratio = J->cfg.extra_verification_ratio;
    walks.clear(); groups.clear(); group_members.clear();
    walks.resize(J->read_walk_begin[read_hi] - J->read_walk_begin[read_lo]);       // zeroed; filled in place
    size_t n_out = 0;
    std::vector<std::vector<uint32_t>> tmp_groups;
    std::vector<int64_t> ref_to_group;
    for (uint32_t ri = read_lo; ri < read_hi; ++ri) {
        fxg_read const& R = J->reads_p[ri];
        const fxg_pex_node* inner = J->nodes_p + R.node_offset;
        const fxg_pex_node* leaves = inner + R.num_inner;
        fxg_pex_node const& root = R.num_inner ? inner[0] : leaves[0];
        for (int orient = 0; orient < 2; ++orient) {
            uint32_t const a0 = uint32_t(R.anchor_offset) + (orient ? R.num_anchors_forward : 0);
            uint32_t const na = orient ? R.num_anchors_reverse : R.num_anchors_forward;
            if (ivopt) { tmp_groups.clear(); ref_to_group.assign(c->refs.len.size(), -1); }
            uint32_t const group_base = uint32_t(groups.size());
            for (uint32_t q = 0; q < na; ++q) {
                fxg_anchor const& A = J->anchors_p[a0 + q];
                fxg_pex_node const& leaf = leaves[A.pex_leaf_index];
                Walk& wk = walks[n_out];
                wk.read = ri; wk.anchor = a0 + q; wk.orient = uint8_t(orient); wk.state = W_WAITING;
                wk.node = (direct || leaf.parent_id == FXG_NULL_ID) ? &root : &inner[leaf.parent_id];
                // the root window is needed up front only by the interval optimisation (and by walks that start at the
                // root); otherwise it is computed when -- and if -- the walk gets there
                if (ivopt || wk.node == &root) {
                    wk.root_span = compute_span(A.reference_position, root, leaf.query_index_from, c->refs.len[A.reference_id], ratio);
                    wk.r_start = wk.root_span.offset; wk.r_end = wk.root_span.offset + wk.root_span.length;
                    wk.t_start = wk.r_start; wk.t_end = wk.r_end;
                    trim(wk.t_start, wk.t_end, wk.root_span.extra);
                    wk.have_root_span = true;
                }
                if (ivopt) {
                    if (ref_to_group[A.reference_id] < 0) { ref_to_group[A.reference_id] = int64_t(tmp_groups.size()); tmp_groups.emplace_back(); }
                    wk.group = group_base + uint32_t(ref_to_group[A.reference_id]);
                    tmp_groups[size_t(ref_to_group[A.reference_id])].push_back(uint32_t(n_out));
                }
                ++n_out;
            }
            if (ivopt) {
                for (auto const& g : tmp_groups) {
                    groups.push_back(Group{uint32_t(group_members.size()), uint32_t(g.size())});
                    group_members.insert(group_members.end(), g.begin(), g.end());
                }
            }
        }
    }
}

int validate_reads_range(fxg_ctx* c, std::string& err, const fxg_read* reads, size_t lo, size_t hi, size_t pool_len,
                         const fxg_pex_node* nodes, size_t n_nodes, const fxg_anchor* anchors, size_t n_anchors, bool with_anchors);

// every read's ranges, tree shape and anchors; large batches on several threads.  with_anchors = false: the reads' anchors
// are not known yet (fxg_seed_verify_reads checks the batch before it seeds; the seeder's anchors are valid by construction)
int validate_reads(fxg_ctx* c, std::string& err, const fxg_read* reads, size_t lo, size_t hi, size_t pool_len,
                   const fxg_pex_node* nodes, size_t n_nodes, const fxg_anchor* anchors, size_t n_anchors, bool with_anchors = true) {
    size_t const n_threads = (n_nodes + n_anchors) < (size_t(1) << 20) ? 1 : std::min<size_t>({size_t(8), hi - lo, std::max<size_t>(1, std::thread::hardware_concurrency() / 2)});
    if (n_threads <= 1) return validate_reads_range(c, err, reads, lo, hi, pool_len, nodes, n_nodes, anchors, n_anchors, with_anchors);
    std::vector<int> rcs(n_threads, FXG_OK); std::vector<std::string> errs(n_threads);
    std::vector<std::thread> threads;
    for (size_t t = 0; t < n_threads; ++t) {
        size_t const a = lo + (hi - lo) * t / n_threads, b = lo + (hi - lo) * (t + 1) / n_threads;
        threads.emplace_back([&, t, a, b] { rcs[t] = validate_reads_range(c, errs[t], reads, a, b, pool_len, nodes, n_nodes, anchors, n_anchors, with_anchors); });
    }
    for (auto& th : threads) th.join();
    for (size_t t = 0; t < n_threads; ++t) if (rcs[t] != FXG_OK) { err = errs[t]; tls_last_error = err; return rcs[t]; }
    return FXG_OK;
}

int validate_reads_range(fxg_ctx* c, std::string& err, const fxg_read* reads, size_t lo, size_t hi, size_t pool_len,
                         const fxg_pex_node* nodes, size_t n_nodes, const fxg_anchor* anchors, size_t n_anchors, bool with_anchors) {
    for (size_t i = lo; i < hi; ++i) {
        fxg_read const& R = reads[i];
        if (R.query_offset + R.query_len > pool_len) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: query outside the pool", i);
        if (R.query_len > FXG_MAX_QUERY_LENGTH) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: longer than %d", i, FXG_MAX_QUERY_LENGTH);
        if (R.node_offset + R.num_inner + R.num_leaves > n_nodes || R.num_leaves == 0) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: bad node range", i);
        if (with_anchors && R.anchor_offset + R.num_anchors_forward + R.num_anchors_reverse > n_anchors) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: bad anchor range", i);
        const fxg_pex_node* nd = nodes + R.node_offset;
        for (uint32_t q = 0; q < R.num_inner + R.num_leaves; ++q) {
            if (nd[q].query_index_to < nd[q].query_index_from || nd[q].query_index_to >= R.query_len) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: node %u outside the query", i, q);
            if (nd[q].parent_id != FXG_NULL_ID && nd[q].parent_id >= R.num_inner) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: node %u has a bad parent", i, q);
        }
        // shape of the tree (pex.hpp:59-76): inner[0] is the root, every other inner node hangs below it
        if (R.num_inner) {
            if (nd[0].parent_id != FXG_NULL_ID) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: inner node 0 is not the root", i);
            // depth[q] = hops to the root, 0xff = not known yet; every chain is followed only as far as a node that is known
            thread_local std::vector<uint8_t> depth;
            depth.assign(R.num_inner, 0xff);
            depth[0] = 0;
            for (uint32_t q = 1; q < R.num_inner; ++q) {
                uint64_t p = q; int hops = 0;
                while (depth[p] == 0xff) {
                    p = nd[p].parent_id;
                    if (p == FXG_NULL_ID || ++hops > 250) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: the parents of inner node %u do not lead to the root", i, q);
                }
                if (int(depth[p]) + hops > 250) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: the tree is deeper than 250 levels", i);
                int d = int(depth[p]) + hops;
                for (uint64_t x = q; depth[x] == 0xff; x = nd[x].parent_id) depth[x] = uint8_t(d--);
            }
        }
        if (!with_anchors) continue;
        const fxg_anchor* an = anchors + R.anchor_offset;
        for (uint32_t q = 0; q < R.num_anchors_forward + R.num_anchors_reverse; ++q) {
            if (an[q].pex_leaf_index >= R.num_leaves) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: anchor %u names leaf %llu", i, q, (unsigned long long)an[q].pex_leaf_index);
            if (an[q].reference_id >= c->refs.len.size()) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: anchor %u names reference %llu", i, q, (unsigned long long)an[q].reference_id);
            if (an[q].reference_position >= c->refs.len[an[q].reference_id]) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: anchor %u outside its reference", i, q);
        }
    }
    return FXG_OK;
}

struct PartOut {
    std::vector<fxg_alignment> alignments;   // cigar offsets index the batch's cigar pool
    std::vector<fxg_stats> stats;            // per member job
    int rc = FXG_OK;
};

// One or more jobs that run together: a job of its own, or the jobs of several callers merged by submit_and_wait.
struct Member { fxg_job* J; uint32_t read0; uint64_t pool_shift; };
struct Batch {
    fxg_verify_config cfg{};
    std::vector<Member> members;
    bool device = false;                 // every member has device records: the walks run on the device
    uint32_t n_reads = 0;
    std::vector<uint32_t> read_walk_begin;   // per read of the batch (+1 sentinel): its first walk
    Pool const* pool = nullptr;          // the Peq planes the passes read: the member's own, or the group's merged ones
    uint64_t pool_len = 0;               // (a job of its own) length of its forward pool
    cudaEvent_t merged_ready = nullptr;  // the merged planes are in place
    // results
    std::vector<fxg_alignment> alignments;
    PinnedBuf* cigars = nullptr; size_t cigars_len = 0;
    std::vector<fxg_stats> stats;
};

// what one part carries from its score phase to its traceback phase
struct PartState {
    std::vector<Walk> walks; std::vector<Group> groups; std::vector<uint32_t> group_members;   // indices local to this part
    uint64_t trace_budget = 0;               // bytes of checkpoint records the part may hold at a time
    std::chrono::steady_clock::time_point t0;
    double cpu0 = 0;                         // the part's thread CPU time at its start (FXG_PROFILE)
    std::vector<ReadRec> part_reads;         // (device-side walks) the part's ReadRecs as the device sees them
    std::vector<fxg_alignment> hits;         // the part's alignments in anchor order, cigar offsets relative to the part's region
    double scale = 1.0;                      // the largest merged batch over this part (buffers are sized for that batch at once)
    size_t n_parts = 1;
    double t_mark[6] = {0, 0, 0, 0, 0, 0};   // (FXG_TRACE_BATCHES) ms since the part began: gathered+enqueued, levels done, units known, scores known, records back
    PartOut out;
};

// hops from an inner node to the root, memoised per read (the trees are small; validate_reads has bounded the chains)
uint8_t node_dist(const fxg_pex_node* inner, std::vector<uint8_t>& memo, uint64_t id) {
    if (memo[id] != 0xff) return memo[id];
    uint8_t d = 0;
    if (inner[id].parent_id != FXG_NULL_ID) d = uint8_t(std::min<int>(254, node_dist(inner, memo, inner[id].parent_id) + 1));
    return memo[id] = d;
}

// ------------------------------------------------------------------------------------------------ prepared jobs
//
// The device-side tree walk (dp_kernels.cuh: walk_init / level_* / decide kernels) reads a job from compact records made
// ONCE per job, on the caller's thread, and kept in HBM: NodeRec per inner node, LeafRec per leaf, ReadRec per read,
// AnchorRec16 per anchor.  A run then touches no per-anchor data on the host: it gathers the records of the jobs it was
// handed (device-to-device), lets the walks climb, and reads back only the walks that verify their root.

// configuration classes are numbered per context, so that the records of different jobs can share a launch
int class_of(fxg_ctx* c, Config const& cf, uint32_t words) {
    std::lock_guard<std::mutex> lock(c->class_mu);
    for (int i = 0; i < c->n_classes; ++i)
        if (c->classes[i].widx == cf.widx && c->classes[i].G == cf.G) { c->classes[i].max_words = std::max(c->classes[i].max_words, words); return i; }
    if (c->n_classes == kMaxLevelClasses) {
        // the table is full (a context that has seen every shape of tree): a class of the same block width with a larger
        // ring runs the pass as well -- the lanes a smaller ring would leave idle cost nothing
        int best = -1;
        for (int i = 0; i < c->n_classes; ++i)
            if (c->classes[i].widx == cf.widx && c->classes[i].G != kWideG && cf.G != kWideG && c->classes[i].G >= cf.G && (best < 0 || c->classes[i].G < c->classes[best].G)) best = i;
        if (best >= 0) c->classes[best].max_words = std::max(c->classes[best].max_words, words);
        return best;
    }
    c->classes[c->n_classes] = ClassDef{cf.widx, cf.G, words};
    return c->n_classes++;
}

// class_of through a table of the calling thread: the context's mutex is taken only for a class the thread has not seen,
// or when a node needs a wider Eq table than the thread has reported for the class
int class_of_cached(fxg_ctx* c, Config const& cf, uint32_t words) {
    struct Seen { uint64_t owner = 0; int id[6][66]; uint32_t words[kMaxLevelClasses]; };
    thread_local Seen seen;
    // (a new context may live at a freed one's address: contexts are told apart by their serial numbers)
    if (seen.owner != c->serial) { seen.owner = c->serial; for (auto& row : seen.id) for (int& x : row) x = -2; for (uint32_t& x : seen.words) x = 0; }
    int& id = seen.id[cf.widx][std::min<int>(cf.G, 65)];
    if (id >= 0 && words <= seen.words[id]) return id;
    id = class_of(c, cf, words);
    if (id >= 0) seen.words[id] = std::max(seen.words[id], words);
    return id;
}

std::vector<ConfigCacheEntry>& thread_config_cache(const fxg_ctx* c) {
    thread_local std::vector<ConfigCacheEntry> cache(8192);
    thread_local uint64_t owner = 0;
    if (owner != c->serial) { for (ConfigCacheEntry& e : cache) e.valid = false; owner = c->serial; }      // (contexts may differ in their knobs)
    return cache;
}

// Where a job's records go in Prepared::dev and its staging: nodes | leaves | reads | anchors, each on a 256-byte boundary.
// Returns the end of the anchors.
size_t carve_records(Prepared& P, uint64_t n_nodes, uint64_t n_leaves, uint64_t n_reads, uint64_t n_walks) {
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t const at = off; off += (bytes + 255) & ~size_t(255); return at; };
    P.o_nodes = carve(n_nodes * sizeof(NodeRec)); P.o_leaves = carve(n_leaves * sizeof(LeafRec));
    P.o_reads = carve(n_reads * sizeof(ReadRec)); P.o_anchors = carve(n_walks * sizeof(AnchorRec16));
    return off;
}

// Builds and uploads the job's records (asynchronously, on the context's staging stream; J->prep.ready marks the end).
// J->prep.ok tells whether the device-side walk can take the job; if not, the host-driven levels run it.
// anchors_on_device: the AnchorRec16 records are already in P.dev at P.o_anchors (fxg_seed_verify_reads wrote them there,
// on a stream its caller has drained); only the nodes, leaves and reads are built and go up.
int prepare_job(fxg_ctx* c, fxg_job* J, std::string& err, fxg_counters& ctr, bool anchors_on_device = false) {
    Prepared& P = J->prep;
    P.ok = false;
    size_t const n_reads = J->n_reads;
    if (n_reads == 0 || !c->device_levels) return FXG_OK;
    uint64_t n_nodes = 0, n_leaves = 0, n_walks = 0;
    for (size_t ri = 0; ri < n_reads; ++ri) {
        fxg_read const& R = J->reads_p[ri];
        if (R.num_inner >= 0xffff) return FXG_OK;
        n_nodes += R.num_inner; n_leaves += R.num_leaves; n_walks += uint64_t(R.num_anchors_forward) + R.num_anchors_reverse;
    }
    if (n_walks == 0 || n_walks >= kMaxDeviceWalks || n_nodes >= (1u << 30) || n_leaves >= (1u << 30) || n_reads >= (1u << 30)) return FXG_OK;
    if (c->refs.total >= (uint64_t(1) << (64 - kWalkBits))) return FXG_OK;
    static_assert(sizeof(AnchorRec16) == 16 && sizeof(ReadRec) == 64 && sizeof(LeafRec) == 8 && sizeof(NodeRec) == 16 && sizeof(WalkRec) == 32 && sizeof(RootEntry) == 16, "record layouts");
    size_t const off = carve_records(P, n_nodes, n_leaves, n_reads, n_walks);
    size_t const up = anchors_on_device ? P.o_anchors : off;          // what goes up from the host
    P.staging.tag = "page-locked job records";
    if (P.staging.ensure(up + 64) != cudaSuccess) return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate staging for the job's records");
    P.used = up;
    if (anchors_on_device && P.dev.cap < off + 64) return fail(err, FXG_ERR_CUDA, "internal: the seeded anchors do not fit the job's record buffer");
    CUDA_TRY(err, P.dev.ensure(off + 64));
    uint8_t* const H = P.staging.as<uint8_t>();
    NodeRec* const nrec = reinterpret_cast<NodeRec*>(H + P.o_nodes);
    LeafRec* const lrec = reinterpret_cast<LeafRec*>(H + P.o_leaves);
    ReadRec* const rrec = reinterpret_cast<ReadRec*>(H + P.o_reads);
    AnchorRec16* const arec = reinterpret_cast<AnchorRec16*>(H + P.o_anchors);
    std::memset(P.level_mask, 0, sizeof P.level_mask);
    P.max_depth = 0;
    double const ratio = J->cfg.extra_verification_ratio;
    // where every read's records go
    uint32_t node_at = 0, leaf_at = 0, walk_at = 0;
    for (size_t ri = 0; ri < n_reads; ++ri) {
        fxg_read const& R = J->reads_p[ri];
        ReadRec& rr = rrec[ri];
        rr.walk_begin = walk_at; rr.n_forward = R.num_anchors_forward; rr.node_base = node_at; rr.leaf_base = leaf_at;
        rr.n_walks = R.num_anchors_forward + R.num_anchors_reverse;
        node_at += R.num_inner; leaf_at += R.num_leaves; walk_at += rr.n_walks;
    }
    // the records themselves: large jobs on several threads, each over a range of reads
    struct ChunkOut { uint32_t level_mask[256]; uint32_t max_depth; int status; };   // status: 0 fine, 1 not for the device path
    auto fill = [&](size_t r_lo, size_t r_hi, ChunkOut& out) {
        std::memset(out.level_mask, 0, sizeof out.level_mask); out.max_depth = 0; out.status = 0;
        std::vector<ConfigCacheEntry>& cache = thread_config_cache(c);
        std::vector<uint8_t> memo;
        // a PEX tree is a function of the read's length and the batch's parameters: reads of equal length have equal trees, and
        // the records of an equal tree are copied instead of rebuilt (the trees are compared, not assumed equal)
        std::unordered_map<uint64_t, uint32_t> first_of_shape;
        for (size_t ri = r_lo; ri < r_hi; ++ri) {
            fxg_read const& R = J->reads_p[ri];
            const fxg_pex_node* inner = J->nodes_p + R.node_offset;
            const fxg_pex_node* leaves = inner + R.num_inner;
            ReadRec& rr = rrec[ri];
            rr.qoff_forward = R.query_offset; rr.qoff_reverse = J->pool_len + R.query_offset;
            fxg_pex_node const& root = R.num_inner ? inner[0] : leaves[0];
            rr.root_from = uint32_t(root.query_index_from); rr.root_m = uint32_t(root.query_index_to - root.query_index_from + 1); rr.root_k = uint32_t(root.num_errors);
            uint64_t const base = uint64_t(rr.root_m) + 2ull * rr.root_k + 1;
            uint64_t const extra = ratio == 0.0 ? 0 : ceil_eps(double(base) * ratio);
            if (extra >= (1u << 30)) { out.status = 1; return; }
            rr.root_extra = uint32_t(extra);
            rr.member = 0; rr.reserved0 = rr.reserved1 = 0;
            {
                // configuration class of the root's score passes, and the widest union window that class takes (root_cluster_kernel)
                Pass p;
                uint64_t const n_root = base + 2 * extra;
                if (n_root >= (uint64_t(1) << 31) || !score_pass_for(0, 0, uint32_t(n_root), rr.root_m, rr.root_k, 0, p)) { out.status = 1; return; }
                Config cf;
                if (!cached_config(cache, p, c->smem_limit, c->force_wide, cf, !J->cfg.without_cigar)) { out.status = 1; return; }   // (with its traceback, if CIGARs are wanted)
                uint32_t const W = uint32_t(kWidths[cf.widx]);
                int const ci = class_of_cached(c, cf, (rr.root_m + 32 * W - 1) / (32 * W) * W);
                if (ci < 0) { out.status = 1; return; }
                rr.reserved0 = uint32_t(ci);
                // ring of G lanes: band B = n - m + 2k + 1 <= ring_band_limit(G, W) (choose_config)
                // (a lane per block, or the multi-warp kernel: any band)
                int64_t const n_cap = (cf.G == kWideG || cf.G >= cf.nb) ? int64_t(1) << 30
                                                                        : int64_t(rr.root_m) - 2 * int64_t(rr.root_k) - 1 + ring_band_limit(cf.G, W);
                rr.reserved1 = uint32_t(std::max<int64_t>(std::min<int64_t>(n_cap, int64_t(1) << 30), int64_t(n_root)));
            }
            uint64_t const shape = (uint64_t(R.query_len) << 32) ^ (uint64_t(R.num_inner) << 16) ^ R.num_leaves;
            auto const ins = first_of_shape.emplace(shape, uint32_t(ri));
            bool copied = false;
            if (!ins.second) {
                fxg_read const& Q = J->reads_p[ins.first->second];
                if (Q.num_inner == R.num_inner && Q.num_leaves == R.num_leaves &&
                    std::memcmp(J->nodes_p + Q.node_offset, inner, (size_t(R.num_inner) + R.num_leaves) * sizeof(fxg_pex_node)) == 0) {
                    ReadRec const& qr = rrec[ins.first->second];
                    std::memcpy(nrec + rr.node_base, nrec + qr.node_base, size_t(R.num_inner) * sizeof(NodeRec));
                    std::memcpy(lrec + rr.leaf_base, lrec + qr.leaf_base, size_t(R.num_leaves) * sizeof(LeafRec));
                    copied = true;
                }
            }
            if (!copied) {
                memo.assign(R.num_inner, 0xff);
                for (uint32_t q = 0; q < R.num_inner; ++q) {
                    fxg_pex_node const& nd = inner[q];
                    NodeRec& r = nrec[rr.node_base + q];
                    r.from = uint32_t(nd.query_index_from); r.m = uint32_t(nd.query_index_to - nd.query_index_from + 1); r.k = uint32_t(nd.num_errors);
                    r.parent = nd.parent_id == FXG_NULL_ID ? uint16_t(0) : uint16_t(nd.parent_id);
                    r.depth = node_dist(inner, memo, q);
                    Pass p;
                    uint64_t const n_full = uint64_t(r.m) + 2ull * r.k + 1;
                    if (!score_pass_for(0, 0, uint32_t(n_full), r.m, r.k, 0, p)) { out.status = 1; return; }
                    Config cf;
                    if (!cached_config(cache, p, c->smem_limit, c->force_wide, cf)) { out.status = 1; return; }
                    uint32_t const W = uint32_t(kWidths[cf.widx]);
                    int const ci = class_of_cached(c, cf, (r.m + 32 * W - 1) / (32 * W) * W);
                    if (ci < 0) { out.status = 1; return; }
                    r.cls = uint8_t(ci);
                    if (q > 0) {                                   // the root is not an inner level
                        out.level_mask[r.depth] |= 1u << ci;
                        out.max_depth = std::max<uint32_t>(out.max_depth, r.depth);
                    }
                }
                for (uint32_t q = 0; q < R.num_leaves; ++q) {
                    lrec[rr.leaf_base + q].from = uint32_t(leaves[q].query_index_from);
                    lrec[rr.leaf_base + q].parent = leaves[q].parent_id == FXG_NULL_ID ? kNoParent : uint32_t(leaves[q].parent_id);
                }
            }
            if (anchors_on_device) continue;
            const fxg_anchor* an = J->anchors_p + R.anchor_offset;
            AnchorRec16* const dst = arec + rr.walk_begin;
            for (uint32_t q = 0; q < rr.n_walks; ++q) {
                dst[q].reference_position = an[q].reference_position; dst[q].pex_leaf_index = uint32_t(an[q].pex_leaf_index); dst[q].reference_id = uint32_t(an[q].reference_id);
            }
        }
    };
    size_t const n_threads = n_walks < (uint64_t(1) << 19) ? 1 : std::min<size_t>({size_t(8), n_reads, std::max<size_t>(1, std::thread::hardware_concurrency() / 2)});
    std::vector<ChunkOut> outs(n_threads);
    if (n_threads == 1) fill(0, n_reads, outs[0]);
    else {
        std::vector<std::thread> threads;
        for (size_t t = 0; t < n_threads; ++t) {
            // (ranges with similar numbers of anchors)
            auto cut = [&](size_t q) { uint64_t const target = n_walks * q / n_threads; size_t lo = 0, hi = n_reads; while (lo < hi) { size_t const mid = (lo + hi) / 2; if (rrec[mid].walk_begin < target) lo = mid + 1; else hi = mid; } return lo; };
            size_t const r_lo = t == 0 ? 0 : cut(t), r_hi = t + 1 == n_threads ? n_reads : cut(t + 1);
            threads.emplace_back(fill, r_lo, r_hi, std::ref(outs[t]));
        }
        for (auto& th : threads) th.join();
    }
    for (ChunkOut const& o : outs) {
        if (o.status) return FXG_OK;
        for (int d = 0; d < 256; ++d) P.level_mask[d] |= o.level_mask[d];
        P.max_depth = std::max(P.max_depth, o.max_depth);
    }
    P.n_nodes = node_at; P.n_leaves = leaf_at; P.n_walks = walk_at; P.n_reads = uint32_t(n_reads);
    P.hreads.assign(rrec, rrec + n_reads);
    if (!P.ready) CUDA_TRY(err, cudaEventCreateWithFlags(&P.ready, cudaEventDisableTiming));
    CUDA_TRY(err, cudaMemcpyAsync(P.dev.p, H, up, cudaMemcpyHostToDevice, c->stage_stream));
    CUDA_TRY(err, cudaEventRecord(P.ready, c->stage_stream));
    ctr.h2d_bytes += up;
    P.ok = true;
    return FXG_OK;
}

// root window of a walk, as the device computes it (dp_kernels.cuh: root_window) and as compute_span does from the nodes
inline Span root_span_of(ReadRec const& R, int64_t diag, uint64_t ref_len) {
    uint64_t const base = uint64_t(R.root_m) + 2ull * R.root_k + 1;
    int64_t const s = diag + int64_t(R.root_from) - int64_t(R.root_k) - int64_t(R.root_extra);
    Span r;
    r.offset = s >= 0 ? uint64_t(s) : 0;
    r.length = std::min<uint64_t>(base + 2ull * R.root_extra, ref_len - r.offset);
    r.extra = R.root_extra;
    return r;
}

// The root level of a part on the device (root_kernels.cuh).  `entries` are the part's root walks on the device, in anchor
// order.  Returns FXG_OK with P.hits filled, an error, or kRootFallback when the part has to take the host's way
// (run_root_passes): a member of a shared pass that the pass cannot vouch for, or more checkpoint records than the budget.
constexpr int kRootFallback = 1;
int root_level_device(fxg_ctx* c, Worker& w, Batch& B, uint32_t r0, uint32_t n_reads, PartState& P, const RootEntry* d_entries, uint32_t n_roots,
                      const ReadRec* d_reads, unsigned long long* d_member_totals, ClassDef const* classes, int n_cls) {
    cudaStream_t const st = w.stream;
    bool const want_cigar = !B.cfg.without_cigar;
    Pool const& pool = *B.pool;
    size_t const n = n_roots, n_members = B.members.size();
    // ---- buffers ----
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t const at = off; off += (bytes + 255) & ~size_t(255); return at; };
    size_t const o_ws = carve(n * 8), o_len = carve(n * 4), o_read = carve(n * 4), o_orient = carve(n), o_key = carve(n * 8), o_idx = carve(n * 4);
    size_t const o_key_s = carve(n * 8), o_idx_s = carve(n * 4), o_ustart = carve(n * 4), o_uof = carve(n * 4), o_pos = carve(n * 4);
    size_t const o_score = carve(n * 4), o_end = carve(n * 4), o_flag = carve(n);
    size_t const o_units = carve(n * sizeof(UnitRec)), o_uwords = carve(n * 8), o_uck = carve(n * 8);
    size_t const o_key2 = carve(n * 8), o_idx2 = carve(n * 4), o_key2_s = carve(n * 8), o_idx2_s = carve(n * 4);
    size_t const o_rep = carve(n * 4), o_tbcap = carve(n * 8), o_tbcig = carve(n * 8), o_tbslot = carve(n * 4);
    size_t const o_hit = carve(n * 4), o_hitat = carve(n * 4), o_ctr = carve(kRootCounters * 4);
    CUDA_TRY(w.err, w.d_root.ensure_scaled(off, P.scale));
    uint8_t* const D = w.d_root.as<uint8_t>();
    size_t tmp_bytes = 0, t1 = 0;
    {   // temporary storage of the sorts and scans
        cub::DeviceRadixSort::SortPairs(nullptr, t1, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr, int(n), 0, 64, st); tmp_bytes = std::max(tmp_bytes, t1);
        cub::DeviceScan::InclusiveSum(nullptr, t1, (const uint32_t*)nullptr, (uint32_t*)nullptr, int(n), st); tmp_bytes = std::max(tmp_bytes, t1);
        cub::DeviceScan::ExclusiveSum(nullptr, t1, (const uint64_t*)nullptr, (uint64_t*)nullptr, int(n), st); tmp_bytes = std::max(tmp_bytes, t1);
        cub::DeviceScan::ExclusiveSum(nullptr, t1, (const uint32_t*)nullptr, (uint32_t*)nullptr, int(n), st); tmp_bytes = std::max(tmp_bytes, t1);
    }
    CUDA_TRY(w.err, w.d_cub.ensure_scaled(tmp_bytes + 256, P.scale));
    RootCtx C{};
    C.entries = d_entries; C.n_roots = n_roots; C.reads = d_reads; C.n_reads = n_reads;
    C.ref_base = c->refs.d_base.as<uint64_t>(); C.ref_len = c->refs.d_len.as<uint64_t>();
    for (int ci = 0; ci < n_cls; ++ci) C.classes[ci] = RootClass{uint32_t(kWidths[classes[ci].widx]), classes[ci].G};
    C.want_cigar = want_cigar ? 1u : 0u; C.share = c->share_root_passes ? 1u : 0u;
    C.ws = reinterpret_cast<uint64_t*>(D + o_ws); C.len = reinterpret_cast<uint32_t*>(D + o_len); C.read = reinterpret_cast<uint32_t*>(D + o_read); C.orient = D + o_orient;
    C.key = reinterpret_cast<uint64_t*>(D + o_key); C.idx = reinterpret_cast<uint32_t*>(D + o_idx);
    C.key_s = reinterpret_cast<uint64_t*>(D + o_key_s); C.idx_s = reinterpret_cast<uint32_t*>(D + o_idx_s);
    C.unit_start = reinterpret_cast<uint32_t*>(D + o_ustart); C.unit_of = reinterpret_cast<uint32_t*>(D + o_uof); C.pos_of = reinterpret_cast<uint32_t*>(D + o_pos);
    C.m_score = reinterpret_cast<int32_t*>(D + o_score); C.m_end = reinterpret_cast<uint32_t*>(D + o_end); C.m_flag = D + o_flag;
    C.units = reinterpret_cast<UnitRec*>(D + o_units); C.unit_words = reinterpret_cast<uint64_t*>(D + o_uwords); C.unit_ck = reinterpret_cast<uint64_t*>(D + o_uck);
    C.key2 = reinterpret_cast<uint64_t*>(D + o_key2); C.idx2 = reinterpret_cast<uint32_t*>(D + o_idx2);
    C.key2_s = reinterpret_cast<uint64_t*>(D + o_key2_s); C.idx2_s = reinterpret_cast<uint32_t*>(D + o_idx2_s);
    C.rep = reinterpret_cast<uint32_t*>(D + o_rep); C.tb_cap = reinterpret_cast<uint64_t*>(D + o_tbcap); C.tb_cig = reinterpret_cast<uint64_t*>(D + o_tbcig);
    C.tb_slot = reinterpret_cast<uint32_t*>(D + o_tbslot);
    C.hit = reinterpret_cast<uint32_t*>(D + o_hit); C.hit_at = reinterpret_cast<uint32_t*>(D + o_hitat);
    C.counters = reinterpret_cast<uint32_t*>(D + o_ctr); C.member_totals = d_member_totals; C.read0 = r0;
    uint32_t const grid = uint32_t((n + 255) / 256);
    size_t const back_bytes = kRootCounters * 4 + n_members * kMemberTotals * 8;
    CUDA_TRY(w.err, w.h_root_back.ensure(back_bytes));
    auto read_back = [&]() -> int {          // counters (and the members' totals) to the host; waits
        CUDA_TRY(w.err, cudaMemcpyAsync(w.h_root_back.p, C.counters, kRootCounters * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(w.err, cudaMemcpyAsync(w.h_root_back.as<uint8_t>() + kRootCounters * 4, d_member_totals, n_members * kMemberTotals * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(w.err, w.wait_for(st));
        w.ctr.d2h_bytes += back_bytes;
        return FXG_OK;
    };
    const uint32_t* const ctr = w.h_root_back.as<uint32_t>();
    auto ctr64 = [&](int at) { uint64_t v; std::memcpy(&v, ctr + at, 8); return v; };

    // ---- windows, units ----
    CUDA_TRY(w.err, cudaMemsetAsync(C.counters, 0, kRootCounters * 4, st));
    CUDA_TRY(w.err, cudaMemsetAsync(C.unit_start, 0, n * 4, st));
    root_prepare_kernel<<<grid, 256, 0, st>>>(C);
    CUDA_TRY(w.err, cub::DeviceRadixSort::SortPairs(w.d_cub.p, tmp_bytes, C.key, const_cast<uint64_t*>(C.key_s), C.idx, const_cast<uint32_t*>(C.idx_s), int(n), 0, 64, st));
    root_cluster_kernel<<<grid, 256, 0, st>>>(C);
    CUDA_TRY(w.err, cub::DeviceScan::InclusiveSum(w.d_cub.p, tmp_bytes, C.unit_start, const_cast<uint32_t*>(C.unit_of), int(n), st));
    CUDA_TRY(w.err, cudaMemsetAsync(C.unit_words, 0, n * 8, st));
    root_units_kernel<<<grid, 256, 0, st>>>(C);
    CUDA_TRY(w.err, cub::DeviceScan::ExclusiveSum(w.d_cub.p, tmp_bytes, C.unit_words, const_cast<uint64_t*>(C.unit_ck), int(n), st));
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches += 6;
    int rc = read_back();
    if (rc != FXG_OK) return rc;
    P.t_mark[2] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count();
    g_prof.lap(w, 7);
    uint32_t const n_feasible = ctr[kCtrFeasible], n_units = ctr[kCtrUnits];
    uint64_t const ck_words = ctr64(kCtrCkWords);
    auto add_root_stats = [&]() {
        const uint64_t* const mt = reinterpret_cast<const uint64_t*>(w.h_root_back.as<uint8_t>() + kRootCounters * 4);
        for (size_t mi = 0; mi < n_members; ++mi) {
            fxg_stats& S = P.out.stats[mi];
            S.n_aligned_root += mt[mi * kMemberTotals + 5]; S.sum_aligned_root += mt[mi * kMemberTotals + 6]; S.cells_root += mt[mi * kMemberTotals + 7];
        }
    };
    if (n_feasible == 0 || n_units == 0) { add_root_stats(); return FXG_OK; }
    uint32_t class_units[kMaxLevelClasses];
    for (int ci = 0; ci < kMaxLevelClasses; ++ci) class_units[ci] = ctr[kCtrClassUnits + ci];
    int timed_class = 0;                                 // the class of the largest launch: timed with an event pair of its own

    // ---- score passes, one launch per class ----
    CUDA_TRY(w.err, w.d_tasks.ensure_scaled(size_t(n_units) * sizeof(DpTask), P.scale));
    CUDA_TRY(w.err, w.d_results.ensure_scaled(size_t(n_units) * sizeof(DpResult), P.scale));
    DevBuf& ckb = w.d_ck[0];
    if (want_cigar && ckb.ensure_scaled(std::max<uint64_t>(ck_words, 4) * 4, P.scale) != cudaSuccess) {
        (void)cudaGetLastError();
        return kRootFallback;                            // no room for all the checkpoint records at once: the host's way works in chunks
    }
    C.tasks = w.d_tasks.as<DpTask>(); C.results = w.d_results.as<DpResult>(); C.ck = ckb.as<uint32_t>();
    root_tasks_kernel<<<(n_units + 255) / 256, 256, 0, st>>>(C, n_units);
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches++;
    {
        // largest class first on the worker's stream, the others beside it
        int order[kMaxLevelClasses]; int n_used = 0;
        for (int ci = 0; ci < n_cls; ++ci) if (class_units[ci]) order[n_used++] = ci;
        std::sort(order, order + n_used, [&](int a, int b) { return class_units[a] > class_units[b]; });
        uint32_t prefix[kMaxLevelClasses + 1] = {0};
        for (int ci = 0; ci < kMaxLevelClasses; ++ci) prefix[ci + 1] = prefix[ci] + class_units[ci];
        CUDA_TRY(w.err, w.fork(st, n_used));
        for (int x = 0; x < n_used; ++x) {
            int const ci = order[x];
            EngineLaunch X;
            rc = engine_launch(c, w, pool, classes[ci], C.tasks + prefix[ci], w.d_results.as<DpResult>(), want_cigar ? ckb.as<uint32_t>() : nullptr,
                               class_units[ci], nullptr, nullptr, 0, X);
            if (rc != FXG_OK) return rc;
            cudaStream_t s2;
            CUDA_TRY(w.err, w.fan_stream(st, x, s2));
            if (x == 0) { timed_class = ci; CUDA_TRY(w.err, cudaEventRecord(w.ev_b0, st)); }
            CUDA_TRY(w.err, launch_dp(X.widx, want_cigar, X.L, X.grid, X.smem, s2));
            if (x == 0) CUDA_TRY(w.err, cudaEventRecord(w.ev_b1, st));
            w.ctr.kernel_launches++;
        }
        CUDA_TRY(w.err, w.join(st, n_used));
    }
    // ---- every member's result; which alignments share a traceback ----
    root_results_kernel<<<grid, 256, 0, st>>>(C);
    w.ctr.kernel_launches++;
    if (want_cigar) {
        CUDA_TRY(w.err, cudaMemsetAsync(C.key2 + n_feasible, 0xff, (n - n_feasible) * 8, st));
        CUDA_TRY(w.err, cub::DeviceRadixSort::SortPairs(w.d_cub.p, tmp_bytes, C.key2, const_cast<uint64_t*>(C.key2_s), C.idx2, const_cast<uint32_t*>(C.idx2_s), int(n), 0, 64, st));
        root_dedup_kernel<<<grid, 256, 0, st>>>(C);
        CUDA_TRY(w.err, cudaMemsetAsync(C.tb_cap + n_feasible, 0, (n - n_feasible) * 8, st));
        root_walk_count_kernel<<<grid, 256, 0, st>>>(C);
        CUDA_TRY(w.err, cub::DeviceScan::ExclusiveSum(w.d_cub.p, tmp_bytes, C.tb_cap, const_cast<uint64_t*>(C.tb_cig), int(n), st));
        w.ctr.kernel_launches += 4;
    }
    CUDA_TRY(w.err, cudaGetLastError());
    rc = read_back();
    if (rc != FXG_OK) return rc;
    {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, w.ev_b0, w.ev_b1) == cudaSuccess) { w.ctr.root_launch_ms += ms; w.ctr.root_launches++; w.ctr.root_launch_word_steps += ctr64(kCtrClassWs + 2 * timed_class); }
    }
    P.t_mark[3] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count();
    g_prof.lap(w, 11);
    if (ctr[kCtrErrors]) return fail(w.err, FXG_ERR_CUDA, "internal: the DP engine lost track of its window buffer");
    if (ctr[kCtrSlow]) return kRootFallback;             // a shared pass cannot vouch for one of its members: the host's way scores it again
    uint32_t const n_accepted = ctr[kCtrAccepted], n_tb = ctr[kCtrTracebacks];
    uint64_t const cig_total = ctr64(kCtrCigars);
    w.ctr.dp_tasks += n_units; w.ctr.dp_word_steps += ctr64(kCtrWordSteps); w.ctr.trace_bytes += ck_words * 4;
    w.ctr.shared_score_passes += ctr[kCtrShared];
    if (want_cigar) w.ctr.shared_tracebacks += n_accepted - n_tb;
    w.ctr.waves++;
    if (n_accepted == 0) { add_root_stats(); return FXG_OK; }
    // ---- tracebacks of the representatives ----
    if (want_cigar) {
        CUDA_TRY(w.err, w.d_wtasks.ensure_scaled(size_t(n_tb) * sizeof(Walk2Task), P.scale));
        CUDA_TRY(w.err, w.d_wresults.ensure_scaled(size_t(n_tb) * sizeof(WalkResult), P.scale));
        if (w.cig_used == 0) CUDA_TRY(w.err, w.d_cigars.ensure_scaled(cig_total * 4, P.scale));
        CUDA_TRY(w.err, w.d_cigars.ensure_preserving((w.cig_used + cig_total) * 4, w.cig_used * 4, st));
        C.wtasks = w.d_wtasks.as<Walk2Task>(); C.wresults = w.d_wresults.as<WalkResult>();
        CUDA_TRY(w.err, cudaMemsetAsync(w.d_cigars.as<uint32_t>() + w.cig_used, 0, cig_total * 4, st));      // (a slot is filled from its end: the unused front stays zero)
        root_walks_kernel<<<grid, 256, 0, st>>>(C, w.cig_used);
        CUDA_TRY(w.err, cudaGetLastError());
        w.ctr.kernel_launches++;
        uint32_t width_tb[6], wprefix[7] = {0};
        int n_launch = 0;
        for (int wi = 0; wi < 6; ++wi) { width_tb[wi] = ctr[kCtrWidthTb + wi]; wprefix[wi + 1] = wprefix[wi] + width_tb[wi]; n_launch += width_tb[wi] != 0; }
        CUDA_TRY(w.err, cudaEventRecord(w.ev_w0, st));
        CUDA_TRY(w.err, w.fork(st, n_launch));
        for (int wi = 0, q = 0; wi < 6; ++wi) {
            if (!width_tb[wi]) continue;
            cudaStream_t s2;
            CUDA_TRY(w.err, w.fan_stream(st, q++, s2));
            CUDA_TRY(w.err, launch_walk(wi, walk_launch(c, w, pool, ckb.as<uint32_t>(), C.wtasks + wprefix[wi], width_tb[wi]), s2));
            w.ctr.kernel_launches++;
        }
        CUDA_TRY(w.err, w.join(st, n_launch));
        CUDA_TRY(w.err, cudaEventRecord(w.ev_w1[0], st));
    }
    // ---- alignment records in anchor order ----
    CUDA_TRY(w.err, w.d_hits.ensure_scaled(size_t(n_accepted) * sizeof(fxg_alignment), P.scale));
    CUDA_TRY(w.err, w.h_hits.ensure_scaled(size_t(n_accepted) * sizeof(fxg_alignment), P.scale));
    C.out = w.d_hits.as<fxg_alignment>();
    root_hits_kernel<<<grid, 256, 0, st>>>(C);
    CUDA_TRY(w.err, cub::DeviceScan::ExclusiveSum(w.d_cub.p, tmp_bytes, C.hit, const_cast<uint32_t*>(C.hit_at), int(n), st));
    root_finish_kernel<<<grid, 256, 0, st>>>(C);
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches += 3;
    CUDA_TRY(w.err, cudaMemcpyAsync(w.h_hits.p, w.d_hits.p, size_t(n_accepted) * sizeof(fxg_alignment), cudaMemcpyDeviceToHost, st));
    w.ctr.d2h_bytes += size_t(n_accepted) * sizeof(fxg_alignment);
    rc = read_back();
    if (rc != FXG_OK) return rc;
    if (want_cigar) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, w.ev_w0, w.ev_w1[0]) == cudaSuccess) w.ctr.trace_kernel_ms += ms;
    }
    P.t_mark[4] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count();
    g_prof.lap(w, 12);
    if (ctr[kCtrErrors]) return fail(w.err, FXG_ERR_CUDA, "internal: the traceback of an alignment disagrees with its score pass");
    add_root_stats();
    P.hits.assign(w.h_hits.as<fxg_alignment>(), w.h_hits.as<fxg_alignment>() + n_accepted);
    w.cig_used += cig_total;
    g_prof.lap(w, 13);
    return FXG_OK;
}

// query_verifier::verify() for every anchor of reads [r0, r1) of a batch: the tree walks on the device, then the root
// level for the walks that verify their root.  On return P.hits holds the part's alignments in anchor order, and the
// statistics have been added to P.out.stats per member.
int run_device_walks(fxg_ctx* c, Worker& w, Batch& B, uint32_t r0, uint32_t r1, PartState& P) {
    g_prof.start(w);
    PartOut& out = P.out;
    cudaStream_t const st = w.stream;
    // ---- the members' slices that make up this part ----
    struct Slice { uint32_t member, a, b; uint32_t walk0, node0, leaf0, read0, n_walks, n_nodes, n_leaves; };
    std::vector<Slice> slices;
    uint32_t n_walks = 0, n_nodes = 0, n_leaves = 0;
    uint32_t level_mask[256] = {0};
    uint32_t max_depth = 0;
    for (size_t mi = 0; mi < B.members.size(); ++mi) {
        Member const& M = B.members[mi];
        Prepared const& R = M.J->prep;
        uint32_t const lo = std::max(r0, M.read0), hi = std::min(r1, M.read0 + R.n_reads);
        if (lo >= hi) continue;
        Slice s{};
        s.member = uint32_t(mi); s.a = lo - M.read0; s.b = hi - M.read0;
        auto walk_at = [&](uint32_t i) { return i < R.n_reads ? R.hreads[i].walk_begin : R.n_walks; };
        auto node_at = [&](uint32_t i) { return i < R.n_reads ? R.hreads[i].node_base : R.n_nodes; };
        auto leaf_at = [&](uint32_t i) { return i < R.n_reads ? R.hreads[i].leaf_base : R.n_leaves; };
        s.walk0 = n_walks; s.node0 = n_nodes; s.leaf0 = n_leaves; s.read0 = lo - r0;
        s.n_walks = walk_at(s.b) - walk_at(s.a); s.n_nodes = node_at(s.b) - node_at(s.a); s.n_leaves = leaf_at(s.b) - leaf_at(s.a);
        n_walks += s.n_walks; n_nodes += s.n_nodes; n_leaves += s.n_leaves;
        for (uint32_t d = 1; d <= R.max_depth; ++d) level_mask[d] |= R.level_mask[d];
        max_depth = std::max(max_depth, R.max_depth);
        slices.push_back(s);
    }
    uint32_t const n_reads = r1 - r0;
    P.walks.clear(); P.hits.clear();
    if (n_walks == 0) return FXG_OK;
    for (uint32_t d = 0; d < 256; ++d)
        if (uint64_t(level_mask[d]) >> c->n_classes) return fail(w.err, FXG_ERR_STATE, "internal: a job's records name a configuration class the context does not have");
    bool const ivopt = B.cfg.interval_optimization != 0;
    bool const direct = B.cfg.verification_kind == FXG_KIND_DIRECT_FULL;
    size_t const n_members = B.members.size();
    // ---- classes (a copy of the context's table as of now: it only grows, and every class of these jobs is in it) ----
    ClassDef classes[kMaxLevelClasses]; int n_cls = 0;
    { std::lock_guard<std::mutex> lock(c->class_mu); n_cls = c->n_classes; std::copy(c->classes, c->classes + n_cls, classes); }
    // ---- device buffers: one allocation, carved up ----
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t const at = off; off += (bytes + 255) & ~size_t(255); return at; };
    size_t const o_nodes = carve(size_t(n_nodes) * sizeof(NodeRec)), o_leaves = carve(size_t(n_leaves) * sizeof(LeafRec));
    size_t const o_reads = carve(size_t(n_reads) * sizeof(ReadRec)), o_anchors = carve(size_t(n_walks) * sizeof(AnchorRec16));
    size_t const o_walks = carve(size_t(n_walks) * sizeof(WalkRec)), o_node = carve(size_t(n_walks) * 4);
    size_t const o_ws = carve(size_t(n_walks) * 8), o_len = carve(size_t(n_walks) * 4), o_flag = carve(n_walks);
    size_t const o_rep = carve(size_t(n_nodes) * 2 * 8), o_rep_min = carve(size_t(n_nodes) * 2 * 8);
    // zeroed together: n_inner | sum_inner | cells_inner | counts | class_active | totals | member totals | n_roots
    size_t const o_zero = off;
    size_t const o_ninner = carve(size_t(n_walks) * 4), o_sum = carve(size_t(n_walks) * 8), o_cells = carve(size_t(n_walks) * 8);
    size_t const o_counts = carve(size_t(kMaxLevelClasses) * 4 * 2);               // counts, then class_active
    size_t const o_back = carve(64 + n_members * kMemberTotals * 8);                // totals (3) | n_roots | member totals: read back together
    size_t const zero_bytes = off - o_zero;
    size_t const o_tasks = carve(size_t(n_walks) * sizeof(DpTask));
    size_t const o_results = carve(size_t(n_walks) * sizeof(DpResult));
    size_t const o_rootflag = carve(n_walks), o_rootcnt = carve(size_t(n_reads) * 2 * 4), o_rootoff = carve(size_t(n_reads) * 2 * 4);
    size_t const o_inserted = carve(ivopt ? size_t(n_walks) * 4 : 0);
    // (only the worker that runs merged batches -- one part per batch -- sizes its buffers for the largest of them)
    P.scale = P.n_parts == 1 ? std::max(1.0, double(c->merge_max_walks) / double(std::max<uint32_t>(n_walks, 1))) : 1.0;
    CUDA_TRY(w.err, w.d_lv.ensure_scaled(off, P.scale));
    uint8_t* const D = w.d_lv.as<uint8_t>();
    size_t const o_member_totals = o_back + 64;
    // ---- gather the members' records (device to device), bases shifted to their place in this part ----
    P.part_reads.resize(n_reads);
    for (Slice const& s : slices) {
        Member const& M = B.members[s.member];
        Prepared const& R = M.J->prep;
        CUDA_TRY(w.err, cudaStreamWaitEvent(st, R.ready, 0));
        if (M.J->pool_ready) CUDA_TRY(w.err, cudaStreamWaitEvent(st, M.J->pool_ready, 0));
        const uint8_t* const S = R.dev.as<uint8_t>();
        ReadRec const& first = R.hreads[s.a];
        if (s.n_nodes) CUDA_TRY(w.err, cudaMemcpyAsync(D + o_nodes + size_t(s.node0) * sizeof(NodeRec), S + R.o_nodes + size_t(first.node_base) * sizeof(NodeRec),
                                                       size_t(s.n_nodes) * sizeof(NodeRec), cudaMemcpyDeviceToDevice, st));
        if (s.n_leaves) CUDA_TRY(w.err, cudaMemcpyAsync(D + o_leaves + size_t(s.leaf0) * sizeof(LeafRec), S + R.o_leaves + size_t(first.leaf_base) * sizeof(LeafRec),
                                                        size_t(s.n_leaves) * sizeof(LeafRec), cudaMemcpyDeviceToDevice, st));
        if (s.n_walks) CUDA_TRY(w.err, cudaMemcpyAsync(D + o_anchors + size_t(s.walk0) * sizeof(AnchorRec16), S + R.o_anchors + size_t(first.walk_begin) * sizeof(AnchorRec16),
                                                       size_t(s.n_walks) * sizeof(AnchorRec16), cudaMemcpyDeviceToDevice, st));
        uint32_t const n = s.b - s.a;
        uint32_t const d_walk = s.walk0 - first.walk_begin, d_node = s.node0 - first.node_base, d_leaf = s.leaf0 - first.leaf_base;   // (modulo 2^32)
        gather_reads_kernel<<<(n + 127) / 128, 128, 0, st>>>(reinterpret_cast<const ReadRec*>(S + R.o_reads) + s.a, reinterpret_cast<ReadRec*>(D + o_reads) + s.read0,
                                                            n, d_walk, d_node, d_leaf, M.pool_shift, s.member);
        CUDA_TRY(w.err, cudaGetLastError());
        w.ctr.kernel_launches++;
        for (uint32_t i = 0; i < n; ++i) {                     // the same on the host (the root level reads it)
            ReadRec r = R.hreads[s.a + i];
            r.walk_begin += d_walk; r.node_base += d_node; r.leaf_base += d_leaf;
            r.qoff_forward += M.pool_shift; r.qoff_reverse += M.pool_shift; r.member = s.member;
            P.part_reads[s.read0 + i] = r;
        }
    }
    if (B.merged_ready) CUDA_TRY(w.err, cudaStreamWaitEvent(st, B.merged_ready, 0));
    CUDA_TRY(w.err, cudaMemsetAsync(D + o_zero, 0, zero_bytes, st));
    walk_init_kernel<<<(n_walks + 255) / 256, 256, 0, st>>>(reinterpret_cast<const AnchorRec16*>(D + o_anchors), reinterpret_cast<const ReadRec*>(D + o_reads), n_reads,
                                                         reinterpret_cast<const LeafRec*>(D + o_leaves), reinterpret_cast<WalkRec*>(D + o_walks),
                                                         reinterpret_cast<uint32_t*>(D + o_node), n_walks, direct ? 1u : 0u);
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches++;

    LevelCtx C{};
    C.walks = reinterpret_cast<const WalkRec*>(D + o_walks); C.nodes = reinterpret_cast<const NodeRec*>(D + o_nodes); C.n_walks = n_walks;
    C.ref_base = c->refs.d_base.as<uint64_t>(); C.ref_len = c->refs.d_len.as<uint64_t>();
    C.node = reinterpret_cast<uint32_t*>(D + o_node);
    C.ask_ws = reinterpret_cast<uint64_t*>(D + o_ws); C.ask_len = reinterpret_cast<uint32_t*>(D + o_len); C.flag = D + o_flag;
    C.rep = reinterpret_cast<unsigned long long*>(D + o_rep); C.rep_min = reinterpret_cast<unsigned long long*>(D + o_rep_min);
    C.n_inner = reinterpret_cast<uint32_t*>(D + o_ninner); C.sum_inner = reinterpret_cast<uint64_t*>(D + o_sum); C.cells_inner = reinterpret_cast<uint64_t*>(D + o_cells);
    C.tasks = reinterpret_cast<DpTask*>(D + o_tasks);
    C.counts = reinterpret_cast<uint32_t*>(D + o_counts); C.class_active = C.counts + kMaxLevelClasses;
    C.results = reinterpret_cast<const DpResult*>(D + o_results);
    C.totals = reinterpret_cast<unsigned long long*>(D + o_back);
    C.infer = c->infer_inner ? 1u : 0u;
    for (int ci = 0; ci < n_cls; ++ci) C.cls_W[ci] = uint8_t(kWidths[classes[ci].widx]);

    uint32_t const wgrid = (n_walks + 255) / 256;
    Pool const& pool = *B.pool;
    auto engine = [&](uint32_t mask) -> int {
        // the classes of a level are independent: the first on the worker's stream, the others beside it
        int const n_launch = __builtin_popcount(mask);           // (mask names classes below n_cls only: checked above)
        CUDA_TRY(w.err, w.fork(st, n_launch));
        for (int ci = 0, q = 0; ci < n_cls; ++ci) {
            if (!(mask >> ci & 1u)) continue;
            EngineLaunch X;
            int const rc = engine_launch(c, w, pool, classes[ci], C.tasks, reinterpret_cast<DpResult*>(D + o_results), nullptr, n_walks, C.counts + ci,
                                         C.class_active, uint32_t(ci), X);
            if (rc != FXG_OK) return rc;
            cudaStream_t s2;
            CUDA_TRY(w.err, w.fan_stream(st, q++, s2));
            CUDA_TRY(w.err, launch_dp(X.widx, false, X.L, X.grid, X.smem, s2));
            w.ctr.kernel_launches++;
        }
        CUDA_TRY(w.err, w.join(st, n_launch));
        return FXG_OK;
    };
    g_prof.lap(w, 2);
    CUDA_TRY(w.err, cudaEventRecord(w.ev0, st));
    for (uint32_t lv = direct ? 0 : max_depth; lv >= 1; --lv) {
        if (level_mask[lv] == 0) continue;
        C.level = lv;
        if (C.infer && n_nodes) {
            CUDA_TRY(w.err, cudaMemsetAsync(C.rep, 0, size_t(n_nodes) * 2 * 8, st));
            CUDA_TRY(w.err, cudaMemsetAsync(C.rep_min, 0xff, size_t(n_nodes) * 2 * 8, st));
        }
        CUDA_TRY(w.err, cudaMemsetAsync(C.counts, 0, size_t(kMaxLevelClasses) * 4 * 2, st));
        level_begin_kernel<<<wgrid, 256, 0, st>>>(C);
        level_first_kernel<<<wgrid, 256, 0, st>>>(C);
        CUDA_TRY(w.err, cudaGetLastError());
        int rc = engine(level_mask[lv]);
        if (rc != FXG_OK) return rc;
        w.ctr.kernel_launches += 2;
        if (C.infer) {
            CUDA_TRY(w.err, cudaMemsetAsync(C.counts, 0, size_t(kMaxLevelClasses) * 4, st));
            level_second_kernel<<<wgrid, 256, 0, st>>>(C);
            CUDA_TRY(w.err, cudaGetLastError());
            rc = engine(level_mask[lv]);
            if (rc != FXG_OK) return rc;
            CUDA_TRY(w.err, cudaMemsetAsync(C.counts, 0, size_t(kMaxLevelClasses) * 4, st));
            level_third_kernel<<<wgrid, 256, 0, st>>>(C);
            CUDA_TRY(w.err, cudaGetLastError());
            rc = engine(level_mask[lv]);                       // (usually nothing is left for it)
            if (rc != FXG_OK) return rc;
            w.ctr.kernel_launches += 2;
        }
        level_advance_kernel<<<wgrid, 256, 0, st>>>(C);
        CUDA_TRY(w.err, cudaGetLastError());
        w.ctr.kernel_launches++;
        w.ctr.waves++;
    }
    CUDA_TRY(w.err, cudaEventRecord(w.ev1, st));
    // ---- which walks count and which verify their root; statistics per member ----
    DecideCtx Dc{};
    Dc.walks = C.walks; Dc.node = C.node; Dc.reads = reinterpret_cast<const ReadRec*>(D + o_reads); Dc.n_reads = n_reads;
    Dc.ref_len = C.ref_len; Dc.n_inner = C.n_inner; Dc.sum_inner = C.sum_inner; Dc.cells_inner = C.cells_inner;
    Dc.root_flag = D + o_rootflag; Dc.root_count = reinterpret_cast<uint32_t*>(D + o_rootcnt);
    Dc.inserted = reinterpret_cast<uint32_t*>(D + o_inserted);
    Dc.member_totals = reinterpret_cast<unsigned long long*>(D + o_member_totals);
    Dc.ivopt = ivopt ? 1u : 0u;
    uint32_t* const d_rootoff = reinterpret_cast<uint32_t*>(D + o_rootoff);
    uint32_t* const d_nroots = reinterpret_cast<uint32_t*>(D + o_back + 24);
    uint32_t const pair_grid = (2 * n_reads * 32 + 127) / 128;
    decide_kernel<<<pair_grid, 128, 0, st>>>(Dc);
    scan_counts_kernel<<<1, 1024, 0, st>>>(Dc.root_count, d_rootoff, 2 * n_reads, d_nroots);
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches += 2;
    size_t const back_bytes = 64 + n_members * kMemberTotals * 8;
    CUDA_TRY(w.err, w.h_lv_back.ensure(back_bytes));
    CUDA_TRY(w.err, cudaMemcpyAsync(w.h_lv_back.p, D + o_back, back_bytes, cudaMemcpyDeviceToHost, st));
    g_prof.lap(w, 6);
    P.t_mark[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count();
    CUDA_TRY(w.err, w.wait_for(st));
    P.t_mark[1] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count();
    float ms = 0;
    CUDA_TRY(w.err, cudaEventElapsedTime(&ms, w.ev0, w.ev1));
    w.ctr.dp_kernel_ms += ms;
    w.ctr.d2h_bytes += back_bytes;
    const uint64_t* const totals = w.h_lv_back.as<uint64_t>();
    w.ctr.dp_tasks += totals[0]; w.ctr.dp_word_steps += totals[1]; w.ctr.inferred_inner += totals[2];
    uint32_t const n_roots = *reinterpret_cast<const uint32_t*>(w.h_lv_back.as<uint8_t>() + 24);
    const uint64_t* const mt = reinterpret_cast<const uint64_t*>(w.h_lv_back.as<uint8_t>() + 64);
    for (size_t mi = 0; mi < n_members; ++mi) {
        fxg_stats& S = out.stats[mi];
        S.n_aligned_inner += mt[mi * kMemberTotals + 0]; S.sum_aligned_inner += mt[mi * kMemberTotals + 1]; S.cells_inner += mt[mi * kMemberTotals + 2];
        S.n_avoided_root += mt[mi * kMemberTotals + 3]; S.sum_avoided_root += mt[mi * kMemberTotals + 4];
    }
    g_prof.lap(w, 8);
    if (n_roots == 0) return FXG_OK;
    if (n_roots > n_walks) return fail(w.err, FXG_ERR_CUDA, "internal: more root walks than walks");
    // ---- the walks that verify their root, in anchor order ----
    CUDA_TRY(w.err, w.d_roots.ensure_scaled(size_t(n_roots) * sizeof(RootEntry), P.scale));
    CUDA_TRY(w.err, w.h_roots.ensure_scaled(size_t(n_roots) * sizeof(RootEntry), P.scale));
    root_emit_kernel<<<pair_grid, 128, 0, st>>>(Dc, d_rootoff, w.d_roots.as<RootEntry>());
    CUDA_TRY(w.err, cudaGetLastError());
    w.ctr.kernel_launches++;
    if (c->device_roots && c->refs.total < (uint64_t(1) << kPosBits) && pool.len < (uint64_t(1) << kPosBits) && n_reads < (1u << 27)) {
        int const rc = root_level_device(c, w, B, r0, n_reads, P, w.d_roots.as<RootEntry>(), n_roots, reinterpret_cast<const ReadRec*>(D + o_reads),
                                         reinterpret_cast<unsigned long long*>(D + o_member_totals), classes, n_cls);
        if (rc != kRootFallback) return rc;
        P.hits.clear();
    }
    // ---- the host's way: the entries come back, one score pass per walk that verifies its root (run_root_passes) ----
    CUDA_TRY(w.err, cudaMemcpyAsync(w.h_roots.p, w.d_roots.p, size_t(n_roots) * sizeof(RootEntry), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(w.err, w.wait_for(st));
    w.ctr.d2h_bytes += size_t(n_roots) * sizeof(RootEntry);
    const RootEntry* const re = w.h_roots.as<RootEntry>();
    g_prof.lap(w, 9);
    // ---- root level (verification.cpp:52-64, 95-109): one score pass per walk that verifies its root, straight from the entries ----
    std::vector<Pass> passes; std::vector<uint32_t> root_k, pass_read, pass_ref; std::vector<uint64_t> span_off; std::vector<uint32_t> span_len; std::vector<uint8_t> pass_orient;
    passes.reserve(n_roots); root_k.reserve(n_roots); pass_read.reserve(n_roots); pass_ref.reserve(n_roots); span_off.reserve(n_roots); span_len.reserve(n_roots); pass_orient.reserve(n_roots);
    bool const want_cigar = !B.cfg.without_cigar;
    uint32_t cur = 0;                                          // read of the entry at hand (entries come in walk order)
    for (uint32_t q = 0; q < n_roots; ++q) {
        RootEntry const& e = re[q];
        while (cur + 1 < n_reads && P.part_reads[cur + 1].walk_begin <= e.walk) ++cur;
        ReadRec const& R = P.part_reads[cur];
        if (e.walk < R.walk_begin || e.walk >= R.walk_begin + R.n_walks || e.ref_id >= c->refs.len.size())
            return fail(w.err, FXG_ERR_CUDA, "internal: a root walk outside its read");
        uint32_t const orient = e.walk - R.walk_begin >= R.n_forward ? 1u : 0u;
        Span const sp = root_span_of(R, e.diag, c->refs.len[e.ref_id]);
        fxg_stats& S = out.stats[R.member];
        S.n_aligned_root++; S.sum_aligned_root += sp.length; S.cells_root += uint64_t(R.root_m) * sp.length;
        Pass p;
        if (score_pass_for(c->refs.base[e.ref_id] + sp.offset, (orient ? R.qoff_reverse : R.qoff_forward) + R.root_from, uint32_t(sp.length), R.root_m, R.root_k,
                           want_cigar ? 0u : kFlagReverse, p)) {
            passes.push_back(p); root_k.push_back(R.root_k); pass_read.push_back(r0 + cur); pass_ref.push_back(e.ref_id);
            span_off.push_back(sp.offset); span_len.push_back(uint32_t(sp.length)); pass_orient.push_back(uint8_t(orient));
        }
    }
    g_prof.lap(w, 2);
    if (passes.empty()) return FXG_OK;
    auto hit = [&](size_t q, uint64_t start, uint32_t errors, uint64_t cigar_offset, uint32_t cigar_len) {
        fxg_alignment a{};
        a.start_in_reference = start; a.cigar_offset = cigar_offset; a.cigar_len = cigar_len;       // (the offset is relative to this part's region for now)
        a.num_errors = errors; a.read_index = pass_read[q]; a.reference_id = pass_ref[q]; a.orientation = pass_orient[q];
        P.hits.push_back(a);
    };
    if (want_cigar) {
        // score pass with checkpoints, then the traceback of the accepted ones
        std::vector<RootOut> root_outs;
        int const rc = run_root_passes(c, w, pool, passes, root_k, P.trace_budget, root_outs);
        if (rc != FXG_OK) return rc;
        g_prof.start(w);
        P.hits.reserve(passes.size());
        for (size_t q = 0; q < passes.size(); ++q)
            if (root_outs[q].score <= int32_t(root_k[q]))
                hit(q, span_off[q] + root_outs[q].begin_col, uint32_t(root_outs[q].score), root_outs[q].cigar_offset, root_outs[q].cigar_len);   // alignment.cpp:175
    } else {
        const DpResult* res = nullptr;
        int const rc = run_passes(c, w, pool, passes, nullptr, nullptr, &res);
        if (rc != FXG_OK) return rc;
        g_prof.start(w);
        for (size_t q = 0; q < passes.size(); ++q)
            if (res[q].score <= int32_t(root_k[q])) hit(q, span_off[q] + (span_len[q] - res[q].end_col), uint32_t(res[q].score), 0, 0);                // alignment.cpp:135-139
    }
    w.ctr.waves++;
    g_prof.lap(w, 13);
    return FXG_OK;
}

// query_verifier::verify() for every anchor of reads [read_lo, read_hi), level-synchronously.
//
// 1. Inner levels.  The walks are advanced deepest node first, so that all alignments of one tree level land in the same
//    wave and fill the machine together; a walk stops at its first failing level (verification.cpp:95-100) or arrives
//    at the root.
// 2. Interval optimisation (verification.cpp:62-64, 106-109, 119-136), exactly as the reference's sequential loop
//    would have it.  Whether a walk reaches the root depends on its inner alignments alone, and the root window is inserted
//    whenever the root is reached (even if the root alignment then fails) -- so once step 1 has run for EVERY walk
//    (speculatively: the sequential loop would not even have started some of them), one pass over each (read, strand,
//    reference) group in anchor order decides everything: a walk whose trimmed root window lies inside the window of an
//    earlier walk that reached the root is avoided (its speculative alignments are discarded, statistics included), any
//    other walk counts, and inserts its window if it reached the root.
// 3. Root level: one wave for the walks that count and reached the root (with checkpoints + tracebacks when CIGARs
//    are wanted).
void verify_part_score(fxg_ctx* c, Worker& w, Batch& B, uint32_t read_lo, uint32_t read_hi, PartState& P) {
    cudaSetDevice(c->device);
    P.t0 = std::chrono::steady_clock::now();
    if (g_prof.on) P.cpu0 = thread_cpu_ms();
    PartOut& out = P.out;
    out.stats.assign(B.members.size(), fxg_stats{});
    g_prof.start(w);
    fxg_job* const J = B.members[0].J;                   // (host-driven levels: the batch is this one job)
    Pool const& pool = *B.pool;
    bool const ivopt = B.cfg.interval_optimization != 0;
    std::vector<Walk>& walks = P.walks; std::vector<Group>& groups = P.groups; std::vector<uint32_t>& group_members = P.group_members;
    std::vector<std::vector<uint32_t>> level;            // walks waiting for the wave of their node's level (0 = root)
    std::vector<uint32_t> active;
    std::vector<Pass> passes; std::vector<uint32_t> pass_walk;
    w.cig_used = 0;

    // The walks climb their trees on the device (run_device_walks): what comes back are the walks that verify their root.
    // A job without device records (limits of prepare_job, or FXG_DEVICE_LEVELS=0) is driven from the host, level by level.
    bool const on_device = B.device;
    if (on_device) {
        walks.clear(); groups.clear(); group_members.clear();
        out.rc = run_device_walks(c, w, B, read_lo, read_hi, P);
        return;
    } else {
        // (fxg_verify_reads) the query pools and their Peq planes were enqueued on the staging stream by the caller's thread
        if (J->pool_ready && cudaStreamWaitEvent(w.stream, J->pool_ready, 0) != cudaSuccess) { out.rc = fail(w.err, FXG_ERR_CUDA, "cannot order the worker behind the upload"); return; }
        build_walks(c, J, read_lo, read_hi, walks, groups, group_members);
        // ---- tree level of every walk's first node ----
        size_t const n_all = walks.size();
        std::vector<uint8_t> memo;
        std::vector<uint8_t> dist(n_all, 0);
        uint32_t cur_read = UINT32_MAX; uint8_t max_dist = 0;
        for (uint32_t i = 0; i < n_all; ++i) {
            Walk const& wk = walks[i];
            fxg_read const& R = J->reads_p[wk.read];
            const fxg_pex_node* inner = J->nodes_p + R.node_offset;
            if (wk.read != cur_read) { cur_read = wk.read; memo.assign(R.num_inner, 0xff); }
            if (R.num_inner && wk.node >= inner && wk.node < inner + R.num_inner) dist[i] = node_dist(inner, memo, uint64_t(wk.node - inner));
            max_dist = std::max(max_dist, dist[i]);
        }
        level.assign(size_t(max_dist) + 1, std::vector<uint32_t>());
        for (uint32_t i = 0; i < n_all; ++i) { level[dist[i]].push_back(i); walks[i].state = W_WALKING; }
    }
    size_t const n_walks = walks.size();
    g_prof.lap(w, 0);

    auto span_of = [&](Walk& wk, bool is_root) -> Span {
        fxg_anchor const& A = J->anchors_p[wk.anchor];
        fxg_read const& R = J->reads_p[wk.read];
        const fxg_pex_node* leaves = J->nodes_p + R.node_offset + R.num_inner;
        if (!is_root) return compute_span(A.reference_position, *wk.node, leaves[A.pex_leaf_index].query_index_from, c->refs.len[A.reference_id], 0.0);
        if (!wk.have_root_span) {
            wk.root_span = compute_span(A.reference_position, *wk.node, leaves[A.pex_leaf_index].query_index_from, c->refs.len[A.reference_id],
                                        J->cfg.extra_verification_ratio);
            wk.have_root_span = true;
        }
        return wk.root_span;
    };

    // ---------------- 1. inner levels, deepest first ----------------
    // Walks of one read and strand that stand at the same tree node (anchors from the same subtree) ask the same question
    // about windows that are a few bases apart -- and an inner alignment is only ever asked whether it EXISTS
    // (alignment.cpp:98-112).  So per node the walk with the rightmost window start goes first; if it finds an alignment
    // (cost <= k, ending at reference position E), every walk of that node whose window ends at or after E has it as
    // well: their windows begin at or before the first one's, so the alignment -- which began somewhere inside the first
    // window -- lies inside theirs.  Identical windows share the answer either way.  Only the walks that remain undecided
    // are computed in a second launch of the level.
    struct Ask { uint64_t ws, qbase; uint32_t len, m, k, wi, key; bool feasible; };
    auto pass_of = [](Ask const& a) {
        Pass p;
        p.ref_base = a.ws; p.query_base = a.qbase; p.n = a.len; p.m = a.m;
        p.dlo = -int32_t(a.k); p.dhi = int32_t(int64_t(a.len) - int64_t(a.m) + int64_t(a.k)); p.flags = 0;   // score_pass_for
        return p;
    };
    // (node, strand) -> the ask that goes first, in a table over the node indices this part's reads use
    uint64_t node_lo = UINT64_MAX, node_hi = 0;
    for (uint32_t ri = read_lo; ri < read_hi && !on_device; ++ri) {
        fxg_read const& R = J->reads_p[ri];
        node_lo = std::min<uint64_t>(node_lo, R.node_offset); node_hi = std::max<uint64_t>(node_hi, R.node_offset + R.num_inner + R.num_leaves);
    }
    bool const infer = !on_device && c->infer_inner && node_hi > node_lo && (node_hi - node_lo) < (uint64_t(1) << 26);
    std::vector<uint32_t> rep_of, rep_stamp;
    if (infer) { rep_of.assign(size_t(node_hi - node_lo) * 2, 0); rep_stamp.assign(size_t(node_hi - node_lo) * 2, 0); }
    uint32_t stamp = 0;
    std::vector<Ask> asks;
    std::vector<uint32_t> first, second;                                // asks computed in the first / second launch
    std::vector<int8_t> verdict;                                         // per ask: -1 undecided, 0 no alignment, 1 alignment exists
    std::vector<uint64_t> rep_end;                                       // per ask computed first: reference position where the alignment found ends
    for (int cur_level = int(level.size()) - 1; cur_level >= 1; --cur_level) {
        g_prof.start(w);
        active.swap(level[size_t(cur_level)]);
        level[size_t(cur_level)].clear();
        if (active.empty()) continue;
        std::vector<uint32_t>& up = level[size_t(cur_level) - 1];
        size_t const NA = active.size();
        asks.resize(NA); verdict.assign(NA, -1); rep_end.resize(NA);
        ++stamp;
        for (size_t q = 0; q < NA; ++q) {
            uint32_t const wi = active[q];
            Walk& wk = walks[wi];
            fxg_anchor const& A = J->anchors_p[wk.anchor];
            Span const sp = span_of(wk, false);
            Ask& a = asks[q];
            a.m = uint32_t(wk.node->query_index_to - wk.node->query_index_from + 1);
            a.k = uint32_t(wk.node->num_errors);
            a.qbase = (wk.orient ? J->pool_len : 0) + J->reads_p[wk.read].query_offset + wk.node->query_index_from;
            a.ws = c->refs.base[A.reference_id] + sp.offset; a.len = uint32_t(sp.length); a.wi = wi;
            // statistics, verification.cpp:238-242 (kept per walk: with the interval optimisation the walk may turn out not to count)
            wk.n_inner++; wk.sum_inner += sp.length; wk.cells_inner += uint64_t(a.m) * sp.length;
            a.feasible = a.m != 0 && int64_t(a.m) - int64_t(a.len) <= int64_t(a.k);          // else more insertions needed than errors allowed
            if (!a.feasible) { verdict[q] = 0; continue; }
            if (infer) {
                a.key = uint32_t(uint64_t(wk.node - J->nodes_p) - node_lo) * 2 + wk.orient;   // the node identifies the read as well
                if (rep_stamp[a.key] != stamp || a.ws > asks[rep_of[a.key]].ws) { rep_stamp[a.key] = stamp; rep_of[a.key] = uint32_t(q); }
            }
        }
        first.clear(); passes.clear();
        for (size_t q = 0; q < NA; ++q)
            if (asks[q].feasible && (!infer || rep_of[asks[q].key] == q)) { first.push_back(uint32_t(q)); passes.push_back(pass_of(asks[q])); }
        g_prof.lap(w, 2);
        if (g_prof.on && w.id == 0 && std::getenv("FXG_TRACE_WAVES"))
            fprintf(stderr, "[fxg] level %d: %zu walks, %zu computed first\n", cur_level, active.size(), passes.size());
        const DpResult* res = nullptr;
        out.rc = run_passes(c, w, pool, passes, nullptr, nullptr, &res);
        if (out.rc != FXG_OK) return;
        w.ctr.waves++;
        g_prof.start(w);
        for (size_t f = 0; f < first.size(); ++f) {
            uint32_t const q = first[f];
            verdict[q] = res[f].score <= int32_t(asks[q].k) ? 1 : 0;
            rep_end[q] = asks[q].ws + res[f].end_col;
        }
        // what follows from the walk that went first for its node
        second.clear(); passes.clear();
        if (infer) {
            for (size_t q = 0; q < NA; ++q) {
                if (verdict[q] != -1) continue;
                Ask const& a = asks[q];
                uint32_t const rep = rep_of[a.key];
                if (a.ws == asks[rep].ws && a.len == asks[rep].len) verdict[q] = verdict[rep];                              // the same window
                else if (verdict[rep] == 1 && a.ws + a.len >= rep_end[rep]) { verdict[q] = 1; w.ctr.inferred_inner++; }      // (ws <= the first one's by choice)
                else { second.push_back(uint32_t(q)); passes.push_back(pass_of(a)); }
            }
        }
        if (g_prof.on && w.id == 0 && std::getenv("FXG_TRACE_WAVES")) {
            size_t yes = 0, same_no = 0;
            for (size_t f = 0; f < first.size(); ++f) yes += verdict[first[f]] == 1;
            for (uint32_t q : second) same_no += verdict[rep_of[asks[q].key]] == 0;
            fprintf(stderr, "[fxg] level %d: %zu of %zu elected found an alignment; %zu computed second, %zu of them because the elected walk found none\n",
                    cur_level, yes, first.size(), second.size(), same_no);
        }
        if (!passes.empty()) {
            out.rc = run_passes(c, w, pool, passes, nullptr, nullptr, &res);
            if (out.rc != FXG_OK) return;
            for (size_t f = 0; f < second.size(); ++f) verdict[second[f]] = res[f].score <= int32_t(asks[second[f]].k) ? 1 : 0;
        }
        for (size_t q = 0; q < NA; ++q) {
            Walk& wk = walks[asks[q].wi];
            if (verdict[q] == 1) {
                fxg_read const& R = J->reads_p[wk.read];
                wk.node = &J->nodes_p[R.node_offset + wk.node->parent_id];      // pex_tree::get_parent_of_child, pex.cpp:70-76
                up.push_back(asks[q].wi);                                        // joins the walks that start one level up
            } else {
                wk.state = W_DONE;
            }
        }
        active.clear();
        g_prof.lap(w, 9);
    }

    // ---------------- 2. which walks count, and which of them verify their root ----------------
    g_prof.start(w);
    std::vector<uint32_t> roots;                         // walks standing at the root that count, in walk order
    fxg_stats& st0 = out.stats[0];
    if (on_device) {
        roots.swap(level[0]);                            // decided on the device (decide_kernel), statistics included
    } else if (!ivopt) {
        roots.swap(level[0]);
        std::sort(roots.begin(), roots.end());
        for (Walk const& wk : walks) { st0.n_aligned_inner += wk.n_inner; st0.sum_aligned_inner += wk.sum_inner; st0.cells_inner += wk.cells_inner; }
    } else {
        std::vector<uint8_t> at_root(n_walks, 0);
        for (uint32_t wi : level[0]) at_root[wi] = 1;
        std::vector<uint32_t> inserted;
        for (Group const& G : groups) {
            inserted.clear();
            const uint32_t* mem = group_members.data() + G.first;
            for (uint32_t q = 0; q < G.count; ++q) {
                uint32_t const wi = mem[q];
                Walk& wk = walks[wi];
                bool avoided = false;
                // verified_intervals::contains over the windows inserted by earlier anchors (intervals.cpp:94-127)
                for (uint32_t ins : inserted)
                    if (walks[ins].r_start <= wk.t_start && walks[ins].r_end >= wk.t_end) { avoided = true; break; }
                if (avoided) {                               // root_was_already_verified, verification.cpp:119-136
                    st0.n_avoided_root++; st0.sum_avoided_root += wk.root_span.length;
                    wk.state = W_DONE;
                    continue;
                }
                st0.n_aligned_inner += wk.n_inner; st0.sum_aligned_inner += wk.sum_inner; st0.cells_inner += wk.cells_inner;
                if (at_root[wi]) { inserted.push_back(wi); roots.push_back(wi); }      // verified_intervals.insert, verification.cpp:106-109 / :40-41
            }
        }
        std::sort(roots.begin(), roots.end());
    }
    if (!on_device) {
        // what the root level needs of a walk (the device-side walks come with it)
        for (uint32_t wi : roots) {
            Walk& wk = walks[wi];
            (void)span_of(wk, true);
            wk.ref_id = uint32_t(J->anchors_p[wk.anchor].reference_id); wk.member = 0;
            wk.rm = uint32_t(wk.node->query_index_to - wk.node->query_index_from + 1); wk.rk = uint32_t(wk.node->num_errors);
            wk.rqbase = (wk.orient ? J->pool_len : 0) + J->reads_p[wk.read].query_offset + wk.node->query_index_from;
        }
    }
    g_prof.lap(w, 1);

    // ---------------- 3. root level ----------------
    g_prof.start(w);
    passes.clear(); pass_walk.clear();
    std::vector<uint32_t> root_k;
    passes.reserve(roots.size()); pass_walk.reserve(roots.size()); root_k.reserve(roots.size());
    bool const want_cigar = !B.cfg.without_cigar;
    for (uint32_t wi : roots) {
        Walk& wk = walks[wi];
        Span const& sp = wk.root_span;
        fxg_stats& S = out.stats[wk.member];
        S.n_aligned_root++; S.sum_aligned_root += sp.length; S.cells_root += uint64_t(wk.rm) * sp.length;
        Pass p;
        if (score_pass_for(c->refs.base[wk.ref_id] + sp.offset, wk.rqbase, uint32_t(sp.length), wk.rm, wk.rk, want_cigar ? 0u : kFlagReverse, p)) {
            passes.push_back(p); pass_walk.push_back(wi); root_k.push_back(wk.rk);
        }
        wk.state = W_DONE;
    }
    g_prof.lap(w, 2);
    if (g_prof.on && w.id == 0 && std::getenv("FXG_TRACE_WAVES")) fprintf(stderr, "[fxg] root level: %zu walks, %zu passes\n", roots.size(), passes.size());
    if (!passes.empty()) {
        if (want_cigar) {
            // score pass with checkpoints, then the traceback of the accepted ones
            std::vector<RootOut> root_outs;
            out.rc = run_root_passes(c, w, pool, passes, root_k, P.trace_budget, root_outs);
            if (out.rc != FXG_OK) return;
            for (size_t q = 0; q < passes.size(); ++q) {
                if (root_outs[q].score > int32_t(root_k[q])) continue;
                Walk& wk = walks[pass_walk[q]];
                wk.hit = true; wk.num_errors = uint32_t(root_outs[q].score);
                wk.start_in_reference = wk.root_span.offset + root_outs[q].begin_col;                 // alignment.cpp:175
                wk.cigar_offset = root_outs[q].cigar_offset; wk.cigar_len = root_outs[q].cigar_len;    // relative to this part's region for now
            }
        } else {
            const DpResult* res = nullptr;
            out.rc = run_passes(c, w, pool, passes, nullptr, nullptr, &res);
            if (out.rc != FXG_OK) return;
            for (size_t q = 0; q < passes.size(); ++q) {
                if (res[q].score > int32_t(root_k[q])) continue;
                Walk& wk = walks[pass_walk[q]];
                wk.hit = true; wk.num_errors = uint32_t(res[q].score);
                wk.start_in_reference = wk.root_span.offset + (wk.root_span.length - res[q].end_col);   // alignment.cpp:135-139
            }
        }
        w.ctr.waves++;
    }
}

// the part's cigars go straight from the device into its region of the job's pool; then the part's alignments
void verify_part_finish(fxg_ctx* c, Worker& w, uint32_t* host_cigars, uint64_t region_base, PartState& P) {
    (void)c;
    PartOut& out = P.out;
    g_prof.start(w);
    out.rc = fetch_cigars(w, host_cigars);
    g_prof.lap(w, 15);
    if (out.rc != FXG_OK) return;
    // ---- emit in anchor order (= insertion order of the reference's single-thread run) ----
    g_prof.start(w);
    for (Walk const& wk : P.walks) {                       // (host-driven levels; the device path has filled P.hits itself)
        if (!wk.hit) continue;
        fxg_alignment a{};
        a.start_in_reference = wk.start_in_reference; a.cigar_offset = wk.cigar_offset; a.cigar_len = wk.cigar_len;
        a.num_errors = wk.num_errors; a.read_index = wk.read; a.reference_id = wk.ref_id;
        a.orientation = wk.orient;
        P.hits.push_back(a);
    }
    for (fxg_alignment& a : P.hits) if (a.cigar_len) a.cigar_offset += region_base;
    out.alignments.swap(P.hits);
    g_prof.lap(w, 13);
    if (g_prof.on) fprintf(stderr, "[fxg] worker %d: %zu walks, %.3f ms (%.3f ms of CPU), %llu waves\n", w.id, P.walks.size(),
                           std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - P.t0).count(), thread_cpu_ms() - P.cpu0,
                           (unsigned long long)w.ctr.waves);
}

// Meeting point of the parts between their score and traceback phases: the last part to arrive sizes the job's
// page-locked cigar pool and hands every part its region.
struct TracePlan {
    std::mutex mu; std::condition_variable cv;
    size_t arrived = 0, n_parts = 0;
    std::vector<uint64_t> caps, bases;
    PinnedBuf* pool = nullptr; size_t* pool_len = nullptr;
    fxg_ctx* ctx = nullptr;
    double scale = 1.0;
    bool failed = false; std::string err;
    void arrive_and_wait(size_t part, uint64_t cap) {
        std::unique_lock<std::mutex> lock(mu);
        caps[part] = cap;
        if (++arrived == n_parts) {
            uint64_t total = 0;
            for (size_t p = 0; p < n_parts; ++p) { bases[p] = total; total += caps[p]; }
            size_t const need = std::max<uint64_t>(total, 1) * 4;
            if (pool->cap < need && ctx) {               // a pool of the right size from the context's spares, if there is one
                std::lock_guard<std::mutex> ctx_lock(ctx->mu);
                PinnedBuf fit = take_pinned_fit(ctx, need);
                if (fit.p) { give_pinned(ctx, *pool); *pool = fit; }
            }
            size_t const cap_before = pool->cap;
            cudaError_t const e = pool->ensure_scaled(need, scale);
            if (e != cudaSuccess) { failed = true; err = std::string("cigar pool allocation: ") + cudaGetErrorString(e); }
            else if (pool->cap != cap_before && scale > 1.0 && ctx) {
                // A pool for merged batches had to be made: as many of them are in use at a time as batches run or wait for
                // their members to pick up their results.  Page-locking takes tens of milliseconds, so the others are made
                // now, in one go (the first merged batches of a context pay; no batch after them does).
                size_t have = 0;
                { std::lock_guard<std::mutex> ctx_lock(ctx->mu); for (PinnedBuf const& b : ctx->spare_pinned) have += b.cap >= pool->cap; }
                size_t const want = size_t(2 * ctx->n_groups);
                for (size_t i = have + 1; i < want && pool->cap <= (size_t(64) << 20); ++i) {
                    PinnedBuf extra; extra.tag = pool->tag;
                    if (extra.exactly(pool->cap) != cudaSuccess) { (void)cudaGetLastError(); break; }
                    std::lock_guard<std::mutex> ctx_lock(ctx->mu);
                    give_pinned(ctx, extra);
                }
            }
            *pool_len = size_t(total);
            cv.notify_all();
        } else {
            cv.wait(lock, [&] { return arrived == n_parts; });
        }
    }
};

// Host workers per group.  A worker mostly waits for its own launches (polling, and yielding the core between polls),
// so two workers per core across the groups of all ranks on this host (torchrun exports LOCAL_WORLD_SIZE) is what
// measured best: 8 groups x 4 workers on the 16 cores of a one-GPU box.  FXG_WORKERS overrides.
int default_workers(int n_groups) {
    if (const char* e = std::getenv("FXG_WORKERS")) { int v = std::atoi(e); if (v >= 1 && v <= 64) return v; }
    unsigned const hc = std::max(1u, std::thread::hardware_concurrency());
    int const ranks = env_int("LOCAL_WORLD_SIZE", 1, 1, 64);
    return int(std::max(1u, std::min(4u, 2 * hc / unsigned(n_groups * ranks))));
}

}  // namespace

// ================================================================================================ C ABI

// Each worker drives its own streams (32 workers and more per context).  With the default of 8 hardware work queues
// the streams share queues and launches of different batches wait for each other without reason (measured on
// config 2: 6.2 -> 5.6 ms per batch with 32 queues).  The variable is read when the CUDA context is created, so it is
// set when the library is loaded, and only if the host application has not chosen a value itself.
__attribute__((constructor)) static void fxg_on_load() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }

extern "C" {

const char* fxg_version(void) { return "floxer_b200 0.2 (sm_100a)"; }

int fxg_create(int device, fxg_ctx** out) {
    if (!out) return FXG_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0 || device < 0 || device >= count) return FXG_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return FXG_ERR_CUDA;
    fxg_ctx* c = new (std::nothrow) fxg_ctx();
    if (!c) return FXG_ERR_OUT_OF_MEMORY;
    c->device = device;
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return FXG_ERR_CUDA; }
    c->num_sms = prop.multiProcessorCount;
    c->smem_limit = prop.sharedMemPerBlockOptin;
    bool ok = cudaStreamCreateWithFlags(&c->stage_stream, cudaStreamNonBlocking) == cudaSuccess && set_all_smem_attrs(c->smem_limit) == cudaSuccess;
    c->root_chunks = env_int("FXG_ROOT_CHUNKS", 1, 1, 64);
    c->infer_inner = env_int("FXG_INFER_INNER", 1, 0, 1) != 0;
    c->force_wide = env_int("FXG_FORCE_WIDE", 0, 0, 1) != 0;
    c->device_roots = env_int("FXG_DEVICE_ROOTS", 1, 0, 1) != 0;
    c->share_root_passes = env_int("FXG_SHARE_ROOTS", 1, 0, 1) != 0;
    c->device_levels = env_int("FXG_DEVICE_LEVELS", 1, 0, 1) != 0;
    c->root_chunk_min = env_int("FXG_ROOT_CHUNK_MIN", 512, 1, 1 << 30);
    c->n_groups = env_int("FXG_GROUPS", 6, 1, fxg_ctx::kMaxGroups);
    c->merge_max_jobs = env_int("FXG_MERGE_JOBS", 16, 1, 4096);
    c->merge_wait_us = env_int("FXG_MERGE_WAIT_US", 300, 0, 1000000);
    c->merged_parts = env_int("FXG_MERGED_PARTS", 1, 1, 64);
    c->merge_max_walks = uint64_t(env_int("FXG_MERGE_WALKS", 1 << 20, 1, int(kMaxDeviceWalks - 1)));
    c->workers_busy = default_workers(c->n_groups);
    // a batch that runs alone is split over 8 workers; the lowest free group is taken, so that is always group 0 and only
    // it owns that many.  An explicit FXG_WORKERS is taken literally.
    int const nw_wide = c->workers_busy;
    for (int gi = 0; gi < c->n_groups; ++gi) {
        WorkerGroup& g = c->groups[gi];
        ok = ok && cudaEventCreate(&g.ev_run0) == cudaSuccess && cudaEventCreate(&g.ev_run1) == cudaSuccess &&
             cudaEventCreateWithFlags(&g.ev_merged, cudaEventDisableTiming) == cudaSuccess;
        int const nw = gi == 0 ? nw_wide : c->workers_busy;
        for (int i = 0; ok && i < nw; ++i) {
            std::unique_ptr<Worker> w(new (std::nothrow) Worker());
            if (!w) { ok = false; break; }
            w->id = i; w->group = &g;
            ok = cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreate(&w->ev0) == cudaSuccess && cudaEventCreate(&w->ev1) == cudaSuccess &&
                 cudaEventCreateWithFlags(&w->ev_fork, cudaEventDisableTiming) == cudaSuccess;
            ok = ok && cudaEventCreate(&w->ev_w0) == cudaSuccess && cudaEventCreate(&w->ev_b0) == cudaSuccess && cudaEventCreate(&w->ev_b1) == cudaSuccess &&
                 cudaEventCreateWithFlags(&w->ev_sleep, cudaEventBlockingSync | cudaEventDisableTiming) == cudaSuccess;
            w->spin_us = env_int("FXG_SPIN_US", 20, 0, 1000000);
            for (int q = 0; ok && q < Worker::kWalkSlots; ++q)
                ok = cudaStreamCreateWithFlags(&w->walk_stream[q], cudaStreamNonBlocking) == cudaSuccess &&
                     cudaEventCreateWithFlags(&w->ev_walk_done[q], cudaEventDisableTiming) == cudaSuccess &&
                     cudaEventCreate(&w->ev_w1[q]) == cudaSuccess;
            for (int q = 0; ok && q < Worker::kSide; ++q)
                ok = cudaStreamCreateWithFlags(&w->side[q], cudaStreamNonBlocking) == cudaSuccess &&
                     cudaEventCreateWithFlags(&w->ev_join[q], cudaEventDisableTiming) == cudaSuccess;
            g.workers.push_back(std::move(w));
        }
    }
    if (!ok) { fxg_destroy(c); return FXG_ERR_CUDA; }
    *out = c;
    return FXG_OK;
}

void fxg_destroy(fxg_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    c->refs.packed.release();
    c->d_tmp.release();
    for (Pool& p : c->spare_pools) p.release();
    for (PinnedBuf& b : c->spare_pinned) b.release();
    for (DevBuf& b : c->spare_dev) b.release();
    for (PinnedBuf& b : c->spare_staging) b.release();
    c->refs.d_base.release(); c->refs.d_len.release();
    for (WorkerGroup& g : c->groups) {
        for (auto& w : g.workers) w->release();
        if (g.ev_run0) cudaEventDestroy(g.ev_run0);
        if (g.ev_run1) cudaEventDestroy(g.ev_run1);
        if (g.ev_merged) cudaEventDestroy(g.ev_merged);
        g.merged.release();
    }
    if (c->stage_stream) cudaStreamDestroy(c->stage_stream);
    delete c;
}

const char* fxg_last_error(const fxg_ctx* c) { return c ? tls_last_error.c_str() : "no context"; }

int fxg_get_counters(const fxg_ctx* c, fxg_counters* out) {
    if (!c || !out) return FXG_ERR_INVALID_ARGUMENT;
    { std::lock_guard<std::mutex> lock(const_cast<fxg_ctx*>(c)->mu); *out = c->ctr; }
    out->alloc_ms = double(g_alloc_ns.load()) * 1e-6 - c->alloc_ms0; out->alloc_calls = g_alloc_calls.load() - c->alloc_calls0;
    return FXG_OK;
}
int fxg_reset_counters(fxg_ctx* c) {
    if (!c) return FXG_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(c->mu);
    c->ctr = fxg_counters{}; c->alloc_ms0 = double(g_alloc_ns.load()) * 1e-6; c->alloc_calls0 = g_alloc_calls.load();
    return FXG_OK;
}

int fxg_set_references(fxg_ctx* c, size_t n_refs, const uint8_t* const* ranks, const uint64_t* lens) {
    if (!c || (n_refs && (!ranks || !lens))) return FXG_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(c->mu);
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    // the store is read by every kernel of every run: it is replaced only while nothing runs or waits
    for (int i = 0; i < c->n_groups; ++i)
        if (c->groups[i].busy) return fail(c->err, FXG_ERR_STATE, "fxg_set_references while a run is in flight");
    if (!c->pending.empty()) return fail(c->err, FXG_ERR_STATE, "fxg_set_references while a run is in flight");
    if (c->seeders_reading) return fail(c->err, FXG_ERR_STATE, "fxg_set_references while a seeding call is in flight");
    // everything new is built beside the old store and takes its place only when every upload has succeeded
    std::vector<uint64_t> base(n_refs, 0), len(lens, lens + n_refs);
    uint64_t total = 0;
    for (size_t i = 0; i < n_refs; ++i) {
        int rc = check_ranks(c->err, ranks[i], lens[i], "reference");
        if (rc != FXG_OK) return rc;
        base[i] = total;
        total += (lens[i] + 31) / 32 * 32;
    }
    DevBuf packed, d_base, d_len;
    auto build = [&]() -> int {
        CUDA_TRY(c->err, packed.ensure(total / 2 + 64));
        CUDA_TRY(c->err, cudaMemsetAsync(packed.p, 0, total / 2 + 64, c->stage_stream));
        for (size_t i = 0; i < n_refs; ++i) {
            uint64_t const slice = uint64_t(256) << 20;        // upload in slices so that the temporary stays small
            for (uint64_t at = 0; at < lens[i]; at += slice) {
                uint64_t const n = std::min<uint64_t>(slice, lens[i] - at);
                int rc = upload_packed(c, ranks[i] + at, n, packed, (base[i] + at) / 8);
                if (rc != FXG_OK) return rc;
            }
        }
        CUDA_TRY(c->err, d_base.ensure(std::max<size_t>(n_refs, 1) * 8));
        CUDA_TRY(c->err, d_len.ensure(std::max<size_t>(n_refs, 1) * 8));
        if (n_refs) {
            CUDA_TRY(c->err, cudaMemcpyAsync(d_base.p, base.data(), n_refs * 8, cudaMemcpyHostToDevice, c->stage_stream));
            CUDA_TRY(c->err, cudaMemcpyAsync(d_len.p, len.data(), n_refs * 8, cudaMemcpyHostToDevice, c->stage_stream));
        }
        CUDA_TRY(c->err, cudaStreamSynchronize(c->stage_stream));
        return FXG_OK;
    };
    int const rc = build();
    c->d_tmp.release();
    if (rc != FXG_OK) { packed.release(); d_base.release(); d_len.release(); return rc; }      // the old store stays as it was
    RefStore& R = c->refs;
    R.packed.release(); R.d_base.release(); R.d_len.release();
    R.packed = packed; R.d_base = d_base; R.d_len = d_len;
    R.base.swap(base); R.len.swap(len); R.total = total; R.version++;
    c->have_refs = true;
    refresh_trace_budget(c);
    return FXG_OK;
}

// ------------------------------------------------------------------------------------------------ align batch

// The DP passes of a batch's tasks, in task order: by chunks of tasks on several threads, then the passes of every chunk
// move to their place.  Called with c->mu held (it reads the reference table).
void build_batch_passes(fxg_ctx* c, fxg_batch* b, uint64_t refs_version) {
    size_t const N = b->tasks.size();
    size_t const T = parallel_threads(N, size_t(1) << 16);
    std::vector<std::vector<Pass>> part_passes(T), part_roots(T);
    std::vector<std::vector<uint32_t>> part_owner(T), part_root_owner(T);
    std::vector<uint64_t> const& ref_bases = c->refs.base;
    parallel_chunks(T, N, [&](size_t th, size_t lo, size_t hi) {
        part_passes[th].reserve(hi - lo); part_owner[th].reserve(hi - lo);
        for (size_t i = lo; i < hi; ++i) {
            fxg_align_task const& t = b->tasks[i];
            if (t.query_len == 0) continue;                  // aligns with zero errors (fxg_align_batch_run)
            uint32_t const flags = (t.mode == FXG_MODE_NO_CIGAR ? kFlagReverse : 0u) | (t.ref_id == FXG_REF_INLINE ? kFlagInlineRef : 0u);
            uint64_t const ref_base = (t.ref_id == FXG_REF_INLINE ? 0 : ref_bases[t.ref_id]) + t.ref_offset;
            Pass p;
            if (!score_pass_for(ref_base, t.query_offset, t.ref_len, t.query_len, t.max_errors, flags, p)) continue;
            if (t.mode == FXG_MODE_CIGAR) { part_roots[th].push_back(p); part_root_owner[th].push_back(uint32_t(i)); }
            else { part_passes[th].push_back(p); part_owner[th].push_back(uint32_t(i)); }
        }
    });
    std::vector<size_t> at(T + 1, 0), root_at(T + 1, 0);
    for (size_t th = 0; th < T; ++th) { at[th + 1] = at[th] + part_passes[th].size(); root_at[th + 1] = root_at[th] + part_roots[th].size(); }
    b->passes.resize(at[T]); b->owner.resize(at[T]); b->root_passes.resize(root_at[T]); b->root_owner.resize(root_at[T]);
    parallel_chunks(T, T, [&](size_t, size_t lo, size_t hi) {
        for (size_t th = lo; th < hi; ++th) {
            std::copy(part_passes[th].begin(), part_passes[th].end(), b->passes.begin() + long(at[th]));
            std::copy(part_owner[th].begin(), part_owner[th].end(), b->owner.begin() + long(at[th]));
            std::copy(part_roots[th].begin(), part_roots[th].end(), b->root_passes.begin() + long(root_at[th]));
            std::copy(part_root_owner[th].begin(), part_root_owner[th].end(), b->root_owner.begin() + long(root_at[th]));
        }
    });
    b->root_k.resize(b->root_owner.size());
    for (size_t q = 0; q < b->root_owner.size(); ++q) b->root_k[q] = b->tasks[b->root_owner[q]].max_errors;
    b->passes_refs_version = refs_version;
}

int fxg_align_batch_stage(fxg_ctx* c, const fxg_align_task* tasks, size_t n_tasks, const uint8_t* query_pool, size_t query_pool_len,
                          const uint8_t* inline_ref_pool, size_t inline_ref_pool_len, fxg_batch** out) {
    if (!c || !out || (n_tasks && !tasks)) return FXG_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(c->mu);
    *out = nullptr;
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    for (size_t i = 0; i < n_tasks; ++i) {
        fxg_align_task const& t = tasks[i];
        if (t.mode > FXG_MODE_CIGAR) return fail(c->err, FXG_ERR_INVALID_ARGUMENT, "task %zu: invalid alignment mode %u", i, unsigned(t.mode));
        if (t.query_offset + t.query_len > query_pool_len) return fail(c->err, FXG_ERR_INVALID_ARGUMENT, "task %zu: query span outside the pool", i);
        if (t.ref_id == FXG_REF_INLINE) {
            if (t.ref_offset + t.ref_len > inline_ref_pool_len) return fail(c->err, FXG_ERR_INVALID_ARGUMENT, "task %zu: inline reference span outside the pool", i);
        } else {
            if (!c->have_refs || t.ref_id >= c->refs.len.size()) return fail(c->err, FXG_ERR_STATE, "task %zu: reference %u not resident", i, t.ref_id);
            if (t.ref_offset + t.ref_len > c->refs.len[t.ref_id]) return fail(c->err, FXG_ERR_INVALID_ARGUMENT, "task %zu: reference span outside reference %u", i, t.ref_id);
        }
    }
    int rc = check_ranks(c->err, query_pool, query_pool_len, "query pool");
    if (rc != FXG_OK) return rc;
    rc = check_ranks(c->err, inline_ref_pool, inline_ref_pool_len, "inline reference pool");
    if (rc != FXG_OK) return rc;
    fxg_batch* b = new (std::nothrow) fxg_batch();
    if (!b) return FXG_ERR_OUT_OF_MEMORY;
    b->tasks.assign(tasks, tasks + n_tasks);
    build_batch_passes(c, b, c->refs.version);
    b->pool = take_pool(c);
    b->cigars = take_pinned(c);
    rc = stage_pool(c, b->pool, query_pool, query_pool_len, nullptr, 0, c->err, c->ctr);
    if (rc == FXG_OK && inline_ref_pool_len) {
        b->pool.inline_len = inline_ref_pool_len;
        cudaError_t e = b->pool.inline_packed.ensure(inline_ref_pool_len / 2 + 64);
        if (e != cudaSuccess) rc = fail(c->err, FXG_ERR_CUDA, "inline pool allocation: %s", cudaGetErrorString(e));
        else {
            cudaMemsetAsync(b->pool.inline_packed.p, 0, inline_ref_pool_len / 2 + 64, c->stage_stream);
            rc = upload_packed(c, inline_ref_pool, inline_ref_pool_len, b->pool.inline_packed, 0);
        }
    }
    if (rc == FXG_OK && cudaStreamSynchronize(c->stage_stream) != cudaSuccess) rc = fail(c->err, FXG_ERR_CUDA, "staging failed");
    if (rc != FXG_OK) { give_pool(c, b->pool); give_pinned(c, b->cigars); delete b; return rc; }
    *out = b;
    return FXG_OK;
}

int fxg_align_batch_run(fxg_ctx* c, fxg_batch* b) {
    if (!c || !b) return FXG_ERR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lock(c->mu);
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    if (b->passes_refs_version != c->refs.version) build_batch_passes(c, b, c->refs.version);    // (the references were replaced since the batch was staged)
    WorkerGroup& grp = acquire_group(c, lock);
    lock.unlock();                                   // the group is this call's own from here on: other callers run beside it
    struct Release { fxg_ctx* c; WorkerGroup& g; ~Release() { std::lock_guard<std::mutex> l(c->mu); release_group(c, g); } } release{c, grp};
    Worker& w = *grp.workers[0];
    w.ctr = fxg_counters{};
    // one batch of independent alignments, one or two waits and nothing else for this thread to do meanwhile: poll longer
    // before sleeping (the event's wake-up latency is 10-20 % of such a call)
    struct Spin { Worker& w; int saved; ~Spin() { w.spin_us = saved; } } spin{w, w.spin_us};
    w.spin_us = std::max(w.spin_us, 1000);
    int rc;
    {
        RunTimer run_timer(grp, w.ctr);
        auto t_mark = std::chrono::steady_clock::now();
        auto mark = [&](const char* what) {              // (FXG_PROFILE) host phases of the call
            if (!g_prof.on) return;
            auto const now = std::chrono::steady_clock::now();
            fprintf(stderr, "[fxg] align_batch_run: %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_mark).count());
            t_mark = now;
        };
        size_t const N = b->tasks.size();
        b->results.resize(N);
        b->cigars_len = 0;
        std::vector<Pass> const& passes = b->passes; std::vector<Pass> const& root_passes = b->root_passes;
        std::vector<uint32_t> const& owner = b->owner; std::vector<uint32_t> const& root_owner = b->root_owner; std::vector<uint32_t> const& root_k = b->root_k;
        size_t const T = parallel_threads(N, size_t(1) << 16);
        parallel_chunks(T, N, [&](size_t, size_t lo, size_t hi) {
            for (size_t i = lo; i < hi; ++i) {
                fxg_align_task const& t = b->tasks[i];
                fxg_align_result r{};
                r.orientation = t.orientation;
                if (t.query_len == 0) {
                    // empty query: aligns with zero errors; the rightmost minimum of an all-zero last row is column n
                    r.exists = 1;
                    if (t.mode == FXG_MODE_CIGAR) r.start_in_reference = t.reference_span_offset + t.ref_len;
                    else if (t.mode == FXG_MODE_NO_CIGAR) r.start_in_reference = t.reference_span_offset;
                }
                b->results[i] = r;
            }
        });
        mark("results reset");
        const DpResult* res = nullptr;
        rc = run_passes(c, w, b->pool, passes, nullptr, nullptr, &res);
        mark("score passes");
        if (rc == FXG_OK) {
            parallel_chunks(T, passes.size(), [&](size_t, size_t lo, size_t hi) {
                for (size_t q = lo; q < hi; ++q) {
                    fxg_align_task const& t = b->tasks[owner[q]];
                    fxg_align_result& r = b->results[owner[q]];
                    if (res[q].score > int32_t(t.max_errors)) continue;
                    r.exists = 1;
                    if (t.mode == FXG_MODE_EXISTS) continue;
                    r.num_errors = uint32_t(res[q].score);
                    r.start_in_reference = t.reference_span_offset + (t.ref_len - res[q].end_col);   // alignment.cpp:135-139
                }
            });
            mark("results of the score passes");
            w.cig_used = 0;
            std::vector<RootOut> outs;
            rc = run_root_passes(c, w, b->pool, root_passes, root_k, trace_budget_bytes(c, 1), outs);
            mark("passes with tracebacks");
            if (rc == FXG_OK) {
                cudaError_t const e = b->cigars.ensure(std::max<uint64_t>(w.cig_used, 1) * 4);
                if (e != cudaSuccess) rc = fail(w.err, FXG_ERR_CUDA, "cigar pool allocation: %s", cudaGetErrorString(e));
            }
            if (rc == FXG_OK) rc = fetch_cigars(w, b->cigars.as<uint32_t>());
            if (rc == FXG_OK) {
                b->cigars_len = size_t(w.cig_used);
                for (size_t q = 0; q < root_passes.size(); ++q) {
                    if (outs[q].score > int32_t(root_k[q])) continue;
                    fxg_align_task const& t = b->tasks[root_owner[q]];
                    fxg_align_result& r = b->results[root_owner[q]];
                    r.exists = 1; r.num_errors = uint32_t(outs[q].score);
                    r.start_in_reference = t.reference_span_offset + outs[q].begin_col;   // alignment.cpp:175
                    r.cigar_offset = outs[q].cigar_offset; r.cigar_len = outs[q].cigar_len;
                }
            }
            mark("cigars and their results");
        }
        if (g_prof.on) g_prof.report();
    }
    { std::lock_guard<std::mutex> l(c->mu); add_counters(c->ctr, w.ctr); if (rc != FXG_OK) c->err = w.err; }
    if (rc != FXG_OK) { tls_last_error = w.err; return rc; }
    b->ran = true;
    return FXG_OK;
}

int fxg_align_batch_fetch(fxg_ctx* c, fxg_batch* b, fxg_align_result* results, uint32_t* cigar_pool, size_t cigar_capacity, size_t* cigar_used) {
    if (!c) return FXG_ERR_INVALID_ARGUMENT;
    if (!b || !b->ran || (b->tasks.size() && !results)) return fail(c->err, FXG_ERR_STATE, "batch has not been run");
    if (cigar_used) *cigar_used = b->cigars_len;
    if (b->cigars_len > cigar_capacity) return fail(c->err, FXG_ERR_OVERFLOW, "cigar pool needs %zu entries, capacity is %zu", b->cigars_len, cigar_capacity);
    if (!b->results.empty()) std::memcpy(results, b->results.data(), b->results.size() * sizeof(fxg_align_result));
    if (b->cigars_len) std::memcpy(cigar_pool, b->cigars.p, b->cigars_len * 4);
    return FXG_OK;
}

void fxg_batch_free(fxg_ctx* c, fxg_batch* b) {
    if (!b) return;
    if (c) { std::lock_guard<std::mutex> lock(c->mu); cudaSetDevice(c->device); give_pool(c, b->pool); give_pinned(c, b->cigars); }
    else b->cigars.release();
    delete b;
}

int fxg_align_batch(fxg_ctx* c, const fxg_align_task* tasks, size_t n_tasks, const uint8_t* query_pool, size_t query_pool_len,
                    const uint8_t* inline_ref_pool, size_t inline_ref_pool_len, fxg_align_result* results,
                    uint32_t* cigar_pool, size_t cigar_capacity, size_t* cigar_used) {
    fxg_batch* b = nullptr;
    int rc = fxg_align_batch_stage(c, tasks, n_tasks, query_pool, query_pool_len, inline_ref_pool, inline_ref_pool_len, &b);
    if (rc != FXG_OK) return rc;
    rc = fxg_align_batch_run(c, b);
    if (rc == FXG_OK) rc = fxg_align_batch_fetch(c, b, results, cigar_pool, cigar_capacity, cigar_used);
    fxg_batch_free(c, b);
    return rc;
}

// ------------------------------------------------------------------------------------------------ verify

namespace {

// reads -> first walk (= anchor) of every read in job order
void index_walks(fxg_job* j) {
    j->read_walk_begin.resize(j->n_reads + 1);
    uint32_t n_walks_total = 0;
    for (size_t ri = 0; ri < j->n_reads; ++ri) {
        j->read_walk_begin[ri] = n_walks_total;
        n_walks_total += j->reads_p[ri].num_anchors_forward + j->reads_p[ri].num_anchors_reverse;
    }
    j->read_walk_begin[j->n_reads] = n_walks_total;
}

// One batch on one worker group, without the context lock (errors and accounting go to the caller's objects).
int run_batch(fxg_ctx* c, WorkerGroup& grp, Batch& B, std::string& err, fxg_counters& ctr) {
    B.alignments.clear(); B.cigars_len = 0; B.stats.assign(B.members.size(), fxg_stats{});
    size_t const n_reads = B.n_reads;
    if (n_reads == 0) return FXG_OK;

    // ---- split the reads into contiguous parts with similar numbers of anchors, one part per worker ----
    std::vector<uint32_t> const& rwb = B.read_walk_begin;
    // (a batch merged from several callers' jobs runs as few parts as possible: its point is launches that fill the machine)
    size_t const max_parts = B.members.size() > 1 ? std::min<size_t>(grp.use_workers, size_t(c->merged_parts)) : grp.use_workers;
    // (the host's share of a batch is small since the walks and the root level run on the device: parts are worth their split
    //  launches only where the phases of one part can hide behind another's -- half a million anchors each at least)
    size_t const n_parts = std::min<size_t>(max_parts, std::max<size_t>(1, std::min<size_t>(n_reads, size_t(rwb[n_reads]) / (B.device ? (size_t(1) << 19) : size_t(4096)) + 1)));
    std::vector<uint32_t> cut(n_parts + 1, 0);
    for (size_t p = 1; p < n_parts; ++p) {
        uint64_t const target = uint64_t(rwb[n_reads]) * p / n_parts;
        auto it = std::lower_bound(rwb.begin(), rwb.begin() + long(n_reads), uint32_t(target));
        cut[p] = std::max(cut[p - 1], uint32_t(it - rwb.begin()));
    }
    cut[n_parts] = uint32_t(n_reads);
    std::vector<PartState> parts(n_parts);
    TracePlan plan;
    plan.n_parts = n_parts; plan.caps.assign(n_parts, 0); plan.bases.assign(n_parts, 0);
    plan.pool = B.cigars; plan.pool_len = &B.cigars_len; plan.ctx = c;
    // (the pool of a batch of several jobs goes back to the context and serves the next such batch, whatever its size; the
    //  pool of a job that ran alone stays with the job, which needs the same amount every time)
    plan.scale = n_parts == 1 && B.members.size() > 1 ? std::max(1.0, double(c->merge_max_walks) / double(std::max<uint32_t>(rwb[n_reads], 1))) : 1.0;
    auto const vt0 = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - vt0).count(); };
    uint64_t const budget = trace_budget_bytes(c, n_parts);
    for (size_t p = 0; p < n_parts; ++p) grp.workers[p]->ctr = fxg_counters{};
    auto run_part = [&](size_t p) {
        Worker& w = *grp.workers[p];
        PartState& P = parts[p];
        P.trace_budget = budget; P.n_parts = n_parts;
        verify_part_score(c, w, B, cut[p], cut[p + 1], P);
        g_prof.start(w);
        plan.arrive_and_wait(p, P.out.rc == FXG_OK ? w.cig_used : 0);        // every part arrives, also a failed one
        g_prof.lap(w, 14);
        if (P.out.rc != FXG_OK) return;
        if (plan.failed) { w.err = plan.err; P.out.rc = FXG_ERR_CUDA; return; }
        verify_part_finish(c, w, B.cigars->as<uint32_t>() + plan.bases[p], plan.bases[p], P);
    };
    {
        RunTimer run_timer(grp, ctr);
        std::vector<std::thread> threads;
        for (size_t p = 1; p < n_parts; ++p) threads.emplace_back(run_part, p);
        run_part(0);
        for (auto& t : threads) t.join();
    }
    double const t_join = since();
    g_prof.report();
    for (size_t p = 0; p < n_parts; ++p) {
        add_counters(ctr, grp.workers[p]->ctr);
        if (parts[p].out.rc != FXG_OK) { err = grp.workers[p]->err; return parts[p].out.rc; }
    }
    {
        size_t n_al = 0;
        for (size_t p = 0; p < n_parts; ++p) n_al += parts[p].out.alignments.size();
        B.alignments.reserve(n_al);
    }
    for (size_t p = 0; p < n_parts; ++p) {
        B.alignments.insert(B.alignments.end(), parts[p].out.alignments.begin(), parts[p].out.alignments.end());
        for (size_t mi = 0; mi < B.members.size(); ++mi) {
            uint64_t* d = reinterpret_cast<uint64_t*>(&B.stats[mi]); const uint64_t* sp = reinterpret_cast<const uint64_t*>(&parts[p].out.stats[mi]);
            for (size_t f = 0; f < sizeof(fxg_stats) / sizeof(uint64_t); ++f) d[f] += sp[f];
        }
    }
    ctr.batches++; ctr.batch_jobs += B.members.size();
    static bool const trace_batches = std::getenv("FXG_TRACE_BATCHES") != nullptr;
    if (trace_batches) {
        static auto const epoch = std::chrono::steady_clock::now();
        fprintf(stderr, "[fxg] batch at %.3f ms: %zu jobs, %u walks, %zu parts%s, %.3f ms (alloc so far %.1f ms in %llu calls); part 0: enqueued %.2f levels %.2f units %.2f scores %.2f records %.2f\n",
                std::chrono::duration<double, std::milli>(vt0 - epoch).count(), B.members.size(), rwb[n_reads], n_parts, B.device ? "" : " (levels driven from the host)", since(),
                double(g_alloc_ns.load()) * 1e-6, (unsigned long long)g_alloc_calls.load(),
                parts[0].t_mark[0], parts[0].t_mark[1], parts[0].t_mark[2], parts[0].t_mark[3], parts[0].t_mark[4]);
    }
    if (g_prof.on) fprintf(stderr, "[fxg] run_batch: %zu jobs, %zu reads, %u walks, %zu parts; parts done %.3f ms, merged %.3f ms\n", B.members.size(), n_reads,
                           rwb[n_reads], n_parts, t_join, since());
    return FXG_OK;
}

// The Peq planes of the members side by side in the group's merged pool: member j's pool positions [0, 2 * pool_len_j)
// move to [shift_j, ...), shift_j a multiple of 32, so whole words are copied (device to device, six rows per member).
// Nothing else of a pool is read by the kernels of a verify run.  Words between the members are never looked at: a pass
// reads up to one block of rows before its piece and one word after it, and masks those bits (dp_task_group: `wild`).
int build_merged_pool(fxg_ctx* c, WorkerGroup& grp, Batch& B, std::string& err) {
    uint64_t at = 0;
    for (Member& M : B.members) { M.pool_shift = at; at += (2 * M.J->pool_len + 31) / 32 * 32; }
    Pool& P = grp.merged;
    P.len = at; P.inline_len = 0;
    P.plane_words = at / 32 + kPeqFrontPadWords + kPeqBackPadWords;
    {
        uint64_t walks = 0;
        for (Member const& M : B.members) walks += M.J->prep.n_walks;
        CUDA_TRY(err, P.peq.ensure_scaled(P.plane_words * kNumSymbols * 4, std::max(1.0, double(c->merge_max_walks) / double(std::max<uint64_t>(walks, 1)))));
    }
    cudaStream_t const st = grp.workers[0]->stream;
    (void)c;
    for (Member const& M : B.members) {
        fxg_job const* J = M.J;
        if (J->pool_ready) CUDA_TRY(err, cudaStreamWaitEvent(st, J->pool_ready, 0));
        uint64_t const words = (2 * J->pool_len + 31) / 32;
        if (!words) continue;
        CUDA_TRY(err, cudaMemcpy2DAsync(P.peq.as<uint32_t>() + kPeqFrontPadWords + M.pool_shift / 32, P.plane_words * 4,
                                        J->pool.peq.as<uint32_t>() + kPeqFrontPadWords, J->pool.plane_words * 4, words * 4, kNumSymbols,
                                        cudaMemcpyDeviceToDevice, st));
    }
    CUDA_TRY(err, cudaEventRecord(grp.ev_merged, st));
    B.merged_ready = grp.ev_merged;
    B.pool = &P;
    return FXG_OK;
}

// A call of fxg_verify_run / fxg_verify_reads waiting in the context's queue.
struct TicketResults {                   // what a merged batch leaves for its members
    std::vector<fxg_alignment> alignments;
    std::shared_ptr<PinnedBuf> cigars;
};
}  // namespace
namespace {
struct Ticket {
    fxg_job* J = nullptr;
    int state = 0;                       // 0 waiting, 1 taken by a batch, 2 done
    bool waited = false;                 // has spent its accumulation window (submit_and_wait)
    int rc = FXG_OK; std::string err;
    std::shared_ptr<TicketResults> shared; size_t al_begin = 0, al_end = 0; uint32_t read0 = 0; fxg_stats stats{};
};

bool same_config(fxg_verify_config const& a, fxg_verify_config const& b) {
    return a.extra_verification_ratio == b.extra_verification_ratio && a.verification_kind == b.verification_kind &&
           a.interval_optimization == b.interval_optimization && a.without_cigar == b.without_cigar;
}

WorkerGroup* try_acquire_group(fxg_ctx* c) {
    int busy = 0;
    for (int i = 0; i < c->n_groups; ++i) busy += c->groups[i].busy;
    for (int i = 0; i < c->n_groups; ++i) if (!c->groups[i].busy) {
        WorkerGroup& g = c->groups[i];
        g.busy = true;
        g.use_workers = std::min(g.workers.size(), size_t(c->workers_busy));     // (the same split whatever else runs: a worker's buffers keep their sizes)
        (void)busy;
        return &g;
    }
    return nullptr;
}

// runs the jobs of `mine` as one batch (or, should that fail, one by one) and leaves every ticket its results
void run_tickets(fxg_ctx* c, WorkerGroup& grp, std::vector<Ticket*> const& mine, PinnedBuf& pinned, fxg_counters& ctr) {
    auto run_some = [&](size_t lo, size_t hi) -> int {
        Batch B;
        B.cfg = mine[lo]->J->cfg;
        B.device = true;
        uint32_t read0 = 0;
        B.read_walk_begin.clear();
        for (size_t i = lo; i < hi; ++i) {
            fxg_job* J = mine[i]->J;
            uint32_t const walk0 = B.read_walk_begin.empty() ? 0u : B.read_walk_begin.back();
            if (!B.read_walk_begin.empty()) B.read_walk_begin.pop_back();
            for (uint32_t x : J->read_walk_begin) B.read_walk_begin.push_back(walk0 + x);
            B.members.push_back(Member{J, read0, 0});
            B.device = B.device && J->prep.ok;
            read0 += uint32_t(J->n_reads);
        }
        B.n_reads = read0;
        B.cigars = &pinned;
        std::string err;
        int rc = FXG_OK;
        if (hi - lo == 1) {
            B.pool = &mine[lo]->J->pool; B.pool_len = mine[lo]->J->pool_len;
            if (!pinned.p) std::swap(pinned, mine[lo]->J->cigars);     // a job that runs alone writes into the pool of its last run
        }
        else rc = build_merged_pool(c, grp, B, err);
        if (rc == FXG_OK) rc = run_batch(c, grp, B, err, ctr);
        if (rc != FXG_OK) {
            cudaDeviceSynchronize();                     // nothing of the failed batch may still be running when its buffers are reused
            for (size_t i = lo; i < hi; ++i) { mine[i]->rc = rc; mine[i]->err = err; }
            return rc;
        }
        if (hi - lo == 1) {
            fxg_job* J = mine[lo]->J;
            J->alignments = std::move(B.alignments);
            std::swap(J->cigars, pinned);                // (the job's previous pool goes back to the context with `pinned`)
            J->cigars_len = B.cigars_len; J->stats = B.stats[0];
            J->use_copy = false;
            mine[lo]->rc = FXG_OK;
            return FXG_OK;
        }
        auto shared = std::make_shared<TicketResults>();
        shared->alignments = std::move(B.alignments);
        shared->cigars = std::shared_ptr<PinnedBuf>(new PinnedBuf(pinned), [c](PinnedBuf* b) {
            { std::lock_guard<std::mutex> lock(c->mu); give_pinned(c, *b); }
            delete b;
        });
        pinned = PinnedBuf{};
        std::vector<fxg_alignment> const& al = shared->alignments;
        size_t at = 0;
        for (size_t i = lo; i < hi; ++i) {
            Ticket& T = *mine[i];
            Member const& M = B.members[i - lo];
            uint32_t const end_read = M.read0 + uint32_t(T.J->n_reads);
            T.al_begin = at;
            while (at < al.size() && al[at].read_index < end_read) ++at;
            T.al_end = at; T.read0 = M.read0; T.stats = B.stats[i - lo]; T.shared = shared; T.rc = FXG_OK;
        }
        return FXG_OK;
    };
    if (run_some(0, mine.size()) != FXG_OK && mine.size() > 1) {
        // one bad job must not fail its neighbours: each on its own
        for (size_t i = 0; i < mine.size(); ++i) {
            run_some(i, i + 1);
        }
    }
}

// a member of a merged batch takes its share of the results (on its own thread)
void take_member_results(fxg_job* J, Ticket& T) {
    std::vector<fxg_alignment> const& al = T.shared->alignments;
    J->alignments.assign(al.begin() + long(T.al_begin), al.begin() + long(T.al_end));
    uint64_t lo = UINT64_MAX, hi = 0;
    for (fxg_alignment const& a : J->alignments) if (a.cigar_len) { lo = std::min(lo, a.cigar_offset); hi = std::max(hi, a.cigar_offset + a.cigar_len); }
    if (lo == UINT64_MAX) lo = hi = 0;
    for (fxg_alignment& a : J->alignments) { a.read_index -= T.read0; if (a.cigar_len) a.cigar_offset -= lo; }
    J->cigars_copy.resize(size_t(hi - lo));
    if (hi > lo) std::memcpy(J->cigars_copy.data(), T.shared->cigars->as<uint32_t>() + lo, size_t(hi - lo) * 4);
    J->use_copy = true;
    J->cigars_len = size_t(hi - lo);
    J->stats = T.stats;
}

// Queues the job and returns when it has run.  A caller that finds a free worker group leads: it takes its own job and
// every compatible one that is waiting (same configuration, device records, within the merge limits) and runs them as
// ONE batch -- their tree levels share launches, and the host-side cost of a batch is paid once.  With as many callers
// as the application has threads and FXG_GROUPS batches in flight, the waiting jobs pile up into batches by themselves.
int submit_and_wait(fxg_ctx* c, fxg_job* J, std::unique_lock<std::mutex>& lock) {
    Ticket T; T.J = J;
    c->pending.push_back(&T);
    for (;;) {
        if (T.state == 2) break;
        if (T.state == 0 && !T.waited && c->merge_wait_us > 0 && c->merge_max_jobs > 1) {
            // while other batches run, the jobs of the callers they will release arrive within a few hundred microseconds of
            // each other: a short wait lets them travel together instead of one by one (a call that finds the context
            // idle starts at once)
            int busy = 0;
            for (int i = 0; i < c->n_groups; ++i) busy += c->groups[i].busy;
            T.waited = true;
            if (busy > 0) { c->cv.wait_for(lock, std::chrono::microseconds(c->merge_wait_us)); continue; }
        }
        WorkerGroup* g = T.state == 0 ? try_acquire_group(c) : nullptr;
        if (!g) { c->cv.wait(lock); continue; }
        std::vector<Ticket*> mine{&T};
        T.state = 1;
        c->pending.erase(std::find(c->pending.begin(), c->pending.end(), &T));
        if (J->prep.ok && c->merge_max_jobs > 1) {
            uint64_t walks = J->prep.n_walks, nodes = J->prep.n_nodes, reads = J->prep.n_reads;
            for (auto it = c->pending.begin(); it != c->pending.end() && mine.size() < size_t(c->merge_max_jobs);) {
                Ticket* t = *it;
                Prepared const& Q = t->J->prep;
                if (t->state == 0 && Q.ok && same_config(t->J->cfg, J->cfg) && walks + Q.n_walks <= c->merge_max_walks &&
                    nodes + Q.n_nodes < (1u << 30) && reads + Q.n_reads < (1u << 30)) {
                    walks += Q.n_walks; nodes += Q.n_nodes; reads += Q.n_reads;
                    t->state = 1; mine.push_back(t);
                    it = c->pending.erase(it);
                } else ++it;
            }
        }
        PinnedBuf pinned;                                // (picked from the context's spares when the batch knows how much it needs)
        pinned.tag = "page-locked cigar pool";
        lock.unlock();
        fxg_counters ctr{};
        run_tickets(c, *g, mine, pinned, ctr);
        lock.lock();
        add_counters(c->ctr, ctr);
        give_pinned(c, pinned);
        for (Ticket* t : mine) t->state = 2;
        g->busy = false;
        c->cv.notify_all();
    }
    if (T.rc != FXG_OK) { c->err = T.err; tls_last_error = T.err; return T.rc; }
    if (T.shared) {
        lock.unlock();
        take_member_results(J, T);
        T.shared.reset();                                // (the last member hands the batch's pool back to the context: not under the lock)
        lock.lock();
    }
    J->ran = true;
    return FXG_OK;
}

int check_verify_call(fxg_ctx* c, const fxg_verify_config* cfg) {
    if (!c->have_refs) return fail(c->err, FXG_ERR_STATE, "fxg_set_references must be called first");
    if (cfg->verification_kind != FXG_KIND_DIRECT_FULL && cfg->verification_kind != FXG_KIND_HIERARCHICAL)
        return fail(c->err, FXG_ERR_INVALID_ARGUMENT, "Internal bug in verification kind (should not happen)");   // verification.cpp:19
    return FXG_OK;
}

void release_job_buffers(fxg_ctx* c, fxg_job* j) {        // call with c->mu held
    give_pool(c, j->pool); give_pinned(c, j->cigars); give_staging(c, j->prep.staging);
    if (j->prep.dev.p && c->spare_dev.size() < size_t(2 * fxg_ctx::kMaxGroups + 64)) c->spare_dev.push_back(j->prep.dev); else j->prep.dev.release();
    j->prep.dev = DevBuf{};
}

// A job of fxg_verify_reads / fxg_seed_verify_reads: it reads the caller's arrays in place during the one call that runs it.
// Call with c->mu held.
fxg_job* new_borrowed_job(fxg_ctx* c, const fxg_verify_config* cfg, const fxg_read* reads, size_t n_reads, const fxg_pex_node* nodes,
                          size_t n_nodes, size_t pool_len) {
    fxg_job* j = new (std::nothrow) fxg_job();
    if (!j) return nullptr;
    j->cfg = *cfg;
    j->reads_p = reads; j->nodes_p = nodes;
    j->n_reads = n_reads; j->n_nodes = n_nodes;
    j->borrowed = true;
    j->pool_len = pool_len;
    j->pool = take_pool(c);
    j->prep.staging = take_staging(c);
    if (!c->spare_dev.empty()) { j->prep.dev = c->spare_dev.back(); c->spare_dev.pop_back(); }
    return j;
}

// The rest of a borrowed job's call once its pools and records are enqueued (rc: how that went): the queue, the check of
// the pools' ranks, and the job handed to the caller -- or released.
int run_borrowed_job(fxg_ctx* c, fxg_job* j, int rc, std::string& err, fxg_counters const& ctr, fxg_job** out) {
    std::unique_lock<std::mutex> lock(c->mu);
    add_counters(c->ctr, ctr);
    if (rc == FXG_OK) {
        rc = submit_and_wait(c, j, lock);
        if (rc != FXG_OK) err = c->err;
    }
    lock.unlock();
    if (rc == FXG_OK) {
        // (waits on an event of its own, asleep: cudaStreamSynchronize would spin -- one core per caller -- until every other
        //  caller's uploads on the staging stream are through as well)
        uint32_t bad_pageable = 0;
        // (into page-locked memory where the job has some: a copy into pageable memory blocks, spinning, as well)
        uint32_t* const bad_p = j->prep.staging.p && j->prep.used ? reinterpret_cast<uint32_t*>(j->prep.staging.as<uint8_t>() + j->prep.used) : &bad_pageable;
        if (cudaMemcpyAsync(bad_p, j->pool.bad_rank.p, 4, cudaMemcpyDeviceToHost, c->stage_stream) != cudaSuccess ||
            cudaEventRecord(j->pool_ready, c->stage_stream) != cudaSuccess ||
            cudaEventSynchronize(j->pool_ready) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "staging failed");
        uint32_t const bad = *bad_p;
        if (rc != FXG_OK) {}
        else if (bad) rc = fail(err, FXG_ERR_INVALID_ARGUMENT, "query pools contain a rank above %d (allowed 0..%d)", FXG_MAX_RANK, FXG_MAX_RANK);
    } else {
        cudaStreamSynchronize(c->stage_stream);          // nothing may still read the caller's arrays when the call returns
    }
    // the caller's arrays are not looked at after this point
    j->reads_p = nullptr; j->nodes_p = nullptr; j->anchors_p = nullptr;
    lock.lock();
    if (rc != FXG_OK) {
        c->err = err; tls_last_error = err;
        release_job_buffers(c, j);
        if (j->prep.ready) cudaEventDestroy(j->prep.ready);
        if (j->pool_ready) cudaEventDestroy(j->pool_ready);
        delete j;
        return rc;
    }
    *out = j;
    return FXG_OK;
}

}  // namespace

int fxg_verify_stage(fxg_ctx* c, const fxg_verify_config* cfg, const fxg_read* reads, size_t n_reads,
                     const uint8_t* fwd, const uint8_t* rc_pool, size_t pool_len,
                     const fxg_pex_node* nodes, size_t n_nodes, const fxg_anchor* anchors, size_t n_anchors, fxg_job** out) {
    if (!c || !cfg || !out) return FXG_ERR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lock(c->mu);
    *out = nullptr;
    int rc = check_verify_call(c, cfg);
    if (rc != FXG_OK) return rc;
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    fxg_job* j = new (std::nothrow) fxg_job();
    if (!j) return FXG_ERR_OUT_OF_MEMORY;
    j->pool = take_pool(c);
    j->prep.staging = take_staging(c);
    if (!c->spare_dev.empty()) { j->prep.dev = c->spare_dev.back(); c->spare_dev.pop_back(); }
    lock.unlock();                       // the rest touches only the job (and the staging stream, which is ordered)
    std::string err; fxg_counters ctr{};
    rc = validate_reads(c, err, reads, 0, n_reads, pool_len, nodes, n_nodes, anchors, n_anchors);
    if (rc == FXG_OK) rc = check_ranks(err, fwd, pool_len, "forward pool");
    if (rc == FXG_OK) rc = check_ranks(err, rc_pool, pool_len, "reverse-complement pool");
    if (rc == FXG_OK) {
        j->cfg = *cfg;
        j->reads.assign(reads, reads + n_reads);
        j->nodes.assign(nodes, nodes + n_nodes);
        j->anchors.assign(anchors, anchors + n_anchors);
        j->reads_p = j->reads.data(); j->nodes_p = j->nodes.data(); j->anchors_p = j->anchors.data();
        j->n_reads = n_reads; j->n_nodes = n_nodes; j->n_anchors = n_anchors;
        j->pool_len = pool_len;
        index_walks(j);
        rc = stage_pool(c, j->pool, fwd, pool_len, rc_pool, pool_len, err, ctr);
    }
    if (rc == FXG_OK) rc = prepare_job(c, j, err, ctr);
    if (rc == FXG_OK && cudaStreamSynchronize(c->stage_stream) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "staging failed");
    lock.lock();
    add_counters(c->ctr, ctr);
    if (rc != FXG_OK) { c->err = err; tls_last_error = err; release_job_buffers(c, j); if (j->prep.ready) cudaEventDestroy(j->prep.ready); delete j; return rc; }
    *out = j;
    return FXG_OK;
}

int fxg_verify_run(fxg_ctx* c, fxg_job* J) {
    if (!c || !J) return FXG_ERR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lock(c->mu);
    if (J->borrowed) return fail(c->err, FXG_ERR_STATE, "a job made by fxg_verify_reads cannot be run again (its inputs belonged to the caller)");
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    return submit_and_wait(c, J, lock);
}

size_t fxg_job_num_alignments(const fxg_job* j) { return j ? j->alignments.size() : 0; }
const fxg_alignment* fxg_job_alignments(const fxg_job* j) { return j ? j->alignments.data() : nullptr; }
size_t fxg_job_cigar_len(const fxg_job* j) { return j ? j->cigars_len : 0; }
const uint32_t* fxg_job_cigar_pool(const fxg_job* j) { return j ? (j->use_copy ? j->cigars_copy.data() : j->cigars.as<uint32_t>()) : nullptr; }
const fxg_stats* fxg_job_stats(const fxg_job* j) { return j ? &j->stats : nullptr; }

void fxg_job_free(fxg_ctx* c, fxg_job* j) {
    if (!j) return;
    if (c) { std::lock_guard<std::mutex> lock(c->mu); cudaSetDevice(c->device); release_job_buffers(c, j); }
    else { j->cigars.release(); j->prep.staging.release(); }
    if (j->prep.ready) cudaEventDestroy(j->prep.ready);
    if (j->pool_ready) cudaEventDestroy(j->pool_ready);
    delete j;
}

// stage + run in one call.  The caller's arrays are used in place (they only have to live until the call returns): the
// query pools and the job's records go up on the caller's thread, asynchronously, and the job joins the queue at once --
// the batch that takes it orders its streams behind those uploads.
int fxg_verify_reads(fxg_ctx* c, const fxg_verify_config* cfg, const fxg_read* reads, size_t n_reads,
                     const uint8_t* fwd, const uint8_t* rc_pool, size_t pool_len,
                     const fxg_pex_node* nodes, size_t n_nodes, const fxg_anchor* anchors, size_t n_anchors, fxg_job** out) {
    if (!c || !cfg || !out) return FXG_ERR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lock(c->mu);
    *out = nullptr;
    int rc = check_verify_call(c, cfg);
    if (rc != FXG_OK) return rc;
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    fxg_job* j = new_borrowed_job(c, cfg, reads, n_reads, nodes, n_nodes, pool_len);
    if (!j) return FXG_ERR_OUT_OF_MEMORY;
    j->anchors_p = anchors; j->n_anchors = n_anchors;
    lock.unlock();
    std::string err; fxg_counters ctr{};
    auto const tp0 = std::chrono::steady_clock::now();
    auto lap_ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count(); };
    rc = validate_reads(c, err, reads, 0, n_reads, pool_len, nodes, n_nodes, anchors, n_anchors);
    double const t_validate = lap_ms();
    if (rc == FXG_OK) {
        index_walks(j);
        // (ranks above 5 in the query pools are detected by the Peq builder on the device and reported after the run:
        //  such a byte simply matches nothing, so no kernel can be led astray by it in the meantime)
        rc = stage_pool(c, j->pool, fwd, pool_len, rc_pool, pool_len, err, ctr, true);
    }
    if (rc == FXG_OK && cudaEventCreateWithFlags(&j->pool_ready, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "cannot create an event");
    if (rc == FXG_OK && cudaEventRecord(j->pool_ready, c->stage_stream) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "staging failed");
    double const t_stage = lap_ms();
    if (rc == FXG_OK) rc = prepare_job(c, j, err, ctr);
    double const t_prepare = lap_ms();
    rc = run_borrowed_job(c, j, rc, err, ctr, out);
    if (g_prof.on) fprintf(stderr, "[fxg] verify_reads: validated %.3f, pools enqueued %.3f, records prepared %.3f, run done %.3f ms\n", t_validate, t_stage, t_prepare, lap_ms());
    return rc;
}

// ------------------------------------------------------------------------------------------------ engine shape

int fxg_engine_shape(uint32_t n, uint32_t m, uint32_t k, int with_traceback, uint32_t* words_per_lane, uint32_t* ring_lanes, uint32_t* blocks,
                     uint64_t* word_steps) {
    Pass p;
    if (!score_pass_for(0, 0, n, m, k, 0, p)) return FXG_ERR_INVALID_ARGUMENT;
    Config cf;
    if (!choose_config(p, size_t(227) * 1024, false, cf, with_traceback != 0)) return FXG_ERR_INVALID_ARGUMENT;
    if (words_per_lane) *words_per_lane = uint32_t(kWidths[cf.widx]);
    if (ring_lanes) *ring_lanes = cf.G;
    if (blocks) *blocks = cf.nb;
    if (word_steps) *word_steps = cf.word_steps;
    return FXG_OK;
}

// ------------------------------------------------------------------------------------------------ int32 peak

int fxg_measure_int32_peak(fxg_ctx* c, double* out) {
    if (!c || !out) return FXG_ERR_INVALID_ARGUMENT;
    std::unique_lock<std::mutex> lock(c->mu);
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    WorkerGroup& grp = acquire_group(c, lock);
    struct Release { fxg_ctx* c; WorkerGroup& g; ~Release() { release_group(c, g); } } release{c, grp};
    Worker& w = *grp.workers[0];
    CUDA_TRY(c->err, c->d_tmp.ensure(64));
    uint32_t const iters = 4096, threads = 256, grid = uint32_t(c->num_sms) * 8;
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(c->err, cudaEventRecord(w.ev0, w.stream));
        int32_peak_kernel<<<grid, threads, 0, w.stream>>>(c->d_tmp.as<uint32_t>(), iters, 12345u + rep);
        CUDA_TRY(c->err, cudaGetLastError());
        CUDA_TRY(c->err, cudaEventRecord(w.ev1, w.stream));
        CUDA_TRY(c->err, cudaStreamSynchronize(w.stream));
        float ms = 0;
        CUDA_TRY(c->err, cudaEventElapsedTime(&ms, w.ev0, w.ev1));
        double const instr = double(grid) * threads * double(iters) * 8.0 * 11.0;
        if (rep > 0) best = std::max(best, instr / (double(ms) * 1e-3));
    }
    *out = best;
    return FXG_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ device seeder

struct fxg_gpu_seeder {
    uint64_t ctx_serial = 0;
    uint64_t refs_version = 0;           // RefStore::version the index was built from
    uint32_t q = 0, n_refs = 0;
    DevBuf bucket, pos;                  // 4^q + 1 offsets, positions in the unpadded concatenation
    DevBuf ubase, pbase, len;            // per reference: unpadded start, start in the store, length
    uint64_t budget = 0;                 // FXG_SEED_CANDIDATES: q-gram occurrences per chunk
    void release() { bucket.release(); pos.release(); ubase.release(); pbase.release(); len.release(); }
};

namespace {

constexpr uint32_t kSeedChunkSeeds = 1u << 27;      // hit keys hold the seed of a chunk in 28 bits

// Keeps the context's packed store in place while a seeding call reads it without holding mu: fxg_set_references
// refuses to replace the store while the count is non-zero.
struct StoreReader {
    fxg_ctx* c;
    bool on = false;
    ~StoreReader() { if (on) { std::lock_guard<std::mutex> lock(c->mu); c->seeders_reading--; } }
};

// a call's own stream, device buffers and page-locked staging; the stream is drained before the buffers go back to the
// pool
struct CallScratch {
    explicit CallScratch(fxg_ctx* ctx) : c(ctx) {}
    fxg_ctx* c;
    cudaStream_t st = nullptr;
    DevBuf bufs[20];
    PinnedBuf host;
    ~CallScratch() {
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
        for (DevBuf& b : bufs) b.release();
        if (host.p) { std::lock_guard<std::mutex> lock(c->mu); give_staging(c, host); }
    }
};

int bits_for(uint64_t v) { int b = 1; while (b < 64 && (v >> b)) ++b; return b; }     // bits that hold 0..v

uint32_t seed_grid(uint64_t n, uint32_t threads = 256) { return uint32_t(std::max<uint64_t>(1, (n + threads - 1) / threads)); }

// the store's tables as the seeder's kernels read them
SeedRefs seed_refs(const fxg_gpu_seeder* S, const uint32_t* packed) {
    return SeedRefs{packed, S->ubase.as<uint64_t>(), S->pbase.as<uint64_t>(), S->len.as<uint64_t>(), S->n_refs};
}

// takes the store for a seeding call: the references must be those the seeder was made from (if it is given)
int take_store(fxg_ctx* c, const fxg_gpu_seeder* S, StoreReader& guard, const uint32_t*& packed, std::vector<uint64_t>* len,
               std::vector<uint64_t>* pbase, uint64_t* version, std::string& err) {
    std::lock_guard<std::mutex> lock(c->mu);
    if (!c->have_refs) return fail(err, FXG_ERR_STATE, "fxg_set_references must be called first");
    if (S && (S->ctx_serial != c->serial || S->refs_version != c->refs.version))
        return fail(err, FXG_ERR_STATE, "the references were replaced after the seeder was made (or it belongs to another context)");
    packed = c->refs.packed.as<uint32_t>();
    if (len) *len = c->refs.len;
    if (pbase) *pbase = c->refs.base;
    if (version) *version = c->refs.version;
    c->seeders_reading++;
    guard.on = true;
    return FXG_OK;
}

// The seeds of a batch, from the reads and their trees, on the host: a read or leaf fxg_seeder_search refuses fails the
// whole call before any device work.
struct SeedPlan {
    std::vector<uint32_t> seed_base, leaf_base;     // per read (+1): first seed, first leaf
    std::vector<uint64_t> leaf_info;                // per (read, leaf): seed_pack(query_offset + from, m, e)
    uint32_t n_seeds = 0;
};

int plan_seeds(const fxg_gpu_seeder* S, const fxg_read* reads, size_t n_reads, size_t pool_len, const fxg_pex_node* nodes, size_t n_nodes,
               SeedPlan& plan, std::string& err) {
    if (pool_len >= (uint64_t(1) << 38)) return fail(err, FXG_ERR_INVALID_ARGUMENT, "query pools of %zu bytes: at most 2^38", pool_len);
    std::vector<uint32_t>& seed_base = plan.seed_base;
    std::vector<uint32_t>& leaf_base = plan.leaf_base;
    seed_base.resize(n_reads + 1); leaf_base.resize(n_reads + 1);
    uint64_t n_leaves = 0;
    for (size_t i = 0; i < n_reads; ++i) {
        fxg_read const& R = reads[i];
        if (R.query_offset > pool_len || R.query_len > pool_len - R.query_offset) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: query outside the pool", i);
        if (R.query_len > FXG_MAX_QUERY_LENGTH) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: longer than %d", i, FXG_MAX_QUERY_LENGTH);
        if (R.node_offset > n_nodes || uint64_t(R.num_inner) + R.num_leaves > n_nodes - R.node_offset)
            return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: bad node range", i);
        leaf_base[i] = uint32_t(n_leaves);
        seed_base[i] = uint32_t(2 * n_leaves);
        n_leaves += R.num_leaves;
        if (2 * n_leaves >= (uint64_t(1) << 31)) return fail(err, FXG_ERR_INVALID_ARGUMENT, "more than 2^30 leaves in one call");
    }
    leaf_base[n_reads] = uint32_t(n_leaves);
    seed_base[n_reads] = uint32_t(2 * n_leaves);
    plan.leaf_info.resize(n_leaves);
    for (size_t i = 0; i < n_reads; ++i) {
        fxg_read const& R = reads[i];
        const fxg_pex_node* lv = nodes + R.node_offset + R.num_inner;
        for (uint32_t li = 0; li < R.num_leaves; ++li) {
            fxg_pex_node const& leaf = lv[li];
            if (leaf.query_index_to < leaf.query_index_from || leaf.query_index_to >= R.query_len)
                return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu, leaf %u: outside the query", i, li);
            uint32_t const m = uint32_t(leaf.query_index_to - leaf.query_index_from + 1), e = uint32_t(leaf.num_errors);
            if (e > uint32_t(kSeedMaxErrors) || m / (e + 1) < S->q)
                return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu, leaf %u: %u bases with %u errors (at most %d errors and q * (errors + 1) = %u bases)",
                            i, li, m, e, kSeedMaxErrors, S->q * (e + 1));
            plan.leaf_info[leaf_base[i] + li] = seed_pack(R.query_offset + leaf.query_index_from, m, e);
        }
    }
    plan.n_seeds = uint32_t(2 * n_leaves);
    return FXG_OK;
}

// Where seed_batch delivers the surviving anchors: a malloc'ed fxg_anchor array (fxg_seed_reads), or -- `dev` set -- a
// verification job's AnchorRec16 records at dev + dev_offset (fxg_seed_verify_reads), in the same order either way.
struct SeedSink {
    DevBuf* dev = nullptr; size_t dev_offset = 0;
    fxg_anchor* host = nullptr;                     // (host) owned by the caller, also when the call fails
    size_t n = 0;                                   // anchors delivered
    std::vector<uint32_t> per_read;                 // per (read, orientation)
    uint64_t h2d_bytes = 0, d2h_bytes = 0;          // what the call copied, besides the query pools
};

// the reads' anchor ranges as the seeder laid the anchors out
void set_read_anchors(fxg_read* reads, size_t n_reads, std::vector<uint32_t> const& per_read) {
    uint64_t at = 0;
    for (size_t i = 0; i < n_reads; ++i) {
        reads[i].anchor_offset = at;
        reads[i].num_anchors_forward = per_read.empty() ? 0 : per_read[2 * i];
        reads[i].num_anchors_reverse = per_read.empty() ? 0 : per_read[2 * i + 1];
        at += uint64_t(reads[i].num_anchors_forward) + reads[i].num_anchors_reverse;
    }
}

// The device seeder on a planned batch (plan.n_seeds > 0) whose query pools -- forward, then reverse complement -- are at
// d_pool on the device, on K's stream (which first waits for `pool_ready`, if given).  Returns with the stream drained.
int seed_batch(fxg_ctx* c, const fxg_gpu_seeder* S, const uint32_t* packed, SeedPlan const& plan, size_t n_reads, CallScratch& K,
               const uint8_t* d_pool, uint64_t pool_len, cudaEvent_t pool_ready, uint64_t max_anchors_hard, uint64_t max_anchors_soft,
               int erase_useless_anchors, SeedSink& out, fxg_seed_stats& st, std::string& err) {
    uint32_t const n_seeds = plan.n_seeds;
    uint64_t const n_leaves = plan.leaf_info.size();
    { std::lock_guard<std::mutex> lock(c->mu); if (!K.host.p) K.host = take_staging(c); }
    DevBuf &d_seed_base = K.bufs[1], &d_leaf_base = K.bufs[2], &d_leaves = K.bufs[3], &d_info = K.bufs[4],
           &d_occ = K.bufs[5], &d_off = K.bufs[6], &d_ctr = K.bufs[7], &d_per_read = K.bufs[8], &d_keys = K.bufs[9], &d_sorted = K.bufs[10],
           &d_uniq = K.bufs[11], &d_nuniq = K.bufs[12], &d_hits = K.bufs[13], &d_hits2 = K.bufs[14], &d_gone = K.bufs[15], &d_at = K.bufs[16],
           &d_out = K.bufs[17], &d_tmp = K.bufs[18];
    cudaStream_t const s = K.st;
    if (pool_ready) CUDA_TRY(err, cudaStreamWaitEvent(s, pool_ready, 0));

    // ---- uploads and the seeds' plan ----
    CUDA_TRY(err, d_seed_base.ensure((n_reads + 1) * 4));
    CUDA_TRY(err, d_leaf_base.ensure((n_reads + 1) * 4));
    CUDA_TRY(err, d_leaves.ensure(n_leaves * 8));
    CUDA_TRY(err, cudaMemcpyAsync(d_seed_base.p, plan.seed_base.data(), (n_reads + 1) * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(err, cudaMemcpyAsync(d_leaf_base.p, plan.leaf_base.data(), (n_reads + 1) * 4, cudaMemcpyHostToDevice, s));
    CUDA_TRY(err, cudaMemcpyAsync(d_leaves.p, plan.leaf_info.data(), n_leaves * 8, cudaMemcpyHostToDevice, s));
    out.h2d_bytes += (n_reads + 1) * 8 + n_leaves * 8;
    CUDA_TRY(err, d_info.ensure(size_t(n_seeds) * 8));
    CUDA_TRY(err, d_occ.ensure(size_t(n_seeds) * 8));
    CUDA_TRY(err, d_off.ensure((size_t(n_seeds) + 1) * 8));
    CUDA_TRY(err, d_ctr.ensure(8 * 8));
    CUDA_TRY(err, d_per_read.ensure(n_reads * 8));
    CUDA_TRY(err, cudaMemsetAsync(d_per_read.p, 0, n_reads * 8, s));
    CUDA_TRY(err, cudaMemsetAsync(d_off.p, 0, 8, s));
    SeedRefs const R = seed_refs(S, packed);
    SeedBatch const B{d_pool, pool_len, d_seed_base.as<uint32_t>(), d_leaf_base.as<uint32_t>(), d_leaves.as<uint64_t>(),
                      uint32_t(n_reads), n_seeds, S->bucket.as<uint32_t>(), S->pos.as<uint32_t>(), S->q};
    seed_plan_kernel<<<seed_grid(n_seeds), 256, 0, s>>>(B, d_info.as<uint64_t>(), d_occ.as<uint64_t>());
    CUDA_TRY(err, cudaGetLastError());
    size_t tmp_bytes = 0;
    CUDA_TRY(err, cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, d_occ.as<uint64_t>(), d_off.as<uint64_t>() + 1, n_seeds, s));
    CUDA_TRY(err, d_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
    CUDA_TRY(err, cub::DeviceScan::InclusiveSum(d_tmp.p, tmp_bytes, d_occ.as<uint64_t>(), d_off.as<uint64_t>() + 1, n_seeds, s));
    CUDA_TRY(err, K.host.ensure(std::max<size_t>(4096, n_reads * 8)));
    uint64_t* h_ctr = K.host.as<uint64_t>();             // (moves when the buffer grows)
    CUDA_TRY(err, cudaMemcpyAsync(h_ctr, d_off.as<uint64_t>() + n_seeds, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(err, cudaStreamSynchronize(s));
    out.d2h_bytes += 8;
    uint64_t const total_occ = h_ctr[0];

    // ---- chunks of whole seeds under the budget of q-gram occurrences (a seed above it gets a chunk of its own) ----
    std::vector<uint64_t> off;                     // host copy of the offsets, only when the batch needs several chunks
    if (total_occ > S->budget || n_seeds > kSeedChunkSeeds) {
        off.resize(size_t(n_seeds) + 1);
        CUDA_TRY(err, cudaMemcpyAsync(off.data(), d_off.p, off.size() * 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        out.d2h_bytes += off.size() * 8;
    }
    auto off_at = [&](uint32_t i) { return off.empty() ? (i == 0 ? 0 : total_occ) : off[i]; };
    for (uint32_t s0 = 0; s0 < n_seeds;) {
        uint32_t s1 = n_seeds;
        if (!off.empty()) {
            s1 = uint32_t(std::upper_bound(off.begin() + s0 + 1, off.end(), off[s0] + S->budget) - off.begin()) - 1;
            s1 = std::min(std::max(s1, s0 + 1), std::min(n_seeds, s0 + kSeedChunkSeeds));
        }
        uint64_t const N = off_at(s1) - off_at(s0);
        uint32_t const ns = s1 - s0;
        if (N == 0) { s0 = s1; continue; }
        if (N >= (uint64_t(1) << 31)) return fail(err, FXG_ERR_INVALID_ARGUMENT, "seeds %u..%u have %llu q-gram occurrences: build the index with a larger q",
                                                  s0, s1 - 1, (unsigned long long)N);
        int const n_items = int(N);
        // candidates: (seed, nominal start) keys, sorted and made unique
        CUDA_TRY(err, d_keys.ensure(N * 8));
        CUDA_TRY(err, d_sorted.ensure(N * 8));
        CUDA_TRY(err, d_uniq.ensure(N * 8));
        CUDA_TRY(err, d_nuniq.ensure(8));
        CUDA_TRY(err, cudaMemsetAsync(d_ctr.p, 0, 64, s));
        unsigned long long* const ctr = d_ctr.as<unsigned long long>();
        seed_emit_kernel<<<seed_grid(ns), 256, 0, s>>>(B, d_info.as<uint64_t>(), d_off.as<uint64_t>(), s0, s1, d_keys.as<uint64_t>(), ctr);
        CUDA_TRY(err, cudaGetLastError());
        int const key_bits = std::min(64, kSeedKeyShift + bits_for(ns - 1));
        size_t sort_bytes = 0, uniq_bytes = 0;
        CUDA_TRY(err, cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, d_keys.as<uint64_t>(), d_sorted.as<uint64_t>(), n_items, 0, key_bits, s));
        CUDA_TRY(err, cub::DeviceSelect::Unique(nullptr, uniq_bytes, d_sorted.as<uint64_t>(), d_uniq.as<uint64_t>(), d_nuniq.as<uint32_t>(), n_items, s));
        CUDA_TRY(err, d_tmp.ensure(std::max(sort_bytes, uniq_bytes)));
        CUDA_TRY(err, cub::DeviceRadixSort::SortKeys(d_tmp.p, sort_bytes, d_keys.as<uint64_t>(), d_sorted.as<uint64_t>(), n_items, 0, key_bits, s));
        CUDA_TRY(err, cub::DeviceSelect::Unique(d_tmp.p, uniq_bytes, d_sorted.as<uint64_t>(), d_uniq.as<uint64_t>(), d_nuniq.as<uint32_t>(), n_items, s));
        // check every distinct start; the hit buffer grows and the check runs again if it was too small
        uint64_t hit_cap = std::max<uint64_t>(d_hits.cap / 8, N + 1024);
        uint64_t n_hits = 0;
        for (;;) {
            CUDA_TRY(err, d_hits.ensure(hit_cap * 8));
            seed_check_kernel<<<seed_grid(N), 256, 0, s>>>(R, B, d_info.as<uint64_t>(), s0, d_uniq.as<uint64_t>(), d_nuniq.as<uint32_t>(),
                                                           d_hits.as<uint64_t>(), hit_cap, ctr);
            CUDA_TRY(err, cudaGetLastError());
            CUDA_TRY(err, cudaMemcpyAsync(h_ctr, ctr, 64, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(err, cudaStreamSynchronize(s));
            out.d2h_bytes += 64;
            n_hits = h_ctr[2];
            if (n_hits <= hit_cap) break;
            hit_cap = n_hits;
            CUDA_TRY(err, cudaMemsetAsync(ctr + 1, 0, 16, s));
        }
        st.candidates += h_ctr[0]; st.checked += h_ctr[1]; st.hits += n_hits;
        if (n_hits == 0) { s0 = s1; continue; }
        // caps on hits ordered by (seed, errors, position), then the kept ones by (seed, position)
        int const hit_items = int(n_hits);
        CUDA_TRY(err, d_hits2.ensure(n_hits * 8));
        CUDA_TRY(err, cub::DeviceRadixSort::SortKeys(nullptr, sort_bytes, d_hits.as<uint64_t>(), d_hits2.as<uint64_t>(), hit_items, 0, 64, s));
        CUDA_TRY(err, d_tmp.ensure(sort_bytes));
        CUDA_TRY(err, cub::DeviceRadixSort::SortKeys(d_tmp.p, sort_bytes, d_hits.as<uint64_t>(), d_hits2.as<uint64_t>(), hit_items, 0,
                                                     std::min(64, kHitKeyShift + bits_for(ns - 1)), s));
        seed_caps_kernel<<<seed_grid(n_hits), 256, 0, s>>>(d_hits2.as<uint64_t>(), n_hits, max_anchors_hard, max_anchors_soft, d_hits.as<uint64_t>(), ctr);
        CUDA_TRY(err, cudaGetLastError());
        CUDA_TRY(err, cub::DeviceRadixSort::SortKeys(d_tmp.p, sort_bytes, d_hits.as<uint64_t>(), d_hits2.as<uint64_t>(), hit_items, 0, 64, s));
        CUDA_TRY(err, cudaMemcpyAsync(h_ctr, ctr, 64, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        out.d2h_bytes += 64;
        st.dropped_hard += h_ctr[3]; st.cut_soft += h_ctr[4];
        uint64_t const n_kept = n_hits - h_ctr[3] - h_ctr[4];
        if (n_kept == 0) { s0 = s1; continue; }
        // erase_useless_anchors, then the survivors in order
        CUDA_TRY(err, d_gone.ensure(n_kept * 4));
        CUDA_TRY(err, d_at.ensure(n_kept * 4));
        CUDA_TRY(err, cudaMemsetAsync(d_gone.p, 0, n_kept * 4, s));
        if (erase_useless_anchors) {
            seed_erase_kernel<<<seed_grid(n_kept), 256, 0, s>>>(R, d_hits2.as<uint64_t>(), n_kept, d_gone.as<uint32_t>());
            CUDA_TRY(err, cudaGetLastError());
        }
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_gone.as<uint32_t>(), d_at.as<uint32_t>(), int(n_kept), s));
        CUDA_TRY(err, d_tmp.ensure(tmp_bytes));
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, d_gone.as<uint32_t>(), d_at.as<uint32_t>(), int(n_kept), s));
        uint64_t n_out = 0;
        if (out.dev) {
            // straight into the job's record buffer, behind the records of the earlier chunks (room for every kept anchor and
            // for the 256-byte rounding of prepare_job's layout; a growing buffer keeps what the earlier chunks wrote)
            size_t const done = out.dev_offset + out.n * sizeof(AnchorRec16);
            size_t const need = out.dev_offset + ((out.n + n_kept) * sizeof(AnchorRec16) + 255) / 256 * 256 + 64;
            CUDA_TRY(err, out.n ? out.dev->ensure_preserving(need, done, s) : out.dev->ensure(need));
            seed_output_kernel<true><<<seed_grid(n_kept), 256, 0, s>>>(R, B, s0, d_hits2.as<uint64_t>(), n_kept, d_gone.as<uint32_t>(), d_at.as<uint32_t>(),
                                                                       out.dev->as<uint8_t>() + done, d_per_read.as<uint32_t>(), ctr);
            CUDA_TRY(err, cudaGetLastError());
            CUDA_TRY(err, cudaMemcpyAsync(h_ctr, ctr, 64, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(err, cudaStreamSynchronize(s));
            out.d2h_bytes += 64;
            n_out = n_kept - h_ctr[5];
        } else {
            CUDA_TRY(err, d_out.ensure(n_kept * sizeof(fxg_anchor)));
            seed_output_kernel<false><<<seed_grid(n_kept), 256, 0, s>>>(R, B, s0, d_hits2.as<uint64_t>(), n_kept, d_gone.as<uint32_t>(), d_at.as<uint32_t>(),
                                                                        d_out.p, d_per_read.as<uint32_t>(), ctr);
            CUDA_TRY(err, cudaGetLastError());
            // back through page-locked memory: the counters, then up to n_kept records
            CUDA_TRY(err, K.host.ensure(64 + n_kept * sizeof(fxg_anchor)));
            uint64_t* const h = h_ctr = K.host.as<uint64_t>();
            CUDA_TRY(err, cudaMemcpyAsync(h, ctr, 64, cudaMemcpyDeviceToHost, s));
            CUDA_TRY(err, cudaMemcpyAsync(h + 8, d_out.p, n_kept * sizeof(fxg_anchor), cudaMemcpyDeviceToHost, s));
            CUDA_TRY(err, cudaStreamSynchronize(s));
            out.d2h_bytes += 64 + n_kept * sizeof(fxg_anchor);
            n_out = n_kept - h[5];
            if (n_out) {
                fxg_anchor* grown = static_cast<fxg_anchor*>(std::realloc(out.host, (out.n + n_out) * sizeof(fxg_anchor)));
                if (!grown) return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate %llu anchors", (unsigned long long)(out.n + n_out));
                out.host = grown;
                std::memcpy(out.host + out.n, h + 8, n_out * sizeof(fxg_anchor));
            }
        }
        st.erased += h_ctr[5];
        out.n += n_out;
        s0 = s1;
    }
    out.per_read.resize(2 * n_reads);
    CUDA_TRY(err, cudaMemcpyAsync(K.host.p, d_per_read.p, n_reads * 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(err, cudaStreamSynchronize(s));
    out.d2h_bytes += n_reads * 8;
    std::memcpy(out.per_read.data(), K.host.p, n_reads * 8);
    uint64_t sum = 0;
    for (uint32_t v : out.per_read) sum += v;
    if (sum != out.n) return fail(err, FXG_ERR_CUDA, "internal: %llu anchors counted per read, %zu written", (unsigned long long)sum, out.n);
    return FXG_OK;
}

}  // namespace

extern "C" {

int fxg_gpu_seeder_create(fxg_ctx* c, uint32_t q, fxg_gpu_seeder** out) {
    if (!c || !out) return FXG_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    std::string err;
    if (q < 4 || q > 14) return fail(err, FXG_ERR_INVALID_ARGUMENT, "q = %u: the index takes q-grams of 4..14 bases", q);
    CUDA_TRY(err, cudaSetDevice(c->device));
    std::unique_ptr<fxg_gpu_seeder> S(new (std::nothrow) fxg_gpu_seeder());
    if (!S) return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate the seeder");
    StoreReader guard{c};
    const uint32_t* packed = nullptr;
    std::vector<uint64_t> len, pbase;
    if (int rc = take_store(c, nullptr, guard, packed, &len, &pbase, &S->refs_version, err)) return rc;
    S->ctx_serial = c->serial;
    S->q = q;
    S->n_refs = uint32_t(len.size());
    std::vector<uint64_t> ubase(len.size());
    uint64_t total = 0;
    for (size_t r = 0; r < len.size(); ++r) { ubase[r] = total; total += len[r]; }
    if (total >= (uint64_t(1) << 32))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "the references hold %llu bases: positions are 32-bit, index below 4 Gbp", (unsigned long long)total);
    S->budget = uint64_t(env_int("FXG_SEED_CANDIDATES", 1 << 26, 1, INT32_MAX));
    CallScratch K{c};
    CUDA_TRY(err, cudaStreamCreateWithFlags(&K.st, cudaStreamNonBlocking));
    size_t const nr = std::max<size_t>(len.size(), 1);
    CUDA_TRY(err, S->ubase.ensure(nr * 8));
    CUDA_TRY(err, S->pbase.ensure(nr * 8));
    CUDA_TRY(err, S->len.ensure(nr * 8));
    if (!len.empty()) {
        CUDA_TRY(err, cudaMemcpyAsync(S->ubase.p, ubase.data(), len.size() * 8, cudaMemcpyHostToDevice, K.st));
        CUDA_TRY(err, cudaMemcpyAsync(S->pbase.p, pbase.data(), len.size() * 8, cudaMemcpyHostToDevice, K.st));
        CUDA_TRY(err, cudaMemcpyAsync(S->len.p, len.data(), len.size() * 8, cudaMemcpyHostToDevice, K.st));
    }
    // counting sort: counts per code, exclusive scan into the buckets, scatter through a copy of the buckets
    size_t const n_codes = size_t(1) << (2 * q);
    DevBuf& counts = K.bufs[0];
    DevBuf& tmp = K.bufs[1];
    CUDA_TRY(err, counts.ensure((n_codes + 1) * 4));
    CUDA_TRY(err, S->bucket.ensure((n_codes + 1) * 4));
    CUDA_TRY(err, cudaMemsetAsync(counts.p, 0, (n_codes + 1) * 4, K.st));
    SeedRefs const R = seed_refs(S.get(), packed);
    uint32_t const grid = uint32_t(std::min<uint64_t>(seed_grid(total), uint64_t(c->num_sms) * 16));
    if (total) {
        seed_index_count_kernel<<<grid, 256, 0, K.st>>>(R, total, q, counts.as<uint32_t>());
        CUDA_TRY(err, cudaGetLastError());
    }
    size_t tmp_bytes = 0;
    CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts.as<uint32_t>(), S->bucket.as<uint32_t>(), n_codes + 1, K.st));
    CUDA_TRY(err, tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
    CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts.as<uint32_t>(), S->bucket.as<uint32_t>(), n_codes + 1, K.st));
    uint32_t n_pos = 0;
    CUDA_TRY(err, cudaMemcpyAsync(&n_pos, S->bucket.as<uint32_t>() + n_codes, 4, cudaMemcpyDeviceToHost, K.st));
    CUDA_TRY(err, cudaStreamSynchronize(K.st));
    CUDA_TRY(err, S->pos.ensure(std::max<size_t>(n_pos, 1) * 4));
    CUDA_TRY(err, cudaMemcpyAsync(counts.p, S->bucket.p, (n_codes + 1) * 4, cudaMemcpyDeviceToDevice, K.st));
    if (n_pos) {
        seed_index_fill_kernel<<<grid, 256, 0, K.st>>>(R, total, q, counts.as<uint32_t>(), S->pos.as<uint32_t>());
        CUDA_TRY(err, cudaGetLastError());
    }
    CUDA_TRY(err, cudaStreamSynchronize(K.st));
    *out = S.release();
    return FXG_OK;
}

void fxg_gpu_seeder_free(fxg_ctx* c, fxg_gpu_seeder* S) {
    if (!S) return;
    if (c) cudaSetDevice(c->device);
    S->release();
    delete S;
}

int fxg_seed_reads(fxg_ctx* c, const fxg_gpu_seeder* S, fxg_read* reads, size_t n_reads,
                   const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                   const fxg_pex_node* nodes, size_t n_nodes,
                   uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                   fxg_anchor** anchors, size_t* n_anchors, fxg_seed_stats* stats) {
    if (!c || !S || !anchors || !n_anchors || (n_reads && !reads) || (pool_len && (!forward_pool || !reverse_complement_pool)) || (n_nodes && !nodes))
        return FXG_ERR_INVALID_ARGUMENT;
    *anchors = nullptr; *n_anchors = 0;
    std::string err;
    SeedPlan plan;
    if (int rc = plan_seeds(S, reads, n_reads, pool_len, nodes, n_nodes, plan, err)) return rc;
    fxg_seed_stats st{};
    st.seeds = plan.n_seeds;
    StoreReader guard{c};
    const uint32_t* packed = nullptr;
    if (int rc = take_store(c, S, guard, packed, nullptr, nullptr, nullptr, err)) return rc;
    SeedSink sink;
    if (plan.n_seeds) {
        CUDA_TRY(err, cudaSetDevice(c->device));
        CallScratch K{c};
        CUDA_TRY(err, cudaStreamCreateWithFlags(&K.st, cudaStreamNonBlocking));
        DevBuf& d_pool = K.bufs[0];
        CUDA_TRY(err, d_pool.ensure(2 * pool_len + 64));
        if (pool_len) {
            CUDA_TRY(err, cudaMemcpyAsync(d_pool.p, forward_pool, pool_len, cudaMemcpyHostToDevice, K.st));
            CUDA_TRY(err, cudaMemcpyAsync(d_pool.as<uint8_t>() + pool_len, reverse_complement_pool, pool_len, cudaMemcpyHostToDevice, K.st));
        }
        int const rc = seed_batch(c, S, packed, plan, n_reads, K, d_pool.as<uint8_t>(), pool_len, nullptr, max_anchors_hard, max_anchors_soft,
                                  erase_useless_anchors, sink, st, err);
        if (rc != FXG_OK) { std::free(sink.host); return rc; }
    }
    set_read_anchors(reads, n_reads, sink.per_read);
    if (stats) *stats = st;
    *anchors = sink.host; *n_anchors = sink.n;
    return FXG_OK;
}

}  // extern "C"

namespace {

// fxg_seed_verify_reads; pool_kind = cudaMemcpyDeviceToDevice: the pools are in device memory (fxg_map_fastq) and fill the
// job's pool from there
int seed_verify(fxg_ctx* c, const fxg_gpu_seeder* S, const fxg_verify_config* cfg, fxg_read* reads, size_t n_reads,
                const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                const fxg_pex_node* nodes, size_t n_nodes,
                uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                fxg_seed_stats* stats, fxg_job** out, cudaMemcpyKind pool_kind) {
    if (!c || !S || !cfg || !out || (n_reads && !reads) || (pool_len && (!forward_pool || !reverse_complement_pool)) || (n_nodes && !nodes))
        return FXG_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    std::string err;
    // ---- what fxg_seed_reads, then fxg_verify_reads would refuse, in that order, before any device work ----
    SeedPlan plan;
    if (int rc = plan_seeds(S, reads, n_reads, pool_len, nodes, n_nodes, plan, err)) return rc;
    StoreReader guard{c};                // (until the job has run: seeding and verification both read the store)
    const uint32_t* packed = nullptr;
    if (int rc = take_store(c, S, guard, packed, nullptr, nullptr, nullptr, err)) return rc;
    std::unique_lock<std::mutex> lock(c->mu);
    if (int rc = check_verify_call(c, cfg)) return rc;
    lock.unlock();
    if (int rc = validate_reads(c, err, reads, 0, n_reads, pool_len, nodes, n_nodes, nullptr, 0, false)) return rc;
    lock.lock();
    CUDA_TRY(c->err, cudaSetDevice(c->device));
    fxg_job* j = new_borrowed_job(c, cfg, reads, n_reads, nodes, n_nodes, pool_len);
    if (!j) return FXG_ERR_OUT_OF_MEMORY;
    lock.unlock();

    // ---- the pools go up once: the seeder reads the job's pool (forward, then reverse complement, as SeedBatch wants) ----
    fxg_counters ctr{};
    int rc = stage_pool(c, j->pool, forward_pool, pool_len, reverse_complement_pool, pool_len, err, ctr, true, pool_kind);
    if (rc == FXG_OK && cudaEventCreateWithFlags(&j->pool_ready, cudaEventDisableTiming | cudaEventBlockingSync) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "cannot create an event");
    if (rc == FXG_OK && cudaEventRecord(j->pool_ready, c->stage_stream) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "staging failed");
    // ---- seeding: the survivors land in the job's record buffer where prepare_job's layout puts the anchors ----
    fxg_seed_stats st{};
    st.seeds = plan.n_seeds;
    SeedSink sink;
    sink.dev = &j->prep.dev;
    {
        uint64_t n_inner = 0;
        for (size_t i = 0; i < n_reads; ++i) n_inner += reads[i].num_inner;
        Prepared layout;
        carve_records(layout, n_inner, plan.leaf_info.size(), n_reads, 0);
        sink.dev_offset = layout.o_anchors;
    }
    if (rc == FXG_OK && plan.n_seeds) {
        CallScratch K{c};
        if (cudaStreamCreateWithFlags(&K.st, cudaStreamNonBlocking) != cudaSuccess) rc = fail(err, FXG_ERR_CUDA, "cannot create a stream");
        if (rc == FXG_OK) rc = seed_batch(c, S, packed, plan, n_reads, K, j->pool.bytes.as<uint8_t>(), pool_len, j->pool_ready, max_anchors_hard,
                                          max_anchors_soft, erase_useless_anchors, sink, st, err);
    }
    ctr.h2d_bytes += sink.h2d_bytes; ctr.d2h_bytes += sink.d2h_bytes;
    if (rc == FXG_OK) {
        set_read_anchors(reads, n_reads, sink.per_read);
        index_walks(j);
        // (seed_batch drained its stream before it returned: Prepared::ready, recorded behind the records' upload, covers
        //  the anchors it wrote as well)
        rc = prepare_job(c, j, err, ctr, true);
    }
    if (rc == FXG_OK && !j->prep.ok && sink.n) {
        // the host-driven levels take the job: they read fxg_anchor records on the host (the walks do not use num_errors)
        std::vector<AnchorRec16> back(sink.n);
        if (cudaMemcpy(back.data(), j->prep.dev.as<uint8_t>() + sink.dev_offset, sink.n * sizeof(AnchorRec16), cudaMemcpyDeviceToHost) != cudaSuccess)
            rc = fail(err, FXG_ERR_CUDA, "cannot copy the anchors back");
        ctr.d2h_bytes += sink.n * sizeof(AnchorRec16);
        j->anchors.resize(sink.n);
        for (size_t i = 0; i < sink.n; ++i) j->anchors[i] = fxg_anchor{back[i].pex_leaf_index, back[i].reference_id, back[i].reference_position, 0};
        j->anchors_p = j->anchors.data(); j->n_anchors = sink.n;
    }
    rc = run_borrowed_job(c, j, rc, err, ctr, out);
    if (rc == FXG_OK && stats) *stats = st;
    return rc;
}

}  // namespace

extern "C" {

int fxg_seed_verify_reads(fxg_ctx* c, const fxg_gpu_seeder* S, const fxg_verify_config* cfg, fxg_read* reads, size_t n_reads,
                          const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                          const fxg_pex_node* nodes, size_t n_nodes,
                          uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                          fxg_seed_stats* stats, fxg_job** out) {
    return seed_verify(c, S, cfg, reads, n_reads, forward_pool, reverse_complement_pool, pool_len, nodes, n_nodes, max_anchors_hard,
                       max_anchors_soft, erase_useless_anchors, stats, out, cudaMemcpyHostToDevice);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ BAM and SAM on the device

namespace {

// The batch as the record kernels read it, and what the format's host writer would refuse.  Both host writers walk the
// reads in order and check a read's alignments before they move on; the first failure they would meet decides the code
// returned here.  bam_output.cpp meets a read's alignments in their stable order by reference id, sam_output.cpp in
// index order.
struct OutPlan {
    std::vector<OutReadRec> reads;
    std::vector<uint64_t> ref_off;                         // (SAM) the reference names, concatenated: n_references + 1 offsets
    std::string header;                                    // the header bytes (empty without it)
    uint64_t cigar_lo = UINT64_MAX, cigar_hi = 0, seq_lo = UINT64_MAX, seq_hi = 0, names_len = 0, quals_len = 0;
    uint64_t n_rec = 0;
};

// (fxg_map_fastq) the reads' SEQ, names and qualities in device memory already: SEQ in the parsed forward pool, the names
// and qualities in the uploaded text at each read's spans.  The record kernels read them there instead of an upload.
struct DeviceReads { const uint8_t* forward_pool; const char* text; const fxg_read_span* spans; };

int plan_output(bool bam, const fxg_alignment* al, size_t n_al, const uint32_t* cigar_pool, size_t n_references,
                const char* const* reference_ids, const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads,
                const fxg_sam_query* queries, int with_header, OutPlan& P, std::string& err, const DeviceReads* dev = nullptr) {
    P.reads.resize(n_reads);
    size_t a = 0;
    for (size_t ri = 0; ri < n_reads; ++ri) {
        size_t const a0 = a;
        while (a < n_al && al[a].read_index == ri) ++a;
        if (a < n_al && al[a].read_index < ri)
            return fail(err, FXG_ERR_STATE, "alignment %zu (read %u) follows read %zu: alignments must be grouped by read", a, al[a].read_index, ri);
        size_t const l_name = (dev ? dev->spans[ri].id_len : std::strlen(queries[ri].id ? queries[ri].id : "*")) + (bam ? 1 : 0);     // BAM names carry their NUL
        if (bam && a == a0 && l_name > 255) return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: the name has %zu characters (254 at most)", ri, l_name - 1);
        // (BAM) the first failing alignment in (reference id, index) order
        uint64_t first = UINT64_MAX;
        int code = FXG_OK;
        for (size_t k = a0; k < a; ++k) {
            fxg_alignment const& A = al[k];
            bool const bad = A.reference_id >= n_references || (A.cigar_len && !cigar_pool);
            if (!bam && bad)
                return fail(err, FXG_ERR_INVALID_ARGUMENT, "read %zu: alignment %zu has a reference id out of range or a CIGAR without a pool", ri, k);
            if (bam) {
                int e = FXG_OK;
                if (bad || l_name > 255) e = FXG_ERR_INVALID_ARGUMENT;
                else if (A.cigar_len > 65535) {
                    int64_t rs = 0, qs = 0;
                    for (uint32_t i = 0; i < A.cigar_len; ++i) {
                        uint32_t const v = cigar_pool[A.cigar_offset + i], op = v & 15u;
                        if (op == FXG_CIGAR_D || op == FXG_CIGAR_EQ || op == FXG_CIGAR_X) rs += v >> 4;
                        if (op == FXG_CIGAR_I || op == FXG_CIGAR_EQ || op == FXG_CIGAR_X) qs += v >> 4;
                    }
                    if (qs >= (int64_t(1) << 28) || rs >= (int64_t(1) << 28)) e = FXG_ERR_OVERFLOW;
                }
                uint64_t const key = uint64_t(A.reference_id) << 32 | (k - a0);
                if (e != FXG_OK && key < first) { first = key; code = e; }
            }
            if (A.cigar_len) { P.cigar_lo = std::min<uint64_t>(P.cigar_lo, A.cigar_offset); P.cigar_hi = std::max<uint64_t>(P.cigar_hi, A.cigar_offset + A.cigar_len); }
        }
        if (code == FXG_ERR_OVERFLOW)
            return fail(err, code, "read %zu: a CIGAR of more than 65535 operations spans 2^28 bases or more (the CG tag's placeholder cannot hold it)", ri);
        if (code != FXG_OK) return fail(err, code, "read %zu: a reference id out of range, a CIGAR without a pool or a name of more than 254 characters", ri);
        fxg_read const& R = reads[ri];
        const char* const q = dev ? nullptr : queries[ri].quality;
        bool const have_q = dev || q;
        size_t const l_q = dev ? dev->spans[ri].quality_len : q ? std::strlen(q) : 0;
        OutReadRec& O = P.reads[ri];
        O.seq = R.query_offset;
        O.name = dev ? dev->spans[ri].id_offset : P.names_len;
        O.qual = dev ? dev->spans[ri].quality_offset : P.quals_len;
        O.l_seq = R.query_len;
        O.l_name = uint32_t(l_name);
        // SAM writes every quality at its own length, BAM only one of exactly query_len characters
        O.l_qual = !have_q ? 0u : !bam ? uint32_t(l_q) : l_q && l_q == R.query_len ? R.query_len : 0u;
        O.al0 = uint32_t(a0); O.n_al = uint32_t(a - a0);
        O.rec0 = uint32_t(P.n_rec);
        P.names_len += O.l_name;
        P.quals_len += O.l_qual;
        if (R.query_len) { P.seq_lo = std::min<uint64_t>(P.seq_lo, R.query_offset); P.seq_hi = std::max<uint64_t>(P.seq_hi, R.query_offset + R.query_len); }
        P.n_rec += std::max<size_t>(a - a0, 1);
    }
    if (a != n_al) return fail(err, FXG_ERR_STATE, "alignment %zu names read %u of %zu: alignments must be grouped by read in read order", a, al[a].read_index, n_reads);
    if (P.n_rec >= (uint64_t(1) << 32) || (bam ? P.names_len : uint64_t(n_al)) >= (uint64_t(1) << 32))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "%llu records: split the batch", (unsigned long long)P.n_rec);
    if (P.seq_lo > P.seq_hi) P.seq_lo = P.seq_hi = 0;
    if (P.cigar_lo > P.cigar_hi) P.cigar_lo = P.cigar_hi = 0;
    for (OutReadRec& O : P.reads) O.seq -= std::min(O.seq, P.seq_lo);
    if (!bam) {
        P.ref_off.resize(n_references + 1);
        for (size_t r = 0; r < n_references; ++r) P.ref_off[r + 1] = P.ref_off[r] + std::strlen(reference_ids[r]);
    }
    if (with_header) {                                     // the host writers' header, byte for byte
        std::string text = "@HD\tVN:1.6\tSO:unknown\tGO:none\n";
        for (size_t r = 0; r < n_references; ++r) { text += "@SQ\tSN:"; text += reference_ids[r]; text += "\tLN:"; text += std::to_string(reference_lengths[r]); text += '\n'; }
        if (!bam) P.header = std::move(text);
        else {                                             // BAM: the text inside the binary header
            auto u32 = [&](uint32_t v) { for (int i = 0; i < 4; ++i) P.header += char(uint8_t(v >> (8 * i))); };
            P.header += "BAM\1";
            u32(uint32_t(text.size())); P.header += text;
            u32(uint32_t(n_references));
            for (size_t r = 0; r < n_references; ++r) {
                size_t const l = std::strlen(reference_ids[r]) + 1;
                u32(uint32_t(l)); P.header.append(reference_ids[r], l);
                u32(uint32_t(std::min<uint64_t>(reference_lengths[r], uint64_t(INT32_MAX))));
            }
        }
    }
    return FXG_OK;
}

constexpr uint8_t kBgzfEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

static_assert(sizeof(DeflateSmem) <= 227 * 1024, "the deflate kernel's shared memory exceeds a block's 227 KB");

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// An output call's scratch: the CallScratch buffers by name, the BGZF tail's apart from the records'
struct OutScratch : CallScratch {
    using CallScratch::CallScratch;
    DevBuf &in = bufs[0], &recs = bufs[1], &sizes = bufs[2], &offs = bufs[3];        // the upload; records, their sizes and offsets
    DevBuf &scan_tmp = bufs[4], &raw = bufs[5];                                      // cub's temporary; the uncompressed output
    DevBuf &work = bufs[6], &slots = bufs[7], &info = bufs[8], &bsize = bufs[9], &boff = bufs[10], &img = bufs[11];     // BGZF
};

// The BGZF image of the uncompressed output K.raw[0, raw_len) (raw_len > 0), on K's stream: deflate per 0xff00-byte
// chunk, block offsets, assembly, and the image copied to the start of K.host (img_len bytes).  h_word is a page-locked
// word for the length's read-back.
int bgzf_image_on_device(OutScratch& K, uint64_t raw_len, uint64_t* h_word, uint64_t& d2h, uint64_t& launches, size_t& img_len,
                         std::string& err) {
    cudaStream_t const s = K.st;
    const uint8_t* const raw = K.raw.as<uint8_t>();
    uint32_t const n_chunks = uint32_t((raw_len + kBgzfChunk - 1) / kBgzfChunk);
    CUDA_TRY(err, K.work.ensure(raw_len * 4));
    CUDA_TRY(err, K.slots.ensure(size_t(n_chunks) * kBgzfSlotWords * 4));
    CUDA_TRY(err, K.info.ensure(size_t(n_chunks) * sizeof(BgzfBlockInfo)));
    CUDA_TRY(err, K.bsize.ensure((size_t(n_chunks) + 2) * 8));
    CUDA_TRY(err, K.boff.ensure((size_t(n_chunks) + 2) * 8));
    CUDA_TRY(err, cudaFuncSetAttribute(bgzf_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(DeflateSmem))));
    bgzf_deflate_kernel<<<n_chunks, kDeflateThreads, sizeof(DeflateSmem), s>>>(raw, raw_len, K.work.as<uint32_t>(), K.slots.as<uint32_t>(),
                                                                              K.info.as<BgzfBlockInfo>(), K.bsize.as<uint64_t>(), n_chunks);
    CUDA_TRY(err, cudaGetLastError());
    size_t tmp_bytes = 0;
    CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, K.bsize.as<uint64_t>(), K.boff.as<uint64_t>(), n_chunks + 2, s));
    CUDA_TRY(err, K.scan_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
    CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(K.scan_tmp.p, tmp_bytes, K.bsize.as<uint64_t>(), K.boff.as<uint64_t>(), n_chunks + 2, s));
    // (the image is at most the raw stream stored, plus framing)
    CUDA_TRY(err, K.img.ensure(raw_len + (uint64_t(n_chunks) + 1) * 31 + 28));
    bgzf_assemble_kernel<<<n_chunks + 1, 256, 0, s>>>(raw, K.slots.as<uint32_t>(), K.info.as<BgzfBlockInfo>(), K.boff.as<uint64_t>(),
                                                      n_chunks, K.img.as<uint8_t>());
    CUDA_TRY(err, cudaGetLastError());
    launches += 2;
    CUDA_TRY(err, cudaMemcpyAsync(h_word, K.boff.as<uint64_t>() + n_chunks + 1, 8, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(err, cudaStreamSynchronize(s));
    d2h += 8;
    img_len = size_t(h_word[0]);
    CUDA_TRY(err, K.host.ensure(img_len));
    CUDA_TRY(err, cudaMemcpyAsync(K.host.p, K.img.p, img_len, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(err, cudaStreamSynchronize(s));
    d2h += img_len;
    return FXG_OK;
}

// a malloc'ed copy of n bytes (and a NUL behind them) for the caller
int hand_out(const void* src, size_t n, uint8_t** bytes, size_t* bytes_len) {
    uint8_t* buf = static_cast<uint8_t*>(std::malloc(n + 1));
    if (!buf) return FXG_ERR_OUT_OF_MEMORY;
    if (n) std::memcpy(buf, src, n);
    buf[n] = 0;
    *bytes = buf; *bytes_len = n;
    return FXG_OK;
}

// fxg_write_bam_device (bam, always bgzf) and fxg_write_sam_device: refusals before any device work, then on a stream of
// the call's own one upload through page-locked staging, the format's size kernel, the scan of the sizes into offsets,
// the header and the format's write kernel, and the output as it is or (bgzf) its BGZF image, malloc'ed for the caller.
// With `dev`, SEQ, names and qualities are read in device memory (forward_pool and queries are not used).
int write_on_device(bool bam, int bgzf, fxg_ctx* c, const fxg_alignment* al, size_t n_al, const uint32_t* cigar_pool, size_t n_references,
                    const char* const* reference_ids, const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads,
                    const uint8_t* forward_pool, const fxg_sam_query* queries, int with_header, uint8_t** bytes, size_t* bytes_len,
                    const DeviceReads* dev = nullptr) {
    std::string err;
    if (!c || !bytes || !bytes_len || (n_al && !al) || (n_reads && (!reads || (!dev && (!forward_pool || !queries)))) ||
        (n_references && (!reference_ids || !reference_lengths)))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "%s: a required argument is null", bam ? "fxg_write_bam_device" : "fxg_write_sam_device");
    *bytes = nullptr; *bytes_len = 0;
    try {
    OutPlan P;
    if (int rc = plan_output(bam, al, n_al, cigar_pool, n_references, reference_ids, reference_lengths, reads, n_reads, queries, with_header, P, err, dev))
        return rc;
    if (P.n_rec == 0 && P.header.empty())                  // no output: nothing but the end-of-file block, or the empty text
        return bgzf ? hand_out(kBgzfEof, sizeof kBgzfEof, bytes, bytes_len) : hand_out(nullptr, 0, bytes, bytes_len);

    // ---- one upload through page-locked staging, every segment at a 256-byte boundary: reads, alignments, CIGAR range,
    //      forward-pool range, names, qualities (these three not with `dev`), (SAM) reference name offsets and names,
    //      header ----
    size_t up = 0;
    auto place = [&up](size_t n) { size_t const at = up; up = align_up(at + n, 256); return at; };
    size_t const o_reads = place(n_reads * sizeof(OutReadRec)), o_al = place(n_al * sizeof(fxg_alignment)),
                 o_cig = place((P.cigar_hi - P.cigar_lo) * 4), o_seq = place(dev ? 0 : P.seq_hi - P.seq_lo),
                 o_names = place(dev ? 0 : P.names_len), o_quals = place(dev ? 0 : P.quals_len), o_refoff = place(P.ref_off.size() * 8),
                 o_refnames = place(P.ref_off.empty() ? 0 : P.ref_off.back()), o_header = place(P.header.size());
    CUDA_TRY(err, cudaSetDevice(c->device));
    OutScratch K{c};
    { std::lock_guard<std::mutex> lock(c->mu); K.host = take_staging(c); }
    CUDA_TRY(err, cudaStreamCreateWithFlags(&K.st, cudaStreamNonBlocking));
    cudaStream_t const s = K.st;
    CUDA_TRY(err, K.host.ensure(up + 64));
    uint8_t* const h = K.host.as<uint8_t>();
    if (n_reads) std::memcpy(h + o_reads, P.reads.data(), n_reads * sizeof(OutReadRec));
    if (n_al) std::memcpy(h + o_al, al, n_al * sizeof(fxg_alignment));
    if (P.cigar_hi > P.cigar_lo) std::memcpy(h + o_cig, cigar_pool + P.cigar_lo, (P.cigar_hi - P.cigar_lo) * 4);
    if (!dev && P.seq_hi > P.seq_lo) std::memcpy(h + o_seq, forward_pool + P.seq_lo, P.seq_hi - P.seq_lo);
    for (size_t ri = 0; ri < (dev ? 0 : n_reads); ++ri) {
        OutReadRec const& O = P.reads[ri];
        std::memcpy(h + o_names + O.name, queries[ri].id ? queries[ri].id : "*", O.l_name);
        if (O.l_qual) std::memcpy(h + o_quals + O.qual, queries[ri].quality, O.l_qual);
    }
    if (!P.ref_off.empty()) std::memcpy(h + o_refoff, P.ref_off.data(), P.ref_off.size() * 8);
    for (size_t r = 0; r + 1 < P.ref_off.size(); ++r) std::memcpy(h + o_refnames + P.ref_off[r], reference_ids[r], P.ref_off[r + 1] - P.ref_off[r]);
    std::memcpy(h + o_header, P.header.data(), P.header.size());
    CUDA_TRY(err, K.in.ensure(up));
    CUDA_TRY(err, cudaMemcpyAsync(K.in.p, h, up, cudaMemcpyHostToDevice, s));
    uint64_t h2d = up, d2h = 0, launches = 0;
    uint8_t* const din = K.in.as<uint8_t>();
    OutArgs A{};
    A.reads = reinterpret_cast<const OutReadRec*>(din + o_reads); A.n_reads = uint32_t(n_reads);
    A.al = reinterpret_cast<const fxg_alignment*>(din + o_al);
    A.cigars = reinterpret_cast<const uint32_t*>(din + o_cig); A.cigar_lo = P.cigar_lo;
    A.seq = din + o_seq; A.names = reinterpret_cast<const char*>(din + o_names); A.quals = reinterpret_cast<const char*>(din + o_quals);
    if (dev) { A.seq = dev->forward_pool + P.seq_lo; A.names = A.quals = dev->text; }
    A.ref_off = reinterpret_cast<const uint64_t*>(din + o_refoff); A.ref_names = reinterpret_cast<const char*>(din + o_refnames);
    auto const size_kernel = bam ? bam_size_kernel : sam_size_kernel;
    auto const write_kernel = bam ? bam_write_kernel : sam_write_kernel;

    // ---- record sizes, their offsets, the output's length ----
    uint32_t const n_rec = uint32_t(P.n_rec);
    uint64_t* const h_word = reinterpret_cast<uint64_t*>(h + up);           // (read-backs go behind the upload)
    uint64_t body = 0;
    if (n_rec) {
        CUDA_TRY(err, K.recs.ensure(size_t(n_rec) * (bam ? sizeof(BamRecord) : sizeof(SamRecord))));
        CUDA_TRY(err, K.sizes.ensure((size_t(n_rec) + 1) * 8));
        CUDA_TRY(err, K.offs.ensure((size_t(n_rec) + 1) * 8));
        CUDA_TRY(err, cudaMemsetAsync(K.sizes.as<uint64_t>() + n_rec, 0, 8, s));
        A.recs = K.recs.p; A.rec_off = K.sizes.as<uint64_t>();
        size_kernel<<<uint32_t((uint64_t(n_reads) * 32 + 255) / 256), 256, 0, s>>>(A);
        CUDA_TRY(err, cudaGetLastError());
        ++launches;
        size_t tmp_bytes = 0;
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, K.sizes.as<uint64_t>(), K.offs.as<uint64_t>(), n_rec + 1, s));
        CUDA_TRY(err, K.scan_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(K.scan_tmp.p, tmp_bytes, K.sizes.as<uint64_t>(), K.offs.as<uint64_t>(), n_rec + 1, s));
        CUDA_TRY(err, cudaMemcpyAsync(h_word, K.offs.as<uint64_t>() + n_rec, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        d2h += 8;
        body = h_word[0];
    }
    uint64_t const raw_len = P.header.size() + body;

    // ---- the uncompressed output: the header, then the records ----
    CUDA_TRY(err, K.raw.ensure(raw_len + 16));
    if (!P.header.empty()) CUDA_TRY(err, cudaMemcpyAsync(K.raw.p, din + o_header, P.header.size(), cudaMemcpyDeviceToDevice, s));
    A.rec_off = K.offs.as<uint64_t>(); A.out = K.raw.as<uint8_t>(); A.body = P.header.size();
    if (n_rec) {
        write_kernel<<<uint32_t((uint64_t(n_rec) * 32 + 255) / 256), 256, 0, s>>>(A, n_rec);
        CUDA_TRY(err, cudaGetLastError());
        ++launches;
    }

    // ---- the output as it is, or its BGZF image ----
    size_t out_len = size_t(raw_len);
    if (bgzf) {
        if (int rc = bgzf_image_on_device(K, raw_len, h_word, d2h, launches, out_len, err)) return rc;
    } else {
        CUDA_TRY(err, cudaStreamSynchronize(s));                           // (the upload may still read the staging)
        CUDA_TRY(err, K.host.ensure(out_len));
        CUDA_TRY(err, cudaMemcpyAsync(K.host.p, K.raw.p, out_len, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        d2h += out_len;
    }
    {
        std::lock_guard<std::mutex> lock(c->mu);
        c->ctr.h2d_bytes += h2d; c->ctr.d2h_bytes += d2h; c->ctr.kernel_launches += launches;
    }
    return hand_out(K.host.p, out_len, bytes, bytes_len);
    } catch (...) { return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate host memory"); }
}

}  // namespace

extern "C" {

int fxg_write_bam_device(fxg_ctx* c, const fxg_alignment* al, size_t n_al, const uint32_t* cigar_pool, size_t n_references,
                         const char* const* reference_ids, const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads,
                         const uint8_t* forward_pool, const fxg_sam_query* queries, int with_header, uint8_t** bytes, size_t* bytes_len) {
    return write_on_device(true, 1, c, al, n_al, cigar_pool, n_references, reference_ids, reference_lengths, reads, n_reads, forward_pool,
                           queries, with_header, bytes, bytes_len);
}

int fxg_job_write_bam_device(fxg_ctx* c, const fxg_job* job, size_t n_references, const char* const* reference_ids,
                             const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool,
                             const fxg_sam_query* queries, int with_header, uint8_t** bytes, size_t* bytes_len) {
    if (!job) return FXG_ERR_INVALID_ARGUMENT;
    return fxg_write_bam_device(c, fxg_job_alignments(job), fxg_job_num_alignments(job), fxg_job_cigar_pool(job), n_references, reference_ids,
                                reference_lengths, reads, n_reads, forward_pool, queries, with_header, bytes, bytes_len);
}

int fxg_write_sam_device(fxg_ctx* c, const fxg_alignment* al, size_t n_al, const uint32_t* cigar_pool, size_t n_references,
                         const char* const* reference_ids, const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads,
                         const uint8_t* forward_pool, const fxg_sam_query* queries, int with_header, int bgzf, uint8_t** bytes,
                         size_t* bytes_len) {
    return write_on_device(false, bgzf, c, al, n_al, cigar_pool, n_references, reference_ids, reference_lengths, reads, n_reads, forward_pool,
                           queries, with_header, bytes, bytes_len);
}

int fxg_job_write_sam_device(fxg_ctx* c, const fxg_job* job, size_t n_references, const char* const* reference_ids,
                             const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool,
                             const fxg_sam_query* queries, int with_header, int bgzf, uint8_t** bytes, size_t* bytes_len) {
    std::string err;
    if (!job) return fail(err, FXG_ERR_INVALID_ARGUMENT, "fxg_job_write_sam_device: no job");
    return fxg_write_sam_device(c, fxg_job_alignments(job), fxg_job_num_alignments(job), fxg_job_cigar_pool(job), n_references, reference_ids,
                                reference_lengths, reads, n_reads, forward_pool, queries, with_header, bgzf, bytes, bytes_len);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ FASTQ input on the device

struct fxg_parsed {
    std::vector<uint8_t> statuses;               // per record
    std::vector<fxg_read> reads;                 // the kept reads, in record order
    std::vector<fxg_read_span> spans;
    std::vector<fxg_pex_node> nodes;
    std::vector<uint8_t> pools;                  // (fxg_parse_fastq) forward, then reverse complement
    uint64_t pool_len = 0;
};

namespace {

// A parse call's scratch.  The text and the pools (forward, then reverse complement) stay on the device for the steps
// that follow in fxg_map_fastq.
struct ParseScratch : CallScratch {
    using CallScratch::CallScratch;
    DevBuf &text = bufs[0], &nl = bufs[1], &n_nl = bufs[2], &recs = bufs[3], &lens = bufs[4], &offs = bufs[5], &scan_tmp = bufs[6],
           &pool = bufs[7], &first_bad = bufs[8];
};

// Parses text[0, text_len) on a stream of K's own into `out` (all but the pools, which stay in K.pool): the text goes up
// once through page-locked staging, the device finds the records, checks and converts them, and the host builds the kept
// reads' trees on several threads while the ranks are written.  The copies and launches are added to ctr.
int parse_on_device(fxg_ctx* c, const fxg_read_config* cfg, const char* text, size_t text_len, ParseScratch& K, fxg_parsed& out,
                    fxg_counters& ctr, std::string& err) {
    if (cfg->build_strategy > 1) return fail(err, FXG_ERR_INVALID_ARGUMENT, "build_strategy %u: 0 (recursive) or 1 (bottom_up)", cfg->build_strategy);
    if (cfg->query_errors == FXG_NULL_ID && !(cfg->error_probability >= 0.0 && cfg->error_probability <= 1.0))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "error_probability %g: it must lie in [0, 1]", cfg->error_probability);
    if (text_len >= (size_t(1) << 31))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "a text of %zu bytes: at most 2^31 - 1, split it at a record boundary", text_len);
    CUDA_TRY(err, cudaSetDevice(c->device));
    { std::lock_guard<std::mutex> lock(c->mu); K.host = take_staging(c); }
    CUDA_TRY(err, cudaStreamCreateWithFlags(&K.st, cudaStreamNonBlocking));
    cudaStream_t const s = K.st;
    size_t const o_word = align_up(text_len, 64);              // read-backs go behind the text in the staging buffer
    CUDA_TRY(err, K.host.ensure(o_word + 64));
    uint64_t* const h_word = reinterpret_cast<uint64_t*>(K.host.as<uint8_t>() + o_word);
    if (text_len) std::memcpy(K.host.p, text, text_len);
    CUDA_TRY(err, K.text.ensure(text_len + 16));
    if (text_len) CUDA_TRY(err, cudaMemcpyAsync(K.text.p, K.host.p, text_len, cudaMemcpyHostToDevice, s));
    ctr.h2d_bytes += text_len;
    const char* const dt = K.text.as<char>();

    // ---- the newlines, the lines, the records ----
    uint64_t n_nl = 0;
    if (text_len) {
        CUDA_TRY(err, K.nl.ensure(text_len * 4));
        CUDA_TRY(err, K.n_nl.ensure(8));
        thrust::counting_iterator<uint32_t> const at(0);
        size_t tmp_bytes = 0;
        CUDA_TRY(err, cub::DeviceSelect::If(nullptr, tmp_bytes, at, K.nl.as<uint32_t>(), K.n_nl.as<uint32_t>(), int(text_len), FastqNewline{dt}, s));
        CUDA_TRY(err, K.scan_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
        CUDA_TRY(err, cub::DeviceSelect::If(K.scan_tmp.p, tmp_bytes, at, K.nl.as<uint32_t>(), K.n_nl.as<uint32_t>(), int(text_len), FastqNewline{dt}, s));
        CUDA_TRY(err, cudaMemcpyAsync(h_word, K.n_nl.p, 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        ctr.d2h_bytes += 4;
        ctr.kernel_launches += 1;
        n_nl = *reinterpret_cast<uint32_t*>(h_word);
    }
    uint64_t const n_lines = n_nl + (text_len && text[text_len - 1] != '\n' ? 1 : 0);
    uint64_t const n_full = n_lines / 4;
    FastqArgs const A{dt, text_len, K.nl.as<uint32_t>(), n_nl, n_full, cfg->error_probability, cfg->query_errors, cfg->seed_errors};
    uint64_t first_bad = n_lines % 4 ? n_full : UINT64_MAX;    // a record cut short can only be the last one
    uint64_t pool_len = 0;
    const FastqRec* recs = nullptr;
    if (n_full) {
        CUDA_TRY(err, K.recs.ensure(n_full * sizeof(FastqRec)));
        CUDA_TRY(err, K.lens.ensure((n_full + 1) * 8));
        CUDA_TRY(err, K.offs.ensure((n_full + 1) * 8));
        CUDA_TRY(err, K.first_bad.ensure(8));
        CUDA_TRY(err, cudaMemsetAsync(K.lens.as<uint64_t>() + n_full, 0, 8, s));
        CUDA_TRY(err, cudaMemsetAsync(K.first_bad.p, 0xff, 8, s));
        fastq_record_kernel<<<uint32_t((n_full + 255) / 256), 256, 0, s>>>(A, K.recs.as<FastqRec>(), K.lens.as<uint64_t>(),
                                                                          K.first_bad.as<unsigned long long>());
        CUDA_TRY(err, cudaGetLastError());
        size_t tmp_bytes = 0;
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, K.lens.as<uint64_t>(), K.offs.as<uint64_t>(), int(n_full + 1), s));
        CUDA_TRY(err, K.scan_tmp.ensure(std::max<size_t>(tmp_bytes, 16)));
        CUDA_TRY(err, cub::DeviceScan::ExclusiveSum(K.scan_tmp.p, tmp_bytes, K.lens.as<uint64_t>(), K.offs.as<uint64_t>(), int(n_full + 1), s));
        ctr.kernel_launches += 2;
        // the records, the first malformed one and the pools' length come back
        size_t const o_recs = o_word + 64;
        CUDA_TRY(err, K.host.ensure(o_recs + n_full * sizeof(FastqRec)));          // (the text's upload is through: the stream was drained)
        uint64_t* const hw = reinterpret_cast<uint64_t*>(K.host.as<uint8_t>() + o_word);
        CUDA_TRY(err, cudaMemcpyAsync(hw, K.first_bad.p, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaMemcpyAsync(hw + 1, K.offs.as<uint64_t>() + n_full, 8, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaMemcpyAsync(K.host.as<uint8_t>() + o_recs, K.recs.p, n_full * sizeof(FastqRec), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(err, cudaStreamSynchronize(s));
        ctr.d2h_bytes += 16 + n_full * sizeof(FastqRec);
        first_bad = std::min<uint64_t>(first_bad, hw[0]);
        pool_len = hw[1];
        recs = reinterpret_cast<const FastqRec*>(K.host.as<uint8_t>() + o_recs);
    }
    if (first_bad != UINT64_MAX) {
        unsigned long long const r = first_bad;
        if (first_bad == n_full) return fail(err, FXG_ERR_INVALID_ARGUMENT, "record %llu is cut short: it has %llu of its 4 lines", r, (unsigned long long)(n_lines % 4));
        if (recs[first_bad].fault == kFastqNoAt) return fail(err, FXG_ERR_INVALID_ARGUMENT, "record %llu: the header line does not start with '@'", r);
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "record %llu: the third line does not start with '+'", r);
    }

    // ---- the ranks into the pools on the device, the kept reads' trees on the host meanwhile ----
    CUDA_TRY(err, K.pool.ensure(2 * pool_len + 64));
    if (pool_len) {
        fastq_ranks_kernel<<<uint32_t((n_full * 32 + 255) / 256), 256, 0, s>>>(A, K.recs.as<FastqRec>(), K.offs.as<uint64_t>(), K.pool.as<uint8_t>());
        CUDA_TRY(err, cudaGetLastError());
        ctr.kernel_launches += 1;
    }
    out.pool_len = pool_len;
    out.statuses.resize(n_full);
    std::vector<uint64_t> kept;
    for (uint64_t r = 0; r < n_full; ++r) {
        out.statuses[r] = recs[r].status;
        if (recs[r].status == FXG_READ_KEPT) kept.push_back(r);
    }
    size_t const n = kept.size();
    out.reads.assign(n, fxg_read{});
    out.spans.resize(n);
    size_t const T = parallel_threads(n, 512);
    std::vector<std::vector<fxg_pex_node>> chunk_nodes(T);
    std::vector<int> chunk_rc(T, FXG_OK);
    parallel_chunks(T, n, [&](size_t t, size_t lo, size_t hi) {
        for (size_t i = lo; i < hi && chunk_rc[t] == FXG_OK; ++i) {
            FastqRec const& F = recs[kept[i]];
            fxg_pex_node *inner = nullptr, *leaves = nullptr;
            size_t ni = 0, nlv = 0;
            chunk_rc[t] = fxg_pex_build(F.l_seq, F.errors, cfg->seed_errors, int(cfg->build_strategy), &inner, &ni, &leaves, &nlv);
            if (chunk_rc[t] == FXG_OK) {
                fxg_read& R = out.reads[i];
                R.node_offset = chunk_nodes[t].size();           // (within the chunk for now)
                R.query_len = F.l_seq; R.num_inner = uint32_t(ni); R.num_leaves = uint32_t(nlv);
                chunk_nodes[t].insert(chunk_nodes[t].end(), inner, inner + ni);
                chunk_nodes[t].insert(chunk_nodes[t].end(), leaves, leaves + nlv);
            }
            fxg_pex_free(inner); fxg_pex_free(leaves);
            out.spans[i] = fxg_read_span{kept[i], F.id, F.qual, F.l_id, F.l_qual};
        }
    });
    for (int rc : chunk_rc) if (rc != FXG_OK) return fail(err, rc, "cannot build the PEX trees");
    std::vector<uint64_t> chunk_base(T + 1, 0);
    for (size_t t = 0; t < T; ++t) chunk_base[t + 1] = chunk_base[t] + chunk_nodes[t].size();
    out.nodes.resize(chunk_base[T]);
    for (size_t t = 0; t < T; ++t) std::copy(chunk_nodes[t].begin(), chunk_nodes[t].end(), out.nodes.begin() + long(chunk_base[t]));
    uint64_t q = 0;
    for (size_t t = 0; t < T; ++t)
        for (size_t i = n * t / T; i < n * (t + 1) / T; ++i) {           // parallel_chunks' split
            out.reads[i].node_offset += chunk_base[t];
            out.reads[i].query_offset = q;
            q += out.reads[i].query_len;
        }
    if (q != pool_len) return fail(err, FXG_ERR_CUDA, "internal: the kept reads hold %llu bases, the pools %llu", (unsigned long long)q, (unsigned long long)pool_len);
    CUDA_TRY(err, cudaStreamSynchronize(s));
    return FXG_OK;
}

void add_call_counters(fxg_ctx* c, fxg_counters const& ctr) {
    std::lock_guard<std::mutex> lock(c->mu);
    c->ctr.h2d_bytes += ctr.h2d_bytes; c->ctr.d2h_bytes += ctr.d2h_bytes; c->ctr.kernel_launches += ctr.kernel_launches;
}

}  // namespace

extern "C" {

int fxg_parse_fastq(fxg_ctx* c, const fxg_read_config* cfg, const char* text, size_t text_len, fxg_parsed** out) {
    std::string err;
    if (!c || !cfg || !out || (text_len && !text)) return fail(err, FXG_ERR_INVALID_ARGUMENT, "fxg_parse_fastq: a required argument is null");
    *out = nullptr;
    try {
        std::unique_ptr<fxg_parsed> P(new fxg_parsed());
        fxg_counters ctr{};
        ParseScratch K{c};
        int rc = parse_on_device(c, cfg, text, text_len, K, *P, ctr, err);
        size_t const n = 2 * P->pool_len;
        if (rc == FXG_OK && n) {                                   // the pools come back
            P->pools.resize(n);
            if (K.host.ensure(n) != cudaSuccess || cudaMemcpyAsync(K.host.p, K.pool.p, n, cudaMemcpyDeviceToHost, K.st) != cudaSuccess ||
                cudaStreamSynchronize(K.st) != cudaSuccess)
                rc = fail(err, FXG_ERR_CUDA, "cannot copy the pools back");
            else std::memcpy(P->pools.data(), K.host.p, n);
            ctr.d2h_bytes += n;
        }
        add_call_counters(c, ctr);
        if (rc == FXG_OK) *out = P.release();
        return rc;
    } catch (...) { return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate host memory"); }
}

int fxg_parsed_get(const fxg_parsed* P, fxg_parsed_view* v) {
    if (!P || !v) return FXG_ERR_INVALID_ARGUMENT;
    v->n_records = P->statuses.size(); v->statuses = P->statuses.data();
    v->n_reads = P->reads.size(); v->reads = P->reads.data(); v->spans = P->spans.data();
    v->pool_len = P->pool_len; v->forward_pool = P->pools.data(); v->reverse_complement_pool = P->pools.data() + P->pool_len;
    v->n_nodes = P->nodes.size(); v->nodes = P->nodes.data();
    return FXG_OK;
}

void fxg_parsed_free(fxg_parsed* P) { delete P; }

int fxg_map_fastq(fxg_ctx* c, const fxg_gpu_seeder* S, const fxg_read_config* rcfg, const fxg_verify_config* vcfg,
                  uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                  const char* text, size_t text_len, size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                  int format, int with_header, uint8_t** bytes, size_t* bytes_len, fxg_map_summary* summary) {
    std::string err;
    if (!c || !S || !rcfg || !vcfg || !bytes || !bytes_len || (text_len && !text) || (n_references && (!reference_ids || !reference_lengths)))
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "fxg_map_fastq: a required argument is null");
    if (format != FXG_FORMAT_BAM && format != FXG_FORMAT_SAM && format != FXG_FORMAT_SAM_BGZF)
        return fail(err, FXG_ERR_INVALID_ARGUMENT, "format %d: FXG_FORMAT_BAM, _SAM or _SAM_BGZF", format);
    *bytes = nullptr; *bytes_len = 0;
    try {
        fxg_parsed P;
        fxg_counters ctr{};
        ParseScratch K{c};
        int rc = parse_on_device(c, rcfg, text, text_len, K, P, ctr, err);
        add_call_counters(c, ctr);
        if (rc != FXG_OK) return rc;
        // ---- the reads the q-gram seeder takes (seeder.cpp:162); the others are counted and not written ----
        std::vector<fxg_read> reads;
        std::vector<fxg_read_span> spans;
        reads.reserve(P.reads.size()); spans.reserve(P.reads.size());
        for (size_t i = 0; i < P.reads.size(); ++i) {
            fxg_read const& R = P.reads[i];
            const fxg_pex_node* lv = P.nodes.data() + R.node_offset + R.num_inner;
            bool ok = true;
            for (uint32_t li = 0; li < R.num_leaves && ok; ++li) {
                uint64_t const m = lv[li].query_index_to - lv[li].query_index_from + 1, e = lv[li].num_errors;
                ok = e <= uint64_t(kSeedMaxErrors) && m / (e + 1) >= S->q;
            }
            if (ok) { reads.push_back(R); spans.push_back(P.spans[i]); }
            else P.statuses[P.spans[i].record] = FXG_READ_UNSEEDABLE;
        }
        // ---- seeding and verification: the job's pool is filled from the parsed pools on the device ----
        fxg_job* job = nullptr;
        fxg_seed_stats st{};
        if (!reads.empty()) {
            const uint8_t* const fwd = K.pool.as<uint8_t>();
            rc = seed_verify(c, S, vcfg, reads.data(), reads.size(), fwd, fwd + P.pool_len, P.pool_len, P.nodes.data(), P.nodes.size(),
                             max_anchors_hard, max_anchors_soft, erase_useless_anchors, &st, &job, cudaMemcpyDeviceToDevice);
            if (rc != FXG_OK) return rc;
        }
        // ---- the records: SEQ from the parsed forward pool, names and qualities from the text, on the device ----
        DeviceReads const dev{K.pool.as<uint8_t>(), K.text.as<char>(), spans.data()};
        size_t const n_al = job ? fxg_job_num_alignments(job) : 0;
        rc = write_on_device(format == FXG_FORMAT_BAM, format != FXG_FORMAT_SAM, c, job ? fxg_job_alignments(job) : nullptr, n_al,
                             job ? fxg_job_cigar_pool(job) : nullptr, n_references, reference_ids, reference_lengths, reads.data(), reads.size(),
                             nullptr, nullptr, with_header, bytes, bytes_len, &dev);
        fxg_job_free(c, job);
        if (rc != FXG_OK) return rc;
        if (summary) {
            *summary = fxg_map_summary{};
            summary->records = P.statuses.size();
            for (uint8_t x : P.statuses) summary->reads[x]++;
            summary->alignments = n_al;
            summary->seed = st;
        }
        return FXG_OK;
    } catch (...) { return fail(err, FXG_ERR_OUT_OF_MEMORY, "cannot allocate host memory"); }
}

}  // extern "C"
