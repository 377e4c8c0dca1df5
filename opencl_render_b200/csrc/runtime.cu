// runtime.cu -- CUDA host runtime behind the C-ABI.  Replaces the OpenCL host setup of
// source/opencl/raytrace.c:283-603: where the reference rebuilds a context, JIT-compiles the kernel and wraps 35
// host arrays as zero-copy buffers on every call, this keeps a Scene resident in HBM (uploaded once, repacked to the
// layout of rt_types.h) and a Frame (camera lists + three 16-bit planes) per camera.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
#include <thread>
#include <utility>
#include <vector>

#include "cam_builder.cuh"
#include "grid_builder.cuh"
#include "pack_kernels.cuh"
#include "rt_kernels.cuh"
#include "rt_query.cuh"
#include "rt_tail.cuh"
#include "rt_trace.cuh"
#include "rt_wavefront.cuh"
#include "runtime.h"

namespace oclr {

#define OCLR_CUDA(call)                                                                              \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            err = std::string(#call) + ": " + cudaGetErrorString(e_);                                \
            return false;                                                                            \
        }                                                                                            \
    } while (0)

// Device memory comes from the stream-ordered pool of the device with the release threshold lifted, so the
// alloc/free pairs of repeated RaytraceAll calls are served from memory the pool already holds.
static void prepare_pool(int device) {
    static bool done[64] = {false};
    if (device < 0 || device >= 64 || done[device]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    done[device] = true;
}

// Host <-> device copies from / to PAGEABLE memory.  The plugin hands RaytraceAll plain new[] arrays (render.cpp:1086-1134) -- 133 MB
// for config 2 -- and cudaMemcpyAsync moves pageable memory through the driver's own bounce buffer at ~10 GB/s on the calling thread
// (the call then spends 14 of its 20 ms uploading).  Here the staging is done by a small pool of copier threads that do NOTHING but
// memcpy (2 MB blocks, caller's array -> a pinned arena that lives as long as the process); every CUDA call stays on the calling
// thread, which enqueues the H2D copy of a block as soon as that block is staged -- so block k crosses PCIe while blocks k+1.. are
// still being staged.  (Round 1's first attempt let every copier thread issue its own cudaMemcpyAsync: 19.8 -> 14.2 ms on average but
// single calls stalled for up to 340 ms on the driver's locks; that is why the CUDA calls are now made by one thread per device.)
// The arena is per device (RaytraceAll on all devices: one uploading thread per GPU, each staging only its 1/N slice) and is reused
// from the start by the next call; a copy that does not fit what is left waits for the stream to drain first.
class CopyPool {
public:
    struct Job {
        void* dst;
        const void* src;
        size_t n;
        std::atomic<int>* done;
    };
    static CopyPool& get() {
        static CopyPool* p = new CopyPool();   // lives until the process ends (its threads are detached)
        return *p;
    }
    void submit(const Job* jobs, size_t count) {
        {
            std::lock_guard<std::mutex> lock(m_);
            for (size_t i = 0; i < count; ++i) q_.push_back(jobs[i]);
            pending_.fetch_add((int)count);
        }
        if (count == 1) cv_.notify_one(); else cv_.notify_all();
    }
    // The calling thread lends a hand while it waits: runs one queued job, if there is one.
    bool help() {
        Job j;
        {
            std::lock_guard<std::mutex> lock(m_);
            if (q_.empty()) return false;
            j = q_.front();
            q_.pop_front();
            pending_.fetch_sub(1);
        }
        run(j);
        return true;
    }
    int threads() const { return threads_; }

private:
    CopyPool() {
        threads_ = 6;
        if (const char* v = getenv("OCLR_STAGING_THREADS")) threads_ = std::max(1, std::min(atoi(v), 32));
        threads_ = std::min<int>(threads_, std::max(1u, std::thread::hardware_concurrency()));
        for (int t = 0; t < threads_; ++t) std::thread([this]() { worker(); }).detach();
    }
    static void run(const Job& j) {
        memcpy(j.dst, j.src, j.n);
        j.done->store(1, std::memory_order_release);
    }
    void worker() {
        for (;;) {
            Job j;
            bool have = false;
            // a call makes a dozen staged copies in a row: stay awake for ~200 us after a job before going back to sleep on the
            // condition variable (a wake-up costs 50-100 us, as much as the block it is woken for)
            const auto until = std::chrono::steady_clock::now() + std::chrono::microseconds(200);
            while (!have && std::chrono::steady_clock::now() < until) {
                if (pending_.load(std::memory_order_acquire) > 0) {
                    std::lock_guard<std::mutex> lock(m_);
                    if (!q_.empty()) {
                        j = q_.front();
                        q_.pop_front();
                        pending_.fetch_sub(1);
                        have = true;
                    }
                } else {
                    std::this_thread::yield();
                }
            }
            if (!have) {
                std::unique_lock<std::mutex> lock(m_);
                cv_.wait(lock, [this] { return !q_.empty(); });
                j = q_.front();
                q_.pop_front();
                pending_.fetch_sub(1);
            }
            run(j);
        }
    }
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<Job> q_;
    std::atomic<int> pending_{0};   // jobs in q_ (read without the lock by workers that are still awake)
    int threads_ = 0;
};

struct StageArena {   // pinned, per device, grow-only up to the cap
    char* p = nullptr;
    size_t bytes = 0, used = 0;
    std::mutex m;   // one staged copy at a time per device (the copier threads are shared anyway)
};
static const size_t kStageBlock = [] { const char* v = getenv("OCLR_STAGING_BLOCK_KB"); return (size_t)(v && atoi(v) >= 64 ? atoi(v) : 512) << 10; }();   // (measured: 512 KB 10.1 ms, 2 MB 12.0 ms, 8 MB 14.1 ms per config-2 call)
static StageArena& stage_arena(int device) {
    static StageArena arenas[64];
    return arenas[device & 63];
}
// Space for n bytes in the device's arena, or nullptr (then the driver's own staging is used).  When the arena has to be recycled or
// regrown the stream is drained first: copies enqueued earlier may still be reading from it.
static char* stage_reserve(int device, size_t n, cudaStream_t st) {
    static const size_t cap = [] { const char* v = getenv("OCLR_STAGING_MB"); return (size_t)(v ? std::max(16, atoi(v)) : 1024) << 20; }();
    StageArena& a = stage_arena(device);
    if (n > cap) return nullptr;
    if (a.used + n > a.bytes) {
        if (cudaDeviceSynchronize() != cudaSuccess) return nullptr;   // (whatever stream earlier staged copies were enqueued on)
        a.used = 0;
        if (n > a.bytes) {
            const size_t want = std::min(cap, std::max(n, std::max<size_t>(a.bytes * 2, 64u << 20)));
            if (a.p) cudaFreeHost(a.p);
            a.p = nullptr;
            a.bytes = 0;
            if (cudaHostAlloc((void**)&a.p, want, cudaHostAllocPortable) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
            a.bytes = want;
        }
    }
    char* p = a.p + a.used;
    a.used += (n + 255) & ~(size_t)255;
    return p;
}
// A new top-level call (RaytraceAll, scene_create) starts from an empty arena: everything the previous one enqueued has completed
// (those calls synchronise before they return).
static void stage_reset(int device) {
    StageArena& a = stage_arena(device);
    std::lock_guard<std::mutex> lock(a.m);
    a.used = 0;
}

static bool is_pageable(const void* p) {
    cudaPointerAttributes attr;
    const bool pageable = cudaPointerGetAttributes(&attr, p) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
    cudaGetLastError();
    return pageable;
}
static bool staging_enabled() {
    static const bool on = [] { const char* v = getenv("OCLR_STAGING"); return !v || atoi(v) != 0; }();
    return on;
}

static bool host_to_device(void* dst, const void* src, size_t n, cudaStream_t st, std::string& err) {
    int device = 0;
    if (staging_enabled() && n >= (1u << 20) && is_pageable(src) && cudaGetDevice(&device) == cudaSuccess) {
        std::lock_guard<std::mutex> lock(stage_arena(device).m);
        char* stage = stage_reserve(device, n, st);
        if (stage) {
            const size_t blocks = (n + kStageBlock - 1) / kStageBlock;
            std::vector<std::atomic<int>> done(blocks);
            std::vector<CopyPool::Job> jobs(blocks);
            for (size_t b = 0; b < blocks; ++b) {
                done[b].store(0);
                const size_t off = b * kStageBlock;
                jobs[b] = {stage + off, (const char*)src + off, std::min(kStageBlock, n - off), &done[b]};
            }
            CopyPool& pool = CopyPool::get();
            pool.submit(jobs.data(), blocks);
            for (size_t b = 0; b < blocks; ++b) {
                while (done[b].load(std::memory_order_acquire) == 0)
                    if (!pool.help()) std::this_thread::yield();
                const size_t off = b * kStageBlock;
                OCLR_CUDA(cudaMemcpyAsync((char*)dst + off, stage + off, jobs[b].n, cudaMemcpyHostToDevice, st));
            }
            return true;
        }
    }
    OCLR_CUDA(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, st));
    return true;
}

// Device -> pageable host memory: one transfer into the arena, then the copier threads (and the caller) spread it out.  Synchronous.
static bool device_to_host(void* dst, const void* src, size_t n, cudaStream_t st, std::string& err) {
    int device = 0;
    if (staging_enabled() && n >= (1u << 20) && is_pageable(dst) && cudaGetDevice(&device) == cudaSuccess) {
        std::lock_guard<std::mutex> lock(stage_arena(device).m);
        char* stage = stage_reserve(device, n, st);
        if (stage) {
            OCLR_CUDA(cudaMemcpyAsync(stage, src, n, cudaMemcpyDeviceToHost, st));
            OCLR_CUDA(cudaStreamSynchronize(st));
            const size_t blocks = (n + kStageBlock - 1) / kStageBlock;
            std::vector<std::atomic<int>> done(blocks);
            std::vector<CopyPool::Job> jobs(blocks);
            for (size_t b = 0; b < blocks; ++b) {
                done[b].store(0);
                const size_t off = b * kStageBlock;
                jobs[b] = {(char*)dst + off, stage + off, std::min(kStageBlock, n - off), &done[b]};
            }
            CopyPool& pool = CopyPool::get();
            pool.submit(jobs.data(), blocks);
            for (size_t b = 0; b < blocks; ++b)
                while (done[b].load(std::memory_order_acquire) == 0)
                    if (!pool.help()) std::this_thread::yield();
            return true;
        }
    }
    OCLR_CUDA(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, st));
    OCLR_CUDA(cudaStreamSynchronize(st));
    return true;
}

// Small pinned blocks (the frames' read-back words) are recycled: cudaHostAlloc / cudaFreeHost cost ~50-100 us each, which a
// RaytraceAll call that creates and destroys its frame would pay every time.  Blocks are 4 KB, portable, never returned to the driver.
static std::mutex g_pinMutex;
static std::vector<void*> g_pinFree;
static void* pinned_block() {
    {
        std::lock_guard<std::mutex> lock(g_pinMutex);
        if (!g_pinFree.empty()) {
            void* p = g_pinFree.back();
            g_pinFree.pop_back();
            return p;
        }
    }
    void* p = nullptr;
    if (cudaHostAlloc(&p, 4096, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
static void pinned_release(void* p) {
    if (!p) return;
    std::lock_guard<std::mutex> lock(g_pinMutex);
    g_pinFree.push_back(p);
}

// ---- per-device caches of driver objects -------------------------------------------------------------------------------------------
// One RaytraceAll call makes ~40 device allocations, as many frees, half a dozen events and a stream -- per GPU.  Each is a driver
// call behind a process-wide lock: cheap alone (2-5 us), but with one host thread per GPU of an 8-GPU box they queue up behind each
// other and were ~1 ms of a 4 ms call (phases "camera lists" 0.5 ms and "release" 0.3-0.5 ms at N = 8, 0.15 ms each at N = 1).  The
// call repeats with the same sizes frame after frame, so: blocks freed inside RaytraceAll go to a free list of their device and the
// next call's allocations of the same size come from there without a driver call; events and streams are recycled the same way.
// Stream-ordered discipline is what cudaMallocAsync already asked for: a block is released only when its last use is complete or
// enqueued on the device's default stream, and every use on another stream is ordered behind an event recorded on that stream.
struct CachedBlock {
    void* p;
    size_t size;             // size it was allocated with
    unsigned long long epoch;   // call during which it was put back
};
struct BlockCache {
    std::mutex m;
    std::vector<CachedBlock> free;
    unsigned long long epoch = 0;                 // RaytraceAll calls on this device so far
    std::vector<cudaEvent_t> events[2];           // [0] timing, [1] cudaEventDisableTiming
    std::vector<cudaStream_t> streams;            // non-blocking
};
static BlockCache& block_cache(int device) {
    static BlockCache caches[64];
    return caches[device & 63];
}
static thread_local int g_cacheDevice = -1;   // >= 0: this thread is inside RaytraceAll on that device (DeviceBuffer uses the free list)
struct CacheScope {
    int saved, device;
    explicit CacheScope(int d) : saved(g_cacheDevice), device(d) { g_cacheDevice = d; }
    ~CacheScope() {
        g_cacheDevice = saved;
        // blocks nobody asked for during the last three calls go back to the driver (a camera sweep changes the list sizes every frame)
        BlockCache& c = block_cache(device);
        std::vector<void*> stale;
        {
            std::lock_guard<std::mutex> lock(c.m);
            ++c.epoch;
            for (size_t i = 0; i < c.free.size();)
                if (c.free[i].epoch + 3 < c.epoch) {
                    stale.push_back(c.free[i].p);
                    c.free[i] = c.free.back();
                    c.free.pop_back();
                } else {
                    ++i;
                }
        }
        if (!stale.empty() && cudaSetDevice(device) == cudaSuccess)
            for (void* p : stale) cudaFreeAsync(p, 0);
    }
};
void* allocation_cache_enter(int device) { return new CacheScope(device); }
void allocation_cache_leave(void* scope) { delete (CacheScope*)scope; }

static cudaError_t make_event(int device, cudaEvent_t* e, bool timing) {
    BlockCache& c = block_cache(device);
    {
        std::lock_guard<std::mutex> lock(c.m);
        auto& v = c.events[timing ? 0 : 1];
        if (!v.empty()) {
            *e = v.back();
            v.pop_back();
            return cudaSuccess;
        }
    }
    return cudaEventCreateWithFlags(e, timing ? cudaEventDefault : cudaEventDisableTiming);
}
static void drop_event(int device, cudaEvent_t e, bool timing) {
    if (!e) return;
    BlockCache& c = block_cache(device);
    std::lock_guard<std::mutex> lock(c.m);
    c.events[timing ? 0 : 1].push_back(e);
}
static cudaError_t make_stream(int device, cudaStream_t* st) {
    BlockCache& c = block_cache(device);
    {
        std::lock_guard<std::mutex> lock(c.m);
        if (!c.streams.empty()) {
            *st = c.streams.back();
            c.streams.pop_back();
            return cudaSuccess;
        }
    }
    return cudaStreamCreateWithFlags(st, cudaStreamNonBlocking);
}
static void drop_stream(int device, cudaStream_t st) {   // (the stream is idle: its owner waited for its work)
    if (!st) return;
    BlockCache& c = block_cache(device);
    std::lock_guard<std::mutex> lock(c.m);
    c.streams.push_back(st);
}

struct DeviceBuffer {
    void* p = nullptr;
    size_t bytes = 0;
    size_t cachedSize = 0;   // != 0: the block belongs to the device's free list (size it was allocated with)
    int cachedDevice = -1;
    bool borrowed = false;   // p points into memory somebody else owns (the shared-upload landing arena): never freed here
    bool alloc(size_t n, std::string& err, cudaStream_t st = 0) {
        bytes = n;
        borrowed = false;
        cachedSize = 0;
        const size_t want = ((n ? n : 16) + 255) & ~(size_t)255;
        if (g_cacheDevice >= 0) {
            BlockCache& c = block_cache(g_cacheDevice);
            {
                std::lock_guard<std::mutex> lock(c.m);
                for (size_t i = 0; i < c.free.size(); ++i)
                    if (c.free[i].size == want) {   // the call repeats with the same sizes: exact fits
                        p = c.free[i].p;
                        c.free[i] = c.free.back();
                        c.free.pop_back();
                        cachedSize = want;
                        cachedDevice = g_cacheDevice;
                        return true;
                    }
            }
            OCLR_CUDA(cudaMallocAsync(&p, want, st));
            cachedSize = want;
            cachedDevice = g_cacheDevice;
            return true;
        }
        OCLR_CUDA(cudaMallocAsync(&p, want, st));
        return true;
    }
    bool upload(const void* src, size_t n, std::string& err, cudaStream_t st = 0) {
        if (!alloc(n, err, st)) return false;
        if (n) return host_to_device(p, src, n, st, err);
        return true;
    }
    void release(cudaStream_t st = 0) {
        if (p && !borrowed) {
            if (cachedSize) {
                BlockCache& c = block_cache(cachedDevice);
                std::lock_guard<std::mutex> lock(c.m);
                if (c.free.size() < 256)
                    c.free.push_back({p, cachedSize, c.epoch});
                else
                    cudaFreeAsync(p, st);
            } else {
                cudaFreeAsync(p, st);
            }
        }
        p = nullptr;
        borrowed = false;
        cachedSize = 0;
    }
};

// ---- one scene, N GPUs of one box: sharded upload + NVLink fan-out ---------------------------------------------------------------------
// RaytraceAll(all devices) used to let every GPU pull the WHOLE scene (133 MB for config 2) over its own PCIe link.  Now GPU k
// uploads the k-th 1/N of every large array into its own landing arena and one kernel stores that slice into the same place of every
// peer's arena over NVLink peer memory (16-byte stores, like push_rows_kernel); events order the consumers behind all N slices.
// PCIe moves every byte once in total instead of once per GPU.  Arrays travel in two groups so that the triangle repack and the
// primary-ray round start while the grid (the larger group) is still in flight.
enum { kMaxPeers = 16, kShardArrays = 12, kShardGroups = 2 };

struct FanoutItem {
    const uint4* src;              // this GPU's slice inside its own buffer
    unsigned long long vecs;       // 16-byte vectors in the slice
    uint4* dst[kMaxPeers];         // the same place inside every peer's buffer
};
struct FanoutTable {
    int items, peers;
    FanoutItem it[kShardArrays];
};
__global__ void __launch_bounds__(256) fanout_kernel(const __grid_constant__ FanoutTable t) {
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (int a = 0; a < t.items; ++a) {
        const FanoutItem& it = t.it[a];
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < it.vecs; i += stride) {
            const uint4 v = it.src[i];
            for (int d = 0; d < t.peers; ++d) it.dst[d][i] = v;
        }
    }
}

struct ShardCtx {
    int world = 0;
    int devices[kMaxPeers] = {0};
    cudaEvent_t pushed[kShardGroups][kMaxPeers] = {};
    void* ptr[kShardArrays][kMaxPeers] = {};
    // spin barrier with a verdict: every thread arrives with its own status, all leave with the AND (a thread that failed keeps
    // arriving at the remaining barriers so that nobody waits for it forever)
    std::atomic<int> arrived{0};
    std::atomic<unsigned> generation{0};
    std::atomic<int> bad{0};
    bool arrive(bool ok) {
        if (!ok) bad.store(1);
        const unsigned gen = generation.load();
        if (arrived.fetch_add(1) + 1 == world) {
            arrived.store(0);
            generation.fetch_add(1);
        } else {
            while (generation.load() == gen) std::this_thread::yield();
        }
        return bad.load() == 0;
    }
};

// Where the shared upload lands: one plain cudaMalloc block per GPU that lives as long as the process (grow-only), carved up anew by
// every call.  Peers store into it over NVLink, so it is classic peer-mapped memory whose addresses never change under a running
// kernel.  (The first version took these buffers from the stream-ordered pool with cudaMemPoolSetAccess: on config 3, where the
// primary-ray round's 5 GB of path state is allocated from the same pool WHILE the peers' grid slices arrive, memory got stomped --
// every array verified correct when checked (OCLR_SHARD_VERIFY) and the fault went away with CUDA_LAUNCH_BLOCKING=1, with the shared
// upload off, or with the early frame off.  Pool memory is no longer written by peers at all.)
struct LandingArena {
    char* p = nullptr;
    size_t bytes = 0;
};
static LandingArena& landing_arena(int device) {
    static LandingArena arenas[64];
    return arenas[device & 63];
}

// Slice k of n bytes cut N ways on 256-byte boundaries.
static inline void shard_range(size_t n, int k, int world, size_t& begin, size_t& end) {
    const size_t per = ((n + (size_t)world - 1) / (size_t)world + 255) & ~(size_t)255;
    begin = std::min(n, per * (size_t)k);
    end = std::min(n, begin + per);
}

// Peer access between the first `world` devices (direct stores into the peers' landing arenas).  Once per process.
static bool ensure_peer_access(int world, std::string& err) {
    static std::mutex m;
    static int enabledFor = 0;
    static bool usable = false;
    std::lock_guard<std::mutex> lock(m);
    if (enabledFor >= world) return usable;
    usable = true;
    for (int i = 0; i < world && usable; ++i) {
        if (cudaSetDevice(i) != cudaSuccess) usable = false;
        prepare_pool(i);
        for (int j = 0; j < world && usable; ++j) {
            if (i == j) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, i, j) != cudaSuccess || !can) {
                usable = false;
                break;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(j, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) usable = false;
            cudaGetLastError();
        }
    }
    cudaGetLastError();
    if (!usable) err = "peer access between the GPUs is not available";
    enabledFor = world;
    return usable;
}

// One worker thread per GPU, alive for the life of the process: RaytraceAll(all devices) hands each its share of the frame.
// (Creating N threads per call costs ~30 us each, serially, in front of a 2 ms call.)
class DevicePool {
public:
    static DevicePool& get() {
        static DevicePool* p = new DevicePool();   // never destroyed: its threads are detached
        return *p;
    }
    // Runs fn(rank) for rank in [0, world) on the worker bound to device rank; returns when all have finished.  One job at a time.
    void run(int world, const std::function<void(int)>& fn) {
        std::lock_guard<std::mutex> job(jobMutex_);
        {
            std::lock_guard<std::mutex> lock(m_);
            while ((int)workers_ < world) {
                const int d = (int)workers_++;
                std::thread([this, d]() { worker(d); }).detach();
            }
            fn_ = &fn;
            world_ = world;
            pending_ = world;
            ++generation_;
            posted_.store(generation_, std::memory_order_release);
        }
        cvJob_.notify_all();
        std::unique_lock<std::mutex> lock(m_);
        cvDone_.wait(lock, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }
    ShardCtx ctx;   // (guarded by the one-job-at-a-time rule)

private:
    void worker(int d) {
        cudaSetDevice(d);
        unsigned long long seen = 0;
        for (;;) {
            const std::function<void(int)>* fn = nullptr;
            {
                // a render loop calls back within a fraction of a millisecond: stay awake that long before sleeping on the condition
                // variable (a wake-up is 50-100 us, paid by every GPU's thread at the start of every call)
                const auto until = std::chrono::steady_clock::now() + std::chrono::microseconds(300);
                while (posted_.load(std::memory_order_acquire) == seen && std::chrono::steady_clock::now() < until) std::this_thread::yield();
                std::unique_lock<std::mutex> lock(m_);
                cvJob_.wait(lock, [&] { return generation_ != seen; });
                seen = generation_;
                if (d < world_) fn = fn_;
            }
            if (!fn) continue;
            (*fn)(d);
            std::lock_guard<std::mutex> lock(m_);
            if (--pending_ == 0) cvDone_.notify_all();
        }
    }
    std::mutex jobMutex_, m_;
    std::condition_variable cvJob_, cvDone_;
    const std::function<void(int)>* fn_ = nullptr;
    unsigned workers_ = 0;
    int world_ = 0, pending_ = 0;
    unsigned long long generation_ = 0;
    std::atomic<unsigned long long> posted_{0};   // == generation_, readable without the lock by workers that are still awake
};

bool run_on_devices(int world, bool shareUpload, const std::function<void(int rank, ShardCtx* share)>& fn, std::string& err) {
    if (world < 1 || world > kMaxPeers || world > device_count()) {
        err = "bad device count";
        return false;
    }
    struct RestoreDevice {   // the caller's current device is its own business (set-up below visits every GPU)
        int d = -1;
        RestoreDevice() {
            if (cudaGetDevice(&d) != cudaSuccess) d = -1;
        }
        ~RestoreDevice() {
            if (d >= 0) cudaSetDevice(d);
            cudaGetLastError();
        }
    } restore;
    DevicePool& pool = DevicePool::get();
    std::string peerErr;
    const bool share = shareUpload && world > 1 && ensure_peer_access(world, peerErr);
    if (shareUpload && world > 1 && !share) {
        static bool said = false;
        if (!said) fprintf(stderr, "[opencl_render_b200] %s: every GPU uploads the whole scene over its own PCIe link\n", peerErr.c_str());
        said = true;
    }
    ShardCtx* ctx = nullptr;
    std::function<void(int)> job = [&](int rank) { fn(rank, ctx); };
    if (!share) {
        pool.run(world, job);
        return true;
    }
    // (the pool's ShardCtx is touched only between its run() calls and by the job itself; run() admits one job at a time, and this
    // function is the only user of ctx, serialised by a mutex of its own)
    static std::mutex shareMutex;
    std::lock_guard<std::mutex> lock(shareMutex);
    ctx = &pool.ctx;
    ctx->world = world;
    ctx->arrived.store(0);
    ctx->bad.store(0);
    for (int d = 0; d < world; ++d) {
        ctx->devices[d] = d;
        if (!ctx->pushed[0][d]) {
            cudaSetDevice(d);
            bool ok = true;
            for (int g = 0; g < kShardGroups; ++g) ok = ok && cudaEventCreateWithFlags(&ctx->pushed[g][d], cudaEventDisableTiming) == cudaSuccess;
            if (!ok) {
                err = "cannot create the upload events";
                cudaGetLastError();
                return false;
            }
        }
    }
    pool.run(world, job);
    return true;
}

struct Scene {
    int device = 0;
    DeviceBuffer triGeo, triShade, bricks, cellRange, cellList, faceMask, planes, matSize, matStart, textures, lights;
    // the walk grid (rt_types.h), when a run of coincident planes collapses; else empty and walkView == view
    DeviceBuffer walkBricks, walkCellRange, walkFaceMask, walkPlanes;
    uint32_t walkTrim = 0;
    SceneView view = {};
    SceneView walkView = {};   // what the production trace stage walks (enqueue_trace)
    size_t bytes = 0;
    int smCount = 148;
    // Ring slots a path of this scene can occupy (rt_wavefront.cuh): only mirror / glass segments (raytrace_opencl.c:682-722) push the
    // ring beyond {current segment, its diffuse bounce} -- a scene in which no material has a reflection or a transparency channel
    // (or only all-black ones, the plugin's 1x1 fallback) never touches slot 2, so its frames allocate 2 slots (96 B per path)
    // instead of kRingSize (576 B)
    int ringSlots = kRingSize;
    bool hasBump = false;   // some material has a BUMP channel: its normals read the camera vectors (radiance queries need a camera)
    uint64_t geometryGen = 0;   // geometry edits so far (scene_update): camera lists built for an older generation are stale
    std::array<DeviceBuffer*, 15> buffers() {
        return {&triGeo, &triShade, &bricks, &cellRange, &cellList, &faceMask, &planes, &matSize, &matStart, &textures, &lights,
                &walkBricks, &walkCellRange, &walkFaceMask, &walkPlanes};
    }
};

// per-round counters of a launch domain: {ray count, cursor, class counts[4], hand-off count, 0, 0, 0, hand-off cursor}, two sets
// alternating between rounds ({hand-off count, 0, 0, 0} doubles as the class counts of the second pass over the rays given up, rt_tail.cuh)
enum { kCounterStride = 2 + kLengthClasses + 5 };
// Wavefront path state of one launch domain (rt_wavefront.cuh WfState, rt_trace.cuh WalkRecords) and its queue counters: stream-ordered
// buffers for up to `capacity` paths, reallocated only when a domain of more paths comes along.
struct PathState {
    DeviceBuffer ctl, rng, colour, ring, carry, rayO, rayD, rayExcl, hit, queue;
    DeviceBuffer recO, recD, recS0, recS1, recOrder;   // walk records in queue order + class order (rt_trace.cuh)
    DeviceBuffer counters;                             // kCounterStride counters x 2, alternating between rounds; then the round log
    uint32_t capacity = 0;
    int ringSlots = 0;   // ring depth the buffers were sized for
    std::array<DeviceBuffer*, 16> buffers() {
        return {&ctl, &rng, &colour, &ring, &carry, &rayO, &rayD, &rayExcl, &hit, &queue, &recO, &recD, &recS0, &recS1, &recOrder, &counters};
    }
    bool reserve(uint32_t Q, int slots, cudaStream_t st, std::string& err) {
        Q = path_state_regrow(capacity, ringSlots, Q, slots);
        if (!Q) return true;
        release(st);
        const size_t q = Q;
        if (!ctl.alloc(sizeof(uint32_t) * q, err, st) || !rng.alloc(sizeof(uint64_t) * q, err, st) || !colour.alloc(sizeof(float4) * q, err, st) ||
            !ring.alloc(sizeof(float4) * q * (size_t)slots * kRingParts, err, st) || !carry.alloc(sizeof(float4) * q * kCarryParts, err, st) ||
            // two ray slots per path (rt_wavefront.cuh: the next segment's closest hit is traced one round ahead)
            !rayO.alloc(sizeof(float4) * 2 * q, err, st) || !rayD.alloc(sizeof(float4) * 2 * q, err, st) ||
            !rayExcl.alloc(sizeof(uint32_t) * 2 * q, err, st) || !hit.alloc(sizeof(float4) * 2 * q, err, st) ||
            !queue.alloc(sizeof(uint32_t) * 2 * q, err, st) || !recO.alloc(sizeof(float4) * 2 * q, err, st) ||
            !recD.alloc(sizeof(float4) * 2 * q, err, st) || !recS0.alloc(sizeof(float4) * 2 * q, err, st) ||
            !recS1.alloc(sizeof(uint4) * 2 * q, err, st) || !recOrder.alloc(sizeof(uint32_t) * 2 * q * kLengthClasses, err, st) ||
            !counters.alloc(sizeof(uint32_t) * (2 * kCounterStride + kRoundLogSize), err, st))
            return false;
        capacity = Q;
        ringSlots = slots;
        return true;
    }
    void release(cudaStream_t st) {
        for (DeviceBuffer* b : buffers()) b->release(st);
        capacity = 0;
        ringSlots = 0;
    }
    size_t bytes() {
        size_t n = 0;
        for (DeviceBuffer* b : buffers()) n += b->bytes;
        return n;
    }
    uint32_t* counter_set(uint32_t round) const { return (uint32_t*)counters.p + kCounterStride * (round & 1u); }
    // A domain of Q <= capacity paths; the queue counters are set per round (RoundDriver).
    void bind(uint32_t Q, int ringSlots, WfState& w, WalkRecords& rec) const {
        w = {Q, (uint32_t*)ctl.p, (uint64_t*)rng.p, (float4*)colour.p, (float4*)ring.p, (uint32_t)ringSlots, (float4*)carry.p, (float4*)rayO.p,
             (float4*)rayD.p, (uint32_t*)rayExcl.p, (float4*)hit.p, (uint32_t*)queue.p, nullptr, nullptr, (uint32_t*)counters.p + 2 * kCounterStride, 0};
        rec = {(float4*)recO.p, (float4*)recD.p, (float4*)recS0.p, (uint4*)recS1.p, (uint32_t*)recOrder.p, nullptr, 2 * Q};   // (two rays per path at most)
    }
};

// One slice of a launch domain (launch_wavefront): its own path state and stream, so the rounds of different slices overlap on the GPU.
enum { kMaxSlices = 8 };
struct WfSlice {
    PathState ps;
    DeviceBuffer tailEntries;                          // hand-off list of a small launch's trace tail (rt_tail.cuh); unallocated for large domains
    DeviceBuffer tailO, tailD, tailS0, tailS1, tailOrder;   // ... as walk records, for the second pass (hand-off mode 2)
    uint32_t tailCapacity = 0;
    uint32_t lastRounds = 4;          // rounds the previous sample needed (first chunk of the next one)
    cudaStream_t stream = nullptr;    // internal stream (slice 0 runs on the caller's stream)
    cudaEvent_t done = nullptr;
    std::vector<cudaEvent_t> traceEvents;   // pairs around the trace launches of the last timed render
    uint32_t traceEventsUsed = 0;
    std::array<DeviceBuffer*, 6> tail_buffers() { return {&tailEntries, &tailO, &tailD, &tailS0, &tailS1, &tailOrder}; }
};

static constexpr uint64_t kNoLists = ~0ull;
struct Frame {
    Scene* scene = nullptr;
    int device = 0;
    Camera cam = {};
    DeviceBuffer camStart, camEnd, camList, planesRGB, ids, flags, counters;
    DeviceBuffer camCheck;           // range-check flag of caller-supplied camera lists (check_camera_lists_kernel); unset for device-built lists
    bool deviceLists = false;        // the lists are built on the device (frame_build_camera_lists), again after a geometry edit
    uint64_t listsGen = 0;           // Scene::geometryGen the lists were made for; kNoLists: the frame has none (a failed frame_set_camera)
    WfSlice slices[kMaxSlices];      // wavefront path state (allocated on first use, sized for the largest slice seen)
    uint32_t* hostCount = nullptr;   // pinned, one per slice
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evFork = nullptr;
    uint32_t lastLaunches = 0;
    size_t camListSize = 0;
    // progressive accumulation + progress (SURVEY.md section 8f-3, 8f-4)
    DeviceBuffer accum;              // float4 per pixel when float accumulation is on (frame_set_accumulation)
    DeviceBuffer doneCount;          // pixel-samples finished by the render call in flight
    cudaStream_t progStream = nullptr;
    unsigned long long* hostDone = nullptr;   // pinned
    std::atomic<unsigned long long> jobPaths{0};   // pixel-samples of the render call in flight (0: none)
    std::mutex progMutex;
    // first logic round started ahead of the render call (frame_prelaunch): it runs on preStream while the scene's grid is uploaded
    cudaStream_t preStream = nullptr;
    cudaEvent_t preReady = nullptr, preDone = nullptr;
    bool prelaunched = false;
    FrameView preView = {};
};

int device_count() {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

bool device_name(int dev, char* buf, size_t len) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    snprintf(buf, len, "CUDA %s (sm_%d%d, %d SMs) #%d", p.name, p.major, p.minor, p.multiProcessorCount, dev);
    return true;
}

// SceneTriangleList::New on the device (grid_builder.cuh) from device-resident vertices / indices; the grid stays in HBM.
struct DeviceGrid {
    DeviceBuffer boxMin, start, list;   // float4 x (n+1), uint32 x (n^3+1), uint32 x total
    uint32_t total = 0;
    void release() {
        boxMin.release();
        start.release();
        list.release();
    }
};

static bool grid_build_on_device(int32_t n, uint32_t V, const float4* dVertexP, uint32_t N, const int4* dIdxP, DeviceGrid& out, std::string& err) {
    const size_t cells = (size_t)n * n * n;
    DeviceBuffer coord, sorted, planes, triCells, slots, offsets, largeList, small, state, queue, keysA, keysB, cellCount, tmp, sortTmp;
    DeviceBuffer &start = out.start, &list = out.list, &boxMin = out.boxMin;
    DeviceBuffer* all[] = {&coord, &sorted, &planes, &triCells, &slots, &offsets, &largeList, &small, &state, &queue, &keysA, &keysB, &cellCount, &tmp, &sortTmp};
    auto done = [&](bool ok) {
        for (DeviceBuffer* b : all) b->release();
        if (!ok) out.release();
        return ok;
    };
    const size_t Vz = V ? V : 1, Nz = N ? N : 1;
    if (!coord.alloc(sizeof(float) * Vz, err) || !sorted.alloc(sizeof(float) * Vz, err) || !planes.alloc(sizeof(float) * 3 * (n + 1), err) ||
        !triCells.alloc(sizeof(TriCells) * Nz, err) || !slots.alloc(sizeof(uint64_t) * (Nz + 1), err) ||
        !offsets.alloc(sizeof(uint64_t) * (Nz + 1), err) || !largeList.alloc(sizeof(uint32_t) * Nz, err) || !small.alloc(sizeof(uint32_t) * 4, err) ||
        !cellCount.alloc(sizeof(uint32_t) * (cells + 1), err) || !start.alloc(sizeof(uint32_t) * (cells + 1), err) ||
        !boxMin.alloc(sizeof(float4) * (n + 1), err))
        return done(false);
    cudaMemsetAsync(planes.p, 0, sizeof(float) * 3 * (n + 1), 0);
    cudaMemsetAsync(small.p, 0, sizeof(uint32_t) * 4, 0);
    cudaMemsetAsync(slots.p, 0, sizeof(uint64_t) * (Nz + 1), 0);
    cudaMemsetAsync(cellCount.p, 0, sizeof(uint32_t) * (cells + 1), 0);
    // 1. split planes at vertex quantiles
    size_t need = 0, tmpBytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, need, (const float*)coord.p, (float*)sorted.p, (int)V);
    tmpBytes = need;
    cub::DeviceScan::ExclusiveSum(nullptr, need, (const uint64_t*)slots.p, (uint64_t*)offsets.p, (int)(N + 1));
    tmpBytes = std::max(tmpBytes, need);
    cub::DeviceScan::ExclusiveSum(nullptr, need, (const uint32_t*)cellCount.p, (uint32_t*)start.p, (int)(cells + 1));
    tmpBytes = std::max(tmpBytes, need);
    if (!tmp.alloc(tmpBytes, err)) return done(false);
    if (V)
        for (int axis = 0; axis < 3; ++axis) {
            grid_coord_kernel<<<(V + 255) / 256, 256>>>(V, dVertexP, axis, (float*)coord.p);
            cub::DeviceRadixSort::SortKeys(tmp.p, tmpBytes, (const float*)coord.p, (float*)sorted.p, (int)V);
            grid_planes_kernel<<<(n + 1 + 127) / 128, 128>>>(V, (const float*)sorted.p, n, (float*)planes.p + (size_t)axis * (n + 1));
        }
    grid_boxmin_kernel<<<(n + 1 + 127) / 128, 128>>>(n, (const float*)planes.p, (float4*)boxMin.p);
    // 2. candidate blocks, slot offsets
    uint32_t* largeCount = (uint32_t*)small.p;
    if (N)
        grid_range_kernel<<<(N + 255) / 256, 256>>>(N, dVertexP, dIdxP, n, (const float*)planes.p, (TriCells*)triCells.p,
                                                   (uint64_t*)slots.p, (uint32_t*)largeList.p, largeCount);
    cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, (const uint64_t*)slots.p, (uint64_t*)offsets.p, (int)(N + 1));
    uint64_t total = 0;
    uint32_t nLarge = 0;
    cudaMemcpyAsync(&total, (const uint64_t*)offsets.p + N, sizeof(uint64_t), cudaMemcpyDeviceToHost, 0);
    cudaMemcpyAsync(&nLarge, largeCount, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    OCLR_CUDA(cudaStreamSynchronize(0));
    if (total > (1ull << 31)) {
        err = "scene-grid builder: more than 2^31 (triangle, cell) candidates";
        return done(false);
    }
    const size_t totalZ = total ? (size_t)total : 1;
    if (!state.alloc(totalZ, err) || !queue.alloc(sizeof(uint16_t) * totalZ, err) || !keysA.alloc(sizeof(uint64_t) * totalZ, err) ||
        !keysB.alloc(sizeof(uint64_t) * totalZ, err))
        return done(false);
    // 3. flood fills -> keys
    const uint64_t sentinel = (uint64_t)cells * (uint64_t)Nz;
    if (N) {
        grid_fill_small_kernel<<<(N + 127) / 128, 128>>>(N, dVertexP, dIdxP, n, (const float*)planes.p,
                                                        (const TriCells*)triCells.p, (const uint64_t*)offsets.p, (uint8_t*)state.p, (uint16_t*)queue.p,
                                                        sentinel, (uint64_t*)keysA.p, (uint32_t*)cellCount.p);
        if (nLarge)
            grid_fill_large_kernel<<<nLarge, 1024>>>(N, dVertexP, dIdxP, n, (const float*)planes.p,
                                                   (const TriCells*)triCells.p, (const uint64_t*)offsets.p, (const uint32_t*)largeList.p,
                                                   (uint8_t*)state.p, sentinel, (uint64_t*)keysA.p, (uint32_t*)cellCount.p);
    }
    // 4. CSR
    cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, (const uint32_t*)cellCount.p, (uint32_t*)start.p, (int)(cells + 1));
    uint32_t real = 0;
    cudaMemcpyAsync(&real, (const uint32_t*)start.p + cells, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    int endBit = 1;
    while (endBit < 64 && (sentinel >> endBit) != 0) ++endBit;
    size_t sortBytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, sortBytes, (const uint64_t*)keysA.p, (uint64_t*)keysB.p, (int64_t)total, 0, endBit);
    if (!sortTmp.alloc(sortBytes, err)) return done(false);
    cub::DeviceRadixSort::SortKeys(sortTmp.p, sortBytes, (const uint64_t*)keysA.p, (uint64_t*)keysB.p, (int64_t)total, 0, endBit);
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        err = std::string("scene-grid builder: ") + cudaGetErrorString(e);
        return done(false);
    }
    if (!list.alloc(sizeof(uint32_t) * (size_t)(real ? real : 1), err)) return done(false);
    if (real) grid_split_kernel<<<(unsigned)((real + 255) / 256), 256>>>((const uint64_t*)keysB.p, real, N, (uint32_t*)list.p);
    out.total = real;
    e = cudaStreamSynchronize(0);
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        err = std::string("scene-grid builder: ") + cudaGetErrorString(e);
        return done(false);
    }
    return done(true);
}

// Same, from host arrays to malloc'ed host arrays (the drop-in form of the host builder).
bool build_scene_grid_device(int device, int32_t n, uint32_t V, const float4* vertex, uint32_t N, const int32_t* triIdx, float4** outBoxMin,
                             uint32_t** outStart, uint32_t** outList, size_t* outListSize, std::string& err) {
    if (n < 1 || (n & (n - 1)) || n > 1024) {
        err = "axesDivCount must be a power of two <= 1024";
        return false;
    }
    if (device < 0 || device >= device_count()) {
        err = "no such CUDA device: " + std::to_string(device);
        return false;
    }
    OCLR_CUDA(cudaSetDevice(device));
    prepare_pool(device);
    const size_t cells = (size_t)n * n * n;
    DeviceBuffer dVertex, dIdx;
    DeviceGrid grid;
    auto done = [&](bool ok) {
        dVertex.release();
        dIdx.release();
        grid.release();
        return ok;
    };
    if (!dVertex.upload(vertex, sizeof(float4) * V, err) || !dIdx.upload(triIdx, sizeof(int32_t) * 4 * (size_t)N, err)) return done(false);
    if (!grid_build_on_device(n, V, (const float4*)dVertex.p, N, (const int4*)dIdx.p, grid, err)) return done(false);
    const uint32_t real = grid.total;
    float4* hBox = (float4*)malloc(sizeof(float4) * (n + 1));
    uint32_t* hStart = (uint32_t*)malloc(sizeof(uint32_t) * (cells + 1));
    uint32_t* hList = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)(real ? real : 1));
    bool ok = hBox && hStart && hList;
    if (ok) {
        cudaError_t e = cudaMemcpy(hBox, grid.boxMin.p, sizeof(float4) * (n + 1), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(hStart, grid.start.p, sizeof(uint32_t) * (cells + 1), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && real) e = cudaMemcpy(hList, grid.list.p, sizeof(uint32_t) * (size_t)real, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            err = std::string("scene-grid builder: ") + cudaGetErrorString(e);
            ok = false;
        }
    } else {
        err = "out of host memory";
    }
    if (!ok) {
        free(hBox);
        free(hStart);
        free(hList);
        return done(false);
    }
    *outBoxMin = hBox;
    *outStart = hStart;
    *outList = hList;
    *outListSize = real;
    return done(true);
}

// Sharded upload (see ShardCtx): the calling thread is `rank` of ctx->world threads that run this same function for the same host
// arrays, one per GPU.  `arrays` lists the large arrays in two groups; buffers are allocated here, slice `rank` goes up over PCIe and
// is fanned out to the peers.  On return (true) the copies are ENQUEUED and the `pushed` events of this rank recorded; the caller
// makes its stream wait for a group with shard_wait_group().  Every rank passes both barriers whatever happens to it.
struct ShardBarriers {   // the two barriers of shard_upload, passed with `false` on scope exit by a rank that never got there
    ShardCtx* ctx;
    int left;
    explicit ShardBarriers(ShardCtx* c) : ctx(c), left(c ? 2 : 0) {}
    ~ShardBarriers() {
        while (left-- > 0) ctx->arrive(false);
    }
    bool arrive(bool ok) {
        --left;
        return ctx->arrive(ok);
    }
};
struct ShardArray {
    DeviceBuffer* buf;
    const void* host;
    size_t bytes;
    int group;
};
static bool shard_upload(ShardCtx* ctx, ShardBarriers& barriers, int rank, ShardArray* arrays, int count, std::string& err) {
    const int world = ctx->world;
    bool ok = count <= kShardArrays;
    // 1. carve the landing arena (256-byte aligned pieces: the fan-out moves whole 16-byte vectors), publish the addresses.  The arena
    //    is free: the previous call synchronised every GPU before it returned, and this call's peers write only after the barrier.
    size_t total = 0;
    for (int a = 0; a < count; ++a) total += (arrays[a].bytes + 255) & ~(size_t)255;
    LandingArena& arena = landing_arena(ctx->devices[rank]);
    if (ok && total > arena.bytes) {
        if (arena.p) {
            cudaDeviceSynchronize();
            cudaFree(arena.p);
        }
        arena.p = nullptr;
        arena.bytes = 0;
        const size_t want = total + total / 4;
        if (cudaMalloc((void**)&arena.p, want) != cudaSuccess) {
            cudaGetLastError();
            err = "out of device memory (shared-upload landing arena)";
            ok = false;
        } else {
            arena.bytes = want;
        }
    }
    size_t off = 0;
    for (int a = 0; ok && a < count; ++a) {
        arrays[a].buf->release();
        arrays[a].buf->p = arena.p + off;
        arrays[a].buf->bytes = arrays[a].bytes;
        arrays[a].buf->borrowed = true;
        ctx->ptr[a][rank] = arrays[a].buf->p;
        off += (arrays[a].bytes + 255) & ~(size_t)255;
    }
    ok = barriers.arrive(ok);
    // 2. own slices up, then out to the peers
    for (int g = 0; g < kShardGroups; ++g) {
        FanoutTable t = {};
        t.peers = world - 1;
        for (int a = 0; ok && a < count; ++a) {
            if (arrays[a].group != g || arrays[a].bytes == 0) continue;
            size_t b0, b1;
            shard_range(arrays[a].bytes, rank, world, b0, b1);
            if (b0 >= b1) continue;
            ok = host_to_device((char*)arrays[a].buf->p + b0, (const char*)arrays[a].host + b0, b1 - b0, 0, err);
            FanoutItem& it = t.it[t.items++];
            it.src = (const uint4*)((const char*)arrays[a].buf->p + b0);
            it.vecs = (b1 - b0 + 15) / 16;
            int k = 0;
            for (int d = 0; d < world; ++d)
                if (d != rank) it.dst[k++] = (uint4*)((char*)ctx->ptr[a][d] + b0);
        }
        if (ok && t.items) {
            int sms = 148;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->devices[rank]);
            fanout_kernel<<<sms * 4, 256>>>(t);
            if (cudaGetLastError() != cudaSuccess) {
                err = "fan-out launch failed";
                ok = false;
            }
        }
        if (ok && cudaEventRecord(ctx->pushed[g][rank], 0) != cudaSuccess) {
            err = "cudaEventRecord failed";
            ok = false;
        }
    }
    // 3. every rank's events are recorded before anybody waits on them (waiting on an unrecorded event is a no-op)
    ok = barriers.arrive(ok);
    if (!ok && err.empty()) err = "the upload failed on another GPU";
    return ok;
}
static bool shard_wait_group(ShardCtx* ctx, int group, std::string& err) {
    for (int d = 0; d < ctx->world; ++d) OCLR_CUDA(cudaStreamWaitEvent(0, ctx->pushed[group][d], 0));
    return true;
}
// Self-test of the shared upload (OCLR_SHARD_VERIFY=1): after the waits every array on this GPU must equal the caller's.
static bool shard_verify(int rank, const ShardArray* arrays, int count, int group, std::string& err) {
    static const bool on = [] { const char* v = getenv("OCLR_SHARD_VERIFY"); return v && atoi(v) != 0; }();
    if (!on) return true;
    OCLR_CUDA(cudaStreamSynchronize(0));
    for (int a = 0; a < count; ++a) {
        if (arrays[a].group != group || arrays[a].bytes == 0) continue;
        std::vector<unsigned char> back(arrays[a].bytes);
        OCLR_CUDA(cudaMemcpy(back.data(), arrays[a].buf->p, arrays[a].bytes, cudaMemcpyDeviceToHost));
        const unsigned char* want = (const unsigned char*)arrays[a].host;
        size_t bad = 0, first = 0;
        for (size_t i = 0; i < arrays[a].bytes; ++i)
            if (back[i] != want[i]) {
                if (!bad) first = i;
                ++bad;
            }
        fprintf(stderr, "[opencl_render_b200] shard verify: rank %d group %d array %d (%zu bytes): %zu bytes differ%s\n", rank, group, a,
                arrays[a].bytes, bad, bad ? (", first at " + std::to_string(first)).c_str() : "");
    }
    return true;
}

// ---- the stages of a scene build, shared by scene_create (scene_upload) and scene_update ------------------------------------------------
// Ring depth of a scene's paths and whether its normals read the camera, from the material tables (host arrays).
static void material_rules(const HostScene& h, int& ringSlots, bool& hasBump) {
    ringSlots = 2;
    for (uint32_t m = 0; m < h.materialCount && ringSlots == 2; ++m)
        for (int ch : {(int)kChReflection, (int)kChTransparency}) {
            // a channel that is present but black everywhere (the plugin's 1x1 fallback for "no reflection") spawns nothing either: the
            // segment multiplier is 0 < 3/256 (:684, :703).  Large maps are not scanned: taken as "may be non-zero"
            const uint2 size = h.matSize[kMaterialChannels * m + ch];
            const size_t texels = (size_t)size.x * size.y;
            if (texels == 0) continue;
            bool black = texels <= ((size_t)1 << 20);
            const uchar4* t = h.textures + h.matStart[kMaterialChannels * m + ch];
            for (size_t i = 0; black && i < texels; ++i) black = (t[i].x | t[i].y | t[i].z) == 0;
            if (!black) ringSlots = kRingSize;
        }
    if (const char* v = getenv("OCLR_RING_SLOTS")) ringSlots = std::max(ringSlots, std::min(atoi(v), (int)kRingSize));   // (test knob: more, never fewer)
    hasBump = false;
    for (uint32_t m = 0; m < h.materialCount; ++m) hasBump |= h.matSize[kMaterialChannels * m + kChBump].x > 0u;
}

static std::string pack_error_message(uint32_t flag) {
    return std::string("scene arrays are inconsistent:") + ((flag & kPackBadVertexIndex) ? " triangleVertexIndex out of range;" : "") +
           ((flag & kPackBadMaterial) ? " triangleMaterialId out of range;" : "") +
           ((flag & kPackBadCsr) ? " scenePixelTriangleListStart is not a monotone CSR;" : "") +
           ((flag & kPackBadListEntry) ? " scenePixelTriangleList entry out of range;" : "") +
           ((flag & kPackListTooLong) ? " a grid cell lists 131072 triangles or more (unsupported);" : "");
}

// The kernels' view of the scene's buffers, and the bytes they hold.
static void bind_view(Scene* s, uint32_t triangleCount, uint32_t materialCount, uint32_t lightCount, int n) {
    SceneView& v = s->view;
    v.triGeo = (const float4*)s->triGeo.p;
    v.triShade = (const float4*)s->triShade.p;
    v.bricks = (const uint4*)s->bricks.p;
    v.cellRange = (const uint2*)s->cellRange.p;
    v.cellList = (const uint32_t*)s->cellList.p;
    v.faceMask = (const uint32_t*)s->faceMask.p;
    v.planes = (const float*)s->planes.p;
    v.matSize = (const uint2*)s->matSize.p;
    v.matStart = (const int32_t*)s->matStart.p;
    v.textures = (const uchar4*)s->textures.p;
    v.lights = (const Light*)s->lights.p;
    v.triangleCount = triangleCount;
    v.materialCount = materialCount;
    v.lightCount = lightCount;
    v.n = n;
    v.nb = n >= 4 ? n / 4 : 1;
    s->walkView = v;
    if (s->walkTrim) {
        SceneView& w = s->walkView;
        w.bricks = (const uint4*)s->walkBricks.p;
        w.cellRange = (const uint2*)s->walkCellRange.p;
        w.faceMask = (const uint32_t*)s->walkFaceMask.p;
        w.planes = (const float*)s->walkPlanes.p;
        w.walkTrim = s->walkTrim;
    }
    s->bytes = 0;
    for (DeviceBuffer* b : s->buffers()) s->bytes += b->bytes;
}

// Triangles: raw reference arrays in device memory -> d->triGeo / d->triShade (pack_triangles_kernel; bad indices and material ids are
// or-ed into error[0]).  Enqueued on the default stream.
static bool pack_stage(Scene* d, uint32_t N, uint32_t V, uint32_t materialCount, const float4* vertex, const int4* triIdx, const int32_t* triMat,
                       const float2* triUv, const float4* triNormal, uint32_t* error, std::string& err) {
    if (!d->triGeo.alloc(sizeof(float4) * 4 * (size_t)N, err) || !d->triShade.alloc(sizeof(float4) * 8 * (size_t)N, err)) return false;
    if (N)
        pack_triangles_kernel<<<(N + 255) / 256, 256>>>(N, V, materialCount, vertex, triIdx, triMat, triUv, triNormal, (float4*)d->triGeo.p,
                                                        (float4*)d->triShade.p, error);
    return true;
}

// Bricks, ranges and face masks of one grid over the reference CSR -- the reference grid (map == nullptr) or a walk grid (map: see
// pack_kernels.cuh grid_ref_id) -- into bricks / cellRange / faceMask, behind `nSuper` zeroed super-brick records.  Synchronises the
// default stream once (the non-empty cell count sizes the ranges).
static bool pack_cells_on_device(int n, const uint32_t* gridStart, uint32_t total, const uint32_t* list, const int32_t* map, size_t nSuper,
                                 DeviceBuffer& bricks, DeviceBuffer& cellRange, DeviceBuffer& faceMask, uint32_t* error, std::string& err) {
    const int nb = n >= 4 ? n / 4 : 1;
    const size_t nBricks = (size_t)nb * nb * nb;
    DeviceBuffer counts, rankBase, scanTmp, cellIds;
    auto done = [&](bool ok) {
        for (DeviceBuffer* b : {&counts, &rankBase, &scanTmp, &cellIds}) b->release();
        return ok;
    };
    if (!bricks.alloc(sizeof(uint4) * (nBricks + nSuper), err) || !counts.alloc(sizeof(uint32_t) * (nBricks + 1), err) ||
        !rankBase.alloc(sizeof(uint32_t) * (nBricks + 1), err))
        return done(false);
    cudaMemsetAsync(counts.p, 0, sizeof(uint32_t) * (nBricks + 1), 0);
    brick_count_kernel<<<(unsigned)((nBricks + 127) / 128), 128>>>(gridStart, n, nb, total, map, (uint32_t*)counts.p, error);
    size_t tmpBytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, (const uint32_t*)counts.p, (uint32_t*)rankBase.p, (int)(nBricks + 1));
    if (!scanTmp.alloc(tmpBytes, err)) return done(false);
    cub::DeviceScan::ExclusiveSum(scanTmp.p, tmpBytes, (const uint32_t*)counts.p, (uint32_t*)rankBase.p, (int)(nBricks + 1));
    uint32_t nonEmpty = 0;
    cudaMemcpyAsync(&nonEmpty, (const uint32_t*)rankBase.p + nBricks, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) {
        err = std::string("scene repack: ") + cudaGetErrorString(e);
        return done(false);
    }
    if (nonEmpty >= (1u << 29)) {
        err = "too many non-empty grid cells (>= 2^29)";
        return done(false);
    }
    const size_t ne = nonEmpty ? nonEmpty : 1;
    if (!cellRange.alloc(sizeof(uint2) * ne, err) || !faceMask.alloc(sizeof(uint32_t) * 6 * ne, err) || !cellIds.alloc(sizeof(uint32_t) * ne, err))
        return done(false);
    brick_write_kernel<<<(unsigned)((nBricks + 127) / 128), 128>>>(gridStart, n, nb, total, map, (const uint32_t*)rankBase.p, (uint4*)bricks.p,
                                                                  (uint2*)cellRange.p, (uint32_t*)cellIds.p, error);
    if (nonEmpty)
        face_mask_kernel<<<(unsigned)(((size_t)nonEmpty * 6 + 255) / 256), 256>>>(gridStart, n, total, nonEmpty, map, (const uint32_t*)cellIds.p,
                                                                                 (const uint2*)cellRange.p, list, (uint32_t*)faceMask.p);
    else
        cudaMemsetAsync(faceMask.p, 0xFF, sizeof(uint32_t) * 6, 0);
    return done(true);   // (the temporaries are freed in stream order behind the kernels that read them)
}

// The grid: given in device memory (boxMin, gridStart and `total` list entries already in d->cellList), or built on the device at n cells
// per axis when gridStart is null; repacked into d->bricks / cellRange / faceMask / planes, and into the walk grid (rt_types.h) when
// a run of coincident planes collapses: the runs are found on the host from the planes, checked on the device (the grid may be the
// caller's), and the walk grid is packed on the device from the cell map of scene_pack.cpp walk_cell_map.  Enqueued on the default
// stream (the builder and the non-empty cell counts synchronise it); problems found on the device are or-ed into error[0], which
// error[1] must be free to use.
static bool grid_stage(Scene* d, int n, uint32_t V, const float4* vertex, uint32_t N, const int4* triIdx, const float4* boxMin,
                       const uint32_t* gridStart, uint32_t total, uint32_t* error, std::string& err) {
    // super-brick records of the three-level walk follow the brick records (rt_walk.h) -- in builds whose trace kernel has that level
    const int superPolicy = OCLR_SUPER_LEVEL ? super_policy(1) : 0;
    const int nb = n >= 4 ? n / 4 : 1;
    const int ns = superPolicy > 0 ? super_bricks_per_axis(n) : 0;
    const size_t nSuper = superPolicy > 0 ? super_brick_records(n) : 0;
    DeviceGrid grid;
    DeviceBuffer runsDev, differs, mapDev;
    auto done = [&](bool ok) {
        for (DeviceBuffer* b : {&grid.boxMin, &grid.start, &runsDev, &differs, &mapDev}) b->release();
        return ok;
    };
    if (!gridStart) {
        // the builder gathers vertices by index before the packer's check has been read: the indices are checked first
        if (N) check_indices_kernel<<<(N + 255) / 256, 256>>>(N, V, triIdx, error + 1);
        uint32_t bad = 0;
        OCLR_CUDA(cudaMemcpy(&bad, error + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost));
        if (bad) {
            err = "scene arrays are inconsistent: triangleVertexIndex out of range;";
            return false;
        }
        if (!grid_build_on_device(n, V, vertex, N, triIdx, grid, err)) return false;
        d->cellList.release();
        d->cellList = grid.list;   // handed over: the buffer an uploaded list would occupy
        grid.list = DeviceBuffer();
        boxMin = (const float4*)grid.boxMin.p;
        gridStart = (const uint32_t*)grid.start.p;
        total = grid.total;
    }
    if (!d->planes.alloc(sizeof(float) * 3 * (n + 1), err)) return done(false);
    split_planes_kernel<<<(n + 1 + 127) / 128, 128>>>(boxMin, n, (float*)d->planes.p);
    if (total) check_list_kernel<<<(total + 255) / 256, 256>>>((const uint32_t*)d->cellList.p, total, N, error);
    std::vector<float> planes(3 * (size_t)(n + 1));
    cudaMemcpyAsync(planes.data(), d->planes.p, sizeof(float) * planes.size(), cudaMemcpyDeviceToHost, 0);   // (read after the next sync)
    if (!pack_cells_on_device(n, gridStart, total, (const uint32_t*)d->cellList.p, nullptr, nSuper, d->bricks, d->cellRange, d->faceMask,
                              error, err))
        return done(false);
    if (nSuper) {
        cudaMemsetAsync((uint4*)d->bricks.p + (size_t)nb * nb * nb, 0, sizeof(uint4) * nSuper, 0);
        super_brick_kernel<<<(unsigned)(ns * ns * ns), 64>>>((uint4*)d->bricks.p, nb, ns);
    }
    // the walk grid
    for (DeviceBuffer* b : {&d->walkBricks, &d->walkCellRange, &d->walkFaceMask, &d->walkPlanes}) b->release();
    d->walkTrim = 0;
    const std::vector<WalkRun> runs = walk_runs(planes.data(), n);
    if (runs.empty()) return done(true);
    std::vector<int3> runs3(runs.size());
    for (size_t i = 0; i < runs.size(); ++i) runs3[i] = make_int3(runs[i].axis, runs[i].first, runs[i].count);
    if (!runsDev.upload(runs3.data(), sizeof(int3) * runs3.size(), err) || !differs.alloc(sizeof(uint32_t) * runs.size(), err)) return done(false);
    cudaMemsetAsync(differs.p, 0, sizeof(uint32_t) * runs.size(), 0);
    run_check_kernel<<<dim3((unsigned)(((size_t)n * n + 255) / 256), (unsigned)runs.size()), 256>>>(
        gridStart, (const uint32_t*)d->cellList.p, n, total, (const int3*)runsDev.p, (uint32_t*)differs.p);
    std::vector<uint32_t> differ(runs.size());
    cudaMemcpyAsync(differ.data(), differs.p, sizeof(uint32_t) * runs.size(), cudaMemcpyDeviceToHost, 0);
    uint32_t packErrors = 0;   // a grid the packers flagged (bad CSR, ...) is refused by the caller: no walk grid is built over it
    cudaMemcpyAsync(&packErrors, error, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) {
        err = std::string("scene repack: ") + cudaGetErrorString(e);
        return done(false);
    }
    if (packErrors) return done(true);
    std::vector<uint8_t> collapses(runs.size());
    bool any = false;
    for (size_t i = 0; i < runs.size(); ++i) any |= (collapses[i] = differ[i] ? 0 : 1) != 0;
    if (!any) return done(true);
    std::vector<int32_t> map;
    const uint32_t trim = walk_cell_map(n, runs, collapses, map);
    if (!trim) return done(true);   // the padding kept every cell again
    std::vector<float> wplanes(planes.size());
    walk_planes(planes.data(), n, map.data(), wplanes.data());
    if (!mapDev.upload(map.data(), sizeof(int32_t) * map.size(), err) || !d->walkPlanes.upload(wplanes.data(), sizeof(float) * wplanes.size(), err) ||
        !pack_cells_on_device(n, gridStart, total, (const uint32_t*)d->cellList.p, (const int32_t*)mapDev.p, 0, d->walkBricks, d->walkCellRange,
                              d->walkFaceMask, error, err))
        return done(false);
    d->walkTrim = trim;
    return done(true);
}

static bool scene_upload(Scene* s, const HostScene& h, std::string& err, const std::function<void(Scene*)>* early, UploadShare* share) {
    ShardCtx* ctx = share ? share->ctx : nullptr;
    ShardBarriers barriers(ctx);   // (any early return below still passes the barriers the other GPUs' threads wait at)
    OCLR_CUDA(cudaSetDevice(s->device));
    int major = 0, minor = 0, sms = 0;   // attribute queries: cudaGetDeviceProperties costs milliseconds per call
    OCLR_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, s->device));
    OCLR_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, s->device));
    OCLR_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, s->device));
    if (major != 10) {   // the library holds sm_100a SASS only (arch-specific: no PTX fallback for sm_12x either)
        err = "this library is built for sm_100a (B200) only; device is sm_" + std::to_string(major) + std::to_string(minor);
        return false;
    }
    s->smCount = sms;
    prepare_pool(s->device);
    stage_reset(s->device);   // (every earlier staged copy of this device has completed: the calls that made them synchronise)
    if (!validate_scene(h, err, true)) return false;
    const bool buildGrid = !h.gridStart;   // no grid given: SceneTriangleList::New runs on the device (grid_builder.cuh)

    const size_t N = h.triangleCount;
    const int n = h.axesDivCount;
    const size_t cells = (size_t)n * n * n;
    // ring depth of this scene's paths (host data only, and decided before the early hook below starts a frame on the scene)
    material_rules(h, s->ringSlots, s->hasBump);
    uint32_t total = buildGrid ? 0u : h.gridStart[cells];
    if (total && !h.gridList) {
        err = "scenePixelTriangleList missing";
        return false;
    }
    std::vector<Light> lights;
    pack_lights(h, lights);

    // 1a. everything the primary-ray round needs -- triangles, materials, lights -- goes first: raw reference arrays -> HBM straight
    //     from the caller's memory (async on the default stream), repacked by pack_triangles_kernel
    DeviceBuffer vertex, triIdx, triMat, triUv, triNormal, boxMin, gridStart, errFlag;
    std::vector<ShardArray> sharded;   // (kept for the self-test of the second group)
    bool ok;
    if (ctx) {
        // one of N GPUs uploading the same arrays: slice + fan-out for the large ones (group 0 = what the triangle repack and the
        // primary-ray round need, the camera lists included; group 1 = the grid), the small tables go up whole
        DeviceBuffer camStart, camEnd, camList;
        const size_t P = share->pixels;
        ShardArray arrays[] = {
            {&vertex, h.vertex, sizeof(float4) * h.vertexCount, 0},
            {&triIdx, h.triIdx, sizeof(int4) * N, 0},
            {&triMat, h.triMat, sizeof(int32_t) * N, 0},
            {&triUv, h.triUv, sizeof(float2) * 3 * N, 0},
            {&triNormal, h.triNormal, sizeof(float4) * 3 * N, 0},
            {&s->textures, h.textures, sizeof(uchar4) * h.texturesSize, 0},
            {&camStart, share->camStart, share->camStart ? sizeof(uint32_t) * P : 0, 0},
            {&camEnd, share->camEnd, share->camStart ? sizeof(uint32_t) * P : 0, 0},
            {&camList, share->camList, share->camStart ? sizeof(uint32_t) * share->camListSize : 0, 0},
            {&gridStart, h.gridStart, buildGrid ? 0 : sizeof(uint32_t) * (cells + 1), 1},
            {&s->cellList, h.gridList, buildGrid ? 0 : sizeof(uint32_t) * total, 1},
        };
        ok = shard_upload(ctx, barriers, share->rank, arrays, (int)(sizeof(arrays) / sizeof(arrays[0])), err);
        if (share->camStart) {   // handed to the frame (frame_create adopts them); no lists given: the frame builds its own on the device
            share->staged.start = camStart.p;
            share->staged.end = camEnd.p;
            share->staged.list = camList.p;
            share->staged.listSize = share->camListSize;
            share->staged.borrowed = camStart.borrowed;
        }
        ok = ok && s->matSize.upload(h.matSize, sizeof(uint2) * kMaterialChannels * h.materialCount, err) &&
             s->matStart.upload(h.matStart, sizeof(int32_t) * (kMaterialChannels * h.materialCount + (h.materialCount ? 1 : 0)), err) &&
             s->lights.upload(lights.data(), sizeof(Light) * lights.size(), err) &&
             (buildGrid || boxMin.upload(h.boxMin, sizeof(float4) * (n + 1), err)) && shard_wait_group(ctx, 0, err);
        sharded.assign(arrays, arrays + sizeof(arrays) / sizeof(arrays[0]));
        ok = ok && shard_verify(share->rank, sharded.data(), (int)sharded.size(), 0, err);
    } else {
        ok = vertex.upload(h.vertex, sizeof(float4) * h.vertexCount, err) && triIdx.upload(h.triIdx, sizeof(int4) * N, err) &&
             triMat.upload(h.triMat, sizeof(int32_t) * N, err) && triUv.upload(h.triUv, sizeof(float2) * 3 * N, err) &&
             triNormal.upload(h.triNormal, sizeof(float4) * 3 * N, err) &&
             s->matSize.upload(h.matSize, sizeof(uint2) * kMaterialChannels * h.materialCount, err) &&
             s->matStart.upload(h.matStart, sizeof(int32_t) * (kMaterialChannels * h.materialCount + (h.materialCount ? 1 : 0)), err) &&
             s->textures.upload(h.textures, sizeof(uchar4) * h.texturesSize, err) &&
             s->lights.upload(lights.data(), sizeof(Light) * lights.size(), err);
    }
    ok = ok && errFlag.alloc(sizeof(uint32_t) * 2, err);
    if (ok) {
        cudaMemsetAsync(errFlag.p, 0, sizeof(uint32_t) * 2, 0);
        ok = pack_stage(s, (uint32_t)N, h.vertexCount, h.materialCount, (const float4*)vertex.p, (const int4*)triIdx.p, (const int32_t*)triMat.p,
                        (const float2*)triUv.p, (const float4*)triNormal.p, (uint32_t*)errFlag.p, err);
    }
    if (ok) {
        bind_view(s, h.triangleCount, h.materialCount, h.lightCount, n);   // the logic kernel's part (the grid part is bound again below)
        // RaytraceAll uploads its camera lists and starts the primary-ray round HERE, on a stream of its own, so that round runs
        // under the upload of the grid (94 of config 2's 133 MB) instead of after it
        if (early && *early) (*early)(s);
    }
    // 1b. the grid
    ok = ok && (buildGrid || (ctx ? (shard_wait_group(ctx, 1, err) && shard_verify(share->rank, sharded.data(), (int)sharded.size(), 1, err))
                                  : (boxMin.upload(h.boxMin, sizeof(float4) * (n + 1), err) &&
                                     gridStart.upload(h.gridStart, sizeof(uint32_t) * (cells + 1), err) &&
                                     s->cellList.upload(h.gridList, sizeof(uint32_t) * total, err))));
    // 2. repack on the device
    ok = ok && grid_stage(s, n, h.vertexCount, (const float4*)vertex.p, (uint32_t)N, (const int4*)triIdx.p, (const float4*)boxMin.p,
                          (const uint32_t*)gridStart.p, total, (uint32_t*)errFlag.p, err);
    uint32_t flag = 0;
    if (ok) cudaMemcpyAsync(&flag, errFlag.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    cudaError_t e = cudaStreamSynchronize(0);
    DeviceBuffer* tmp[] = {&vertex, &triIdx, &triMat, &triUv, &triNormal, &boxMin, &gridStart, &errFlag};
    for (DeviceBuffer* b : tmp) b->release();
    if (!ok) return false;
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        err = std::string("scene upload: ") + cudaGetErrorString(e);
        return false;
    }
    if (flag) {
        err = pack_error_message(flag);
        return false;
    }
    bind_view(s, h.triangleCount, h.materialCount, h.lightCount, n);
    return true;
}

Scene* scene_create(int device, const HostScene& h, std::string& err, const std::function<void(Scene*)>* early, UploadShare* share) {
    if (device < 0 || device >= device_count()) {
        err = "no such CUDA device: " + std::to_string(device) + " (the library has no CPU fallback)";
        ShardBarriers barriers(share ? share->ctx : nullptr);
        return nullptr;
    }
    Scene* s = new Scene();
    s->device = device;
    if (!scene_upload(s, h, err, early, share)) {
        cudaDeviceSynchronize();   // the `early` hook may have started work on another stream that still reads this scene
        scene_destroy(s);
        return nullptr;
    }
    return s;
}

void scene_destroy(Scene* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    for (DeviceBuffer* b : s->buffers()) b->release();
    delete s;
}

size_t scene_device_bytes(const Scene* s) { return s->bytes; }
// Wavefront path state a frame holds in HBM (all slices: ring, carry, ray / hit slots, walk records, queue) -- what a launch domain
// of `capacity` paths costs; 0 before the first render.
size_t frame_state_bytes(Frame* f) {
    size_t n = 0;
    for (WfSlice& sl : f->slices) {
        n += sl.ps.bytes();
        for (DeviceBuffer* b : sl.tail_buffers()) n += b->bytes;
    }
    return n;
}

// Debug/test door: copies one packed device array back (0 triGeo, 1 triShade, 2 bricks, 3 cellRange, 4 planes, 5 cellList, 6 faceMask;
// the walk grid: 7 bricks, 8 cellRange, 9 faceMask, 10 planes -- empty when the scene walks the reference grid -- and 11 its extents,
// three uint32).
size_t scene_debug_read(Scene* s, int which, void* dst, size_t cap) {
    DeviceBuffer* all[] = {&s->triGeo, &s->triShade, &s->bricks, &s->cellRange, &s->planes, &s->cellList, &s->faceMask,
                           &s->walkBricks, &s->walkCellRange, &s->walkFaceMask, &s->walkPlanes};
    if (which == 11) {
        const uint32_t ext[3] = {s->view.n - ((s->walkTrim) & 1023u), s->view.n - ((s->walkTrim >> 10) & 1023u), s->view.n - ((s->walkTrim >> 20) & 1023u)};
        if (dst && cap >= sizeof(ext)) memcpy(dst, ext, sizeof(ext));
        return sizeof(ext);
    }
    if (which < 0 || which > 10) return 0;
    cudaSetDevice(s->device);
    const size_t n = all[which]->bytes;
    if (dst && n && n <= cap) cudaMemcpy(dst, all[which]->p, n, cudaMemcpyDeviceToHost);
    return n;
}
int scene_device(const Scene* s) { return s->device; }

static bool frame_setup_common(Frame* f, std::string& err, bool sync = true) {
    const size_t P = (size_t)f->cam.width * f->cam.height;
    if (!f->planesRGB.alloc(sizeof(uint16_t) * 3 * P, err)) return false;
    if (!f->ids.alloc(sizeof(uint32_t) * P, err)) return false;
    if (!f->flags.alloc(sizeof(uint8_t) * P, err)) return false;
    OCLR_CUDA(cudaMemsetAsync(f->flags.p, 0, f->flags.bytes, 0));
    if (!f->counters.alloc(sizeof(Counters), err)) return false;
    if (!f->doneCount.alloc(sizeof(unsigned long long), err)) return false;
    OCLR_CUDA(cudaMemsetAsync(f->doneCount.p, 0, sizeof(unsigned long long), 0));
    f->hostDone = (unsigned long long*)pinned_block();
    if (!f->hostDone) {
        err = "out of pinned host memory";
        return false;
    }
    OCLR_CUDA(cudaMemsetAsync(f->planesRGB.p, 0, f->planesRGB.bytes, 0));
    OCLR_CUDA(make_event(f->device, &f->ev0, true));
    OCLR_CUDA(make_event(f->device, &f->ev1, true));
    OCLR_CUDA(make_event(f->device, &f->evFork, false));
    if (sync) OCLR_CUDA(cudaStreamSynchronize(0));
    return true;
}

// Caller-supplied (or staged) camera lists into the frame, range-checked on the device.
static bool frame_upload_lists(Frame* f, const uint32_t* camStart, const uint32_t* camEnd, const uint32_t* camList, size_t listSize,
                               std::string& err, StagedCamLists* staged) {
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    const size_t P = (size_t)f->cam.width * f->cam.height;
    if (staged && staged->start && !staged->adopted) {   // already in HBM (uploaded together with the scene, shard_upload)
        staged->adopted = true;
        f->camStart.p = staged->start;
        f->camStart.bytes = sizeof(uint32_t) * P;
        f->camEnd.p = staged->end;
        f->camEnd.bytes = sizeof(uint32_t) * P;
        f->camList.p = staged->list;
        f->camList.bytes = sizeof(uint32_t) * staged->listSize;
        f->camStart.borrowed = f->camEnd.borrowed = f->camList.borrowed = staged->borrowed;
        listSize = staged->listSize;
    } else {
        if (!camStart || !camEnd || (listSize && !camList)) {
            err = "camera triangle lists missing";
            return false;
        }
        if (!f->camStart.upload(camStart, sizeof(uint32_t) * P, err)) return false;
        if (!f->camEnd.upload(camEnd, sizeof(uint32_t) * P, err)) return false;
        if (!f->camList.upload(camList, sizeof(uint32_t) * listSize, err)) return false;
    }
    f->camListSize = listSize;
    if (listSize > 0xFFFFFFFFull) {
        err = "camera triangle list too long";
        return false;
    }
    // range check on the device, stream-ordered in front of every kernel that reads the lists (no host round trip: the kernels look
    // at the flag themselves, the host reports it at its next synchronisation -- launch_wavefront / frame_launch)
    if (!f->camCheck.alloc(sizeof(uint32_t), err)) return false;
    OCLR_CUDA(cudaMemsetAsync(f->camCheck.p, 0, sizeof(uint32_t), 0));
    check_camera_lists_kernel<<<(unsigned)std::min<size_t>((std::max(P, listSize) + 255) / 256, (size_t)f->scene->smCount * 8), 256>>>(
        (const uint32_t*)f->camStart.p, (const uint32_t*)f->camEnd.p, (const uint32_t*)f->camList.p, (uint32_t)P, (uint32_t)listSize,
        f->scene->view.triangleCount, (uint32_t*)f->camCheck.p);
    f->deviceLists = false;
    f->listsGen = f->scene->geometryGen;
    return true;
}

// CameraTriangleList::New on the device (cam_builder.cuh): the frame's camera lists are built from the resident scene.
static bool frame_build_camera_lists(Frame* f, std::string& err) {
    Scene* s = f->scene;
    OCLR_CUDA(cudaSetDevice(s->device));
    for (DeviceBuffer* b : {&f->camStart, &f->camEnd, &f->camList, &f->camCheck}) b->release();   // (a rebuild: the old lists go)
    f->camListSize = 0;
    f->deviceLists = true;
    f->listsGen = kNoLists;
    const uint32_t W = f->cam.width, H = f->cam.height, N = s->view.triangleCount;
    const uint32_t P = W * H;
    if ((uint64_t)W * H >= 0xFFFFFFFFull) {
        err = "image too large for the device camera-list builder";
        return false;
    }
    CamProjD c;
    c.eye = mk3(f->cam.eye);
    c.tl = mk3(f->cam.eyeToTopLeft);
    c.lr = mk3(f->cam.leftToRight);
    c.tb = mk3(f->cam.topToBottom);
    c.screenN = cross3(c.lr, c.tb);        // host arithmetic, g++/nvcc host side with -ffp-contract=off like builders.cpp
    c.tlDotN = dot3(c.tl, c.screenN);
    c.psiSq = f->cam.pixelSizeInv * f->cam.pixelSizeInv;
    c.W = W;
    c.H = H;
    DeviceBuffer screen, slots, offsets, largeList, small, keysA, keysB, pixelCount, startInc, tmp, listRaw, parent, keptLen, keptStart;
    DeviceBuffer* all[] = {&screen, &slots, &offsets, &largeList, &small, &keysA, &keysB, &pixelCount, &startInc, &tmp, &listRaw, &parent, &keptLen, &keptStart};
    auto done = [&](bool ok) {
        for (DeviceBuffer* b : all) b->release();
        return ok;
    };
    const size_t Nz = N ? N : 1;
    if (!screen.alloc(sizeof(TriScreen) * Nz, err) || !slots.alloc(sizeof(uint64_t) * (Nz + 1), err) ||
        !offsets.alloc(sizeof(uint64_t) * (Nz + 1), err) || !largeList.alloc(sizeof(uint32_t) * Nz, err) ||
        !small.alloc(sizeof(uint32_t) * 4, err) || !pixelCount.alloc(sizeof(uint32_t) * ((size_t)P + 1), err) ||
        !startInc.alloc(sizeof(uint32_t) * ((size_t)P + 1), err))
        return done(false);
    cudaMemsetAsync(small.p, 0, sizeof(uint32_t) * 4, 0);
    cudaMemsetAsync(slots.p, 0, sizeof(uint64_t) * (Nz + 1), 0);
    cudaMemsetAsync(pixelCount.p, 0, sizeof(uint32_t) * ((size_t)P + 1), 0);
    uint32_t* largeCount = (uint32_t*)small.p;
    if (N)
        cam_project_kernel<<<(N + 255) / 256, 256>>>(c, N, s->view.triShade, (TriScreen*)screen.p, (uint64_t*)slots.p, (uint32_t*)largeList.p,
                                                    largeCount);
    size_t tmpBytes = 0, need = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, need, (const uint64_t*)slots.p, (uint64_t*)offsets.p, (int)(N + 1));
    tmpBytes = need;
    cub::DeviceScan::ExclusiveSum(nullptr, need, (const uint32_t*)pixelCount.p, (uint32_t*)startInc.p, (int)(P + 1));
    tmpBytes = std::max(tmpBytes, need);
    if (!tmp.alloc(tmpBytes, err)) return done(false);
    cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, (const uint64_t*)slots.p, (uint64_t*)offsets.p, (int)(N + 1));
    uint64_t total = 0;
    uint32_t nLarge = 0;
    cudaMemcpyAsync(&total, (const uint64_t*)offsets.p + N, sizeof(uint64_t), cudaMemcpyDeviceToHost, 0);
    cudaMemcpyAsync(&nLarge, largeCount, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    OCLR_CUDA(cudaStreamSynchronize(0));
    if (total > (1ull << 31)) {
        err = "camera-list builder: more than 2^31 (triangle, pixel) candidates";
        return done(false);
    }
    const size_t totalZ = total ? (size_t)total : 1;
    if (!keysA.alloc(sizeof(uint64_t) * totalZ, err) || !keysB.alloc(sizeof(uint64_t) * totalZ, err)) return done(false);
    const uint64_t sentinel = (uint64_t)P * (uint64_t)(N ? N : 1);
    if (N) {
        cam_raster_small_kernel<<<(N + 127) / 128, 128>>>(N, W, sentinel, (const TriScreen*)screen.p, (const uint64_t*)offsets.p,
                                                         (uint64_t*)keysA.p, (uint32_t*)pixelCount.p);
        if (nLarge)
            cam_raster_large_kernel<<<dim3(nLarge, 32), 256>>>(N, W, sentinel, (const TriScreen*)screen.p, (const uint64_t*)offsets.p,
                                                              (const uint32_t*)largeList.p, (uint64_t*)keysA.p, (uint32_t*)pixelCount.p);
    }
    cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, (const uint32_t*)pixelCount.p, (uint32_t*)startInc.p, (int)(P + 1));
    uint32_t real = 0;
    cudaMemcpyAsync(&real, (const uint32_t*)startInc.p + P, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    int endBit = 1;
    while (endBit < 64 && (sentinel >> endBit) != 0) ++endBit;
    size_t sortBytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, sortBytes, (const uint64_t*)keysA.p, (uint64_t*)keysB.p, (int64_t)total, 0, endBit);
    DeviceBuffer sortTmp;
    if (!sortTmp.alloc(sortBytes, err)) return done(false);
    cub::DeviceRadixSort::SortKeys(sortTmp.p, sortBytes, (const uint64_t*)keysA.p, (uint64_t*)keysB.p, (int64_t)total, 0, endBit);
    cudaError_t e = cudaStreamSynchronize(0);
    sortTmp.release();
    if (e != cudaSuccess) {
        err = std::string("camera-list builder: ") + cudaGetErrorString(e);
        return done(false);
    }
    const size_t realZ = real ? real : 1;
    if (!listRaw.alloc(sizeof(uint32_t) * realZ, err) || !parent.alloc(sizeof(uint32_t) * (size_t)P, err) ||
        !keptLen.alloc(sizeof(uint32_t) * ((size_t)P + 1), err) || !keptStart.alloc(sizeof(uint32_t) * ((size_t)P + 1), err))
        return done(false);
    if (real) cam_split_kernel<<<(unsigned)((real + 255) / 256), 256>>>((const uint64_t*)keysB.p, real, N, (uint32_t*)listRaw.p);
    // storage compression against the left / upper neighbour
    cudaMemsetAsync(keptLen.p, 0, sizeof(uint32_t) * ((size_t)P + 1), 0);
    cam_equal_kernel<<<(P + 255) / 256, 256>>>(W, P, (const uint32_t*)startInc.p, (const uint32_t*)listRaw.p, (uint32_t*)parent.p,
                                              (uint32_t*)keptLen.p);
    cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, (const uint32_t*)keptLen.p, (uint32_t*)keptStart.p, (int)(P + 1));
    uint32_t kept = 0;
    cudaMemcpyAsync(&kept, (const uint32_t*)keptStart.p + P, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    int jumps = 1;
    while ((1u << jumps) < W + H) ++jumps;
    for (int k = 0; k < jumps; ++k) cam_jump_kernel<<<(P + 255) / 256, 256>>>(P, (uint32_t*)parent.p, largeCount + 1);
    OCLR_CUDA(cudaStreamSynchronize(0));
    if (!f->camStart.alloc(sizeof(uint32_t) * (size_t)P, err) || !f->camEnd.alloc(sizeof(uint32_t) * (size_t)P, err) ||
        !f->camList.alloc(sizeof(uint32_t) * (size_t)(kept ? kept : 1), err))
        return done(false);
    cam_finish_kernel<<<(P + 255) / 256, 256>>>(P, (const uint32_t*)startInc.p, (const uint32_t*)parent.p, (const uint32_t*)keptStart.p,
                                               (const uint32_t*)listRaw.p, (uint32_t*)f->camStart.p, (uint32_t*)f->camEnd.p,
                                               (uint32_t*)f->camList.p);
    f->camListSize = kept;
    e = cudaStreamSynchronize(0);
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        err = std::string("camera-list builder: ") + cudaGetErrorString(e);
        return done(false);
    }
    f->listsGen = s->geometryGen;
    return done(true);
}

// Lists for the scene's current geometry, before anything reads them: device-built lists are rebuilt after a geometry edit; caller
// lists made for older geometry may name triangles that no longer exist, so the frame refuses until it is given new ones.
static bool frame_lists_current(Frame* f, std::string& err) {
    if (f->listsGen == f->scene->geometryGen) return true;
    if (f->deviceLists) return frame_build_camera_lists(f, err);
    err = f->listsGen == kNoLists ? "the frame has no camera triangle lists (its last camera change failed): set a camera again"
                                  : "the scene's geometry changed since the frame's camera triangle lists were made: give the frame new lists "
                                    "(oclr_frame_set_camera_lists) or let the device build them (oclr_frame_set_camera)";
    return false;
}

void staged_release(StagedCamLists& st) {
    if (st.adopted || st.borrowed) return;
    if (st.start) cudaFreeAsync(st.start, 0);
    if (st.end) cudaFreeAsync(st.end, 0);
    if (st.list) cudaFreeAsync(st.list, 0);
    st = StagedCamLists();
}

Frame* frame_create(Scene* s, const Camera& cam, const uint32_t* camStart, const uint32_t* camEnd, const uint32_t* camList,
                    size_t camListSize, std::string& err, bool sync, StagedCamLists* staged) {
    if (!s) {
        err = "null scene";
        return nullptr;
    }
    if (cam.width == 0 || cam.height == 0 || (uint64_t)cam.width * cam.height > 0xFFFFFFFFull) {
        err = "bad image dimension";
        return nullptr;
    }
    Frame* f = new Frame();
    f->scene = s;
    f->device = s->device;
    f->cam = cam;
    const bool ok = (camStart || (staged && staged->start))
                        ? frame_upload_lists(f, camStart, camEnd, camList, camListSize, err, staged) && frame_setup_common(f, err, sync)
                        : (frame_build_camera_lists(f, err) && frame_setup_common(f, err));   // no lists given: build them on the device
    if (!ok) {
        frame_destroy(f);
        return nullptr;
    }
    return f;
}

size_t frame_camera_list_size(Frame* f) {
    std::string ignored;   // (frame_read_camera_lists reports why stale lists cannot be read)
    return f && frame_lists_current(f, ignored) ? f->camListSize : 0;
}

bool frame_read_camera_lists(Frame* f, uint32_t* start, uint32_t* end, uint32_t* list, std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    if (!frame_lists_current(f, err)) return false;
    const size_t P = (size_t)f->cam.width * f->cam.height;
    OCLR_CUDA(cudaMemcpy(start, f->camStart.p, sizeof(uint32_t) * P, cudaMemcpyDeviceToHost));
    OCLR_CUDA(cudaMemcpy(end, f->camEnd.p, sizeof(uint32_t) * P, cudaMemcpyDeviceToHost));
    if (f->camListSize) OCLR_CUDA(cudaMemcpy(list, f->camList.p, sizeof(uint32_t) * f->camListSize, cudaMemcpyDeviceToHost));
    return true;
}

void frame_destroy(Frame* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    if (f->prelaunched && f->preDone) cudaEventSynchronize(f->preDone);   // a round started ahead that no render call picked up
    DeviceBuffer* all[] = {&f->camStart, &f->camEnd, &f->camList, &f->planesRGB, &f->ids, &f->flags, &f->counters, &f->accum, &f->doneCount,
                           &f->camCheck};
    for (DeviceBuffer* b : all) b->release();
    drop_stream(f->device, f->progStream);
    pinned_release(f->hostDone);
    drop_stream(f->device, f->preStream);
    drop_event(f->device, f->preReady, false);
    drop_event(f->device, f->preDone, false);
    for (WfSlice& sl : f->slices) {
        sl.ps.release(0);
        for (DeviceBuffer* b : sl.tail_buffers()) b->release();
        drop_stream(f->device, sl.stream);
        drop_event(f->device, sl.done, false);
        for (cudaEvent_t e : sl.traceEvents) drop_event(f->device, e, true);
    }
    pinned_release(f->hostCount);
    drop_event(f->device, f->ev0, true);
    drop_event(f->device, f->ev1, true);
    drop_event(f->device, f->evFork, false);
    delete f;
}

uint32_t band_owned_rows(uint32_t height, uint32_t bandRows, uint32_t rank, uint32_t world) {
    if (world <= 1) return height;
    uint32_t owned = 0;
    for (uint32_t b0 = rank * bandRows; b0 < height; b0 += bandRows * world) owned += (b0 + bandRows <= height) ? bandRows : height - b0;
    return owned;
}

// Slices of a launch domain.  The trace kernel is a persistent grid that owns every SM; the end of each launch is a tail in which
// a few long walks keep a few warps busy (profiles/README.md), and the logic kernel between two trace launches is latency-bound.
// The domain is therefore cut into slices -- sub-band sets of the rows -- with their own path state, queue counters and stream:
// the rounds of one slice are still strictly ordered, but the CTAs of another slice's kernels move into the SMs a draining
// launch gives up.  Pixels are independent, so the cut is invisible in the output.
// Measured (B200, gpurun_out/slices*.log): config 3 (8.3 M paths) 24.4 -> 23.7 ms with 2 slices, flat to 4, worse at 8; config 2
// (2.1 M paths) 4.51 ms with 1 or 2 slices and slower beyond -- every slice's launches end in their own partly filled warps, which
// costs what the overlap wins.  Default: one slice per 3 M paths, at most 4 (OCLR_SLICES=k forces k; round 2: config 3, 8.3 M paths, 23.5 -> 22.8 ms with 2).
// Tracing one round ahead (rt_wavefront.cuh): 0 never, 1 for every segment but the camera's, 2 for all.  -1 = automatic.
static std::atomic<int> g_aheadMode(-2);
void set_ahead_mode(int m) { g_aheadMode.store(m < -1 || m > 2 ? -1 : m); }
static int ahead_mode_for(uint32_t paths) {
    if (g_aheadMode.load() == -2) {
        const char* v = getenv("OCLR_AHEAD");
        set_ahead_mode(v ? atoi(v) : -1);
    }
    const int m = g_aheadMode.load();
    if (m >= 0) return m;
    // Measured on a B200 (scripts/ahead_probe.py, gpurun_out/ahead_probe*.log): config 2, 2.07 M paths: 4.54 / 4.54 / 4.52 ms for
    // modes 0 / 1 / 2; its 1/8 band share 1.28 / 1.26 / 0.97 ms (two latency floors instead of three); config 3, 8.3 M paths:
    // 24.7 / 24.7 / 25.4 ms (shadow and bounce rays of 8 M paths in one launch thrash the L2-resident working set); the mirror
    // chains of config 5 need 48 launches per frame instead of 90 with mode 1 or 2 (27 -> 12 ms per frame).
    return paths < 3000000u ? 2 : 1;
}

// Shadow rays of lights on the side of the surface the segment does not see (rt_wavefront.cuh, GO_LIGHTS): skipped (1, default) or traced
// like the reference (0).  The planes are the same either way; 0 is for A/B runs.
static std::atomic<bool> g_cullHidden(true);
void set_cull_hidden_lights(int on) { g_cullHidden.store(on != 0); }

static std::atomic<int> g_sliceCount(-1);   // -1: not yet read from OCLR_SLICES; 0: automatic
void set_slice_count(int k) { g_sliceCount.store(std::max(0, std::min(k, (int)kMaxSlices))); }
static int slice_count_for(uint32_t rows, uint32_t width) {
    if (g_sliceCount.load() < 0) {
        const char* v = getenv("OCLR_SLICES");
        set_slice_count(v ? atoi(v) : 0);
    }
    const int forced = g_sliceCount.load();
    if (forced) return forced;
    const uint64_t paths = (uint64_t)rows * width;
    return (int)std::min<uint64_t>(4, std::max<uint64_t>(1, paths / (3ull << 20)));   // (config 3's 8.3 M paths: 2 slices, 23.5 -> 22.8 ms)
}

static bool same_request(const FrameView& a, const FrameView& b);
static std::string cam_check_message(uint32_t flag);
// A round started ahead by frame_prelaunch is continued only by the identical request rendered as ONE slice (the only case started
// ahead).  frame_launch and launch_wavefront both decide with this, so the progress counter and the round agree.
static int slice_count_for(uint32_t rows, uint32_t width);
static bool resumes_prelaunch(const Frame* f, const FrameView& F);

// ---- the trace stage (rt_trace.cuh), shared by frames and ray queries --------------------------------------------------------------
// Scheduling knobs of wf_pipe_kernel.
static const TraceTuning& trace_tuning() {
    // (function-local static built by a lambda: initialised once, thread-safe -- RaytraceAll's all-devices mode launches from one
    // host thread per GPU)
    static const TraceTuning tune = [] {
        auto env = [](const char* k, int d) { const char* v = getenv(k); return v && atoi(v) > 0 ? atoi(v) : d; };
        TraceTuning t = {0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 1, 16, 12};
        t.refillMin = env("OCLR_REFILL_MIN", 4);
        t.hierarchical = getenv("OCLR_HIERARCHICAL") ? atoi(getenv("OCLR_HIERARCHICAL")) : 2;
        t.drainMin = std::min(env("OCLR_DRAIN_MIN", 64), (int)kCellQCap - 31);   // (round 2 sweep: 64 is ~1 % faster than 48 on configs 2 and 3)
        t.walkMin3 = env("OCLR_WALK_MIN3", 8);
        t.switchMin = env("OCLR_SWITCH_MIN", 6);
        t.tailDrain = env("OCLR_TAIL_DRAIN", 8);
        t.splitMin = getenv("OCLR_SPLIT_MIN") ? atoi(getenv("OCLR_SPLIT_MIN")) : 0;   // 0: never cut a walk (default, see rt_trace.cuh)
        t.splitPart = env("OCLR_SPLIT_PART", 16);
        t.splitEarly = getenv("OCLR_SPLIT_EARLY") ? atoi(getenv("OCLR_SPLIT_EARLY")) : 0;
        t.handoffAfter = getenv("OCLR_HANDOFF_AFTER") ? atoi(getenv("OCLR_HANDOFF_AFTER")) : 2;
        t.handoffMode = getenv("OCLR_HANDOFF_MODE") ? atoi(getenv("OCLR_HANDOFF_MODE")) : 1;
        if (t.handoffMode == 1 && getenv("OCLR_TAIL_BRICKS") && atoi(getenv("OCLR_TAIL_BRICKS")) == 0) t.handoffMode = 3;   // cell-plane bursts
        t.handoffLanes = getenv("OCLR_HANDOFF_LANES") ? atoi(getenv("OCLR_HANDOFF_LANES")) : (t.handoffMode == 2 ? 16 : 32);
        t.handoffBurst = env("OCLR_HANDOFF_BURST", 12);
        return t;
    }();
    return tune;
}

// Persistent grid of the trace kernel: as many CTAs as are resident on the device at once.
static bool trace_grid(const SceneView& S, int smCount, bool counting, unsigned& grid, std::string& err) {
    const size_t shBytes = sizeof(float) * 3 * (S.n + 1);
    int perSm = 0;
    if (counting)
        OCLR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, wf_pipe_kernel<true, false>, 128, shBytes));
    else
        OCLR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, wf_pipe_kernel<false, false>, 128, shBytes));
    if (perSm < 1) perSm = 1;
    if (getenv("OCLR_TRACE_CTAS") && atoi(getenv("OCLR_TRACE_CTAS")) > 0) perSm = std::min(perSm, atoi(getenv("OCLR_TRACE_CTAS")));
    grid = (unsigned)(smCount * perSm);
    return true;
}

// Enqueues one round of the trace stage on `ks`: walk records of the rays queued in w (wf_setup_kernel), the trace (wf_pipe_kernel,
// instantiation chosen from the tuning), and the hand-off of its tail when `tq` has room (tq.capacity != 0).  Every kernel reads the ray
// count from device memory, so a round with nothing queued costs only its launches.  The production instantiations walk `walkGrid`
// (Scene::walkView); the off-by-default experiments -- run-time split, tail hand-off, super-brick level -- the reference grid `S`.
static void enqueue_trace(const SceneView& reference, const SceneView& walkGrid, const WfState& w, const WalkRecords& rec, const TailQueue& tq,
                          unsigned setupGrid, unsigned traceGrid, int smCount, Counters* dcnt, cudaStream_t ks, uint32_t& launches) {
    const TraceTuning& tune = trace_tuning();
    // (the run-time split of long walks is an instantiation of its own: compiled into the production kernel it cost
    // 10 % through register pressure even when switched off)
    // (so is the hand-off of the tail to wf_tail_kernel: only the launches of small domains run that instantiation)
    const bool handoff = tq.capacity != 0 && tune.splitMin <= 0;
    const SceneView& S = (OCLR_SUPER_LEVEL || tune.splitMin > 0 || handoff) ? reference : walkGrid;
    const size_t shBytes = sizeof(float) * 3 * (S.n + 1);
    wf_setup_kernel<<<setupGrid, 256, shBytes, ks>>>(S, w, rec);
    ++launches;
    if (dcnt && tune.splitMin > 0)
        wf_pipe_kernel<true, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (dcnt && handoff)
        wf_pipe_kernel<true, false, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (dcnt && S.walkTrim)
        wf_pipe_kernel<true, false, false, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (dcnt)
        wf_pipe_kernel<true, false><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (tune.splitMin > 0)
        wf_pipe_kernel<false, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (handoff)
        wf_pipe_kernel<false, false, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else if (S.walkTrim)
        wf_pipe_kernel<false, false, false, true><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    else
        wf_pipe_kernel<false, false><<<traceGrid, 128, shBytes, ks>>>(S, w, rec, tune, dcnt, tq);
    if (handoff && tune.handoffMode == 2) {   // second pass: the same kernel over the rays given up, as their own little queue
        WfState w2 = w;
        w2.queueCount = tq.count;
        w2.queueCursor = tq.cursor;
        WalkRecords rec2 = {tq.o, tq.d, tq.s0, tq.s1, tq.order, tq.count, tq.capacity};
        if (dcnt)
            wf_pipe_kernel<true, false><<<traceGrid, 128, shBytes, ks>>>(S, w2, rec2, tune, dcnt, tq);
        else
            wf_pipe_kernel<false, false><<<traceGrid, 128, shBytes, ks>>>(S, w2, rec2, tune, dcnt, tq);
        ++launches;
    } else if (handoff) {   // one ray per warp: bursts over brick planes (default) or over cell planes (OCLR_TAIL_BRICKS=0)
        if (tune.handoffMode == 1)
            wf_tail_brick_kernel<<<(unsigned)(smCount * 4), 128, shBytes, ks>>>(S, w, tq);
        else
            wf_tail_kernel<<<(unsigned)(smCount * 4), 128, shBytes, ks>>>(S, w, tq);
        ++launches;
    }
    ++launches;
}

// Every walk of the trace stage is the packed walk (rt_walk.h).
static bool packed_walk_ok(const SceneView& S, std::string& err) {
    if (S.n > 1024) {
        err = "axesDivCount > 1024 is not supported by the packed walk";
        return false;
    }
    return true;
}

// ---- the round driver of the path state machine (rt_wavefront.cuh), shared by frames and radiance queries ---------------------------
// One launch domain: its bound path state, stream and round history.
struct RoundDomain {
    const PathState* ps = nullptr;
    WfState w = {};       // ps bound (PathState::bind); the driver points the queue counters at each round's set
    WalkRecords rec = {};
    TailQueue tail = {};  // hand-off buffers of the trace tail (capacity 0: none); the driver points its counters at each round's set
    cudaStream_t st = nullptr;
    uint32_t* lastRounds = nullptr;                    // rounds the previous sample needed: the length of the next one's first chunk
    std::vector<cudaEvent_t>* traceEvents = nullptr;   // set: a timing event pair around every round's trace stage
    uint32_t* traceEventsUsed = nullptr;
};
// Enqueues the entry kernel(s) of round r of domain k on `ks`, behind the clearing of the round's counter set; `prev` is the previous
// round's set (null at r = 0).  Counted as one launch.
using RoundEntry = std::function<void(int k, uint32_t r, const WfState& w, const uint32_t* prev, cudaStream_t ks)>;
struct RoundDriver {
    const SceneView& S;
    const SceneView& walkS;   // the grid the production trace stage walks (Scene::walkView)
    int device, smCount;
    unsigned traceGrid;
    Counters* dcnt;
    uint32_t* host;           // pinned: per domain kRoundLogSize + 1 words, then the camera-check word
    const uint32_t* camBad;   // optional device word read back with every chunk's round logs (FrameView::camBad)
    const char* what;         // "<what> did not converge"
    int K = 0;
    RoundDomain dom[kMaxSlices];
    uint32_t launches = 0, rounds = 0;
    bool run(cudaEvent_t resume, const RoundEntry& entry, std::string& err);
};
static_assert(sizeof(uint32_t) * (kMaxSlices * (kRoundLogSize + 1) + 1) <= 4096, "round logs + camera-check word fit one pinned block");

// Rounds of one sample (entry -> setup -> trace) until no path of any domain waits for a ray.  Rounds are enqueued ahead in chunks
// without a host round trip: every kernel reads the ray count of its round from device memory and returns at once when there is
// nothing to do.  The host reads the round log once per chunk; the first chunk is as long as the previous sample needed.  Domains are
// enqueued round by round, alternating, so that their launches interleave on the device.  `resume`: round 0 of domain 0 was enqueued
// ahead (frame_prelaunch) and has already queued its rays; the stream waits for it instead of clearing the counters and entering again.
bool RoundDriver::run(cudaEvent_t resume, const RoundEntry& entry, std::string& err) {
    uint32_t round[kMaxSlices] = {0};
    bool live[kMaxSlices];
    unsigned setupGrid[kMaxSlices];
    for (int k = 0; k < K; ++k) {
        live[k] = true;
        setupGrid[k] = (unsigned)std::min<uint64_t>((uint64_t)smCount * 8, (2 * (uint64_t)dom[k].w.Q + 255) / 256);
    }
    for (;;) {
        uint32_t chunk[kMaxSlices], maxChunk = 0;
        for (int k = 0; k < K; ++k) {
            chunk[k] = !live[k] ? 0u : (round[k] == 0 ? std::max<uint32_t>(*dom[k].lastRounds, 2) : 2u);
            maxChunk = std::max(maxChunk, chunk[k]);
        }
        if (maxChunk == 0) return true;
        for (uint32_t c = 0; c < maxChunk; ++c) {
            for (int k = 0; k < K; ++k) {
                if (c >= chunk[k]) continue;
                RoundDomain& d = dom[k];
                const uint32_t r = round[k];
                d.w.queueCount = d.ps->counter_set(r);
                d.w.queueCursor = d.w.queueCount + 1;
                d.w.roundIndex = r;
                d.rec.classCount = d.w.queueCount + 2;
                d.tail.count = d.w.queueCount + 2 + kLengthClasses;
                d.tail.cursor = d.w.queueCount + 6 + kLengthClasses;
                if (resume && k == 0 && r == 0) {
                    OCLR_CUDA(cudaStreamWaitEvent(d.st, resume, 0));
                } else {
                    OCLR_CUDA(cudaMemsetAsync(d.w.queueCount, 0, sizeof(uint32_t) * kCounterStride, d.st));
                    entry(k, r, d.w, r ? d.ps->counter_set(r - 1) : nullptr, d.st);
                    ++launches;
                }
                if (d.traceEvents) {
                    while (d.traceEvents->size() < (size_t)*d.traceEventsUsed + 2) {
                        cudaEvent_t e;
                        OCLR_CUDA(make_event(device, &e, true));
                        d.traceEvents->push_back(e);
                    }
                    OCLR_CUDA(cudaEventRecord((*d.traceEvents)[*d.traceEventsUsed], d.st));
                }
                enqueue_trace(S, walkS, d.w, d.rec, d.tail, setupGrid[k], traceGrid, smCount, dcnt, d.st, launches);
                if (d.traceEvents) {
                    OCLR_CUDA(cudaEventRecord((*d.traceEvents)[*d.traceEventsUsed + 1], d.st));
                    *d.traceEventsUsed += 2;
                }
                ++round[k];
                ++rounds;
            }
        }
        // one read per chunk: the round log (rays queued by every round so far; the last enqueued round decides) and, beyond the log,
        // the live counter of the last enqueued round
        for (int k = 0; k < K; ++k) {
            if (!chunk[k]) continue;
            uint32_t* log = host + k * (kRoundLogSize + 1);
            OCLR_CUDA(cudaMemcpyAsync(log, dom[k].w.roundLog, sizeof(uint32_t) * std::min<uint32_t>(round[k], kRoundLogSize),
                                      cudaMemcpyDeviceToHost, dom[k].st));
            if (round[k] > kRoundLogSize)
                OCLR_CUDA(cudaMemcpyAsync(log + kRoundLogSize, dom[k].ps->counter_set(round[k] - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                          dom[k].st));
        }
        uint32_t* camFlag = host + kMaxSlices * (kRoundLogSize + 1);
        *camFlag = 0;
        if (camBad) OCLR_CUDA(cudaMemcpyAsync(camFlag, camBad, sizeof(uint32_t), cudaMemcpyDeviceToHost, dom[0].st));
        for (int k = 0; k < K; ++k)
            if (chunk[k]) OCLR_CUDA(cudaStreamSynchronize(dom[k].st));
        if (*camFlag) {
            err = cam_check_message(*camFlag);
            return false;
        }
        for (int k = 0; k < K; ++k) {
            if (!chunk[k]) continue;
            const uint32_t* log = host + k * (kRoundLogSize + 1);
            bool finished = false;
            uint32_t needed = round[k];
            if (round[k] <= kRoundLogSize) {
                finished = log[round[k] - 1] == 0;
                for (uint32_t r = 0; r < round[k]; ++r)
                    if (log[r] == 0) {   // the first round that queued no ray is the last one that had anything to do
                        needed = r + 1;
                        break;
                    }
            } else {
                finished = log[kRoundLogSize] == 0;
            }
            if (finished) {
                live[k] = false;
                *dom[k].lastRounds = needed;
            } else if (round[k] > 100000) {
                err = std::string(what) + " did not converge";
                return false;
            }
        }
    }
}

// Wavefront driver: alternate the logic and trace kernels until no path is waiting for a ray (rt_wavefront.cuh).
// `prelaunchOnly`: allocate the path state and enqueue nothing but the first logic round of the first sample, on the frame's own
// stream behind everything already enqueued on `st` (frame_prelaunch).  A later normal call with the same view finds
// f->prelaunched set, skips that round's logic launch and orders its first setup kernel behind it.
// Launch domains of at most OCLR_HANDOFF_MAX_PATHS paths hand the tail of their trace launches to wf_tail_kernel (rt_tail.cuh).  Off by
// default (0): exact, but a 1/8 share of config 2 gets slower (0.93 -> 0.97-1.08 ms) -- what a small launch loses is not a few very long
// rays but the decaying lane fill of every warp's last batch, and one warp per ray is the wrong cure for that (profiles/r02_super_level.txt).
static bool handoff_domain(uint32_t Q) {
    static const uint32_t maxPaths = [] { const char* v = getenv("OCLR_HANDOFF_MAX_PATHS"); return v ? (uint32_t)strtoul(v, nullptr, 10) : 0u; }();
    return Q <= maxPaths;
}
static bool launch_wavefront(Frame* f, const SceneView& S, const FrameView& Fall, int smCount, Counters* dcnt, cudaStream_t st,
                             uint32_t& launches, bool timeTrace, std::string& err, bool prelaunchOnly = false) {
    const uint32_t W = Fall.cam.width;
    if (!packed_walk_ok(S, err)) return false;
    // ---- cut the launch domain into slices -------------------------------------------------------------------------------------------
    const uint32_t rowsAll = launch_rows(Fall);
    int K = slice_count_for(rowsAll, W);
    FrameView FV[kMaxSlices];
    if (Fall.bandWorld <= 1) {   // contiguous row ranges, multiples of 8 rows (the logic kernel's tile height)
        const uint32_t per = ((rowsAll + (uint32_t)K - 1) / (uint32_t)K + 7u) / 8u * 8u;
        int used = 0;
        for (uint32_t r0 = 0; r0 < rowsAll; r0 += per, ++used) {
            FV[used] = Fall;
            FV[used].rowBegin = Fall.rowBegin + r0;
            FV[used].rowEnd = Fall.rowBegin + std::min(rowsAll, r0 + per);
            FV[used].ownedRows = FV[used].rowEnd - FV[used].rowBegin;
        }
        K = used;
    } else {   // band set of rank r in world N -> sub-band sets r + N*k in world N*K (b % (N*K) == r + N*k implies b % N == r)
        int used = 0;
        for (int k = 0; k < K; ++k) {
            FrameView v = Fall;
            v.bandWorld = Fall.bandWorld * (uint32_t)K;
            v.bandRank = Fall.bandRank + Fall.bandWorld * (uint32_t)k;
            v.ownedRows = band_owned_rows(Fall.cam.height, v.bandRows, v.bandRank, v.bandWorld);
            if (v.ownedRows) FV[used++] = v;
        }
        K = used;
    }
    if (K == 0) return true;
    const bool resumePre = !prelaunchOnly && K == 1 && resumes_prelaunch(f, Fall);
    if (!prelaunchOnly && f->prelaunched && !resumePre) {   // a prelaunched round nobody can use: wait it out and start over
        OCLR_CUDA(cudaStreamWaitEvent(st, f->preDone, 0));
        f->prelaunched = false;
    }
    if (prelaunchOnly && K != 1) return true;   // (only the one-slice case is started ahead)

    RoundDriver drv = {S, f->scene->walkView, f->device, smCount, 0u, dcnt, nullptr, Fall.camBad, "wavefront"};
    drv.K = K;
    dim3 logicGrid[kMaxSlices];
    int aheadMode[kMaxSlices];
    const bool cull = g_cullHidden.load();
    for (int k = 0; k < K; ++k) {
        WfSlice& sl = f->slices[k];
        const uint32_t rows = launch_rows(FV[k]);
        const uint64_t Q64 = (uint64_t)((rows + 7) / 8 * 8) * W;
        if (Q64 > 0x7FFFFFF0ull) {   // ray indices are slot * Q + path
            err = "launch domain too large";
            return false;
        }
        const uint32_t Q = (uint32_t)Q64;
        if (path_state_regrow(sl.ps.capacity, sl.ps.ringSlots, Q, f->scene->ringSlots)) {
            for (DeviceBuffer* b : sl.tail_buffers()) b->release(st);
            if (!sl.ps.reserve(Q, f->scene->ringSlots, st, err)) return false;
            sl.tailCapacity = 0;
            if (handoff_domain(sl.ps.capacity)) {   // small launch domain: its trace tail is handed to wf_tail_kernel (rt_tail.cuh)
                sl.tailCapacity = 2 * sl.ps.capacity;   // (every ray of a round could be given up: the list cannot overflow)
                const size_t c = sl.tailCapacity;
                if (!sl.tailEntries.alloc(sizeof(uint4) * c, err, st) || !sl.tailO.alloc(sizeof(float4) * c, err, st) ||
                    !sl.tailD.alloc(sizeof(float4) * c, err, st) || !sl.tailS0.alloc(sizeof(float4) * c, err, st) ||
                    !sl.tailS1.alloc(sizeof(uint4) * c, err, st) || !sl.tailOrder.alloc(sizeof(uint32_t) * c, err, st))
                    return false;
            }
        }
        if (k > 0 && !sl.stream) OCLR_CUDA(make_stream(f->device, &sl.stream));
        if (!sl.done) OCLR_CUDA(make_event(f->device, &sl.done, false));
        sl.traceEventsUsed = 0;
        RoundDomain& d = drv.dom[k];
        d.ps = &sl.ps;
        sl.ps.bind(Q, f->scene->ringSlots, d.w, d.rec);
        d.tail = {(uint4*)sl.tailEntries.p, nullptr, nullptr, sl.tailCapacity, (float4*)sl.tailO.p, (float4*)sl.tailD.p, (float4*)sl.tailS0.p,
                  (uint4*)sl.tailS1.p, (uint32_t*)sl.tailOrder.p};
        d.st = k == 0 ? st : sl.stream;
        d.lastRounds = &sl.lastRounds;
        if (timeTrace) {
            d.traceEvents = &sl.traceEvents;
            d.traceEventsUsed = &sl.traceEventsUsed;
        }
        aheadMode[k] = ahead_mode_for(Q);
        logicGrid[k] = dim3((W + 15) / 16, (rows + 7) / 8);
    }
    for (int k = K; k < kMaxSlices; ++k) f->slices[k].traceEventsUsed = 0;
    if (!f->hostCount) f->hostCount = (uint32_t*)pinned_block();
    if (!f->hostCount) {
        err = "out of pinned host memory";
        return false;
    }
    drv.host = f->hostCount;

    if (!trace_grid(S, smCount, dcnt != nullptr, drv.traceGrid, err)) return false;
    if (Fall.flagOut && !resumePre) OCLR_CUDA(cudaMemsetAsync(Fall.flagOut, 0, (size_t)Fall.cam.width * Fall.cam.height, st));
    if (prelaunchOnly) {
        if (!f->preStream) {
            OCLR_CUDA(make_stream(f->device, &f->preStream));
            OCLR_CUDA(make_event(f->device, &f->preReady, false));
            OCLR_CUDA(make_event(f->device, &f->preDone, false));
        }
        WfState& w = drv.dom[0].w;
        w.queueCount = f->slices[0].ps.counter_set(0);
        w.queueCursor = w.queueCount + 1;
        OCLR_CUDA(cudaEventRecord(f->preReady, st));
        OCLR_CUDA(cudaStreamWaitEvent(f->preStream, f->preReady, 0));
        OCLR_CUDA(cudaMemsetAsync(w.queueCount, 0, sizeof(uint32_t) * kCounterStride, f->preStream));
        wf_logic_kernel<false><<<logicGrid[0], 128, 0, f->preStream>>>(S, FV[0], w, Fall.sampleBegin, 1u, nullptr, nullptr, aheadMode[0], cull);
        OCLR_CUDA(cudaGetLastError());
        OCLR_CUDA(cudaEventRecord(f->preDone, f->preStream));
        f->prelaunched = true;
        f->preView = Fall;
        ++launches;
        return true;
    }
    // fork: the internal streams start after everything already enqueued on the caller's stream
    if (K > 1) {
        OCLR_CUDA(cudaEventRecord(f->evFork, st));
        for (int k = 1; k < K; ++k) OCLR_CUDA(cudaStreamWaitEvent(drv.dom[k].st, f->evFork, 0));
    }
    for (uint32_t s = Fall.sampleBegin; s < Fall.sampleEnd; ++s) {
        const RoundEntry logic = [&](int k, uint32_t r, const WfState& w, const uint32_t* prev, cudaStream_t ks) {
            if (dcnt)
                wf_logic_kernel<true><<<logicGrid[k], 128, 0, ks>>>(S, FV[k], w, s, r == 0 ? 1u : 0u, prev, dcnt, aheadMode[k], false);
            else
                wf_logic_kernel<false><<<logicGrid[k], 128, 0, ks>>>(S, FV[k], w, s, r == 0 ? 1u : 0u, prev, dcnt, aheadMode[k], cull);
        };
        // the first logic round of the request may already be running (or done) on the frame's own stream: frame_prelaunch
        const cudaEvent_t resume = resumePre && s == Fall.sampleBegin ? f->preDone : nullptr;
        if (resume) f->prelaunched = false;
        if (!drv.run(resume, logic, err)) return false;
    }
    launches += drv.launches;
    // join: later work on the caller's stream (plane reads, gathers) follows every slice
    for (int k = 1; k < K; ++k) {
        OCLR_CUDA(cudaEventRecord(f->slices[k].done, drv.dom[k].st));
        OCLR_CUDA(cudaStreamWaitEvent(st, f->slices[k].done, 0));
    }
    return true;
}

static bool resumes_prelaunch(const Frame* f, const FrameView& F) {
    return f->prelaunched && same_request(f->preView, F) && slice_count_for(launch_rows(F), F.cam.width) == 1;
}

static void fill_view(Frame* f, FrameView& F) {
    const size_t P = (size_t)f->cam.width * f->cam.height;
    F.cam = f->cam;
    F.camStart = (const uint32_t*)f->camStart.p;
    F.camEnd = (const uint32_t*)f->camEnd.p;
    F.camList = (const uint32_t*)f->camList.p;
    F.outR = (uint16_t*)f->planesRGB.p;
    F.outG = F.outR + P;
    F.outB = F.outG + P;
    F.idOut = (uint32_t*)f->ids.p;
    F.flagOut = (uint8_t*)f->flags.p;
    F.accum = (float4*)f->accum.p;   // nullptr unless float accumulation is on
    F.doneCount = (unsigned long long*)f->doneCount.p;
    F.camBad = (const uint32_t*)f->camCheck.p;
}

static std::string cam_check_message(uint32_t flag) {
    return std::string("camera triangle lists are inconsistent:") + ((flag & kCamBadRange) ? " Start <= End <= list size violated;" : "") +
           ((flag & kCamBadEntry) ? " list entry >= triangleCount;" : "");
}

// Two render requests are the same job (a round started ahead by frame_prelaunch may be continued): field by field -- the structs
// carry padding, memcmp would compare it.
static bool same_request(const FrameView& a, const FrameView& b) {
    return memcmp(&a.cam, &b.cam, sizeof(Camera)) == 0 && a.camStart == b.camStart && a.camEnd == b.camEnd && a.camList == b.camList &&
           a.sampleCount == b.sampleCount && a.sampleBegin == b.sampleBegin && a.sampleEnd == b.sampleEnd && a.rowBegin == b.rowBegin &&
           a.rowEnd == b.rowEnd && a.bandRows == b.bandRows && a.bandRank == b.bandRank && a.bandWorld == b.bandWorld &&
           a.ownedRows == b.ownedRows && a.outR == b.outR && a.outG == b.outG && a.outB == b.outB && a.idOut == b.idOut &&
           a.flagOut == b.flagOut && a.accum == b.accum && a.doneCount == b.doneCount && a.camBad == b.camBad;
}

static bool frame_launch(Frame* f, FrameView& F, int variant, bool count, void* stream, RenderStats* stats, std::string& err) {
    Scene* s = f->scene;
    cudaStream_t st = (cudaStream_t)stream;
    fill_view(f, F);
    if (F.accum && variant == kKernelSimple) {
        err = "float accumulation is implemented by the wavefront pipeline only";
        return false;
    }
    // (a first round started ahead by frame_prelaunch for exactly this request has already counted its finished paths)
    const bool continuesPre = variant == kKernelPipe && !count && resumes_prelaunch(f, F);
    if (f->prelaunched && !continuesPre) {
        // The round started ahead belongs to another request: wait it out and start over.  It rendered sample 0 of ITS job into the
        // planes (sample 0 overwrites), so a request that continues an earlier job (sampleBegin > 0) has lost those samples.
        if (F.sampleBegin > 0) {
            err = "a first round started ahead (frame_prelaunch) for another request has overwritten the planes this request continues";
            return false;
        }
        OCLR_CUDA(cudaStreamWaitEvent(st, f->preDone, 0));
        f->prelaunched = false;
    }
    if (!continuesPre) OCLR_CUDA(cudaMemsetAsync(F.doneCount, 0, sizeof(unsigned long long), st));
    f->jobPaths.store((unsigned long long)launch_rows(F) * f->cam.width * (F.sampleEnd - F.sampleBegin));
    Counters* dcnt = (Counters*)f->counters.p;
    if (count) OCLR_CUDA(cudaMemsetAsync(dcnt, 0, sizeof(Counters), st));
    const size_t shBytes = sizeof(float) * 3 * (s->view.n + 1);
    uint32_t launches = 0;
    if (stats) OCLR_CUDA(cudaEventRecord(f->ev0, st));
    if (variant == kKernelSimple) {
        dim3 grid((f->cam.width + 15) / 16, (launch_rows(F) + 7) / 8);
        if (count)
            raytrace_simple_kernel<true><<<grid, 128, shBytes, st>>>(s->view, F, dcnt);
        else
            raytrace_simple_kernel<false><<<grid, 128, shBytes, st>>>(s->view, F, dcnt);
        launches = 1;
    } else if (variant == kKernelPipe) {
        if (!launch_wavefront(f, s->view, F, s->smCount, count ? dcnt : nullptr, st, launches, stats != nullptr, err)) return false;
    } else {
        err = "unknown kernel variant";
        return false;
    }
    if (F.accum) {
        resolve_accum_kernel<<<dim3((f->cam.width + 255) / 256, launch_rows(F)), 256, 0, st>>>(F);
        ++launches;
    }
    OCLR_CUDA(cudaGetLastError());
    f->lastLaunches = launches;
    if (stats) {
        OCLR_CUDA(cudaEventRecord(f->ev1, st));
        OCLR_CUDA(cudaEventSynchronize(f->ev1));
        OCLR_CUDA(cudaEventElapsedTime(&stats->deviceMs, f->ev0, f->ev1));
        stats->launches = launches;
        stats->traceMs = 0.f;
        stats->traceLaunches = 0;
        // Trace-stage time = length of the union of the [setup start, trace end] intervals of all slices (their launches overlap),
        // measured against ev0 on the device clock.
        std::vector<std::pair<float, float>> spans;
        for (WfSlice& sl : f->slices) {
            for (uint32_t k = 0; variant != kKernelSimple && k + 1 < sl.traceEventsUsed; k += 2) {
                float t0 = 0.f, ms = 0.f;
                OCLR_CUDA(cudaEventElapsedTime(&t0, f->ev0, sl.traceEvents[k]));
                OCLR_CUDA(cudaEventElapsedTime(&ms, sl.traceEvents[k], sl.traceEvents[k + 1]));
                if (ms > 0.015f) {   // rounds enqueued ahead that found no ray return at once (~6 us): not counted
                    ++stats->traceLaunches;
                    spans.emplace_back(t0, t0 + ms);
                }
            }
        }
        std::sort(spans.begin(), spans.end());
        float covered = -1.f;
        for (const auto& sp : spans) {
            const float from = std::max(sp.first, covered);
            if (sp.second > from) stats->traceMs += sp.second - from;
            covered = std::max(covered, sp.second);
        }
        if (count) OCLR_CUDA(cudaMemcpy(&stats->counters, dcnt, sizeof(Counters), cudaMemcpyDeviceToHost));
        if (variant == kKernelSimple && F.camBad) {
            uint32_t flag = 0;
            OCLR_CUDA(cudaMemcpy(&flag, F.camBad, sizeof(uint32_t), cudaMemcpyDeviceToHost));
            if (flag) {
                err = cam_check_message(flag);
                return false;
            }
        }
    }
    return true;
}

bool frame_render(Frame* f, uint32_t sampleCount, uint32_t sampleBegin, uint32_t sampleEnd, uint32_t rowBegin, uint32_t rowEnd, int variant,
                  bool count, void* stream, RenderStats* stats, std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    if (rowEnd > f->cam.height) rowEnd = f->cam.height;
    if (sampleCount == 0 || rowBegin >= rowEnd || sampleBegin >= sampleEnd || sampleEnd > sampleCount) {
        err = "empty render request";
        return false;
    }
    if (!frame_lists_current(f, err)) return false;
    FrameView F = {};
    F.sampleCount = sampleCount;
    F.sampleBegin = sampleBegin;
    F.sampleEnd = sampleEnd;
    F.rowBegin = rowBegin;
    F.rowEnd = rowEnd;
    F.bandRows = 0;
    F.bandRank = 0;
    F.bandWorld = 1;
    F.ownedRows = rowEnd - rowBegin;
    return frame_launch(f, F, variant, count, stream, stats, err);
}

bool frame_render_bands(Frame* f, uint32_t sampleCount, uint32_t sampleBegin, uint32_t sampleEnd, uint32_t bandRows, uint32_t rank, uint32_t world,
                        int variant, bool count, void* stream, RenderStats* stats, std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    if (sampleCount == 0 || bandRows == 0 || world == 0 || rank >= world || sampleBegin >= sampleEnd || sampleEnd > sampleCount) {
        err = "bad band request";
        return false;
    }
    if (world == 1) return frame_render(f, sampleCount, sampleBegin, sampleEnd, 0, f->cam.height, variant, count, stream, stats, err);
    if (!frame_lists_current(f, err)) return false;
    FrameView F = {};
    F.sampleCount = sampleCount;
    F.sampleBegin = sampleBegin;
    F.sampleEnd = sampleEnd;
    F.rowBegin = 0;
    F.rowEnd = f->cam.height;
    F.bandRows = bandRows;
    F.bandRank = rank;
    F.bandWorld = world;
    F.ownedRows = band_owned_rows(f->cam.height, bandRows, rank, world);
    if (F.ownedRows == 0) {
        if (stats) *stats = RenderStats();
        return true;
    }
    return frame_launch(f, F, variant, count, stream, stats, err);
}

// Starts the first logic round (ray generation, camera-list scan, shading of the primary hits) of the request
// frame_render_bands(f, sampleCount, 0, sampleCount, bandRows, rank, world, kKernelPipe, ...) would make, on a stream of the frame's own
// behind everything enqueued on the default stream so far.  Needs only the triangle / material / light part of the scene (see
// scene_create's `early` hook).  The matching render call continues from there; any other request waits the round out and starts over.
bool frame_prelaunch(Frame* f, uint32_t sampleCount, uint32_t bandRows, uint32_t rank, uint32_t world, std::string& err) {
    if (!f || sampleCount == 0 || world == 0 || rank >= world || bandRows == 0) {
        err = "bad prelaunch request";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    if (!frame_lists_current(f, err)) return false;
    FrameView F = {};
    F.sampleCount = sampleCount;
    F.sampleBegin = 0;
    F.sampleEnd = sampleCount;
    if (world == 1) {
        F.rowBegin = 0;
        F.rowEnd = f->cam.height;
        F.bandRows = 0;
        F.bandRank = 0;
        F.bandWorld = 1;
        F.ownedRows = f->cam.height;
    } else {
        F.rowBegin = 0;
        F.rowEnd = f->cam.height;
        F.bandRows = bandRows;
        F.bandRank = rank;
        F.bandWorld = world;
        F.ownedRows = band_owned_rows(f->cam.height, bandRows, rank, world);
        if (F.ownedRows == 0) return true;
    }
    fill_view(f, F);
    if (F.accum) return true;
    OCLR_CUDA(cudaMemsetAsync(F.doneCount, 0, sizeof(unsigned long long), 0));
    uint32_t launches = 0;
    return launch_wavefront(f, f->scene->view, F, f->scene->smCount, nullptr, 0, launches, false, err, true);
}

bool frame_read(Frame* f, uint32_t rowBegin, uint32_t rowEnd, uint16_t* outR, uint16_t* outG, uint16_t* outB, void* stream,
                std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (rowEnd > f->cam.height) rowEnd = f->cam.height;
    if (rowBegin >= rowEnd) return true;
    const size_t P = (size_t)f->cam.width * f->cam.height;
    const size_t off = (size_t)rowBegin * f->cam.width, cnt = (size_t)(rowEnd - rowBegin) * f->cam.width;
    const uint16_t* d = (const uint16_t*)f->planesRGB.p;
    if (staging_enabled() && cnt * 2 >= (1u << 20) && is_pageable(outR + off)) {   // pageable planes: pinned arena + copier threads
        return device_to_host(outR + off, d + off, cnt * 2, st, err) && device_to_host(outG + off, d + P + off, cnt * 2, st, err) &&
               device_to_host(outB + off, d + 2 * P + off, cnt * 2, st, err);
    }
    OCLR_CUDA(cudaMemcpyAsync(outR + off, d + off, cnt * 2, cudaMemcpyDeviceToHost, st));
    OCLR_CUDA(cudaMemcpyAsync(outG + off, d + P + off, cnt * 2, cudaMemcpyDeviceToHost, st));
    OCLR_CUDA(cudaMemcpyAsync(outB + off, d + 2 * P + off, cnt * 2, cudaMemcpyDeviceToHost, st));
    OCLR_CUDA(cudaStreamSynchronize(st));
    return true;
}

// ---- read-back of a band set (RaytraceAll on all devices) --------------------------------------------------------------------------
// A rank's rows are bands scattered over the frame.  Copying them band by band into the caller's pageable planes is 3 blocking
// copies per band; instead the rows are compacted on the device ([plane][owned row][W]), cross PCIe in ONE transfer into a pinned
// block that lives as long as the process, and the calling thread scatters them (N threads do that side by side).
__global__ void __launch_bounds__(256) compact_rows_kernel(const uint16_t* __restrict__ planes, uint16_t* __restrict__ out, uint32_t W, uint32_t H,
                                                           uint32_t bandRows, uint32_t rank, uint32_t world, uint32_t ownedRows) {
    const size_t P = (size_t)W * H;
    const uint64_t total = (uint64_t)ownedRows * W * 3u;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t x = (uint32_t)(i % W);
        const uint64_t rowPlane = i / W;
        const uint32_t k = (uint32_t)(rowPlane % ownedRows), plane = (uint32_t)(rowPlane / ownedRows);
        const uint32_t y = (k / bandRows) * (bandRows * world) + rank * bandRows + (k % bandRows);   // map_row()
        out[i] = planes[plane * P + (size_t)y * W + x];
    }
}

struct PinnedStage {
    void* p = nullptr;
    size_t bytes = 0;
};
static PinnedStage& read_stage(int device, size_t need) {
    static PinnedStage stages[64];
    PinnedStage& st = stages[device & 63];
    if (st.bytes < need) {   // (one render at a time per device: RaytraceAll's worker thread)
        if (st.p) cudaFreeHost(st.p);
        st.p = nullptr;
        st.bytes = 0;
        if (cudaHostAlloc(&st.p, need, cudaHostAllocPortable) == cudaSuccess)
            st.bytes = need;
        else
            cudaGetLastError();
    }
    return st;
}

bool frame_read_bands(Frame* f, uint32_t bandRows, uint32_t rank, uint32_t world, uint16_t* outR, uint16_t* outG, uint16_t* outB,
                      std::string& err) {
    if (!f || bandRows == 0 || world == 0 || rank >= world) {
        err = "bad read request";
        return false;
    }
    const uint32_t W = f->cam.width, H = f->cam.height;
    if (world == 1) return frame_read(f, 0, H, outR, outG, outB, nullptr, err);
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    const uint32_t owned = band_owned_rows(H, bandRows, rank, world);
    if (owned == 0) return true;
    if (!staging_enabled() || !is_pageable(outR)) {
        // page-locked planes: every band is one contiguous piece per plane, copied straight to where it belongs
        const size_t P = (size_t)W * H;
        const uint16_t* d = (const uint16_t*)f->planesRGB.p;
        uint16_t* out[3] = {outR, outG, outB};
        for (uint32_t k = 0; k < owned; k += bandRows) {
            const uint32_t y = (k / bandRows) * (bandRows * world) + rank * bandRows;
            const size_t off = (size_t)y * W, cnt = (size_t)std::min(bandRows, owned - k) * W;
            for (int plane = 0; plane < 3; ++plane)
                OCLR_CUDA(cudaMemcpyAsync(out[plane] + off, d + plane * P + off, cnt * sizeof(uint16_t), cudaMemcpyDeviceToHost, 0));
        }
        OCLR_CUDA(cudaStreamSynchronize(0));
        return true;
    }
    const size_t bytes = sizeof(uint16_t) * 3 * (size_t)owned * W;
    PinnedStage& st = read_stage(f->scene->device, bytes);
    if (!st.p) {
        err = "out of pinned host memory";
        return false;
    }
    DeviceBuffer pack;
    if (!pack.alloc(bytes, err)) return false;
    const uint64_t total = (uint64_t)owned * W * 3u;
    compact_rows_kernel<<<(unsigned)std::min<uint64_t>((total + 255) / 256, (uint64_t)f->scene->smCount * 8), 256>>>(
        (const uint16_t*)f->planesRGB.p, (uint16_t*)pack.p, W, H, bandRows, rank, world, owned);
    cudaError_t e = cudaMemcpyAsync(st.p, pack.p, bytes, cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    pack.release();
    if (e != cudaSuccess) {
        err = std::string("frame_read_bands: ") + cudaGetErrorString(e);
        return false;
    }
    // scatter: one job per band and plane, shared out among the copier threads (and this one)
    const uint16_t* src = (const uint16_t*)st.p;
    uint16_t* dst[3] = {outR, outG, outB};
    const size_t bands = (owned + bandRows - 1) / bandRows;
    std::vector<std::atomic<int>> done(3 * bands);
    std::vector<CopyPool::Job> jobs;
    jobs.reserve(3 * bands);
    for (int plane = 0; plane < 3; ++plane)
        for (uint32_t k = 0; k < owned; k += bandRows) {   // one band = consecutive frame rows
            const uint32_t y = (k / bandRows) * (bandRows * world) + rank * bandRows;
            const uint32_t rows = std::min(bandRows, owned - k);
            done[jobs.size()].store(0);
            jobs.push_back({dst[plane] + (size_t)y * W, src + ((size_t)plane * owned + k) * W, sizeof(uint16_t) * (size_t)rows * W, &done[jobs.size()]});
        }
    CopyPool& pool = CopyPool::get();
    pool.submit(jobs.data(), jobs.size());
    for (size_t b = 0; b < jobs.size(); ++b)
        while (done[b].load(std::memory_order_acquire) == 0)
            if (!pool.help()) std::this_thread::yield();
    return true;
}

// Host -> device copy of rows [rowBegin,rowEnd) of the three planes: restores a checkpoint taken with frame_read after k samples;
// the job then continues with frame_render(sampleBegin = k).
bool frame_write(Frame* f, uint32_t rowBegin, uint32_t rowEnd, const uint16_t* inR, const uint16_t* inG, const uint16_t* inB, void* stream,
                 std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (rowEnd > f->cam.height) rowEnd = f->cam.height;
    if (rowBegin >= rowEnd) return true;
    const size_t P = (size_t)f->cam.width * f->cam.height;
    const size_t off = (size_t)rowBegin * f->cam.width, cnt = (size_t)(rowEnd - rowBegin) * f->cam.width;
    uint16_t* d = (uint16_t*)f->planesRGB.p;
    OCLR_CUDA(cudaMemcpyAsync(d + off, inR + off, cnt * 2, cudaMemcpyHostToDevice, st));
    OCLR_CUDA(cudaMemcpyAsync(d + P + off, inG + off, cnt * 2, cudaMemcpyHostToDevice, st));
    OCLR_CUDA(cudaMemcpyAsync(d + 2 * P + off, inB + off, cnt * 2, cudaMemcpyHostToDevice, st));
    OCLR_CUDA(cudaStreamSynchronize(st));
    return true;
}

// Accumulation mode: 0 = the reference's 16-bit planes with per-sample truncation, 1 = fp32 sums (allocates 16 B per pixel).
bool frame_set_accumulation(Frame* f, int mode, std::string& err) {
    if (!f || (mode != 0 && mode != 1)) {
        err = "bad accumulation mode";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    if (mode == 0) {
        f->accum.release();
        f->accum.bytes = 0;
        return true;
    }
    if (!f->accum.p) {
        const size_t P = (size_t)f->cam.width * f->cam.height;
        if (!f->accum.alloc(sizeof(float4) * P, err)) return false;
        OCLR_CUDA(cudaMemsetAsync(f->accum.p, 0, sizeof(float4) * P, 0));
        OCLR_CUDA(cudaStreamSynchronize(0));
    }
    return true;
}

// The fp32 accumulator, (sum r, sum g, sum b, samples) per pixel: read (checkpoint / float output) or write (resume).
bool frame_accum_copy(Frame* f, float* host, bool toHost, std::string& err) {
    if (!f || !f->accum.p || !host) {
        err = "float accumulation is not enabled on this frame";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    const size_t bytes = sizeof(float4) * (size_t)f->cam.width * f->cam.height;
    if (toHost)
        OCLR_CUDA(cudaMemcpy(host, f->accum.p, bytes, cudaMemcpyDeviceToHost));
    else
        OCLR_CUDA(cudaMemcpy(f->accum.p, host, bytes, cudaMemcpyHostToDevice));
    return true;
}

// Progress of the render call in flight on this frame: pixel-samples finished / pixel-samples requested.  Safe to call from another
// thread while frame_render runs (raytrace.c:156-173 polls from the UI thread); reads a device counter through its own stream.
bool frame_progress(Frame* f, unsigned long long* done, unsigned long long* total) {
    if (!f) return false;
    std::lock_guard<std::mutex> lock(f->progMutex);
    *total = f->jobPaths.load();
    *done = 0;
    if (*total == 0) return true;
    if (cudaSetDevice(f->device) != cudaSuccess) return false;
    if (!f->progStream && make_stream(f->device, &f->progStream) != cudaSuccess) {   // first poll of this frame
        cudaGetLastError();
        f->progStream = nullptr;
        return false;
    }
    if (cudaMemcpyAsync(f->hostDone, f->doneCount.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, f->progStream) != cudaSuccess ||
        cudaStreamSynchronize(f->progStream) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    *done = std::min(*f->hostDone, *total);
    return true;
}

bool frame_read_ids(Frame* f, uint32_t* ids, std::string& err) {
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    OCLR_CUDA(cudaMemcpy(ids, f->ids.p, f->ids.bytes, cudaMemcpyDeviceToHost));
    return true;
}

bool frame_read_flags(Frame* f, uint8_t* flags, std::string& err) {
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    OCLR_CUDA(cudaMemcpy(flags, f->flags.p, f->flags.bytes, cudaMemcpyDeviceToHost));
    return true;
}

uint32_t frame_last_launches(const Frame* f) { return f ? f->lastLaunches : 0; }

// ---- frame assembly over NVLink peer memory (SURVEY.md section 8e: the path's only exchange step) -------------------------------------
// Every rank owns the rows y with (y / bandRows) % world == rank.  Instead of packing them, calling an all-gather and unpacking,
// one kernel STORES the rank's finished rows straight into the full-frame planes of every GPU of the box -- its own and its
// peers', whose buffers are mapped into this process (NVLink 5 / NVSwitch peer access) -- at the place they belong.  16-byte
// stores, one row segment of 8 pixels per thread and destination; the caller puts a cross-GPU barrier behind it.
struct PeerPlanes {
    uint16_t* p[kMaxPeers];
};
__global__ void __launch_bounds__(256) push_rows_kernel(const uint16_t* __restrict__ src, PeerPlanes dst, int world, uint32_t W, uint32_t H,
                                                        uint32_t bandRows, uint32_t rank, uint32_t ownedRows) {
    const uint32_t vecPerRow = (W + 7u) / 8u;   // 8 pixels = 16 bytes
    const uint64_t total = (uint64_t)ownedRows * vecPerRow * 3u;
    const size_t P = (size_t)W * H;
    const bool aligned = (W % 8u) == 0u;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = (uint32_t)(i % vecPerRow);
        const uint64_t rowPlane = i / vecPerRow;
        const uint32_t k = (uint32_t)(rowPlane % ownedRows), plane = (uint32_t)(rowPlane / ownedRows);
        const uint32_t y = (k / bandRows) * (bandRows * (uint32_t)world) + rank * bandRows + (k % bandRows);   // map_row()
        const size_t off = plane * P + (size_t)y * W + (size_t)v * 8u;
        if (aligned) {
            const uint4 val = *reinterpret_cast<const uint4*>(src + off);
            for (int d = 0; d < world; ++d) *reinterpret_cast<uint4*>(dst.p[d] + off) = val;
        } else {
            const uint32_t n = min(8u, W - v * 8u);
            for (uint32_t e = 0; e < n; ++e) {
                const uint16_t val = src[off + e];
                for (int d = 0; d < world; ++d) dst.p[d][off + e] = val;
            }
        }
    }
}

bool frame_push_rows(Frame* f, uint32_t bandRows, uint32_t rank, uint32_t world, void* const* peerPlanes, void* stream, std::string& err) {
    if (!f || !peerPlanes || bandRows == 0 || world == 0 || world > kMaxPeers || rank >= world) {
        err = "bad push request";
        return false;
    }
    OCLR_CUDA(cudaSetDevice(f->scene->device));
    const uint32_t owned = band_owned_rows(f->cam.height, bandRows, rank, world);
    if (owned == 0) return true;
    PeerPlanes dst = {};
    for (uint32_t d = 0; d < world; ++d) {
        if (!peerPlanes[d]) {
            err = "null peer plane pointer";
            return false;
        }
        dst.p[d] = (uint16_t*)peerPlanes[d];
    }
    const uint64_t total = (uint64_t)owned * ((f->cam.width + 7u) / 8u) * 3u;
    const unsigned grid = (unsigned)std::min<uint64_t>((total + 255) / 256, (uint64_t)f->scene->smCount * 8);
    push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)f->planesRGB.p, dst, (int)world, f->cam.width, f->cam.height, bandRows,
                                                             rank, owned);
    OCLR_CUDA(cudaGetLastError());
    return true;
}

void frame_device_planes(Frame* f, void** r, void** g, void** b) {
    const size_t P = (size_t)f->cam.width * f->cam.height;
    uint16_t* d = (uint16_t*)f->planesRGB.p;
    *r = d;
    *g = d + P;
    *b = d + 2 * P;
}

// ---- batched ray queries (rt_query.cuh) ------------------------------------------------------------------------------------------------
// A device pointer the trace stage may read with 16-byte loads: device memory of the scene's device, aligned to `align`.
static bool query_pointer_ok(const Scene* s, const void* p, size_t align, const char* what, std::string& err) {
    if ((uintptr_t)p % align != 0) {
        err = std::string(what) + " is not " + std::to_string(align) + "-byte aligned";
        return false;
    }
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        err = std::string(what) + " is not a CUDA pointer";
        return false;
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != s->device) {
        err = std::string(what) + " is not device memory of the scene's device (" + std::to_string(s->device) + ")";
        return false;
    }
    return true;
}

// Caller rays of one query call (scene_query, scene_radiance): the argument checks, the host-memory staging of each batch, the result
// download and the call's statistics.  Buffers are stream-ordered and released on the call's stream whichever way the call ends, so that
// calls on one scene from different streams share nothing.
struct CallerRays {
    Scene* s;
    size_t count;
    const float* origin4;
    const float* direction4;
    const uint32_t* excluded;
    float* out4;
    uint8_t* flags;   // radiance's optional per-ray flags
    bool deviceMemory;
    cudaStream_t st;
    DeviceBuffer inO, inD, inExcl, out, outFlags, counters;
    Counters* dcnt = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint32_t* pinned = nullptr;   // read-back words of the call's rounds
    ~CallerRays() {
        for (DeviceBuffer* b : {&inO, &inD, &inExcl, &out, &outFlags, &counters}) b->release(st);
        if (s) {
            drop_event(s->device, ev0, true);
            drop_event(s->device, ev1, true);
        }
        pinned_release(pinned);
    }
    // True with nothing checked beyond the scene when there are no rays.
    bool check(const char* outName, RenderStats* stats, std::string& err) {
        if (!s) {
            err = "null scene";
            return false;
        }
        if (stats) *stats = RenderStats();
        if (count == 0) return true;
        if (!origin4 || !direction4 || !out4) {
            err = "null origin, direction or output array";
            return false;
        }
        OCLR_CUDA(cudaSetDevice(s->device));
        if (deviceMemory && (!query_pointer_ok(s, origin4, 16, "origin", err) || !query_pointer_ok(s, direction4, 16, "direction", err) ||
                             !query_pointer_ok(s, out4, 16, outName, err) || (excluded && !query_pointer_ok(s, excluded, 4, "excluded", err)) ||
                             (flags && !query_pointer_ok(s, flags, 1, "flags", err))))
            return false;
        return packed_walk_ok(s->view, err);
    }
    // Staging for batches of up to b rays and the counters block, then the start of the call's timing.
    bool begin(size_t b, bool counting, RenderStats* stats, std::string& err) {
        if ((counting && !counters.alloc(sizeof(Counters), err, st)) ||
            (!deviceMemory && (!inO.alloc(sizeof(float4) * b, err, st) || !inD.alloc(sizeof(float4) * b, err, st) ||
                               (excluded && !inExcl.alloc(sizeof(uint32_t) * b, err, st)) || !out.alloc(sizeof(float4) * b, err, st) ||
                               (flags && !outFlags.alloc(b, err, st)))))
            return false;
        dcnt = counting ? (Counters*)counters.p : nullptr;
        if (dcnt) OCLR_CUDA(cudaMemsetAsync(dcnt, 0, sizeof(Counters), st));
        if (stats) {
            OCLR_CUDA(make_event(s->device, &ev0, true));
            OCLR_CUDA(make_event(s->device, &ev1, true));
            OCLR_CUDA(cudaEventRecord(ev0, st));
        }
        return true;
    }
    // The rays of batch [off, off + n) as device arrays (host memory: uploaded into the staging buffers).
    bool rays(size_t off, uint32_t n, const float4*& origin, const float4*& direction, const uint32_t*& excl, std::string& err) {
        if (deviceMemory) {
            origin = (const float4*)origin4 + off;
            direction = (const float4*)direction4 + off;
            excl = excluded ? excluded + off : nullptr;
            return true;
        }
        if (!host_to_device(inO.p, origin4 + 4 * off, sizeof(float4) * n, st, err) ||
            !host_to_device(inD.p, direction4 + 4 * off, sizeof(float4) * n, st, err) ||
            (excluded && !host_to_device(inExcl.p, excluded + off, sizeof(uint32_t) * n, st, err)))
            return false;
        origin = (const float4*)inO.p;
        direction = (const float4*)inD.p;
        excl = excluded ? (const uint32_t*)inExcl.p : nullptr;
        return true;
    }
    float4* result(size_t off) const { return deviceMemory ? (float4*)out4 + off : (float4*)out.p; }
    uint8_t* flag_out(size_t off) const { return !flags ? nullptr : deviceMemory ? flags + off : (uint8_t*)outFlags.p; }
    // Results of batch [off, off + n) back to host memory (device memory is written in place).
    bool download(size_t off, uint32_t n, std::string& err) {
        return deviceMemory || (device_to_host(out4 + 4 * off, out.p, sizeof(float4) * n, st, err) &&
                                (!flags || device_to_host(flags + off, outFlags.p, n, st, err)));
    }
    bool finish(RenderStats* stats, uint32_t launches, uint32_t rounds, std::string& err) {
        if (!stats) return true;
        OCLR_CUDA(cudaEventRecord(ev1, st));
        OCLR_CUDA(cudaEventSynchronize(ev1));
        OCLR_CUDA(cudaEventElapsedTime(&stats->deviceMs, ev0, ev1));
        stats->launches = launches;
        stats->traceLaunches = rounds;
        if (dcnt) OCLR_CUDA(cudaMemcpy(&stats->counters, dcnt, sizeof(Counters), cudaMemcpyDeviceToHost));
        return true;
    }
};

// Scratch of one query call besides its caller rays, stream-ordered like them.
struct QueryScratch {
    DeviceBuffer recO, recD, recS0, recS1, order, queue, excl, counters, hit, rayO;
    cudaStream_t st = nullptr;
    ~QueryScratch() {
        for (DeviceBuffer* b : {&recO, &recD, &recS0, &recS1, &order, &queue, &excl, &counters, &hit, &rayO}) b->release(st);
    }
};

static bool scene_query(Scene* s, bool transmit, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded,
                        float* out4, bool deviceMemory, bool counting, void* stream, RenderStats* stats, std::string& err) {
    cudaStream_t st = (cudaStream_t)stream;
    CallerRays rays = {s, count, origin4, direction4, excluded, out4, nullptr, deviceMemory, st};
    if (!rays.check(transmit ? "att" : "hit", stats, err)) return false;
    if (count == 0) return true;
    const SceneView& S = s->view;
    QueryScratch q;
    q.st = st;
    const uint32_t B = (uint32_t)std::min<size_t>(count, kQueryBatch);
    const size_t b = B;
    if (!q.recO.alloc(sizeof(float4) * b, err, st) || !q.recD.alloc(sizeof(float4) * b, err, st) || !q.recS0.alloc(sizeof(float4) * b, err, st) ||
        !q.recS1.alloc(sizeof(uint4) * b, err, st) || !q.order.alloc(sizeof(uint32_t) * b * kLengthClasses, err, st) ||
        !q.queue.alloc(sizeof(uint32_t) * b * (transmit ? 2 : 1), err, st) || !q.excl.alloc(sizeof(uint32_t) * b, err, st) ||
        !q.counters.alloc(sizeof(uint32_t) * (2 * kCounterStride + kRoundLogSize), err, st) ||
        (transmit && (!q.hit.alloc(sizeof(float4) * b, err, st) || !q.rayO.alloc(sizeof(float4) * b, err, st))) ||
        !rays.begin(b, counting, stats, err))
        return false;
    Counters* dcnt = rays.dcnt;
    unsigned traceGrid = 0;
    if (!trace_grid(S, s->smCount, counting, traceGrid, err)) return false;
    const unsigned setupGrid = (unsigned)std::min<uint64_t>((uint64_t)s->smCount * 8, (b + 255) / 256);
    const unsigned rayGrid = (unsigned)std::min<uint64_t>((uint64_t)s->smCount * 16, (b + 127) / 128);
    uint32_t* counters = (uint32_t*)q.counters.p;
    const uint32_t cstride = kCounterStride;
    if (transmit && !(rays.pinned = (uint32_t*)pinned_block())) {
        err = "out of pinned host memory";
        return false;
    }
    uint32_t launches = 0, rounds = 0;
    for (size_t off = 0; off < count; off += b) {
        const uint32_t n = (uint32_t)std::min<size_t>(b, count - off);
        QueryBatch qb;
        qb.count = n;
        qb.excl = (uint32_t*)q.excl.p;
        if (!rays.rays(off, n, qb.origin, qb.direction, qb.excluded, err)) return false;
        float4* result = rays.result(off);
        qb.hit = transmit ? (float4*)q.hit.p : result;
        qb.rayO = transmit ? (float4*)q.rayO.p : nullptr;
        qb.att = transmit ? result : nullptr;
        WfState w = {};
        w.Q = B;
        w.rayO = transmit ? qb.rayO : (float4*)qb.origin;   // (the trace stage only reads rayO / rayD / rayExcl)
        w.rayD = (float4*)qb.direction;
        w.rayExcl = qb.excl;
        w.hit = qb.hit;
        w.roundLog = counters + 2 * cstride;
        WalkRecords rec = {(float4*)q.recO.p, (float4*)q.recD.p, (float4*)q.recS0.p, (uint4*)q.recS1.p, (uint32_t*)q.order.p, nullptr, B};
        auto use_set = [&](WfState& v, uint32_t r) {
            v.queue = (uint32_t*)q.queue.p + (transmit ? (size_t)(r & 1u) * b : 0);
            v.queueCount = counters + cstride * (r & 1u);
            v.queueCursor = v.queueCount + 1;
        };
        use_set(w, 0);
        OCLR_CUDA(cudaMemsetAsync(w.queueCount, 0, sizeof(uint32_t) * cstride, st));
        query_screen_kernel<<<rayGrid, 128, 0, st>>>(qb, w);
        ++launches;
        // Rounds (trace -> transmit) are enqueued ahead in chunks without a host round trip, as frames do (RoundDriver): every kernel
        // reads its ray count from device memory and returns at once when there is nothing to do.  One read per chunk: the count the last
        // transmit round queued.
        for (uint32_t r = 0;;) {
            const uint32_t chunk = transmit ? 3u : 1u;
            for (uint32_t c = 0; c < chunk; ++c, ++r) {
                use_set(w, r);
                w.roundIndex = r;
                rec.classCount = w.queueCount + 2;
                const TailQueue tq = {nullptr, w.queueCount + 2 + kLengthClasses, w.queueCount + 6 + kLengthClasses, 0u,
                                      nullptr, nullptr, nullptr, nullptr, nullptr};
                enqueue_trace(S, s->walkView, w, rec, tq, setupGrid, traceGrid, s->smCount, dcnt, st, launches);
                ++rounds;
                if (!transmit) break;
                WfState next = w;
                use_set(next, r + 1);
                OCLR_CUDA(cudaMemsetAsync(next.queueCount, 0, sizeof(uint32_t) * cstride, st));
                query_transmit_kernel<<<rayGrid, 128, 0, st>>>(S, qb, w.queue, w.queueCount, next);
                ++launches;
            }
            if (!transmit) break;
            OCLR_CUDA(cudaMemcpyAsync(rays.pinned, counters + cstride * (r & 1u), sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            OCLR_CUDA(cudaStreamSynchronize(st));
            if (*rays.pinned == 0) break;
            if (r > 100000) {
                err = "transmittance did not converge";
                return false;
            }
        }
        OCLR_CUDA(cudaGetLastError());
        if (!rays.download(off, n, err)) return false;
    }
    return rays.finish(stats, launches, rounds, err);
}

bool scene_intersect(Scene* s, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded, float* hit4,
                     bool deviceMemory, bool counting, void* stream, RenderStats* stats, std::string& err) {
    return scene_query(s, false, count, origin4, direction4, excluded, hit4, deviceMemory, counting, stream, stats, err);
}

bool scene_transmittance(Scene* s, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded, float* att4,
                         bool deviceMemory, bool counting, void* stream, RenderStats* stats, std::string& err) {
    return scene_query(s, true, count, origin4, direction4, excluded, att4, deviceMemory, counting, stream, stats, err);
}

// ---- radiance along caller rays (rt_query.cuh radiance_start_kernel, then the frame's wf_logic_kernel) ---------------------------------
// Scratch of one radiance call besides its caller rays: the path state of one batch and its per-ray sums, stream-ordered like them.
struct RadianceScratch {
    PathState ps;
    DeviceBuffer accum, firstHit;
    cudaStream_t st = nullptr;
    ~RadianceScratch() {
        ps.release(st);
        accum.release(st);
        firstHit.release(st);
    }
};

bool scene_radiance(Scene* s, const Camera* cam, size_t count, const float* origin4, const float* direction4, const uint32_t* excluded,
                    unsigned long long indexBase, uint32_t sampleCount, float* rgb4, uint8_t* flags, bool deviceMemory, bool counting,
                    void* stream, RenderStats* stats, std::string& err) {
    // (a null scene is refused by CallerRays::check)
    if (s && sampleCount < 1) {
        err = "sampleCount must be at least 1";
        return false;
    }
    if (s && !cam && s->hasBump) {
        err = "null camera: the scene has bump-mapped materials, whose normals read the camera's leftToRight / topToBottom / pixelSizeInv";
        return false;
    }
    cudaStream_t st = (cudaStream_t)stream;
    CallerRays rays = {s, count, origin4, direction4, excluded, rgb4, flags, deviceMemory, st};
    if (!rays.check("rgb", stats, err)) return false;
    if (count == 0) return true;
    const SceneView& S = s->view;
    RadianceScratch q;
    q.st = st;
    const uint32_t B = (uint32_t)std::min<size_t>(count, kRadianceBatch);
    const size_t b = B;
    const uint32_t W = kRadianceRowWidth, Q = (B + W - 1) / W * W;   // paths: the batch as a W-wide image (rt_query.cuh)
    if (!q.ps.reserve(Q, s->ringSlots, st, err) || !q.accum.alloc(sizeof(float4) * Q, err, st) ||
        !q.firstHit.alloc(sizeof(uint32_t) * Q, err, st) || !rays.begin(b, counting, stats, err))
        return false;
    if (!(rays.pinned = (uint32_t*)pinned_block())) {
        err = "out of pinned host memory";
        return false;
    }
    Counters* dcnt = rays.dcnt;
    RoundDriver drv = {S, s->walkView, s->device, s->smCount, 0u, dcnt, rays.pinned, nullptr, "radiance query"};
    if (!trace_grid(S, s->smCount, counting, drv.traceGrid, err)) return false;
    const int aheadMode = ahead_mode_for(Q);   // (no camera segments: modes 1 and 2 coincide)
    const bool cull = g_cullHidden.load();
    uint32_t lastRounds = 4;
    drv.K = 1;
    RoundDomain& d = drv.dom[0];
    d.ps = &q.ps;
    q.ps.bind(Q, s->ringSlots, d.w, d.rec);
    d.st = st;
    d.lastRounds = &lastRounds;
    FrameView F = {};   // the logic kernel's view of a batch: camera vectors, sample count, accumulator, flags (rt_query.cuh)
    if (cam) F.cam = *cam;
    F.cam.width = W;
    F.sampleCount = sampleCount;
    F.accum = (float4*)q.accum.p;
    for (size_t off = 0; off < count; off += b) {
        const uint32_t n = (uint32_t)std::min<size_t>(b, count - off);
        RayBatch R;
        R.count = n;
        R.indexBase = indexBase + off;
        if (!rays.rays(off, n, R.origin, R.direction, R.excluded, err)) return false;
        F.flagOut = rays.flag_out(off);
        if (F.flagOut) OCLR_CUDA(cudaMemsetAsync(F.flagOut, 0, n, st));
        const uint32_t rows = (n + W - 1) / W;
        F.cam.height = rows;
        F.rowBegin = 0;
        F.rowEnd = rows;
        const dim3 logicGrid(1, (rows + 7) / 8);
        const unsigned startGrid = (rows * W + 127) / 128, rayGrid = (n + 127) / 128;
        for (uint32_t smp = 0; smp < sampleCount; ++smp) {
            // round 0 enters at radiance_start_kernel instead of the logic kernel's kWfNew
            const RoundEntry entry = [&](int, uint32_t r, const WfState& w, const uint32_t* prev, cudaStream_t ks) {
                if (r == 0) {
                    if (dcnt)
                        radiance_start_kernel<true><<<startGrid, 128, 0, ks>>>(R, w, smp, sampleCount, dcnt);
                    else
                        radiance_start_kernel<false><<<startGrid, 128, 0, ks>>>(R, w, smp, sampleCount, dcnt);
                    return;
                }
                if (r == 1 && smp == 0)   // the trace of round 0 holds each ray's own closest hit
                    radiance_first_hit_kernel<<<rayGrid, 128, 0, ks>>>(n, w.hit, (uint32_t*)q.firstHit.p);
                if (dcnt)
                    wf_logic_kernel<true><<<logicGrid, 128, 0, ks>>>(S, F, w, smp, 0u, prev, dcnt, aheadMode, false);
                else
                    wf_logic_kernel<false><<<logicGrid, 128, 0, ks>>>(S, F, w, smp, 0u, prev, dcnt, aheadMode, cull);
            };
            if (!drv.run(nullptr, entry, err)) return false;
        }
        radiance_resolve_kernel<<<rayGrid, 128, 0, st>>>(R, (const float4*)q.accum.p, (const uint32_t*)q.firstHit.p, sampleCount,
                                                          rays.result(off));
        ++drv.launches;
        OCLR_CUDA(cudaGetLastError());
        if (!rays.download(off, n, err)) return false;
    }
    return rays.finish(stats, drv.launches, drv.rounds, err);
}

// ---- edits of a resident scene and of a frame's camera -----------------------------------------------------------------------------------
bool frame_set_camera(Frame* f, const Camera& cam, const uint32_t* camStart, const uint32_t* camEnd, const uint32_t* camList, size_t listSize,
                      std::string& err) {
    if (!f) {
        err = "null frame";
        return false;
    }
    if (cam.width != f->cam.width || cam.height != f->cam.height) {
        err = "the new camera is " + std::to_string(cam.width) + "x" + std::to_string(cam.height) + ", the frame " + std::to_string(f->cam.width) +
              "x" + std::to_string(f->cam.height) + ": a frame keeps its image size (create a new frame)";
        return false;
    }
    // From here on the frame holds the new camera; whatever fails below leaves it without lists (it refuses to render until a camera is
    // set successfully), never with the old camera's lists under the new camera.
    f->cam = cam;
    f->deviceLists = false;
    f->listsGen = kNoLists;
    OCLR_CUDA(cudaSetDevice(f->device));
    // every launch that may read the old lists has finished (a round started ahead included) before they are replaced
    OCLR_CUDA(cudaDeviceSynchronize());
    f->prelaunched = false;
    for (DeviceBuffer* b : {&f->camStart, &f->camEnd, &f->camList, &f->camCheck}) b->release();
    f->camListSize = 0;
    if (!camStart) return frame_build_camera_lists(f, err);
    if (!frame_upload_lists(f, camStart, camEnd, camList, listSize, err, nullptr)) {
        f->listsGen = kNoLists;
        return false;
    }
    OCLR_CUDA(cudaStreamSynchronize(0));   // (the caller's arrays may go once the call returns)
    return true;
}

// The device arrays of a geometry update: caller device memory used in place, or host arrays uploaded.
struct GeometryInputs {
    DeviceBuffer vertex, triIdx, triMat, triUv, triNormal, boxMin, gridStart;
    const void* p[7] = {};   // the arrays in that order, in device memory
    ~GeometryInputs() {
        for (DeviceBuffer* b : {&vertex, &triIdx, &triMat, &triUv, &triNormal, &boxMin, &gridStart}) b->release();
    }
};

bool scene_update(Scene* s, const HostScene& h, unsigned parts, bool deviceMemory, std::string& err) {
    if (!s) {
        err = "null scene";
        return false;
    }
    const bool lights = parts & kSceneLights, materials = parts & kSceneMaterials, geometry = parts & kSceneGeometry;
    // The arrays of the parts named, checked like a scene of their own (the resident grid size stands in when the geometry stays).
    HostScene v;
    if (geometry) {
        v.vertexCount = h.vertexCount;
        v.vertex = h.vertex;
        v.triangleCount = h.triangleCount;
        v.triIdx = h.triIdx;
        v.triMat = h.triMat;
        v.triUv = h.triUv;
        v.triNormal = h.triNormal;
        v.axesDivCount = h.axesDivCount;
        v.boxMin = h.boxMin;
        v.gridStart = h.gridStart;
        v.gridList = h.gridList;
    } else {
        v.axesDivCount = s->view.n;
    }
    if (materials) {
        v.materialCount = h.materialCount;
        v.matSize = h.matSize;
        v.matStart = h.matStart;
        v.texturesSize = h.texturesSize;
        v.textures = h.textures;
    }
    if (lights) {
        v.lightCount = h.lightCount;
        v.lightType = h.lightType;
        v.lightPos = h.lightPos;
        v.lightDir = h.lightDir;
        v.lightColour = h.lightColour;
        v.lightRadius = h.lightRadius;
        v.lightHalf = h.lightHalf;
    }
    if (!validate_scene(v, err, true)) return false;
    OCLR_CUDA(cudaSetDevice(s->device));
    const int n = v.axesDivCount;
    const size_t N = v.triangleCount, cells = (size_t)n * n * n;
    const bool buildGrid = geometry && !v.gridStart;
    if (geometry && deviceMemory) {
        const struct {
            const void* p;
            size_t align;
            const char* what;
        } arrays[] = {{v.vertex, 16, "vertex"}, {v.triIdx, 16, "triangleVertexIndex"}, {v.triMat, 4, "triangleMaterialId"},
                      {v.triUv, 8, "triangleUv"}, {v.triNormal, 16, "triangleNormal"}, {v.boxMin, 16, "sceneBoxMin"},
                      {v.gridStart, 4, "scenePixelTriangleListStart"}, {v.gridList, 4, "scenePixelTriangleList"}};
        for (const auto& a : arrays)
            if (a.p && !query_pointer_ok(s, a.p, a.align, a.what, err)) return false;
    }
    // every piece of work already enqueued on the device (renders and queries on this scene among it) ends before anything changes
    OCLR_CUDA(cudaDeviceSynchronize());
    stage_reset(s->device);
    // The new parts are built beside the resident ones and swapped in on success.  The scratch owns whatever it holds when the call
    // ends: the new buffers after a failure (whichever way it returns), the replaced ones after a success.
    struct Scratch {
        Scene t;
        DeviceBuffer errFlag;
        ~Scratch() {
            cudaDeviceSynchronize();   // (staged copies and kernels that touch the buffers have ended)
            for (DeviceBuffer* b : t.buffers()) b->release();
            errFlag.release();
        }
    } x;
    Scene& t = x.t;
    t.device = s->device;
    GeometryInputs in;
    std::vector<Light> packed;
    if (!x.errFlag.alloc(sizeof(uint32_t) * 2, err)) return false;
    OCLR_CUDA(cudaMemsetAsync(x.errFlag.p, 0, sizeof(uint32_t) * 2, 0));
    uint32_t* flagDev = (uint32_t*)x.errFlag.p;
    if (lights) {
        pack_lights(v, packed);
        if (!t.lights.upload(packed.data(), sizeof(Light) * packed.size(), err)) return false;
    }
    const uint32_t M = materials ? v.materialCount : s->view.materialCount;
    if (materials) {
        material_rules(v, t.ringSlots, t.hasBump);
        if (!t.matSize.upload(v.matSize, sizeof(uint2) * kMaterialChannels * M, err) ||
            !t.matStart.upload(v.matStart, sizeof(int32_t) * (kMaterialChannels * M + (M ? 1 : 0)), err) ||
            !t.textures.upload(v.textures, sizeof(uchar4) * v.texturesSize, err))
            return false;
        if (!geometry && s->view.triangleCount)   // the resident triangles against the new material count
            check_materials_kernel<<<(s->view.triangleCount + 255) / 256, 256>>>(s->view.triangleCount, M, s->view.triShade, flagDev);
    }
    if (geometry) {
        uint32_t total = 0;
        if (!buildGrid) {
            if (deviceMemory)
                OCLR_CUDA(cudaMemcpy(&total, v.gridStart + cells, sizeof(uint32_t), cudaMemcpyDeviceToHost));
            else
                total = v.gridStart[cells];
            if (total && !v.gridList) {
                err = "scenePixelTriangleList missing";
                return false;
            }
        }
        const size_t bytes[7] = {sizeof(float4) * v.vertexCount, sizeof(int4) * N, sizeof(int32_t) * N, sizeof(float2) * 3 * N,
                                 sizeof(float4) * 3 * N, buildGrid ? 0 : sizeof(float4) * (n + 1), buildGrid ? 0 : sizeof(uint32_t) * (cells + 1)};
        const void* src[7] = {v.vertex, v.triIdx, v.triMat, v.triUv, v.triNormal, v.boxMin, v.gridStart};
        DeviceBuffer* dst[7] = {&in.vertex, &in.triIdx, &in.triMat, &in.triUv, &in.triNormal, &in.boxMin, &in.gridStart};
        for (int i = 0; i < 7; ++i) {
            if (deviceMemory) {
                in.p[i] = src[i];
            } else {
                if (!dst[i]->upload(src[i], bytes[i], err)) return false;
                in.p[i] = bytes[i] ? dst[i]->p : nullptr;
            }
        }
        if (!buildGrid && !t.cellList.alloc(sizeof(uint32_t) * total, err)) return false;
        if (total) {
            if (deviceMemory)
                OCLR_CUDA(cudaMemcpyAsync(t.cellList.p, v.gridList, sizeof(uint32_t) * total, cudaMemcpyDeviceToDevice, 0));
            else if (!host_to_device(t.cellList.p, v.gridList, sizeof(uint32_t) * total, 0, err))
                return false;
        }
        if (!pack_stage(&t, (uint32_t)N, v.vertexCount, M, (const float4*)in.p[0], (const int4*)in.p[1], (const int32_t*)in.p[2],
                        (const float2*)in.p[3], (const float4*)in.p[4], flagDev, err) ||
            !grid_stage(&t, n, v.vertexCount, (const float4*)in.p[0], (uint32_t)N, (const int4*)in.p[1], (const float4*)in.p[5],
                        (const uint32_t*)in.p[6], total, flagDev, err))
            return false;
    }
    uint32_t flag = 0;
    cudaMemcpyAsync(&flag, flagDev, sizeof(uint32_t), cudaMemcpyDeviceToHost, 0);
    cudaError_t e = cudaStreamSynchronize(0);
    if (e != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        err = std::string("scene update: ") + cudaGetErrorString(e);
        return false;
    }
    if (flag) {
        err = pack_error_message(flag);
        return false;
    }
    // success: the new parts in, the old ones out
    if (lights) std::swap(s->lights, t.lights);
    if (materials) {
        for (DeviceBuffer Scene::*b : {&Scene::matSize, &Scene::matStart, &Scene::textures}) std::swap(s->*b, t.*b);
        s->ringSlots = t.ringSlots;
        s->hasBump = t.hasBump;
    }
    if (geometry) {
        for (DeviceBuffer Scene::*b : {&Scene::triGeo, &Scene::triShade, &Scene::bricks, &Scene::cellRange, &Scene::cellList, &Scene::faceMask,
                                       &Scene::planes, &Scene::walkBricks, &Scene::walkCellRange, &Scene::walkFaceMask, &Scene::walkPlanes})
            std::swap(s->*b, t.*b);
        s->walkTrim = t.walkTrim;
        ++s->geometryGen;
    }
    bind_view(s, geometry ? v.triangleCount : s->view.triangleCount, M, lights ? v.lightCount : s->view.lightCount, n);
    return true;   // (the scratch releases the replaced buffers)
}

}  // namespace oclr
