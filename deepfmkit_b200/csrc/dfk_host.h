// Host-side internals shared by the translation units of libdfk_b200.so: the context, error reporting, scratch
// buffers, the staged host -> device copy.  Not part of the ABI (include/dfk_b200.h is).
#pragma once
#include "../../include/dfk_b200.h"

#include <cuda_runtime.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include <algorithm>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>


inline thread_local char g_err[512] = "";

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define DFK_CUDA(call)                                                                              \
    do {                                                                                            \
        const cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                      \
            return fail(DFK_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

struct DevBuf {
    void* ptr = nullptr;
    size_t bytes = 0;
};


struct dfk_ctx {
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;
    int smem_per_sm = 0;
    cudaStream_t own_stream = nullptr, copy_stream = nullptr, aux_stream = nullptr, user_stream = nullptr;
    bool use_user = false;
    cudaEvent_t copied[2] = {nullptr, nullptr}, consumed[2] = {nullptr, nullptr};
    cudaEvent_t fork = nullptr, join = nullptr;
    // pageable host records are staged through pinned buffers filled by a few copy threads
    static constexpr int kStagers = 8;               // allocated on first use, as many as HostCopyTuning::stagers
    static constexpr size_t kStageBytes = 64u << 20;
    void* stager[kStagers] = {};
    cudaEvent_t stager_free[kStagers] = {};
    DevBuf qi, dc, retry, counters, slab[2], rows, stats, stats_part, misc, qi_seed, dc_seed;
    DevBuf cov;  // covariance rows of a host record (dfk_nls_fit_cov_host)
    static constexpr int kPostBufs = 8;
    DevBuf post[kPostBufs];  // scratch of the ingest / spectra / generator entries (dfk_post.cu, dfk_ingest.cu)
    int64_t launches = 0;
    // text record resident in post[3] between dfk_text_load* and dfk_text_parse_dev (dfk_ingest.cu)
    int64_t text_bytes = 0, text_rows = 0, text_chunks = 0;
    int text_first = 0;
    bool stats_ready = false;      // ctx->stats already holds whole-record moments (streamed EKF)
    size_t host_slab_bytes = 0;    // 0 = defaults; else the slab size of the host-pointer entries (tests force streaming)
    // optional per-kernel-class timing (bench.py's roofline figures): event pairs recorded around the
    // demod launch [0], the LM launches [1], the side-stream seed fits [2] and the EKF kernel [3], summed on read
    bool profiling = false;
    static constexpr int kProfSlots = 512;
    cudaEvent_t prof_ev[DFK_PROFILE_KINDS][kProfSlots][2] = {};
    int prof_used[DFK_PROFILE_KINDS] = {};
    double prof_ms[DFK_PROFILE_KINDS] = {};
    int64_t prof_n[DFK_PROFILE_KINDS] = {};
    cudaStream_t stream() const { return use_user ? user_stream : own_stream; }
};


inline int ensure(dfk_ctx* ctx, DevBuf& b, size_t bytes) {
    if (b.bytes >= bytes) return DFK_OK;
    if (b.ptr) {
        // scratch may still be in use by kernels queued on the stream
        DFK_CUDA(cudaStreamSynchronize(ctx->stream()));
        DFK_CUDA(cudaFree(b.ptr));
        b.ptr = nullptr;
        b.bytes = 0;
    }
    const size_t want = std::max(bytes, static_cast<size_t>(256));
    const cudaError_t e = cudaMalloc(&b.ptr, want);
    if (e != cudaSuccess) {
        b.ptr = nullptr;
        return fail(e == cudaErrorMemoryAllocation ? DFK_ERR_NOMEM : DFK_ERR_CUDA, "cudaMalloc(%zu) failed: %s", want,
                    cudaGetErrorString(e));
    }
    b.bytes = want;
    return DFK_OK;
}

inline int prof_drain(dfk_ctx* ctx) {  // fold recorded event pairs into the totals (synchronises)
    for (int k = 0; k < DFK_PROFILE_KINDS; ++k) {
        for (int i = 0; i < ctx->prof_used[k]; ++i) {
            DFK_CUDA(cudaEventSynchronize(ctx->prof_ev[k][i][1]));
            float ms = 0.f;
            DFK_CUDA(cudaEventElapsedTime(&ms, ctx->prof_ev[k][i][0], ctx->prof_ev[k][i][1]));
            ctx->prof_ms[k] += ms;
            ctx->prof_n[k]++;
        }
        ctx->prof_used[k] = 0;
    }
    return DFK_OK;
}

struct ProfScope {  // records an event pair around the launches issued while it lives
    dfk_ctx* ctx;
    int kind, slot;
    cudaStream_t st;
    ProfScope(dfk_ctx* c, int k, cudaStream_t s) : ctx(c), kind(k), slot(-1), st(s) {
        if (!ctx->profiling) return;
        if (ctx->prof_used[kind] == dfk_ctx::kProfSlots && prof_drain(ctx) != DFK_OK) return;
        slot = ctx->prof_used[kind];
        for (int e = 0; e < 2; ++e)
            if (!ctx->prof_ev[kind][slot][e] && cudaEventCreate(&ctx->prof_ev[kind][slot][e]) != cudaSuccess) {
                slot = -1;
                return;
            }
        cudaEventRecord(ctx->prof_ev[kind][slot][0], st);
    }
    ~ProfScope() {
        if (slot < 0) return;
        cudaEventRecord(ctx->prof_ev[kind][slot][1], st);
        ctx->prof_used[kind] = slot + 1;
    }
};

struct Guard {  // make the context's device current for the duration of a call
    int prev = -1;
    bool ok = false;
    explicit Guard(const dfk_ctx* ctx) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(ctx->device) == cudaSuccess;
    }
    ~Guard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Host-pointer entries enqueue DMA from caller memory and from the pinned stagers on three streams.  If such a call
// leaves early on an error, everything already queued must drain before the caller may free or reuse its record.
struct HostCallGuard {
    dfk_ctx* ctx;
    bool finished = false;
    explicit HostCallGuard(dfk_ctx* c) : ctx(c) {}
    void done() { finished = true; }
    ~HostCallGuard() {
        if (finished) return;
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(ctx->aux_stream);
        cudaStreamSynchronize(ctx->stream());
    }
};

#define DFK_ENTER(ctx)                                             \
    if (!(ctx)) return fail(DFK_ERR_ARG, "null context");          \
    Guard guard_(ctx);                                             \
    if (!guard_.ok) return fail(DFK_ERR_CUDA, "cudaSetDevice(%d) failed", (ctx)->device)

inline bool is_pageable(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return attr.type == cudaMemoryTypeUnregistered;
}

// A small persistent pool for the host-side halves of the staged copies (memcpy of pageable memory, pread of files
// into the pinned stagers).  Spawning threads per 64 MiB stage cost a quarter of the staged path's time.
class CopyPool {
public:
    static CopyPool& instance() {
        // never destroyed: its threads end with the process, so nothing is joined during static destruction (or in a
        // forked child, where the threads do not exist)
        static CopyPool* pool = new CopyPool();
        return *pool;
    }
    // run fn(t) for t in [0, n) on the pool's threads (the caller takes a share) and wait
    template <class Fn>
    void run(int n, Fn fn) {
        if (n <= 1) {
            if (n == 1) fn(0);
            return;
        }
        std::unique_lock<std::mutex> call(call_mutex_);  // one parallel region at a time
        {
            std::lock_guard<std::mutex> lk(m_);
            task_ = [&](int t) { fn(t); };
            next_ = 0;
            total_ = n;
            pending_ = n;
            ++generation_;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [&] { return pending_ == 0; });
        task_ = nullptr;
    }
    int size() const { return static_cast<int>(threads_.size()) + 1; }

private:
    CopyPool() {
        unsigned hw = std::thread::hardware_concurrency();
        const int n = static_cast<int>(hw ? std::min(hw, 32u) : 4u) - 1;
        for (int i = 0; i < n; ++i) threads_.emplace_back([this] { loop(); });
    }
    ~CopyPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }
    void work() {
        for (;;) {
            int t;
            {
                std::lock_guard<std::mutex> lk(m_);
                if (next_ >= total_) return;
                t = next_++;
            }
            task_(t);
            std::lock_guard<std::mutex> lk(m_);
            if (--pending_ == 0) done_.notify_all();
        }
    }
    void loop() {
        unsigned long long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return stop_ || generation_ != seen; });
                if (stop_) return;
                seen = generation_;
            }
            work();
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_, call_mutex_;
    std::condition_variable cv_, done_;
    std::function<void(int)> task_;
    int next_ = 0, total_ = 0, pending_ = 0;
    unsigned long long generation_ = 0;
    bool stop_ = false;
};

// Geometry of the staged copies (development overrides DFK_STAGE_KB, DFK_STAGERS, DFK_COPY_NT, DFK_COPY_THREADS).
struct HostCopyTuning {
    size_t stage_bytes = dfk_ctx::kStageBytes;
    int stagers = 3;
    int nt = 0;        // 1: non-temporal stores into the stager (no read-for-ownership of its lines)
    int threads = 16;  // copy threads per stage (the pool holds min(hardware, 32))
};
inline HostCopyTuning& host_copy_tuning() {
    static HostCopyTuning t;
    return t;
}

// memcpy with streaming stores; dst 32-byte aligned
#if defined(__x86_64__)
__attribute__((target("avx2"))) inline void stream_copy(char* dst, const char* src, size_t bytes) {
    size_t i = 0;
    for (; i + 128 <= bytes; i += 128) {
        const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i));
        const __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i + 32));
        const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i + 64));
        const __m256i d = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i + 96));
        _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + i), a);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + i + 32), b);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + i + 64), c);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(dst + i + 96), d);
    }
    _mm_sfence();
    if (i < bytes) std::memcpy(dst + i, src + i, bytes - i);
}
inline bool have_stream_copy() { return __builtin_cpu_supports("avx2"); }
#else
inline void stream_copy(char* dst, const char* src, size_t bytes) { std::memcpy(dst, src, bytes); }
inline bool have_stream_copy() { return false; }
#endif

inline void parallel_memcpy(void* dst, const void* src, size_t bytes) {
    CopyPool& pool = CopyPool::instance();
    const HostCopyTuning& tune = host_copy_tuning();
    const int nt = static_cast<int>(
        std::min<size_t>(static_cast<size_t>(std::min(pool.size(), std::max(1, tune.threads))), bytes / (1u << 20) + 1));
    static const bool have_avx2 = have_stream_copy();
    const bool streaming = tune.nt && have_avx2 && (reinterpret_cast<uintptr_t>(dst) & 31) == 0;
    if (nt <= 1) {
        std::memcpy(dst, src, bytes);
        return;
    }
    const size_t chunk = ((bytes / nt) + 4095) & ~static_cast<size_t>(4095);
    pool.run(nt, [=](int t) {
        const size_t lo = std::min(bytes, chunk * t), hi = std::min(bytes, chunk * (t + 1));
        if (hi <= lo) return;
        if (streaming)
            stream_copy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo);
        else
            std::memcpy(static_cast<char*>(dst) + lo, static_cast<const char*>(src) + lo, hi - lo);
    });
}

// Host -> device copy of one slab on the copy stream.  Pinned (or registered) memory goes by DMA directly; pageable
// memory -- what a numpy array from pandas is -- would make cudaMemcpyAsync stage it synchronously at ~10 GB/s, so
// it is copied by a few threads into pinned staging buffers whose DMA overlaps the next buffer's fill.
inline int copy_slab_to_device(dfk_ctx* ctx, void* dst, const void* src, size_t bytes, bool pageable) {
    if (!pageable) {
        DFK_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
        return DFK_OK;
    }
    const HostCopyTuning& tune = host_copy_tuning();
    for (int i = 0; i < tune.stagers; ++i) {
        if (!ctx->stager[i]) {
            DFK_CUDA(cudaHostAlloc(&ctx->stager[i], dfk_ctx::kStageBytes, cudaHostAllocDefault));
            DFK_CUDA(cudaEventCreateWithFlags(&ctx->stager_free[i], cudaEventDisableTiming));
        }
    }
    int k = 0;
    for (size_t off = 0; off < bytes; off += tune.stage_bytes, k = (k + 1) % tune.stagers) {
        const size_t n = std::min(tune.stage_bytes, bytes - off);
        DFK_CUDA(cudaEventSynchronize(ctx->stager_free[k]));  // (a never-recorded event counts as complete)
        parallel_memcpy(ctx->stager[k], static_cast<const char*>(src) + off, n);
        DFK_CUDA(cudaMemcpyAsync(static_cast<char*>(dst) + off, ctx->stager[k], n, cudaMemcpyHostToDevice, ctx->copy_stream));
        DFK_CUDA(cudaEventRecord(ctx->stager_free[k], ctx->copy_stream));
    }
    return DFK_OK;
}
