// common.cuh -- shared host/device helpers for libeast_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#define EAST_TERM_BASE 0x0A00u  // east/consts.py:24 UNICODE_SPECIAL_SYMBOLS_START
#define EAST_NUM_SMS 148        // B200: 2 dies x 74 SMs; grids are sized in multiples of this

namespace east {

struct Error : public std::runtime_error {
    int status;
    Error(int st, const std::string &m) : std::runtime_error(m), status(st) {}
};

#define EAST_CUDA(expr)                                                                      \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess)                                                               \
            throw ::east::Error(-2, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

extern thread_local int64_t g_launches;
extern thread_local int g_time_kernels;     // option "time_kernels": CUDA events around every launch
extern thread_local double g_next_bytes;    // algorithmic bytes of the next launch (roofline numerator)
void ktime_begin(const char *name, cudaStream_t s);
void ktime_end(cudaStream_t s);
void ktime_collect();
void host_debug_mark(const char *what);   // EAST_DEBUG_TIMING: host timestamp on stderr  // after a stream sync: fold the pending event pairs into the per-kernel table

// every kernel launch of the library goes through this macro so bench.py can report
// "gpu_launches" from a real count and per-kernel device time measured live with CUDA events
#define EAST_LAUNCH(kernel, grid, block, smem, stream, ...)                                  \
    do {                                                                                     \
        if (::east::g_time_kernels) ::east::ktime_begin(#kernel, (stream));                  \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                          \
        if (::east::g_time_kernels) ::east::ktime_end((stream));                             \
        ++::east::g_launches;                                                                \
        ::east::g_next_bytes = 0.0;                                                          \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess)                                                               \
            throw ::east::Error(-2, std::string(#kernel) + " launch: " + cudaGetErrorString(_e)); \
    } while (0)
// the same for an instance of a kernel template, counted and timed under `name` (every instance under one name)
#define EAST_LAUNCH_AS(name, kernel, grid, block, smem, stream, ...)                         \
    do {                                                                                     \
        if (::east::g_time_kernels) ::east::ktime_begin((name), (stream));                   \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__);                          \
        if (::east::g_time_kernels) ::east::ktime_end((stream));                             \
        ++::east::g_launches;                                                                \
        ::east::g_next_bytes = 0.0;                                                          \
        cudaError_t _e = cudaGetLastError();                                                 \
        if (_e != cudaSuccess)                                                               \
            throw ::east::Error(-2, std::string(name) + " launch: " + cudaGetErrorString(_e)); \
    } while (0)
#define EAST_BYTES(b) (::east::g_next_bytes = (double)(b))

// Stream-ordered allocations from two library-private memory pools per device (the device's default pool and its
// attributes are left alone: the caller's framework allocates there).  `big`: the arena of an index and the text
// buffers -- a few large blocks whose sizes repeat from call to call, so a freed block is reused whole; everything else
// (scratch of a build or score call) comes from the other pool.  Both keep freed memory up to a bounded release
// threshold; east_trim() gives it back.
void *dev_alloc(size_t bytes, cudaStream_t s, bool big = false);
void dev_free(void *p, cudaStream_t s);

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaStream_t s = 0;
    bool owned = true;   // false: a slice of an index arena (freed with the arena)
    DevBuf() {}
    DevBuf(size_t n_, cudaStream_t s_) : n(n_), s(s_) {
        const size_t bytes = sizeof(T) * (n_ ? n_ : 1);
        p = (T *)dev_alloc(bytes, s_, bytes >= ((size_t)32 << 20));   // large scratch: the library's own block cache
    }
    DevBuf(T *slice, size_t n_) : p(slice), n(n_), owned(false) {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n), s(o.s), owned(o.owned) { o.p = nullptr; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; s = o.s; owned = o.owned; o.p = nullptr; }
        return *this;
    }
    void release() { if (p) { if (owned) dev_free(p, s); p = nullptr; } }
    ~DevBuf() { release(); }
};

// One allocation that holds every array of an index (suffix array, tables, byte text, bucket tables ...): a bump
// allocator over an upper bound computed before the build.  take() falls back to an allocation of its own when the
// bound turns out too small; rewind() gives back what a failed pass (speculative pipelined build, bucket overflow) took.
struct Arena {
    uint8_t *base = nullptr;
    size_t cap = 0, used = 0;
    template <typename T>
    DevBuf<T> take(size_t count, cudaStream_t s) {
        const size_t bytes = (sizeof(T) * (count ? count : 1) + 255) & ~(size_t)255;
        if (base && used + bytes <= cap) {
            T *p = reinterpret_cast<T *>(base + used);
            used += bytes;
            return DevBuf<T>(p, count);
        }
        return DevBuf<T>(count, s);
    }
    bool holds(const void *p) const { return base && (const uint8_t *)p >= base && (const uint8_t *)p < base + cap; }
    static size_t padded(size_t bytes) { return (bytes + 255) & ~(size_t)255; }
};

// per-stage device timing with CUDA events on the launching stream
struct StageTimer {
    cudaStream_t s;
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> names;
    explicit StageTimer(cudaStream_t s_) : s(s_) {}
    void mark(const char *name);  // closes the previous stage, opens `name`
    void finish();                // closes the last stage
    void collect();               // after stream sync: publish to the thread-local table
    ~StageTimer();
};

static inline int bits_for(uint64_t v) {  // number of bits needed to represent v (0 -> 0)
    int b = 0;
    while (v) { ++b; v >>= 1; }
    return b;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device setting: a process that indexes on several devices
// (the `device` argument of the C ABI) must opt in on each of them, once
static inline void ensure_dynamic_smem(const void *kernel, int bytes) {
    static std::mutex m;
    static std::set<std::pair<const void *, int>> done;
    int dev = 0;
    EAST_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> g(m);
    if (done.count({kernel, dev})) return;
    EAST_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.insert({kernel, dev});
}

static inline int grid_for(int64_t work_items, int per_block, int max_waves = 8) {
    int64_t g = (work_items + per_block - 1) / per_block;
    if (g < 1) g = 1;
    int64_t cap = (int64_t)EAST_NUM_SMS * max_waves;
    if (g > cap) g = cap;
    return (int)g;
}

}  // namespace east

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
#ifdef __CUDACC__
namespace east {

// largest d with doc_off[d] <= x   (doc_off has D+1 entries, doc_off[0]==0, x < doc_off[D])
__device__ __forceinline__ int doc_of(const int32_t *__restrict__ doc_off, int D, int32_t x) {
    int lo = 0, hi = D - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (__ldg(doc_off + mid) <= x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

}  // namespace east
#endif
