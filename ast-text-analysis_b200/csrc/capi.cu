// capi.cu -- the C ABI of libeast_b200.so (declared in include/east_b200.h).
#include <algorithm>
#include <array>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <map>
#include <memory>
#include <mutex>
#include <string>

#include "../../include/east_b200.h"
#include "sa_build.h"
#include "kp_prep.h"

namespace east {

thread_local int64_t g_launches = 0;
thread_local int g_time_kernels = 0;
thread_local double g_next_bytes = 0.0;

struct KernelStat { int64_t launches = 0; double ms = 0.0; double bytes = 0.0; };
struct PendingLaunch { std::string name; cudaEvent_t a, b; double bytes; };
static thread_local std::map<std::string, KernelStat> g_kstats;
static thread_local std::vector<PendingLaunch> g_pending;
static thread_local std::vector<cudaEvent_t> g_event_pool;

static cudaEvent_t pool_event() {
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e;
    EAST_CUDA(cudaEventCreate(&e));
    return e;
}
static thread_local bool g_last_timed = false;
void ktime_begin(const char *name, cudaStream_t s) {
    // level 2: only the per-document kernel (the dominant one of a table step) gets its event pair -- 40 event records
    // around the ~20 small launches of a step are host and device time of their own inside a timed region
    g_last_timed = g_time_kernels == 1 || !strcmp(name, "k_doc_suffix_sort");
    if (!g_last_timed) return;
    PendingLaunch p{name, pool_event(), pool_event(), g_next_bytes};
    EAST_CUDA(cudaEventRecord(p.a, s));
    g_pending.push_back(p);
}
void ktime_end(cudaStream_t s) { if (g_last_timed) EAST_CUDA(cudaEventRecord(g_pending.back().b, s)); }
void ktime_collect() {
    // EAST_DEBUG_TIMELINE (with option time_kernels): start offset of every launch from the first one collected
    static const bool timeline = getenv("EAST_DEBUG_TIMELINE") != nullptr;
    std::vector<PendingLaunch> still;
    for (auto &p : g_pending) {
        float ms = 0.f;
        cudaError_t e = cudaEventElapsedTime(&ms, p.a, p.b);
        if (timeline && e == cudaSuccess) {
            float off = 0.f;
            if (cudaEventElapsedTime(&off, g_pending.front().a, p.a) != cudaSuccess) cudaGetLastError();
            fprintf(stderr, "[east] timeline %8.3f ms  +%7.3f ms  %s\n", off, ms, p.name.c_str());
        }
        if (e == cudaErrorNotReady) {  // launched on the auxiliary stream and not finished yet: keep for later
            cudaGetLastError();
            still.push_back(p);
            continue;
        }
        if (e == cudaSuccess) {
            KernelStat &k = g_kstats[p.name];
            k.launches += 1; k.ms += ms; k.bytes += p.bytes;
        } else {
            cudaGetLastError();
        }
        g_event_pool.push_back(p.a);
        g_event_pool.push_back(p.b);
    }
    g_pending.swap(still);
}
static thread_local std::string g_error;
static thread_local std::vector<float> g_stage_ms;
static thread_local std::vector<std::string> g_stage_names;

static std::mutex g_opt_mutex;
static std::map<std::string, int64_t> g_options;

static int64_t get_option(const char *name, int64_t dflt) {
    std::lock_guard<std::mutex> g(g_opt_mutex);
    auto it = g_options.find(name);
    return (it == g_options.end() || it->second == 0) ? dflt : it->second;
}

// two library-private pools per device: [0] scratch, [1] large repeating blocks (index arenas, text buffers)
static std::mutex g_pool_mutex;
static std::map<int, std::array<cudaMemPool_t, 2>> g_pools;

static cudaMemPool_t pool_for(bool big) {
    int dev = 0;
    EAST_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> g(g_pool_mutex);
    auto it = g_pools.find(dev);
    if (it == g_pools.end()) {
        std::array<cudaMemPool_t, 2> pools{};
        size_t free_b = 0, total_b = 0;
        EAST_CUDA(cudaMemGetInfo(&free_b, &total_b));
        for (int k = 0; k < 2; ++k) {
            cudaMemPoolProps props = {};
            props.allocType = cudaMemAllocationTypePinned;
            props.handleTypes = cudaMemHandleTypeNone;
            props.location.type = cudaMemLocationTypeDevice;
            props.location.id = dev;
            EAST_CUDA(cudaMemPoolCreate(&pools[k], &props));
            // freed blocks stay for the next call up to this much (build/score steps reuse them); east_trim() drops them
            uint64_t thr = (uint64_t)total_b / 4;
            EAST_CUDA(cudaMemPoolSetAttribute(pools[k], cudaMemPoolAttrReleaseThreshold, &thr));
        }
        it = g_pools.emplace(dev, pools).first;
    }
    return it->second[big ? 1 : 0];
}

// Large blocks (index arenas, text buffers) are kept by the library itself when they are freed and handed out again to
// the next request of (nearly) the same size: measured on B200, a 2 GB cudaMallocFromPoolAsync costs 0.3-0.55 ms of host
// time even when the pool holds a free block of exactly that size -- a tenth of a whole table call.  A cached block
// carries the event after which its previous user is done with it.
struct BigBlock { void *p; size_t bytes; cudaEvent_t idle; };
static std::map<int, std::vector<BigBlock>> g_big_cache;     // per device, free blocks
static std::map<const void *, size_t> g_big_live;            // blocks handed out: size
static std::map<int, size_t> g_big_cached_bytes;             // per device, bytes held by the free blocks
static const size_t BIG_CACHE_BLOCKS = 48;                   // and at most a third of the device memory

static void *big_cache_take(size_t bytes, cudaStream_t s) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    BigBlock hit{nullptr, 0, nullptr};
    {
        std::lock_guard<std::mutex> g(g_pool_mutex);
        auto &v = g_big_cache[dev];
        size_t best = v.size();
        for (size_t i = 0; i < v.size(); ++i)
            if (v[i].bytes >= bytes && v[i].bytes - bytes <= bytes / 8 && (best == v.size() || v[i].bytes < v[best].bytes)) best = i;
        if (best == v.size()) return nullptr;
        hit = v[best];
        v.erase(v.begin() + best);
        g_big_cached_bytes[dev] -= hit.bytes;
        g_big_live[hit.p] = hit.bytes;
    }
    cudaStreamWaitEvent(s, hit.idle, 0);
    cudaEventDestroy(hit.idle);
    return hit.p;
}

// true: the block was kept (or freed) here
static bool big_cache_put(void *p, cudaStream_t s) {
    int dev = 0;
    size_t bytes = 0;
    {
        std::lock_guard<std::mutex> g(g_pool_mutex);
        auto it = g_big_live.find(p);
        if (it == g_big_live.end()) return false;
        bytes = it->second;
        g_big_live.erase(it);
    }
    cudaEvent_t ev = nullptr;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventRecord(ev, s) != cudaSuccess) {
        cudaGetLastError();
        if (ev) cudaEventDestroy(ev);
        cudaFreeAsync(p, s);
        return true;
    }
    std::vector<BigBlock> evict;
    {
        static size_t limit = 0;
        if (!limit) { size_t free_b = 0, total_b = 0; limit = cudaMemGetInfo(&free_b, &total_b) == cudaSuccess ? total_b / 3 : ((size_t)32 << 30); }
        std::lock_guard<std::mutex> g(g_pool_mutex);
        auto &v = g_big_cache[dev];
        size_t &held = g_big_cached_bytes[dev];
        v.push_back(BigBlock{p, bytes, ev});
        held += bytes;
        while (v.size() > 1 && (v.size() > BIG_CACHE_BLOCKS || held > limit)) {   // the oldest go back to the pool
            evict.push_back(v.front());
            held -= v.front().bytes;
            v.erase(v.begin());
        }
    }
    for (auto &b : evict) { cudaStreamWaitEvent(s, b.idle, 0); cudaEventDestroy(b.idle); cudaFreeAsync(b.p, s); }
    return true;
}

static void big_cache_drop(int dev) {
    std::vector<BigBlock> v;
    {
        std::lock_guard<std::mutex> g(g_pool_mutex);
        v.swap(g_big_cache[dev]);
        g_big_cached_bytes[dev] = 0;
    }
    for (auto &b : v) { cudaEventDestroy(b.idle); cudaFreeAsync(b.p, 0); }
}

void *dev_alloc(size_t bytes, cudaStream_t s, bool big) {
    void *p = nullptr;
    if (big && (p = big_cache_take(bytes, s)) != nullptr) return p;
    cudaError_t e = cudaMallocFromPoolAsync(&p, bytes, pool_for(big), s);
    if (e == cudaErrorMemoryAllocation && big) {   // give the cached blocks back and try once more
        cudaGetLastError();
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceSynchronize();
        big_cache_drop(dev);
        e = cudaMallocFromPoolAsync(&p, bytes, pool_for(big), s);
    }
    if (e == cudaSuccess && big) { std::lock_guard<std::mutex> g(g_pool_mutex); g_big_live[p] = bytes; }
    if (e != cudaSuccess) {
        cudaGetLastError();
        throw Error(e == cudaErrorMemoryAllocation ? -3 : -2,
                    std::string("cudaMallocFromPoolAsync(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    }
    return p;
}
void dev_free(void *p, cudaStream_t s) {
    if (!p) return;
    // an exception is unwinding the build: kernels that use the buffer may still run on the auxiliary, helper, prep or
    // copy streams (non-blocking: `s` does not order them) -- let the device finish before anything goes back to the pool
    if (std::uncaught_exceptions() > 0) cudaDeviceSynchronize();
    if (big_cache_put(p, s)) return;
    cudaFreeAsync(p, s);
}

static double host_now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
void host_debug_mark(const char *what) {
    static const bool debug = getenv("EAST_DEBUG_TIMING") != nullptr;
    if (debug) fprintf(stderr, "[east] host %.3f ms  . %s\n", host_now_ms(), what);
}
void StageTimer::mark(const char *name) {
    static const bool debug = getenv("EAST_DEBUG_TIMING") != nullptr;
    if (debug) fprintf(stderr, "[east] host %.3f ms  -> %s\n", host_now_ms(), name);
    cudaEvent_t e;
    EAST_CUDA(cudaEventCreate(&e));
    EAST_CUDA(cudaEventRecord(e, s));
    ev.push_back(e);
    names.push_back(name);
}
void StageTimer::finish() { mark(""); }
void StageTimer::collect() {
    ktime_collect();
    g_stage_ms.clear();
    g_stage_names.clear();
    for (size_t i = 0; i + 1 < ev.size(); ++i) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ev[i], ev[i + 1]) != cudaSuccess) { cudaGetLastError(); ms = -1.f; }
        g_stage_ms.push_back(ms);
        g_stage_names.push_back(names[i]);
    }
}
StageTimer::~StageTimer() { for (auto e : ev) cudaEventDestroy(e); }

static void use_device(int device) {
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        throw Error(-2, "no CUDA device available (libeast_b200 has no CPU fallback)");
    }
    if (device < 0 || device >= cnt) throw Error(-1, "bad device ordinal");
    EAST_CUDA(cudaSetDevice(device));
}

}  // namespace east

using namespace east;

struct east_index {
    int device = 0;
    int32_t n_docs = 0;
    int32_t n = 0;
    int64_t m_total = 0;
    std::vector<int32_t> doc_off;  // host copies
    std::vector<int32_t> doc_m;
    Arena arena;                    // one allocation: every array below except an owned text
    bool owns_text = false;
    uint32_t *text = nullptr;
    int32_t *d_doc_off = nullptr, *d_doc_m = nullptr;
    int32_t *sa = nullptr, *lcp = nullptr, *up = nullptr, *down = nullptr, *next = nullptr, *ann = nullptr;
    uint8_t *t8 = nullptr;          // fast path: dense byte codes of the text
    uint32_t *bkt = nullptr;        // fast path: 2-gram bucket table
    uint32_t *bkt3 = nullptr;       // per-document kernel, 5-bit symbols: 3-gram bucket table
    uint32_t *sk = nullptr;         // fast path: text bytes at offsets 2..5 of every suffix, in rank order
    std::vector<uint8_t> code_table;
    int sym_bits = 0, term_code = 0;
    int rounds = 0, fast_path = 0, key_chars = 0, key_bits = 0, doc_sorted = 0, doc_sort_overflow = 0, tables_fused = 0, pipelined = 0, pipeline_miss = 0, alphabet_miss = 0, alphabet_guessed = 0;
    uint32_t active_after_round0 = 0;
    // LCP / child / annotation tables are produced on an auxiliary stream after the suffix array is
    // final, so a score call (which needs only SA + text) overlaps them; readers wait on ev_tables
    std::unique_ptr<StageTimer> build_timer;
    cudaEvent_t ev_tables = nullptr;
    bool tables_pending = false;
    bool sk_pending = false;          // sk is allocated but not (completely) filled yet: indexes built by the global sort, and
                                      // documents the per-document kernel scored itself; ensure_suffix_keys() makes it
};

// per-device auxiliary (non-blocking) stream for the table kernels
static cudaStream_t aux_stream(int device) {
    static std::mutex m;
    static std::map<int, cudaStream_t> streams;
    std::lock_guard<std::mutex> g(m);
    auto it = streams.find(device);
    if (it != streams.end()) return it->second;
    cudaStream_t st;
    EAST_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    streams[device] = st;
    return st;
}

// per-device high-priority stream: small preparatory kernels of the pipelined build
static cudaStream_t prep_stream(int device) {
    static std::mutex m;
    static std::map<int, cudaStream_t> streams;
    std::lock_guard<std::mutex> g(m);
    auto it = streams.find(device);
    if (it != streams.end()) return it->second;
    int least = 0, greatest = 0;
    EAST_CUDA(cudaDeviceGetStreamPriorityRange(&least, &greatest));
    cudaStream_t st;
    EAST_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, greatest));
    streams[device] = st;
    return st;
}

// per-device copy stream of the pipelined host build
static cudaStream_t copy_stream(int device) {
    static std::mutex m;
    static std::map<int, cudaStream_t> streams;
    std::lock_guard<std::mutex> g(m);
    auto it = streams.find(device);
    if (it != streams.end()) return it->second;
    cudaStream_t st;
    EAST_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    streams[device] = st;
    return st;
}

// block until the tables of `idx` are complete; publishes the build's stage timings once
static void wait_tables(const east_index *cidx) {
    // an index is immutable for its users, but "the tables are complete" is published here, once: concurrent
    // east_index_copy / east_index_devptr / score calls on one index take turns
    static std::mutex m;
    std::lock_guard<std::mutex> g(m);
    east_index *idx = const_cast<east_index *>(cidx);
    if (!idx->tables_pending) return;
    EAST_CUDA(cudaEventSynchronize(idx->ev_tables));
    idx->tables_pending = false;
    if (idx->build_timer) idx->build_timer->collect();
}

// the scorer's per-rank key words of an index built by the global sort: filled by the first scoring call (on its stream)
static void ensure_suffix_keys(const east_index *cidx, cudaStream_t s) {
    static std::mutex m;
    std::lock_guard<std::mutex> g(m);
    east_index *idx = const_cast<east_index *>(cidx);
    if (!idx->sk_pending) return;
    fill_suffix_keys(idx->t8, idx->sa, idx->n, idx->sk, s);
    EAST_CUDA(cudaStreamSynchronize(s));   // later calls may use other streams
    idx->sk_pending = false;
}

static int fail(const Error &e) { g_error = e.what(); return e.status; }
static int fail(int st, const char *msg) { g_error = msg; return st; }

#define EAST_API_BEGIN try {
#define EAST_API_END                                                        \
    }                                                                       \
    catch (const Error &e) { return fail(e); }                              \
    catch (const std::bad_alloc &) { return fail(EAST_ERR_NOMEM, "host out of memory"); } \
    catch (const std::exception &e) { return fail(EAST_ERR_INVALID, e.what()); }           \
    return EAST_OK;

extern "C" {

static void drop_kp_cache();   // defined with the cache, below

const char *east_last_error(void) { return g_error.c_str(); }
const char *east_version(void) { return "east_b200 0.1 (sm_100a)"; }

int east_device_count(void) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess) { cudaGetLastError(); return 0; }
    return cnt;
}

int east_set_option(const char *name, int64_t value) {
    if (!name) return fail(EAST_ERR_INVALID, "option name is NULL");
    if (!strcmp(name, "time_kernels")) {  // per-thread: events around every launch; value 0 also clears the table
        g_time_kernels = value == 2 ? 2 : (value ? 1 : 0);   // 2: the dominant kernel only
        if (!value) g_kstats.clear();
        return EAST_OK;
    }
    if (!strcmp(name, "drop_kp_cache")) {   // per-thread: forget the keyphrase preparation kept for the score calls
        if (value) drop_kp_cache();
        return EAST_OK;
    }
    if (!strcmp(name, "forget_alphabet_guess")) {   // per-thread: the next batch of small documents scans for its alphabet
        if (value) alphabet_guess_forget();
        return EAST_OK;
    }
    std::lock_guard<std::mutex> g(g_opt_mutex);
    g_options[name] = value;
    return EAST_OK;
}

int64_t east_launch_count(int reset) {
    int64_t v = g_launches;
    if (reset) g_launches = 0;
    return v;
}

int east_last_timings(float *ms, char *names, int32_t cap, int32_t names_cap) {
    int n = (int)g_stage_ms.size();
    int32_t w = 0;
    for (int i = 0; i < n; ++i) {
        if (ms && i < cap) ms[i] = g_stage_ms[i];
        if (names) {
            const std::string &s = g_stage_names[i];
            if (w + (int32_t)s.size() + 1 <= names_cap) {
                memcpy(names + w, s.c_str(), s.size() + 1);
                w += (int32_t)s.size() + 1;
            }
        }
    }
    return n;
}

int east_kernel_stats(char *names, int32_t names_cap, double *ms, int64_t *launches, double *bytes, int32_t cap) {
    int i = 0;
    int32_t w = 0;
    for (auto &kv : g_kstats) {
        if (i < cap) {
            if (ms) ms[i] = kv.second.ms;
            if (launches) launches[i] = kv.second.launches;
            if (bytes) bytes[i] = kv.second.bytes;
            if (names && w + (int32_t)kv.first.size() + 1 <= names_cap) {
                memcpy(names + w, kv.first.c_str(), kv.first.size() + 1);
                w += (int32_t)kv.first.size() + 1;
            }
        }
        ++i;
    }
    return i;
}

static void free_index(east_index *idx) {
    if (!idx) return;
    cudaSetDevice(idx->device);
    if (std::uncaught_exceptions() > 0) cudaDeviceSynchronize();   // error path: see dev_free
    if (idx->tables_pending) { cudaEventSynchronize(idx->ev_tables); idx->tables_pending = false; }
    if (idx->build_timer) { try { idx->build_timer->collect(); } catch (...) {} idx->build_timer.reset(); }
    if (idx->ev_tables) cudaEventDestroy(idx->ev_tables);
    if (idx->owns_text && idx->text) dev_free(idx->text, 0);
    for (void *p : {(void *)idx->d_doc_off, (void *)idx->d_doc_m, (void *)idx->sa, (void *)idx->lcp,
                    (void *)idx->up, (void *)idx->down, (void *)idx->next, (void *)idx->ann, (void *)idx->t8,
                    (void *)idx->bkt, (void *)idx->bkt3, (void *)idx->sk})
        if (p && !idx->arena.holds(p)) cudaFreeAsync(p, 0);   // a slice the arena had no room for
    if (idx->arena.base) dev_free(idx->arena.base, 0);
    delete idx;
}

struct ChunkPlan {   // pipelined host build: runs of whole documents and the events of their copies
    std::vector<int32_t> doc;          // n_chunks + 1 document boundaries
    std::vector<cudaEvent_t> ready;
    ~ChunkPlan() { for (auto e : ready) cudaEventDestroy(e); }
};

// what east_table_host hangs on the pipelined build: a hook called after every run of documents, and where
// to publish the index under construction (its text / suffix-array / offset pointers are final from the start)
struct RunHook {
    void (*begin)(void *ctx, const RunReady &run, DocScore &score) = nullptr;
    void (*fn)(void *ctx, const RunReady &run, int in_kernel) = nullptr;
    void (*scan_queued)(void *ctx) = nullptr;
    void *ctx = nullptr;
    const east_index **building = nullptr;
};

static int build_common(const uint32_t *text_dev, bool owns_text, const int64_t *doc_off, const int32_t *doc_m,
                        int32_t n_docs, int device, cudaStream_t s, east_index **out, const ChunkPlan *chunks = nullptr,
                        const RunHook *hook = nullptr, const uint8_t *text8_dev = nullptr /* one byte per code point: text_dev is filled from it */) {
    std::unique_ptr<east_index, void (*)(east_index *)> idx(new east_index(), free_index);
    // pipelined build: whatever happens, the copy stream must be done with the text before the index
    // (declared above, destroyed after this guard) can free it
    struct CopyGuard {
        cudaStream_t cs; bool armed;
        ~CopyGuard() { if (armed) cudaStreamSynchronize(cs); }
    } copy_guard{chunks ? copy_stream(device) : (cudaStream_t)0, chunks != nullptr};
    idx->device = device;
    idx->n_docs = n_docs;
    idx->text = const_cast<uint32_t *>(text_dev);
    idx->owns_text = owns_text;
    const int64_t n64 = doc_off[n_docs];
    idx->n = (int32_t)n64;
    const int32_t n = idx->n;
    idx->doc_off.resize(n_docs + 1);
    idx->doc_m.assign(doc_m, doc_m + n_docs);
    for (int i = 0; i <= n_docs; ++i) idx->doc_off[i] = (int32_t)doc_off[i];
    for (int i = 0; i < n_docs; ++i) idx->m_total += doc_m[i];

    // ---- one arena for everything the index keeps: an upper bound that does not depend on the alphabet
    int32_t max_doc_n = 0;
    for (int i = 0; i < n_docs; ++i) max_doc_n = std::max<int32_t>(max_doc_n, (int32_t)(doc_off[i + 1] - doc_off[i]));
    if (!get_option("no_arena", 0)) {
        const size_t words = sizeof(int32_t) * (size_t)n;
        size_t need = Arena::padded(sizeof(int32_t) * ((size_t)n_docs + 1)) + Arena::padded(sizeof(int32_t) * (size_t)n_docs) +
                      7 * Arena::padded(words) + Arena::padded((size_t)n + 128);
        // 2-gram table: n_docs << 2b entries with b <= 7, kept only up to 2n + 4096; 3-gram table: the per-document
        // kernel with 3 symbols per bucket id (b = 4, 5), kept up to 8 GB
        need += Arena::padded(sizeof(uint32_t) * (std::min<size_t>((size_t)n_docs << 14, (size_t)2 * n + 4096) + 1));
        const size_t e3 = ((size_t)n_docs << 15) + 1;
        if (max_doc_n <= 65535 && !get_option("no_doc_sort", 0) && !get_option("no_bkt3", 0) && e3 * sizeof(uint32_t) <= ((size_t)8 << 30) + 4)
            need += Arena::padded(sizeof(uint32_t) * e3);
        host_debug_mark("arena alloc");
        idx->arena.base = (uint8_t *)dev_alloc(need, s, true);
        idx->arena.cap = need;
        host_debug_mark("arena alloc done");
    }
    auto take32 = [&](size_t count) { DevBuf<int32_t> b = idx->arena.take<int32_t>(count, s); int32_t *p = b.p; b.p = nullptr; return p; };
    idx->d_doc_off = take32((size_t)n_docs + 1);
    idx->d_doc_m = take32((size_t)n_docs);
    EAST_CUDA(cudaMemcpyAsync(idx->d_doc_off, idx->doc_off.data(), sizeof(int32_t) * (n_docs + 1),
                              cudaMemcpyHostToDevice, s));
    EAST_CUDA(cudaMemcpyAsync(idx->d_doc_m, idx->doc_m.data(), sizeof(int32_t) * n_docs, cudaMemcpyHostToDevice, s));
    idx->sa = take32((size_t)n);
    idx->lcp = take32((size_t)n);
    idx->up = take32((size_t)n);
    idx->down = take32((size_t)n);
    idx->next = take32((size_t)n);
    idx->ann = take32((size_t)n);

    if (text8_dev && !chunks) {   // not pipelined: the code points first, then the ordinary build
        DevBuf<uint32_t> bad(1, s);
        EAST_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(uint32_t), s));
        expand_text8(text8_dev, idx->d_doc_off, idx->d_doc_m, n_docs, idx->text, bad.p, s);
        uint32_t h_bad = 0;
        EAST_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        EAST_CUDA(cudaStreamSynchronize(s));
        if (h_bad) throw Error(EAST_ERR_INVALID, "one-byte text: a document does not hold exactly doc_m string ends (0xFF) or does not end with one");
    }
    idx->build_timer.reset(new StageTimer(s));
    StageTimer &tm = *idx->build_timer;
    const bool overlap = get_option("sync_build", 0) == 0;
    {
        SaInput in;
        in.text = idx->text; in.doc_off = idx->d_doc_off; in.doc_m = idx->d_doc_m;
        in.n = n; in.n_docs = n_docs; in.m_total = idx->m_total;
        in.key_chars = (int)get_option("key_chars", 0);
        in.force_general = (int)get_option("force_general", 0);
        in.rs_variant = (int)get_option("rs_variant", 0);
        in.doc_off_host = idx->doc_off.data();
        in.sort_batch_elems = get_option("sort_batch_elems", 0);
        in.local_group_sort = get_option("doubling_radix", 0) ? 0 : 1;
        in.segmented_sort = get_option("global_sort", 0) ? 0 : 1;
        // the per-document shared-memory sort is the default for small documents; any tuning option of
        // the global prefix-doubling sort (and "no_doc_sort") selects the global sort instead
        in.doc_sort = (get_option("no_doc_sort", 0) || in.key_chars || in.rs_variant || in.sort_batch_elems ||
                       !in.segmented_sort || !in.local_group_sort) ? 0 : 1;
        in.want_bkt3 = get_option("no_bkt3", 0) ? 0 : 1;
        in.light_scan = get_option("no_light_scan", 0) ? 0 : 1;
        // device-resident batches: alphabet from the first 2 M code points (option alphabet_sample; -1 = the whole text)
        { const int64_t smp = get_option("alphabet_sample", (int64_t)1 << 21); in.alphabet_sample = smp < 0 ? 0 : smp; }
        // ... or from the thread's previous batch on this device (option no_alphabet_guess = 1: always scan)
        in.alphabet_guess = get_option("no_alphabet_guess", 0) ? 0 : 1;
        in.fused_encode = get_option("no_fused_encode", 0) ? 0 : 1;
        if (!get_option("no_suffix_keys", 0)) {
            idx->sk = (uint32_t *)take32((size_t)n);
            in.sk = idx->sk;
        }
        if (!get_option("no_fused_tables", 0)) {
            in.lcp = idx->lcp; in.up = idx->up; in.down = idx->down; in.next = idx->next; in.ann = idx->ann;
        }
        in.arena = idx->arena.base ? &idx->arena : nullptr;
        in.helper_stream = aux_stream(device);
        if (!get_option("no_prep_stream", 0)) in.prep_stream = prep_stream(device);
        if (hook && hook->fn) {
            in.run_begin = hook->begin; in.run_hook = hook->fn; in.run_ctx = hook->ctx; in.scan_queued = hook->scan_queued;
            if (hook->building) *hook->building = idx.get();
        }
        if (chunks && text8_dev) {
            if (!in.doc_sort || !in.fused_encode) throw Error(EAST_ERR_INVALID, "internal: the one-byte pipelined build needs the per-document kernel");
            in.text8 = text8_dev;
        }
        if (chunks && in.doc_sort) {
            in.n_chunks = (int)chunks->ready.size();
            in.chunk_doc = chunks->doc.data();
            in.chunk_ready = chunks->ready.data();
        } else if (chunks) {   // the global sort needs the whole text: wait for every copy
            for (auto e : chunks->ready) EAST_CUDA(cudaStreamWaitEvent(s, e, 0));
        }
        SaOutput so;
        so.sa = idx->sa;
        build_suffix_array(in, so, tm, s);
        idx->pipelined = so.pipelined; idx->pipeline_miss = so.pipeline_miss; idx->alphabet_miss = so.alphabet_miss; idx->alphabet_guessed = so.alphabet_guessed;
        idx->rounds = so.rounds; idx->fast_path = so.fast_path; idx->key_chars = so.key_chars;
        idx->key_bits = so.key_bits; idx->active_after_round0 = so.active_after_round0;
        idx->doc_sorted = so.doc_sorted; idx->doc_sort_overflow = so.doc_sort_overflow;
        idx->t8 = so.t8.p; so.t8.p = nullptr;      // ownership moves to the index
        idx->bkt = so.bkt.p; so.bkt.p = nullptr;
        idx->bkt3 = so.bkt3.p; so.bkt3.p = nullptr;
        idx->code_table = so.code_table; idx->sym_bits = so.sym_bits; idx->term_code = so.term_code;
        idx->tables_fused = so.tables_done;
        if (idx->sk && so.sk_done && so.sk_skipped && idx->t8) idx->sk_pending = true;   // made by the first later score call
        if (idx->sk && !so.sk_done) {
            // global sort: the scorer's per-rank key words are not part of the structure (SA, LCP, child table, annotation):
            // they are made by the first call that scores against the index (ensure_suffix_keys), not by the build
            if (idx->t8) idx->sk_pending = true;
            else { if (!idx->arena.holds(idx->sk)) dev_free(idx->sk, s); idx->sk = nullptr; }   // general path: no byte text
        }
        if (so.tables_done) {
            tm.finish();   // the per-document kernel produced every table: nothing is pending
        } else {
            // the suffix array is final here (the doubling loop ended on a host sync)
            cudaStream_t ts = s;
            if (overlap) {
                ts = aux_stream(device);
                cudaEvent_t fork;
                EAST_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
                EAST_CUDA(cudaEventRecord(fork, s));
                EAST_CUDA(cudaStreamWaitEvent(ts, fork, 0));
                EAST_CUDA(cudaEventDestroy(fork));
                tm.s = ts;
            }
            build_lcp_tables(idx->text, idx->t8, idx->term_code, idx->sa, idx->d_doc_off, idx->d_doc_m, n_docs, n, idx->lcp, idx->up,
                             idx->down, idx->next, idx->ann, tm, ts, (int)get_option("child_variant", 0));
            tm.finish();
            if (overlap) {
                EAST_CUDA(cudaEventCreateWithFlags(&idx->ev_tables, cudaEventDisableTiming));
                EAST_CUDA(cudaEventRecord(idx->ev_tables, ts));
                idx->tables_pending = true;
            }
        }
    }
    if (!overlap) {
        EAST_CUDA(cudaStreamSynchronize(s));
        tm.collect();
    }
    *out = idx.release();
    return EAST_OK;
}

static void check_documents(const void *text, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs) {
    if (!text || !doc_off || !doc_m) throw Error(EAST_ERR_INVALID, "NULL argument");
    if (n_docs <= 0) throw Error(EAST_ERR_INVALID, "n_docs must be positive");
    if (doc_off[0] != 0) throw Error(EAST_ERR_INVALID, "doc_off[0] must be 0");
    for (int i = 0; i < n_docs; ++i) {
        if (doc_off[i + 1] <= doc_off[i]) throw Error(EAST_ERR_INVALID, "empty document (a packed document has at least one terminator)");
        if (doc_m[i] <= 0) throw Error(EAST_ERR_INVALID, "document without strings (EmptyStringsCollectionException in the reference)");
        if (doc_m[i] > doc_off[i + 1] - doc_off[i]) throw Error(EAST_ERR_INVALID, "doc_m larger than the document");
    }
    if (doc_off[n_docs] >= (1ll << 30)) throw Error(EAST_ERR_RANGE, "more than 2^30 code points in one index; split the batch");
}

static void build_host_impl(const void *text_any, int width /* bytes per code point on the host: 4, or 1 (0xFF = end of a string) */,
                            const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                            int device, east_index **out, const RunHook *hook) {
    const uint32_t *text = static_cast<const uint32_t *>(text_any);
    const uint8_t *text8 = static_cast<const uint8_t *>(text_any);
    static const bool debug = getenv("EAST_DEBUG_TIMING") != nullptr;
    if (debug) fprintf(stderr, "[east] host %.3f ms  east_build_host enter\n", host_now_ms());
    if (!out) throw Error(EAST_ERR_INVALID, "NULL argument");
    check_documents(text_any, doc_off, doc_m, n_docs);
    use_device(device);
    const int64_t n = doc_off[n_docs];
    const size_t bytes = sizeof(uint32_t) * (size_t)n;
    // stream-ordered pool allocation (cudaMalloc/cudaFree take device-wide locks and synchronise)
    DevBuf<uint8_t> d_text8;
    if (width == 1) {
        d_text8 = DevBuf<uint8_t>((uint8_t *)dev_alloc((size_t)n + 256, 0, true), (size_t)n + 256);   // 16-byte groups are read whole
        d_text8.owned = true;
        EAST_CUDA(cudaMemsetAsync(d_text8.p + n, 0, 256, 0));
    }
    host_debug_mark("text alloc");
    uint32_t *d_text = (uint32_t *)dev_alloc(bytes, 0, true);
    host_debug_mark("text alloc done");
    // Large batches of small documents: copy in runs of whole documents on a copy stream so that the
    // per-document kernels of run c overlap the copy of run c+1 (worth it with pinned host memory)
    int64_t max_doc = 0;
    for (int32_t d = 0; d < n_docs; ++d) max_doc = std::max(max_doc, doc_off[d + 1] - doc_off[d]);
    const int64_t chunk_target = get_option("pipeline_chunk", (int64_t)1 << 22);
    int want = (int)std::min<int64_t>(16, n / chunk_target);
    if (width == 1) want = (int)std::min<int64_t>(16, n / (chunk_target / 4));   // the same runs of documents for a quarter of the bytes
    const bool tuned_sort = get_option("key_chars", 0) || get_option("rs_variant", 0) || get_option("sort_batch_elems", 0) ||
                            get_option("global_sort", 0) || get_option("doubling_radix", 0);
    const bool pipelined = want >= 2 && n_docs >= 2 * EAST_NUM_SMS && max_doc <= 65535 && !get_option("no_pipeline", 0) &&
                           !get_option("no_doc_sort", 0) && (width == 4 || (!get_option("no_fused_encode", 0) && !tuned_sort));
    cudaError_t e = cudaSuccess;
    if (!pipelined) {
        e = width == 1 ? cudaMemcpyAsync(d_text8.p, text8, (size_t)n, cudaMemcpyHostToDevice, 0)
                       : cudaMemcpyAsync(d_text, text, bytes, cudaMemcpyHostToDevice, 0);
        if (e != cudaSuccess) { dev_free(d_text, 0); throw Error(EAST_ERR_CUDA, cudaGetErrorString(e)); }
        build_common(d_text, true, doc_off, doc_m, n_docs, device, 0, out, nullptr, hook, d_text8.p);  // owns d_text from here on
    } else {
        ChunkPlan plan;
        cudaStream_t cs = copy_stream(device);
        try {
            // the allocation was made on stream 0: the copy stream must not run ahead of it
            cudaEvent_t alloc_done;
            EAST_CUDA(cudaEventCreateWithFlags(&alloc_done, cudaEventDisableTiming));
            EAST_CUDA(cudaEventRecord(alloc_done, 0));
            EAST_CUDA(cudaStreamWaitEvent(cs, alloc_done, 0));
            EAST_CUDA(cudaEventDestroy(alloc_done));
            // runs of whole documents, a multiple of the SM count each: one per-document CTA per SM and wave,
            // so a run costs exactly its waves (10 runs of 100 documents on 148 SMs would cost 10 waves, not 7)
            const int32_t per_run = (int32_t)(((int64_t)(n_docs + want - 1) / want + EAST_NUM_SMS - 1) / EAST_NUM_SMS) * EAST_NUM_SMS;
            // the device idles until the first run is resident and its alphabet known: the first wave's documents
            // come as a short run (a quarter of the SMs) followed by the rest of the wave
            // ... unless the alphabet is a guess (nothing waits for run 0 on the host then): the short run would only be
            // one more launch and a split first wave (measured: 3.45 against 3.56 ms per call without it)
            uint8_t guessed_table[EAST_TERM_BASE];
            const bool will_guess = !get_option("no_alphabet_guess", 0) && alphabet_guess_code_table(guessed_table);
            const int32_t lead = (get_option("no_lead_run", 0) || will_guess) ? 0 : EAST_NUM_SMS / 4;
            plan.doc.push_back(0);
            for (int32_t d = 0; d < n_docs;) {
                const int32_t step = (lead > 0 && d == 0) ? lead : ((lead > 0 && d == lead) ? per_run - lead : per_run);
                const int32_t d1 = std::min(n_docs, d + step);
                const int64_t e0 = doc_off[d], e1 = doc_off[d1];
                if (width == 1) EAST_CUDA(cudaMemcpyAsync(d_text8.p + e0, text8 + e0, (size_t)(e1 - e0), cudaMemcpyHostToDevice, cs));
                else EAST_CUDA(cudaMemcpyAsync(d_text + e0, text + e0, sizeof(uint32_t) * (size_t)(e1 - e0), cudaMemcpyHostToDevice, cs));
                cudaEvent_t ev;
                EAST_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                plan.ready.push_back(ev);
                EAST_CUDA(cudaEventRecord(ev, cs));
                plan.doc.push_back(d1);
                d = d1;
            }
        } catch (...) {
            cudaStreamSynchronize(cs);
            dev_free(d_text, 0);
            throw;
        }
        if (debug) fprintf(stderr, "[east] host %.3f ms  copies queued\n", host_now_ms());
        build_common(d_text, true, doc_off, doc_m, n_docs, device, 0, out, &plan, hook, d_text8.p);
        if (debug) fprintf(stderr, "[east] host %.3f ms  build_common done\n", host_now_ms());
    }
}

int east_build_host(const uint32_t *text, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                    int device, east_index **out) {
    EAST_API_BEGIN
    build_host_impl(text, 4, doc_off, doc_m, n_docs, device, out, nullptr);
    EAST_API_END
}

int east_build_host_u8(const uint8_t *text8, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                       int device, east_index **out) {
    EAST_API_BEGIN
    build_host_impl(text8, 1, doc_off, doc_m, n_docs, device, out, nullptr);
    EAST_API_END
}

int east_build_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                   int device, void *stream, east_index **out) {
    EAST_API_BEGIN
    if (!out) throw Error(EAST_ERR_INVALID, "NULL argument");
    check_documents(text_dev, doc_off, doc_m, n_docs);
    use_device(device);
    build_common(text_dev, false, doc_off, doc_m, n_docs, device, (cudaStream_t)stream, out);
    EAST_API_END
}

void east_free(east_index *idx) { free_index(idx); }

int east_index_info(const east_index *idx, int32_t *n_docs, int64_t *n_total, int32_t *device, int32_t *rounds,
                    int32_t *fast_path) {
    if (!idx) return fail(EAST_ERR_INVALID, "NULL index");
    if (n_docs) *n_docs = idx->n_docs;
    if (n_total) *n_total = idx->n;
    if (device) *device = idx->device;
    if (rounds) *rounds = idx->rounds;
    if (fast_path) *fast_path = idx->fast_path;
    return EAST_OK;
}

int east_index_doc(const east_index *idx, int32_t doc, int64_t *offset, int64_t *n, int32_t *m) {
    if (!idx || doc < 0 || doc >= idx->n_docs) return fail(EAST_ERR_INVALID, "bad index/doc");
    if (offset) *offset = idx->doc_off[doc];
    if (n) *n = idx->doc_off[doc + 1] - idx->doc_off[doc];
    if (m) *m = idx->doc_m[doc];
    return EAST_OK;
}

int east_index_stat(const east_index *idx, const char *name, int64_t *value) {
    if (!idx || !name || !value) return fail(EAST_ERR_INVALID, "NULL argument");
    if (!strcmp(name, "doc_sorted")) *value = idx->doc_sorted;
    else if (!strcmp(name, "doc_sort_overflow")) *value = idx->doc_sort_overflow;
    else if (!strcmp(name, "tables_fused")) *value = idx->tables_fused;
    else if (!strcmp(name, "bkt3")) *value = idx->bkt3 != nullptr;
    else if (!strcmp(name, "pipelined")) *value = idx->pipelined;
    else if (!strcmp(name, "pipeline_miss")) *value = idx->pipeline_miss;
    else if (!strcmp(name, "alphabet_miss")) *value = idx->alphabet_miss;
    else if (!strcmp(name, "alphabet_guessed")) *value = idx->alphabet_guessed;
    else if (!strcmp(name, "key_chars")) *value = idx->key_chars;
    else if (!strcmp(name, "key_bits")) *value = idx->key_bits;
    else if (!strcmp(name, "rounds")) *value = idx->rounds;
    else if (!strcmp(name, "active_after_round0")) *value = idx->active_after_round0;
    else if (!strcmp(name, "fast_path")) *value = idx->fast_path;
    else return fail(EAST_ERR_INVALID, "unknown stat name");
    return EAST_OK;
}

static const int32_t *array_of(const east_index *idx, int which) {
    switch (which) {
        case EAST_SUFTAB: return idx->sa;
        case EAST_LCPTAB: return idx->lcp;
        case EAST_CHILDTAB_UP: return idx->up;
        case EAST_CHILDTAB_DOWN: return idx->down;
        case EAST_CHILDTAB_NEXT_L_INDEX: return idx->next;
        case EAST_ANNTAB: return idx->ann;
        default: return nullptr;
    }
}

int east_index_copy(const east_index *idx, int32_t doc, int which, int32_t *dst_host) {
    EAST_API_BEGIN
    if (!idx || !dst_host || doc < 0 || doc >= idx->n_docs) throw Error(EAST_ERR_INVALID, "bad index/doc/destination");
    const int32_t *src = which == EAST_PACKED_TEXT ? reinterpret_cast<const int32_t *>(idx->text) : array_of(idx, which);
    if (!src) throw Error(EAST_ERR_INVALID, "unknown array id");
    EAST_CUDA(cudaSetDevice(idx->device));
    wait_tables(idx);
    const int32_t off = idx->doc_off[doc], n = idx->doc_off[doc + 1] - off;
    EAST_CUDA(cudaMemcpy(dst_host, src + off, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost));
    if (which == EAST_SUFTAB)
        for (int32_t i = 0; i < n; ++i) dst_host[i] -= off;  // global text position -> position in the document
    EAST_API_END
}

int east_index_devptr(const east_index *idx, int which, const void **ptr) {
    if (!idx || !ptr) return fail(EAST_ERR_INVALID, "NULL argument");
    if (which == 100) { *ptr = idx->text; return EAST_OK; }
    try { wait_tables(idx); } catch (const Error &e) { return fail(e); }
    const int32_t *p = array_of(idx, which);
    if (!p) return fail(EAST_ERR_INVALID, "unknown array id");
    *ptr = p;
    return EAST_OK;
}

// ---- scoring ----------------------------------------------------------------------------
// Everything the scorer derives from the keyphrases alone (and the index's alphabet): built once and
// kept for the next call -- keyphrases_table scores the same keyphrases against one index after the
// other (document tiles, ranks, benchmark steps).  A hit is confirmed by comparing the code points.
struct KpPrepared {
    int device = -1;
    bool dedup = false, fast = false, finished = false;
    int sym_bits = 0;
    std::vector<uint32_t> kp;          // host copy of the code points (cache key; host preparation)
    std::vector<int64_t> off;          // K + 1 offsets (cache key)
    std::vector<uint8_t> code_table;   // alphabet of the index the dense codes were made for (cache key)
    int64_t n_uniq = 0;
    KpDevice dev;                      // d_off, d_uniq_of, d_recs, d_q8: filled by kp_prep.cu (or by the host variant)
};
static thread_local std::unique_ptr<KpPrepared> g_kp_cache;
static void drop_kp_cache() {
    if (!g_kp_cache) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(g_kp_cache->device);
    cudaDeviceSynchronize();
    g_kp_cache.reset();
    cudaSetDevice(cur);
}

// The host variant of kp_prep.cu (round 1; option "kp_prep_host" = 1, kept as the cross-check of the device pipeline):
// hashing, sorting and coding on the host, four uploads and a stream sync.
static void prepare_keyphrases_host(KpPrepared *c, bool fast, int sym_bits, const std::vector<uint8_t> &code_table,
                                    const int64_t *kp_off, int32_t K, bool dedup, cudaStream_t s) {
    const int64_t total = kp_off[K];
    const std::vector<uint32_t> &kp_host = c->kp;
    struct { const std::vector<uint8_t> &code_table; int sym_bits; } view{code_table, sym_bits};
    auto *idx = &view;
    std::vector<int32_t> off32(K + 1), suf_kp((size_t)total);
    for (int32_t k = 0; k <= K; ++k) off32[k] = (int32_t)kp_off[k];
    for (int32_t k = 0; k < K; ++k)
        for (int64_t p = kp_off[k]; p < kp_off[k + 1]; ++p) suf_kp[(size_t)p] = k;

    // ---- identical query suffixes are walked once.  A suffix result depends only on the code points
    // from its start to the end of its keyphrase (easa.py:98-131), and keyphrases built from a
    // vocabulary share most word tails: 47 % distinct at 10^5 Zipf keyphrases, 72 % at 10^3.
    // Suffix hashes are built backwards (h(s[i:]) from code[i] and h(s[i+1:])), equal hashes are
    // confirmed by comparing the code points.
    std::vector<int32_t> uniq_of((size_t)total), uniq_rep;
    if (!dedup) {
        uniq_rep.resize((size_t)total);
        for (int64_t p = 0; p < total; ++p) { uniq_of[(size_t)p] = (int32_t)p; uniq_rep[(size_t)p] = (int32_t)p; }
    } else {
        std::vector<uint64_t> hash((size_t)total);
        for (int32_t k = 0; k < K; ++k) {
            uint64_t h = 0x9e3779b97f4a7c15ull;
            for (int64_t p = kp_off[k + 1] - 1; p >= kp_off[k]; --p) {
                h = h * 0x100000001b3ull + (uint64_t)kp_host[(size_t)p] + 0x632be59bd9b4e019ull;
                h ^= h >> 29;
                hash[(size_t)p] = h;
            }
        }
        std::vector<int32_t> by_hash((size_t)total);
        for (int64_t p = 0; p < total; ++p) by_hash[(size_t)p] = (int32_t)p;
        auto suffix_len = [&](int32_t p) { return (int32_t)(kp_off[suf_kp[(size_t)p] + 1] - p); };
        auto same = [&](int32_t a, int32_t b) {
            const int32_t la = suffix_len(a);
            return la == suffix_len(b) && std::equal(kp_host.begin() + a, kp_host.begin() + a + la, kp_host.begin() + b);
        };
        std::sort(by_hash.begin(), by_hash.end(), [&](int32_t a, int32_t b) {
            return hash[(size_t)a] != hash[(size_t)b] ? hash[(size_t)a] < hash[(size_t)b] : a < b;
        });
        for (size_t i = 0; i < by_hash.size();) {
            size_t j = i;
            while (j < by_hash.size() && hash[(size_t)by_hash[j]] == hash[(size_t)by_hash[i]]) ++j;
            // one hash value: almost always one distinct suffix; a collision splits the run
            const size_t first_id = uniq_rep.size();
            for (size_t a = i; a < j; ++a) {
                const int32_t pa = by_hash[a];
                int32_t id = -1;
                for (size_t q = first_id; q < uniq_rep.size() && id < 0; ++q)
                    if (same(uniq_rep[q], pa)) id = (int32_t)q;
                if (id < 0) { id = (int32_t)uniq_rep.size(); uniq_rep.push_back(pa); }
                uniq_of[(size_t)pa] = id;
            }
            i = j;
        }
    }
    const int64_t n_uniq = (int64_t)uniq_rep.size();
    c->n_uniq = n_uniq;
    std::vector<uint8_t> q8((size_t)total, 0), generic((size_t)total, 1);
    std::vector<int32_t> order((size_t)n_uniq);
    if (fast) {
        // dense byte codes of the queries + per-suffix "contains a code point >= 0x0A00" flag
        for (int32_t k = 0; k < K; ++k) {
            uint8_t weird = 0;
            for (int64_t p = kp_off[k + 1] - 1; p >= kp_off[k]; --p) {
                const uint32_t cp = kp_host[(size_t)p];
                if (cp >= EAST_TERM_BASE) { weird = 1; q8[(size_t)p] = 0; }
                else q8[(size_t)p] = idx->code_table[cp];
                generic[(size_t)p] = weird;
            }
        }
    }
    if (fast && dedup) {
        // visiting order of the distinct suffixes: counting sort by their first three dense symbols, so the
        // threads of a warp walk neighbouring SA intervals (cache locality, less divergence).  (Without
        // de-duplication the caller wants per-suffix results: they stay in suffix order.)
        const int b = idx->sym_bits;
        const int nsym = (3 * b <= 18) ? 3 : ((2 * b <= 18) ? 2 : 1);
        std::vector<uint32_t> bin((size_t)n_uniq);
        std::vector<uint32_t> count(((size_t)1 << (nsym * b)) + 1, 0u);
        for (int64_t u = 0; u < n_uniq; ++u) {
            const int64_t p = uniq_rep[(size_t)u], pe = kp_off[suf_kp[(size_t)p] + 1];
            uint32_t key = 0;
            for (int q = 0; q < nsym; ++q) key = (key << b) | ((p + q < pe) ? q8[(size_t)(p + q)] : 0u);
            bin[(size_t)u] = key;
            ++count[key + 1];
        }
        for (size_t i = 1; i < count.size(); ++i) count[i] += count[i - 1];
        std::vector<uint32_t> first(count.begin(), count.end() - 1);   // first position of every bin
        for (int64_t u = 0; u < n_uniq; ++u) order[count[bin[(size_t)u]]++] = (int32_t)u;
        // inside a bin: full lexicographic order of the dense codes, so that the lanes of a warp share as
        // long a prefix (= as much of their control flow and of their loads) as possible
        auto lex_less = [&](int32_t a, int32_t b2) {
            const int64_t pa = uniq_rep[(size_t)a], pb = uniq_rep[(size_t)b2];
            const int64_t la = kp_off[suf_kp[(size_t)pa] + 1] - pa, lb = kp_off[suf_kp[(size_t)pb] + 1] - pb;
            const int cmp = memcmp(q8.data() + pa, q8.data() + pb, (size_t)std::min(la, lb));
            return cmp != 0 ? cmp < 0 : la < lb;
        };
        if (!get_option("score_bin_order", 0))
            for (size_t x = 0; x < first.size(); ++x)
                if (count[x] - first[x] > 1) std::sort(order.begin() + first[x], order.begin() + count[x], lex_less);
    } else {
        for (int64_t u = 0; u < n_uniq; ++u) order[(size_t)u] = (int32_t)u;
    }
    // one record per distinct suffix in visiting order; every suffix points at the position of its twin
    std::vector<SufRec> recs((size_t)n_uniq);
    std::vector<int32_t> pos_of((size_t)n_uniq);
    for (int64_t pos = 0; pos < n_uniq; ++pos) {
        const int32_t u = order[(size_t)pos];
        const int64_t p = uniq_rep[(size_t)u], pe = kp_off[suf_kp[(size_t)p] + 1];
        pos_of[(size_t)u] = (int32_t)pos;
        SufRec r;
        r.q8_first = 0;
        for (int q = 0; q < 8 && p + q < pe; ++q) r.q8_first |= (uint64_t)q8[(size_t)(p + q)] << (8 * q);
        r.sidx = (int32_t)p;
        if (pe - p > 0xffff) throw Error(EAST_ERR_RANGE, "keyphrase longer than 65535 code points");
        r.len = (uint16_t)(pe - p);
        r.generic = generic[(size_t)p];
        r.pad = 0;
        recs[(size_t)pos] = r;
    }
    for (int64_t p = 0; p < total; ++p) uniq_of[(size_t)p] = pos_of[(size_t)uniq_of[(size_t)p]];
    KpDevice &d = c->dev;
    d.total = (int32_t)total; d.K = K; d.dedup = dedup;
    d.d_off = DevBuf<int32_t>(K + 1, s);
    d.d_uniq_of = DevBuf<int32_t>((size_t)total, s);
    d.d_recs = DevBuf<SufRec>((size_t)n_uniq, s);
    EAST_CUDA(cudaMemcpyAsync(d.d_off.p, off32.data(), sizeof(int32_t) * (K + 1), cudaMemcpyHostToDevice, s));
    EAST_CUDA(cudaMemcpyAsync(d.d_uniq_of.p, uniq_of.data(), sizeof(int32_t) * (size_t)total, cudaMemcpyHostToDevice, s));
    EAST_CUDA(cudaMemcpyAsync(d.d_recs.p, recs.data(), sizeof(SufRec) * (size_t)n_uniq, cudaMemcpyHostToDevice, s));
    if (fast) {
        d.d_q8 = DevBuf<uint8_t>((size_t)total + 16, s);   // the scorer reads the queries 8 bytes at a time
        EAST_CUDA(cudaMemsetAsync(d.d_q8.p + total, 0, 16, s));
        EAST_CUDA(cudaMemcpyAsync(d.d_q8.p, q8.data(), (size_t)total, cudaMemcpyHostToDevice, s));
    }
    EAST_CUDA(cudaStreamSynchronize(s));   // the host staging vectors end here
}

// Keyphrase preparation in two steps.  kp_begin: everything that does not depend on an index (queued on `s`, nothing
// waits: east_table_host runs it on a side stream under the transfer of the text).  kp_finish: the dense codes for the
// alphabet of an index, queued on `s`; returns with n_uniq known.  kp_finish may be repeated for another alphabet.
static std::unique_ptr<KpPrepared> kp_begin(int device, const uint32_t *kp_dev, const uint32_t *kp_host_in, const int64_t *kp_off,
                                            int32_t K, bool dedup, bool keep_host_copy, cudaStream_t s,
                                            const uint8_t *likely_code_table = nullptr /* of the index to come, if anyone knows */) {
    std::unique_ptr<KpPrepared> c(new KpPrepared());
    const int64_t total = kp_off[K];
    const bool host_prep = get_option("kp_prep_host", 0) != 0;
    c->device = device; c->dedup = dedup;
    c->off.assign(kp_off, kp_off + K + 1);
    if (keep_host_copy || host_prep) {
        c->kp.resize((size_t)total);
        if (kp_host_in) {   // the caller's host copy: no round trip through the device
            std::copy(kp_host_in, kp_host_in + total, c->kp.begin());
        } else {
            EAST_CUDA(cudaMemcpyAsync(c->kp.data(), kp_dev, sizeof(uint32_t) * (size_t)total, cudaMemcpyDeviceToHost, s));
            EAST_CUDA(cudaStreamSynchronize(s));
        }
    }
    if (!host_prep) kp_stage1(c->dev, kp_dev, kp_host_in, kp_off, K, dedup, s, (int32_t)get_option("kp_small_max", 1 << 30), likely_code_table);
    return c;
}

static void kp_finish(KpPrepared *c, const uint32_t *kp_dev, bool fast, int sym_bits, const std::vector<uint8_t> &code_table,
                      cudaStream_t s) {
    const int32_t K = (int32_t)c->off.size() - 1;
    c->fast = fast; c->sym_bits = sym_bits;
    if (fast) c->code_table = code_table; else c->code_table.clear();
    if (get_option("kp_prep_host", 0) != 0 || !c->dev.done) {
        prepare_keyphrases_host(c, fast, sym_bits, code_table, c->off.data(), K, c->dedup, s);
    } else {
        kp_stage2(c->dev, kp_dev, fast ? code_table.data() : nullptr, s);
        c->n_uniq = c->dev.n_uniq;
    }
    c->finished = true;
}

// ---- what a call scores, where its results go, where its documents come from ---------------------------------------
// The keyphrases of a call -- or, grouped, the synonym variants of east_*_groups_*: K variants in G groups and a row G
// wide.  kp_off and group_off are host arrays; the code points come from the host (uploaded by the call into kp_dev)
// or from the device (kp_host: an optional host copy).
struct Query {
    const uint32_t *kp_dev = nullptr, *kp_host = nullptr;
    bool on_host = false;
    const int64_t *kp_off = nullptr;
    int32_t K = 0;
    int normalized = 0;
    bool grouped = false;
    const int64_t *group_off = nullptr;
    int32_t G = 0;
    DevBuf<int32_t> d_groups;   // the device copy of group_off (upload_groups)
    Query(const uint32_t *kp, bool on_host_, const uint32_t *kp_host_copy, const int64_t *kp_off_, int32_t K_, int normalized_,
          bool grouped_ = false, const int64_t *group_off_ = nullptr, int32_t G_ = 0)
        : kp_dev(on_host_ ? nullptr : kp), kp_host(on_host_ ? kp : kp_host_copy), on_host(on_host_), kp_off(kp_off_), K(K_),
          normalized(grouped_ ? 1 : (normalized_ ? 1 : 0)),   // groups are always normalized, as the reference's synonym branch
          grouped(grouped_), group_off(grouped_ ? group_off_ : nullptr), G(grouped_ ? G_ : 0) {}
    int32_t cols() const { return grouped ? G : K; }
    int64_t total() const { return kp_off[K]; }
    // the device copy of host code points, queued on `s`
    DevBuf<uint32_t> upload(cudaStream_t s) {
        DevBuf<uint32_t> d((size_t)total(), s);
        EAST_CUDA(cudaMemcpyAsync(d.p, kp_host, sizeof(uint32_t) * (size_t)total(), cudaMemcpyHostToDevice, s));
        kp_dev = d.p;
        return d;
    }
    // int32 offsets: < 2^31 variants, each has a code point of the keyphrase buffer (check_keyphrases); uploaded once, on
    // `s` (the pageable host vector is staged before the copy call returns)
    void upload_groups(cudaStream_t s) {
        if (!grouped || d_groups.p) return;
        const std::vector<int32_t> g32(group_off, group_off + G + 1);
        d_groups = DevBuf<int32_t>((size_t)G + 1, s);
        EAST_CUDA(cudaMemcpyAsync(d_groups.p, g32.data(), sizeof(int32_t) * ((size_t)G + 1), cudaMemcpyHostToDevice, s));
    }
};

// tcgen05 kernel of the co-occurrence counts (option cooc_variant: 2 = the 128 x 128 kernel, 3 = the cp.async pipeline,
// otherwise the TMA-fed cluster kernel; 1 selects the AND + POPC kernel of east_cooc_*, which reads the score table)
static int cooc_tc_kernel() {
    const int64_t v = get_option("cooc_variant", 0);
    return v == 2 ? 1 : (v == 3 ? 2 : 0);
}

// ---- keyphrase graphs: relevance bytes instead of a score table ------------------------------------------------------
// A graph call fills B[k][d] = (score of document d in column k >= threshold), the zero-padded Kp x Dp byte matrix of the
// co-occurrence GEMM (cooc_tc.cu), and never a documents x keyphrases table: the per-document kernel stores its column of
// bytes itself (k_doc_suffix_sort_graph); every other path scores tiles of documents into an fp64 scratch bounded by the
// score_tmp_doubles budget and thresholds each tile into its columns (graph_enqueue).
struct GraphOut {
    double threshold = 0.0;
    int32_t *C = nullptr;   // device: cols x cols counts
    DevBuf<uint8_t> B;
    int64_t Dp = 0;
    int32_t Kp = 0;
    void begin(int32_t n_docs, int32_t cols, cudaStream_t s) {
        cooc_padding(n_docs, cols, &Dp, &Kp);
        B = DevBuf<uint8_t>((size_t)Kp * (size_t)Dp, s);
        EAST_CUDA(cudaMemsetAsync(B.p, 0, (size_t)Kp * (size_t)Dp, s));   // padding rows / columns stay zero
    }
    void finish(int32_t cols, cudaStream_t s) const { cooc_counts_bytes(B.p, Dp, Kp, cols, C, s, cooc_tc_kernel()); }
};

// Where a call's results go: the rows of a table on the device (the caller's; host entries: the call's own, copied to
// the host), optionally stored into the other ranks' tables too, or the counts of a keyphrase graph (to a device
// pointer, or copied to a host pointer).
struct Output {
    double *rows = nullptr;              // device, n_docs x cols
    bool to_host = false;
    double *rows_host = nullptr;         // to_host: the host copy of the rows
    double *const *peer_rows = nullptr;  // sharded table: where this rank's rows start in every other rank's table
    int32_t n_peers = 0;
    bool is_graph = false;
    GraphOut graph;                      // is_graph: counts into graph.C ...
    int32_t *counts_host = nullptr;      // ... or, given this, into the call's own buffer and then here
    DevBuf<double> own_rows;
    DevBuf<int32_t> own_counts;

    static Output table_dev(double *rows, double *const *peer_rows = nullptr, int32_t n_peers = 0) {
        Output o;
        o.rows = rows; o.peer_rows = peer_rows; o.n_peers = n_peers;
        return o;
    }
    // rows_dev: where the rows also go on the device (NULL: a buffer of the call)
    static Output table_host(double *host, double *rows_dev = nullptr, double *const *peer_rows = nullptr, int32_t n_peers = 0) {
        Output o = table_dev(rows_dev, peer_rows, n_peers);
        o.to_host = true; o.rows_host = host;
        return o;
    }
    static Output counts(double threshold, int32_t *C_dev, int32_t *C_host) {
        Output o;
        o.is_graph = true; o.graph.threshold = threshold; o.graph.C = C_dev; o.counts_host = C_host;
        return o;
    }
    void begin(int32_t n_docs, int32_t cols, cudaStream_t s) {
        if (is_graph) {
            if (counts_host) {
                own_counts = DevBuf<int32_t>((size_t)cols * cols, s);
                graph.C = own_counts.p;
            }
            graph.begin(n_docs, cols, s);
        } else if (!rows) {
            own_rows = DevBuf<double>((size_t)n_docs * cols, s);
            rows = own_rows.p;
        }
    }
};

// Where a build-and-score call's documents come from: packed text on the host (width 4: uint32 code points, 1: one byte
// per code point), packed text on the device, or raw UTF-8 texts (doc_off: their byte offsets) that the call packs on
// the device into a text the index then owns, also returning the packed offsets and string counts when asked.
struct Source {
    enum Kind { HOST, DEVICE, TEXTS } kind;
    const void *text;
    int width;                           // HOST: 4 or 1 (text_width); DEVICE: 4; TEXTS: 1
    const int64_t *doc_off;
    const int32_t *doc_m;                // TEXTS: NULL
    int32_t n_docs;
    int device;
    cudaStream_t stream = 0;
    int64_t *doc_off_out = nullptr;      // TEXTS, optional
    int32_t *doc_m_out = nullptr;
};

static void check_keyphrases(const int64_t *kp_off, int32_t K) {
    if (kp_off[K] >= (1ll << 31)) throw Error(EAST_ERR_RANGE, "keyphrase buffer too large");
    for (int32_t k = 0; k < K; ++k) {
        if (kp_off[k + 1] <= kp_off[k]) throw Error(EAST_ERR_ZERODIV, "empty query: float division by zero");
        if (kp_off[k + 1] - kp_off[k] > 0xffff) throw Error(EAST_ERR_RANGE, "keyphrase longer than 65535 code points");
    }
}

// the host-side checks of raw UTF-8 texts (texts_to_packed)
static void check_texts(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts) {
    if (!utf8 || !text_off || n_texts <= 0) throw Error(EAST_ERR_INVALID, "bad argument");
    if (text_off[0] != 0) throw Error(EAST_ERR_INVALID, "text_off[0] must be 0");
    for (int32_t i = 0; i < n_texts; ++i)
        if (text_off[i + 1] < text_off[i]) throw Error(EAST_ERR_INVALID, "text offsets must not decrease");
    if (text_off[n_texts] >= (1ll << 31)) throw Error(EAST_ERR_RANGE, "more than 2^31 bytes of text in one call; split the collection");
}

// The argument checks of every build-and-score and score entry, made before its first CUDA call, in one order (see
// include/east_b200.h): the output, peers and text_width; the documents (raw texts: their offsets; a score call on an
// index: the index and the document range [doc_begin, doc_begin + doc_count)); the groups; the keyphrases.
static void validate(const Output &out, const Source *src, const Query &q, const east_index *idx = nullptr,
                     int32_t doc_begin = 0, int32_t doc_count = 0) {
    if (out.is_graph ? !out.graph.C && !out.counts_host : !(out.to_host ? out.rows_host : out.rows))
        throw Error(EAST_ERR_INVALID, "bad argument");
    if (out.n_peers < 0 || out.n_peers > DocScore::MAX_PEERS || (out.n_peers > 0 && !out.peer_rows))
        throw Error(EAST_ERR_INVALID, "bad peer list");
    if (src && src->width != 1 && src->width != 4) throw Error(EAST_ERR_INVALID, "text_width must be 1 or 4");
    if (!src) {
        if (!idx) throw Error(EAST_ERR_INVALID, "bad argument");
        if (doc_begin < 0 || doc_count <= 0 || (int64_t)doc_begin + doc_count > idx->n_docs) throw Error(EAST_ERR_INVALID, "bad document range");
    } else if (src->kind == Source::TEXTS) {
        check_texts(static_cast<const uint8_t *>(src->text), src->doc_off, src->n_docs);
    } else {
        check_documents(src->text, src->doc_off, src->doc_m, src->n_docs);
    }
    if (q.grouped) {   // V variants in G groups, every group non-empty, the offsets ending at V
        if (!q.group_off || q.G < 1) throw Error(EAST_ERR_INVALID, "no groups of variants");
        if (q.group_off[0] != 0 || q.group_off[q.G] != q.K) throw Error(EAST_ERR_INVALID, "group offsets must run from 0 to the number of variants");
        for (int32_t g = 0; g < q.G; ++g)
            if (q.group_off[g + 1] <= q.group_off[g]) throw Error(EAST_ERR_INVALID, "empty group of variants");
    }
    if (!q.kp_off || q.K <= 0) throw Error(EAST_ERR_INVALID, "bad argument");
    check_keyphrases(q.kp_off, q.K);
    if (!(q.on_host ? q.kp_host : q.kp_dev)) throw Error(EAST_ERR_INVALID, "bad argument");
}

// score calls on an existing index: what was prepared for the previous call is kept (exact match of the code points)
static KpPrepared *prepare_keyphrases(const east_index *idx, const uint32_t *kp_dev, const uint32_t *kp_host_in,
                                      const int64_t *kp_off, int32_t K, bool dedup, cudaStream_t s) {
    const int64_t total = kp_off[K];
    const bool fast = idx->bkt && idx->t8 && !get_option("score_generic", 0);
    std::vector<uint32_t> kp_host;
    const uint32_t *kh = kp_host_in;
    if (!kh) {
        kp_host.resize((size_t)total);
        EAST_CUDA(cudaMemcpyAsync(kp_host.data(), kp_dev, sizeof(uint32_t) * (size_t)total, cudaMemcpyDeviceToHost, s));
        EAST_CUDA(cudaStreamSynchronize(s));
        kh = kp_host.data();
    }
    KpPrepared *c = g_kp_cache.get();
    if (c && c->finished && c->device == idx->device && c->dedup == dedup && c->fast == fast && (int64_t)c->off.size() == (int64_t)K + 1 &&
        (int64_t)c->kp.size() == total && std::equal(c->kp.begin(), c->kp.end(), kh) && std::equal(c->off.begin(), c->off.end(), kp_off) &&
        (!fast || (c->sym_bits == idx->sym_bits && c->code_table == idx->code_table)))
        return c;
    if (c) { cudaSetDevice(c->device); cudaDeviceSynchronize(); g_kp_cache.reset(); cudaSetDevice(idx->device); }
    g_kp_cache = kp_begin(idx->device, kp_dev, kh, kp_off, K, dedup, true, s, fast ? idx->code_table.data() : nullptr);
    c = g_kp_cache.get();
    kp_finish(c, kp_dev, fast, idx->sym_bits, idx->code_table, s);
    EAST_CUDA(cudaStreamSynchronize(s));
    // the entry outlives this call: whoever drops it frees on the legacy stream of its device, after a device sync
    for (cudaStream_t *ps : {&c->dev.d_off.s, &c->dev.d_uniq_of.s, &c->dev.d_recs.s, &c->dev.d_q8.s, &c->dev.d_n_uniq.s}) *ps = 0;
    return c;
}

// The launches that score documents [doc_begin, doc_begin + doc_count) of `idx` (tile_docs at a time through the
// scratch tmp[tile_docs][n_uniq]) into out_dev[(d - doc_begin) * cols + column]; with groups, q's groups must have been
// uploaded.  Nothing here waits for the device.
static void score_enqueue(const east_index *idx, const KpPrepared *kp, const Query &q, double *out_dev, int32_t doc_begin,
                          int32_t doc_count, cudaStream_t s, double *tmp, int32_t tile_docs, unsigned long long *probe_count,
                          double *const *peer_rows = nullptr /* sharded table: rows of document doc_begin in the peers' tables */,
                          int32_t n_peers = 0) {
    ensure_suffix_keys(idx, s);
    const int32_t cols = q.cols();   // columns of out_dev
    ScoreInput in;
    in.text = idx->text; in.sa = idx->sa;
    in.doc_off = idx->d_doc_off + doc_begin; in.doc_m = idx->d_doc_m + doc_begin; in.n_docs = doc_count;
    in.kp = q.kp_dev; in.kp_off = kp->dev.d_off.p; in.K = q.K; in.total_suffixes = (int32_t)q.total();
    in.uniq_of = kp->dev.d_uniq_of.p; in.recs = kp->dev.d_recs.p; in.n_uniq = (int32_t)kp->n_uniq;
    in.normalized = q.normalized;
    if (kp->fast) {
        in.t8 = idx->t8; in.sk = idx->sk; in.q8 = kp->dev.d_q8.p; in.sym_bits = idx->sym_bits;
        in.bkt = idx->bkt + ((size_t)doc_begin << (2 * idx->sym_bits));
        if (idx->bkt3 && !get_option("score_no_bkt3", 0)) in.bkt3 = idx->bkt3 + ((size_t)doc_begin << (3 * idx->sym_bits));
    }
    in.algorithmic_bytes = (double)get_option("score_bytes", 0);
    in.probe_count = probe_count;
    in.group_off = q.d_groups.p; in.G = q.G;
    auto tile = [&](int32_t d0, int32_t cnt) {
        ScoreInput part = in;
        part.n_docs = cnt;
        part.doc_off = in.doc_off + d0;
        part.doc_m = in.doc_m + d0;
        if (in.bkt) part.bkt = in.bkt + ((size_t)d0 << (2 * in.sym_bits));
        if (in.bkt3) part.bkt3 = in.bkt3 + ((size_t)d0 << (3 * in.sym_bits));
        part.algorithmic_bytes = in.algorithmic_bytes * ((double)part.n_docs / (double)doc_count);
        part.n_peers = n_peers;
        for (int32_t pi = 0; pi < n_peers; ++pi) part.peer_out[pi] = peer_rows[pi] + (size_t)d0 * cols;
        return part;
    };
    const int32_t n_tiles = (doc_count + tile_docs - 1) / tile_docs;
    if (n_tiles <= 2 || tile_docs < 2 || probe_count || get_option("score_no_overlap", 0)) {
        for (int32_t d0 = 0; d0 < doc_count; d0 += tile_docs) {
            const ScoreInput part = tile(d0, std::min(tile_docs, doc_count - d0));
            score_table(part, tmp, out_dev + (size_t)d0 * cols, s);
        }
        return;
    }
    // Many tiles (large K: the scratch holds a few hundred documents at a time): the keyphrase sums of tile t -- and, in a
    // sharded run, the peer stores of its rows, bound by NVLink, not by the SMs -- run on the auxiliary stream while the
    // walks of tile t + 1 keep the SMs busy; the scratch is used in two halves.
    const int32_t half = tile_docs / 2;
    cudaStream_t aux = aux_stream(idx->device);
    cudaEvent_t walked[2], summed[2];
    for (int i = 0; i < 2; ++i) {
        EAST_CUDA(cudaEventCreateWithFlags(&walked[i], cudaEventDisableTiming));
        EAST_CUDA(cudaEventCreateWithFlags(&summed[i], cudaEventDisableTiming));
    }
    int t = 0;
    for (int32_t d0 = 0; d0 < doc_count; d0 += half, ++t) {
        const int b = t & 1;
        const ScoreInput part = tile(d0, std::min(half, doc_count - d0));
        double *buf = tmp + (size_t)b * (size_t)half * (size_t)in.n_uniq;
        if (t >= 2) EAST_CUDA(cudaStreamWaitEvent(s, summed[b], 0));   // the sums that read this half two tiles ago
        score_suffixes(part, buf, s);
        EAST_CUDA(cudaEventRecord(walked[b], s));
        EAST_CUDA(cudaStreamWaitEvent(aux, walked[b], 0));
        score_combine(part, buf, out_dev + (size_t)d0 * cols, aux);
        EAST_CUDA(cudaEventRecord(summed[b], aux));
    }
    for (int i = 0; i < 2; ++i) {
        EAST_CUDA(cudaStreamWaitEvent(s, summed[i], 0));
        EAST_CUDA(cudaEventDestroy(walked[i]));     // released once they have fired
        EAST_CUDA(cudaEventDestroy(summed[i]));
    }
}

// documents per tile of a graph call's fp64 scratch
static int32_t graph_tile_docs(int32_t doc_count, int32_t cols) {
    const int64_t budget = get_option("score_tmp_doubles", (int64_t)1 << 27);
    return (int32_t)std::max<int64_t>(1, std::min<int64_t>(doc_count, budget / std::max<int32_t>(1, cols)));
}

// score_enqueue for a graph: documents [doc_begin, doc_begin + doc_count) tile by tile into S[S_docs][cols], each tile
// thresholded into its columns of g.B (stream-ordered: the next tile overwrites S after the previous one is read)
static void graph_enqueue(const east_index *idx, const KpPrepared *kp, const Query &q, int32_t doc_begin, int32_t doc_count,
                          cudaStream_t s, double *tmp, int32_t tile_docs, const GraphOut &g, double *S, int32_t S_docs) {
    for (int32_t d0 = 0; d0 < doc_count; d0 += S_docs) {
        const int32_t cnt = std::min(S_docs, doc_count - d0);
        score_enqueue(idx, kp, q, S, doc_begin + d0, cnt, s, tmp, tile_docs, nullptr);
        threshold_bytes(S, cnt, q.cols(), g.threshold, g.B.p, g.Dp, (int64_t)doc_begin + d0, s);
    }
}

// documents [doc_begin, doc_begin + doc_count) of `idx` scored into out_dev, or into the relevance bytes of `graph`
static void score_common(const east_index *idx, Query &q, double *out_dev, const GraphOut *graph, int32_t doc_begin,
                         int32_t doc_count, cudaStream_t s,
                         double *suffix_out_dev = nullptr /* optional: per-suffix results of the doc range */,
                         int64_t *probes_out = nullptr /* optional: run the probe-counting scorer */) {
    // per-suffix results wanted (return_suffix_scores): every suffix is its own "distinct" suffix
    const bool dedup = !suffix_out_dev && !get_option("score_no_dedup", 0);
    KpPrepared *kp = prepare_keyphrases(idx, q.kp_dev, q.kp_host, q.kp_off, q.K, dedup, s);
    const int64_t n_uniq = kp->n_uniq;

    // per-suffix results tmp[doc][distinct suffix] are produced and consumed tile by tile over the documents,
    // so the scratch stays <= ~1 GB however large K x D is (config 4: 0.63 M distinct suffixes x 12 500 docs)
    DevBuf<double> tmp_own;
    double *tmp = suffix_out_dev;
    int32_t tile_docs = doc_count;
    if (!tmp) {
        const int64_t budget = get_option("score_tmp_doubles", (int64_t)1 << 27);
        tile_docs = (int32_t)std::max<int64_t>(1, std::min<int64_t>(doc_count, budget / std::max<int64_t>(1, n_uniq)));
        tmp_own = DevBuf<double>((size_t)tile_docs * (size_t)n_uniq, s);
        tmp = tmp_own.p;
    }
    q.upload_groups(s);
    DevBuf<unsigned long long> d_probes;
    if (probes_out) {
        d_probes = DevBuf<unsigned long long>(1, s);
        EAST_CUDA(cudaMemsetAsync(d_probes.p, 0, sizeof(unsigned long long), s));
    }
    StageTimer tm(s);
    tm.mark("score");
    if (graph) {
        const int32_t S_docs = graph_tile_docs(doc_count, q.cols());
        DevBuf<double> S((size_t)S_docs * q.cols(), s);
        graph_enqueue(idx, kp, q, doc_begin, doc_count, s, tmp, tile_docs, *graph, S.p, S_docs);
    } else {
        score_enqueue(idx, kp, q, out_dev, doc_begin, doc_count, s, tmp, tile_docs, d_probes.p);
    }
    tm.finish();
    if (probes_out) {
        unsigned long long h = 0;
        EAST_CUDA(cudaMemcpyAsync(&h, d_probes.p, sizeof(h), cudaMemcpyDeviceToHost, s));
        EAST_CUDA(cudaStreamSynchronize(s));
        *probes_out = (int64_t)h;
    }
    EAST_CUDA(cudaStreamSynchronize(s));
    tm.collect();
}

// The score calls on an index: checked, then scored; the host entries upload the code points and copy the rows back.
static void score_index(const east_index *idx, Query q, Output out, int32_t doc_begin, int32_t doc_count, void *stream,
                        int64_t *probes = nullptr) {
    validate(out, nullptr, q, idx, doc_begin, doc_count);
    EAST_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    DevBuf<uint32_t> d_kp;
    if (q.on_host) d_kp = q.upload(s);
    out.begin(doc_count, q.cols(), s);
    score_common(idx, q, out.rows, nullptr, doc_begin, doc_count, s, nullptr, probes);
    if (out.to_host) EAST_CUDA(cudaMemcpy(out.rows_host, out.rows, sizeof(double) * (size_t)doc_count * q.cols(), cudaMemcpyDeviceToHost));
}

int east_score_table_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off, int32_t K,
                         int normalized, double *out_DxK_dev, void *stream) {
    EAST_API_BEGIN
    score_index(idx, Query(kp_dev, false, nullptr, kp_off, K, normalized), Output::table_dev(out_DxK_dev), 0,
                idx ? idx->n_docs : 0, stream);
    EAST_API_END
}

int east_score_range_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off, int32_t K, int normalized,
                         int32_t doc_begin, int32_t doc_count, double *out_dev, void *stream) {
    EAST_API_BEGIN
    score_index(idx, Query(kp_dev, false, nullptr, kp_off, K, normalized), Output::table_dev(out_dev), doc_begin, doc_count,
                stream);
    EAST_API_END
}

int east_score_probes_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off, int32_t K,
                          double *out_DxK_dev, void *stream, int64_t *probes) {
    EAST_API_BEGIN
    score_index(idx, Query(kp_dev, false, nullptr, kp_off, K, 1),
                Output::table_dev(probes ? out_DxK_dev : nullptr /* the probe count is an output too */), 0,
                idx ? idx->n_docs : 0, stream, probes);
    EAST_API_END
}

int east_score_groups_dev(const east_index *idx, const uint32_t *kp_dev, const int64_t *kp_off, int32_t V,
                          const int64_t *group_off, int32_t G, int32_t doc_begin, int32_t doc_count, double *out_dev,
                          void *stream) {
    EAST_API_BEGIN
    score_index(idx, Query(kp_dev, false, nullptr, kp_off, V, 1, true, group_off, G), Output::table_dev(out_dev), doc_begin,
                doc_count, stream);
    EAST_API_END
}

int east_score_groups_host(const east_index *idx, const uint32_t *kp, const int64_t *kp_off, int32_t V,
                           const int64_t *group_off, int32_t G, int32_t doc_begin, int32_t doc_count, double *out_host) {
    EAST_API_BEGIN
    score_index(idx, Query(kp, true, nullptr, kp_off, V, 1, true, group_off, G), Output::table_host(out_host), doc_begin,
                doc_count, 0);
    EAST_API_END
}

int east_score_table_host(const east_index *idx, const uint32_t *kp, const int64_t *kp_off, int32_t K,
                          int normalized, double *out_DxK) {
    EAST_API_BEGIN
    score_index(idx, Query(kp, true, nullptr, kp_off, K, normalized), Output::table_host(out_DxK), 0, idx ? idx->n_docs : 0, 0);
    EAST_API_END
}

int east_score_one(const east_index *idx, int32_t doc, const uint32_t *q, int32_t len, int normalized,
                   double *score, double *suffix_scores) {
    EAST_API_BEGIN
    const int64_t off[2] = {0, q ? len : 0};   // no code points: the empty query
    Query query(q, true, nullptr, off, 1, normalized);
    validate(Output::table_host(score), nullptr, query, idx, doc, 1);
    EAST_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = 0;
    DevBuf<uint32_t> d_q = query.upload(s);
    DevBuf<double> d_out(1, s), d_suf(len, s);
    score_common(idx, query, d_out.p, nullptr, doc, 1, s, d_suf.p);
    EAST_CUDA(cudaMemcpy(score, d_out.p, sizeof(double), cudaMemcpyDeviceToHost));
    if (suffix_scores) EAST_CUDA(cudaMemcpy(suffix_scores, d_suf.p, sizeof(double) * len, cudaMemcpyDeviceToHost));
    EAST_API_END
}

// ---- device preprocessing (tokenize.cu) -----------------------------------------------------
namespace {
struct PackedTexts {
    uint32_t *text = nullptr;          // device, owned until released
    std::vector<int64_t> doc_off;
    std::vector<int32_t> doc_m;
    ~PackedTexts() { if (text) dev_free(text, 0); }
};

// raw UTF-8 texts (host; check_texts has accepted them) -> packed documents on the device; throws EAST_ERR_UNSUPPORTED
// when a text needs the host path
void texts_to_packed(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, cudaStream_t s, PackedTexts &out) {
    const int64_t bytes = text_off[n_texts];
    DevBuf<uint8_t> d_raw((size_t)bytes + 16, s);
    DevBuf<int64_t> d_off((size_t)n_texts + 1, s), d_doc_off((size_t)n_texts + 1, s);
    DevBuf<int32_t> d_sizes(3 * (size_t)n_texts, s);
    if (bytes) EAST_CUDA(cudaMemcpyAsync(d_raw.p, utf8, (size_t)bytes, cudaMemcpyHostToDevice, s));
    EAST_CUDA(cudaMemcpyAsync(d_off.p, text_off, sizeof(int64_t) * ((size_t)n_texts + 1), cudaMemcpyHostToDevice, s));
    tokenize_texts(d_raw.p, d_off.p, n_texts, d_sizes.p, s);
    std::vector<int32_t> sizes(3 * (size_t)n_texts);
    EAST_CUDA(cudaMemcpyAsync(sizes.data(), d_sizes.p, sizeof(int32_t) * sizes.size(), cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaStreamSynchronize(s));
    out.doc_off.assign((size_t)n_texts + 1, 0);
    out.doc_m.resize((size_t)n_texts);
    for (int32_t i = 0; i < n_texts; ++i) {
        if (sizes[3 * (size_t)i + 2])
            throw Error(EAST_ERR_UNSUPPORTED, "text " + std::to_string(i) + " has characters outside ASCII / U+0400-045F (or invalid UTF-8): "
                                              "use the host preprocessing");
        out.doc_off[(size_t)i + 1] = out.doc_off[(size_t)i] + sizes[3 * (size_t)i];
        out.doc_m[(size_t)i] = sizes[3 * (size_t)i + 1];
    }
    if (out.doc_off.back() >= (1ll << 30)) throw Error(EAST_ERR_RANGE, "more than 2^30 code points in one index; split the batch");
    EAST_CUDA(cudaMemcpyAsync(d_doc_off.p, out.doc_off.data(), sizeof(int64_t) * out.doc_off.size(), cudaMemcpyHostToDevice, s));
    out.text = (uint32_t *)dev_alloc(sizeof(uint32_t) * (size_t)out.doc_off.back(), s, true);
    tokenize_emit(d_raw.p, d_off.p, n_texts, d_doc_off.p, out.text, s);
    EAST_CUDA(cudaStreamSynchronize(s));   // the staging buffers (and the pageable doc_off upload) end here
}
}  // namespace

int east_texts_to_packed_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device, uint32_t *packed_out,
                              int64_t packed_cap, int64_t *doc_off_out, int32_t *doc_m_out) {
    EAST_API_BEGIN
    if (!doc_off_out || !doc_m_out) throw Error(EAST_ERR_INVALID, "NULL argument");
    check_texts(utf8, text_off, n_texts);
    use_device(device);
    PackedTexts pt;
    texts_to_packed(utf8, text_off, n_texts, 0, pt);
    std::copy(pt.doc_off.begin(), pt.doc_off.end(), doc_off_out);
    std::copy(pt.doc_m.begin(), pt.doc_m.end(), doc_m_out);
    if (pt.doc_off.back() > packed_cap || !packed_out) throw Error(EAST_ERR_RANGE, "packed_out is too small (doc_off_out holds the sizes)");
    EAST_CUDA(cudaMemcpy(packed_out, pt.text, sizeof(uint32_t) * (size_t)pt.doc_off.back(), cudaMemcpyDeviceToHost));
    EAST_API_END
}

// ---- build + score in one call ------------------------------------------------------------
// applications.keyphrases_table (applications.py:43-52) builds the structure of a text and scores every
// keyphrase against it, text after text.  Here: while the pipelined host build is still receiving the
// later runs of documents, the runs that are already sorted are scored on the stream that sorted them
// and their rows of the table go back to the host -- copy-in, sort, score and copy-out overlap.
struct TableRun {
    Query &q;
    Output &out;
    const east_index *building = nullptr;
    double *host_out = nullptr;           // the host build: each run's rows are copied here as they are scored
    // the batched scorer's rows of a graph call go through the per-stream scratch rows[] of rows_docs documents
    DevBuf<double> rows[2];
    int32_t rows_docs[2] = {0, 0};
    int32_t docs_sent = 0;                // documents whose rows have reached the peers (current pass)
    std::unique_ptr<KpPrepared> kp_own;   // prepared for this call only (a table call is made once per collection)
    // device builds: stage 1 of the preparation is queued from the build's scan_queued hook (its ~15 launches are host
    // time that hides under the round trip of the alphabet scan); everything it needs:
    int device = 0;
    bool dedup = !get_option("score_no_dedup", 0);
    cudaStream_t kp_stream = nullptr, caller_stream = nullptr;
    cudaEvent_t kp_ready = nullptr;       // dense codes of the current pass queued
    KpPrepared *kp = nullptr;
    east_index view;                 // non-owning: the pointers of the index under construction + the run's tables
    cudaStream_t lane[2] = {nullptr, nullptr};
    bool lane_used[2] = {false, false};
    DevBuf<double> tmp[2];           // per-stream scratch of the scorer: [documents of a run][distinct suffixes]
    int64_t tmp_docs[2] = {0, 0};
    int32_t docs_scored = 0;         // of the current pass over the batch (a pass starts with document 0)
    int final_pass = 0;              // the last pass was not speculative
    bool failed = false;
    TableRun(Query &q_, Output &out_, int device_) : q(q_), out(out_), device(device_) {}
    ~TableRun() { if (kp_ready) cudaEventDestroy(kp_ready); }
};

// the code table a table call's build is expected to end up with: that of the guessed alphabet (sa_build.cu), if any
static const uint8_t *likely_code_table() {
    static thread_local uint8_t table[EAST_TERM_BASE];
    if (get_option("no_alphabet_guess", 0)) return nullptr;
    return alphabet_guess_code_table(table) ? table : nullptr;
}

static void table_kp_begin(void *vctx) {
    TableRun &t = *static_cast<TableRun *>(vctx);
    if (t.kp_own) return;
    try {
        cudaEvent_t inputs_ready;   // the keyphrases may have been produced on the caller's stream
        EAST_CUDA(cudaEventCreateWithFlags(&inputs_ready, cudaEventDisableTiming));
        EAST_CUDA(cudaEventRecord(inputs_ready, t.caller_stream));
        EAST_CUDA(cudaStreamWaitEvent(t.kp_stream, inputs_ready, 0));
        EAST_CUDA(cudaEventDestroy(inputs_ready));
        t.kp_own = kp_begin(t.device, t.q.kp_dev, t.q.kp_host, t.q.kp_off, t.q.K, t.dedup, false, t.kp_stream, likely_code_table());
    } catch (...) {
        t.failed = true;
    }
}

static int table_lane(TableRun &t, cudaStream_t s) {
    for (int i = 0; i < 2; ++i)
        if (t.lane_used[i] && t.lane[i] == s) return i;
    for (int i = 0; i < 2; ++i)
        if (!t.lane_used[i]) { t.lane_used[i] = true; t.lane[i] = s; return i; }
    throw Error(EAST_ERR_INVALID, "the build used more than two streams");
}

// before the per-document kernel of a run is launched: have it score the run itself when the scratch fits
static void table_run_begin(void *vctx, const RunReady &r, DocScore &score) {
    TableRun &t = *static_cast<TableRun *>(vctx);
    const Query &q = t.q;
    try {
        if (r.doc_begin == 0) {   // a new pass over the batch (the first, or the ordinary build after a failed speculation)
            t.failed = false;
            t.docs_scored = 0;
            t.docs_sent = 0;
            t.final_pass = r.speculative ? 0 : 1;
            const east_index *b = t.building;
            east_index &v = t.view;
            v.device = b->device; v.n_docs = b->n_docs; v.n = b->n;
            v.text = b->text; v.sa = b->sa; v.sk = b->sk; v.d_doc_off = b->d_doc_off; v.d_doc_m = b->d_doc_m;
            v.t8 = const_cast<uint8_t *>(r.t8);
            v.bkt = const_cast<uint32_t *>(r.bkt);
            v.bkt3 = const_cast<uint32_t *>(r.bkt3);
            v.sym_bits = r.sym_bits;
            v.code_table = *r.code_table;
            const bool fast = v.bkt && v.t8 && !get_option("score_generic", 0);
            table_kp_begin(&t);   // (the builds that do not scan first -- pipelined host build -- have queued it long ago)
            if (!t.kp_own) return;
            host_debug_mark("kp_finish begin");
            kp_finish(t.kp_own.get(), q.kp_dev, fast, v.sym_bits, v.code_table, r.stream);
            t.kp = t.kp_own.get();
            if (!t.kp_ready) EAST_CUDA(cudaEventCreateWithFlags(&t.kp_ready, cudaEventDisableTiming));
            EAST_CUDA(cudaEventRecord(t.kp_ready, r.stream));
            host_debug_mark("kp_finish end");
        }
        if (t.failed || !t.kp) return;
        EAST_CUDA(cudaStreamWaitEvent(r.stream, t.kp_ready, 0));   // the other lane: the dense codes were queued on the first
        const int li = table_lane(t, r.stream);
        const int64_t n_uniq = std::max<int64_t>(1, t.kp->n_uniq);
        const int64_t budget = get_option("score_tmp_doubles", (int64_t)1 << 27);
        const bool in_kernel = t.kp->fast && (int64_t)r.doc_count * n_uniq <= budget && !get_option("no_fused_score", 0) &&
                               (!q.grouped || q.G <= DocScore::MAX_GROUPS);   // the groups' maxima fit the shared memory
        const int64_t want = in_kernel ? r.doc_count : std::max<int64_t>(1, std::min<int64_t>(r.doc_count, budget / n_uniq));
        if (t.tmp_docs[li] < want) {
            t.tmp[li] = DevBuf<double>((size_t)want * (size_t)n_uniq, r.stream);
            t.tmp_docs[li] = want;
        }
        if (in_kernel) {
            score.recs = t.kp->dev.d_recs.p; score.n_uniq = (int32_t)t.kp->n_uniq; score.q8 = t.kp->dev.d_q8.p; score.kp = q.kp_dev;
            score.tmp = t.tmp[li].p; score.normalized = q.normalized;
            score.kp_off = t.kp->dev.d_off.p; score.uniq_of = t.kp->dev.d_uniq_of.p; score.K = q.K;
            if (t.out.is_graph) {
                score.graph = t.out.graph.B.p; score.graph_pitch = t.out.graph.Dp; score.graph_col0 = r.doc_begin;
                score.threshold = t.out.graph.threshold;
            } else {
                score.out = t.out.rows + (size_t)r.doc_begin * q.cols();
            }
            if (q.grouped) { score.group_off = q.d_groups.p; score.G = q.G; }
            score.skip_suffix_keys = get_option("eager_suffix_keys", 0) ? 0 : 1;
            score.n_peers = t.out.n_peers;
            for (int32_t pi = 0; pi < t.out.n_peers; ++pi) score.peer_out[pi] = t.out.peer_rows[pi] + (size_t)r.doc_begin * q.cols();
            score.algorithmic_bytes = (double)get_option("score_bytes", 0) * ((double)r.doc_count / (double)t.view.n_docs);
        }
    } catch (...) {
        t.failed = true;   // the ordinary score call after the build reports whatever this was
    }
}

// after the launch: the batched scorer if the kernel did not score the run itself, and the rows of the table on
// their way to the host
static void table_run_done(void *vctx, const RunReady &r, int in_kernel) {
    TableRun &t = *static_cast<TableRun *>(vctx);
    if (t.failed || !t.kp) return;
    try {
        const int li = table_lane(t, r.stream);
        const int32_t cols = t.q.cols();
        if (t.out.is_graph) {
            if (!in_kernel) {
                const int32_t S_docs = graph_tile_docs(r.doc_count, cols);
                if (t.rows_docs[li] < S_docs) {
                    t.rows[li] = DevBuf<double>((size_t)S_docs * cols, r.stream);
                    t.rows_docs[li] = S_docs;
                }
                graph_enqueue(&t.view, t.kp, t.q, r.doc_begin, r.doc_count, r.stream, t.tmp[li].p, (int32_t)t.tmp_docs[li],
                              t.out.graph, t.rows[li].p, t.rows_docs[li]);
            }
            t.docs_scored += r.doc_count;
            return;
        }
        double *rows = t.out.rows + (size_t)r.doc_begin * cols;
        if (!in_kernel) {
            std::vector<double *> peers((size_t)t.out.n_peers);
            for (int32_t pi = 0; pi < t.out.n_peers; ++pi) peers[(size_t)pi] = t.out.peer_rows[pi] + (size_t)r.doc_begin * cols;
            score_enqueue(&t.view, t.kp, t.q, rows, r.doc_begin, r.doc_count, r.stream, t.tmp[li].p, (int32_t)t.tmp_docs[li],
                          nullptr, peers.data(), t.out.n_peers);
        }
        t.docs_sent += r.doc_count;   // the rows reach the peers from the kernels that produce them, on either path
        if (t.host_out)
            EAST_CUDA(cudaMemcpyAsync(t.host_out + (size_t)r.doc_begin * cols, rows, sizeof(double) * (size_t)r.doc_count * cols,
                                      cudaMemcpyDeviceToHost, r.stream));
        t.docs_scored += r.doc_count;
    } catch (...) {
        t.failed = true;
    }
}

// Every build-and-score entry: checks, builds the index of `src` with `q` scored into `out` on the way, and re-scores the
// index when the rows scored during the build do not stand.
static void run_table(Source src, Query q, Output out, east_index **out_idx) {
    validate(out, &src, q);
    use_device(src.device);
    cudaStream_t s = src.stream;
    TableRun run(q, out, src.device);
    RunHook hook;
    hook.begin = table_run_begin; hook.fn = table_run_done; hook.ctx = &run; hook.building = &run.building;
    DevBuf<uint32_t> d_kp;   // the host code points, uploaded
    PackedTexts pt;          // raw texts: the packed text, owned here until the index takes it over
    east_index *built = nullptr;
    if (src.kind == Source::HOST) {
        // the keyphrases go first, on a side stream: hashing, ordering and de-duplication of their suffixes (kp_prep.cu)
        // run there while the text is on its way
        cudaStream_t ps = prep_stream(src.device);
        d_kp = q.upload(ps);
        out.begin(src.n_docs, q.cols(), s);
        run.kp_own = kp_begin(src.device, q.kp_dev, q.kp_host, q.kp_off, q.K, run.dedup, false, ps, likely_code_table());
        q.upload_groups(s);
        run.host_out = out.rows_host;
        build_host_impl(src.text, src.width, src.doc_off, src.doc_m, src.n_docs, src.device, &built, &hook);
    } else {
        if (src.kind == Source::TEXTS) {
            texts_to_packed(static_cast<const uint8_t *>(src.text), src.doc_off, src.n_docs, s, pt);
            if (src.doc_off_out) std::copy(pt.doc_off.begin(), pt.doc_off.end(), src.doc_off_out);
            if (src.doc_m_out) std::copy(pt.doc_m.begin(), pt.doc_m.end(), src.doc_m_out);
            d_kp = q.upload(s);
            src.text = pt.text; src.doc_off = pt.doc_off.data(); src.doc_m = pt.doc_m.data();
        }
        out.begin(src.n_docs, q.cols(), s);
        q.upload_groups(s);
        // keyphrase preparation on a side stream, queued from the build once its alphabet scan is on its way
        run.kp_stream = prep_stream(src.device); run.caller_stream = s;
        hook.scan_queued = table_kp_begin;
        if (get_option("kp_upfront", 0)) table_kp_begin(&run);   // A/B: queue the preparation before the build starts
        const bool owns_text = src.kind == Source::TEXTS;
        pt.text = nullptr;   // build_common's index owns it from its first statement on
        build_common(static_cast<const uint32_t *>(src.text), owns_text, src.doc_off, src.doc_m, src.n_docs, src.device, s,
                     &built, nullptr, &hook);
    }
    std::unique_ptr<east_index, void (*)(east_index *)> guard(built, free_index);
    // Rows scored on the way stand if the pass that produced them is the one the index came from: the speculative
    // pipelined pass of a host build (pipelined = 1: the build ended on a host sync after both streams, the rows are in
    // place) or the ordinary per-document pass (its copies are still in flight on stream s).
    const int32_t n_docs = src.n_docs, cols = q.cols();
    const bool stands = !run.failed && run.docs_scored == n_docs &&
                        ((built->pipelined && !run.final_pass) || (built->doc_sorted && !built->pipelined && run.final_pass));
    if (!stands) score_common(built, q, out.rows, out.is_graph ? &out.graph : nullptr, 0, n_docs, s);
    if (out.to_host && !(stands && run.host_out))   // the rows did not go to the host run by run
        EAST_CUDA(cudaMemcpyAsync(out.rows_host, out.rows, sizeof(double) * (size_t)n_docs * cols, cudaMemcpyDeviceToHost, s));
    if (out.n_peers > 0 && !(stands && run.docs_sent == n_docs))   // rows (also) produced by the batched scorer: plain peer copies
        for (int32_t pi = 0; pi < out.n_peers; ++pi)
            EAST_CUDA(cudaMemcpyAsync(out.peer_rows[pi], out.rows, sizeof(double) * (size_t)n_docs * cols, cudaMemcpyDefault, s));
    if (out.is_graph) {
        out.graph.finish(cols, s);
        if (out.counts_host)
            EAST_CUDA(cudaMemcpyAsync(out.counts_host, out.graph.C, sizeof(int32_t) * (size_t)cols * cols, cudaMemcpyDeviceToHost, s));
    }
    EAST_CUDA(cudaStreamSynchronize(s));
    if (out_idx) *out_idx = guard.release();
}

int east_table_host(const uint32_t *text, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                    const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized, double *out_DxK,
                    east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::HOST, text, 4, doc_off, doc_m, n_docs, device},
              Query(kp, true, nullptr, kp_off, K, normalized), Output::table_host(out_DxK), out_idx);
    EAST_API_END
}

int east_table_host_u8(const uint8_t *text8, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                       const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized, double *out_DxK,
                       east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::HOST, text8, 1, doc_off, doc_m, n_docs, device},
              Query(kp, true, nullptr, kp_off, K, normalized), Output::table_host(out_DxK), out_idx);
    EAST_API_END
}

int east_table_host_gather(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                           int device, const uint32_t *kp, const int64_t *kp_off, int32_t K, int normalized, double *out_DxK,
                           double *own_rows_dev, double *const *peer_rows, int32_t n_peers, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::HOST, text, text_width, doc_off, doc_m, n_docs, device},
              Query(kp, true, nullptr, kp_off, K, normalized),
              Output::table_host(out_DxK, own_rows_dev, peer_rows, n_peers), out_idx);
    EAST_API_END
}

int east_table_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                   const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t K, int normalized,
                   double *out_DxK_dev, void *stream, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::DEVICE, text_dev, 4, doc_off, doc_m, n_docs, device, (cudaStream_t)stream},
              Query(kp_dev, false, kp_host, kp_off, K, normalized), Output::table_dev(out_DxK_dev), out_idx);
    EAST_API_END
}

int east_table_dev_gather(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                          const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t K, int normalized,
                          double *out_DxK_dev, double *const *peer_rows, int32_t n_peers, void *stream, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::DEVICE, text_dev, 4, doc_off, doc_m, n_docs, device, (cudaStream_t)stream},
              Query(kp_dev, false, kp_host, kp_off, K, normalized), Output::table_dev(out_DxK_dev, peer_rows, n_peers), out_idx);
    EAST_API_END
}

int east_table_texts_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device, const uint32_t *kp,
                          const int64_t *kp_off, int32_t K, int normalized, double *out_DxK, int64_t *doc_off_out,
                          int32_t *doc_m_out, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::TEXTS, utf8, 1, text_off, nullptr, n_texts, device, 0, doc_off_out, doc_m_out},
              Query(kp, true, nullptr, kp_off, K, normalized), Output::table_host(out_DxK), out_idx);
    EAST_API_END
}

// ---- synonym-expanded tables in one call: the per-document kernel keeps the best variant of every group ------------
int east_table_groups_host(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                           int device, const uint32_t *kp, const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G,
                           double *out_DxG, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::HOST, text, text_width, doc_off, doc_m, n_docs, device},
              Query(kp, true, nullptr, kp_off, V, 1, true, group_off, G), Output::table_host(out_DxG), out_idx);
    EAST_API_END
}

int east_table_groups_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                          const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t V,
                          const int64_t *group_off, int32_t G, double *out_DxG_dev, double *const *peer_rows, int32_t n_peers,
                          void *stream, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::DEVICE, text_dev, 4, doc_off, doc_m, n_docs, device, (cudaStream_t)stream},
              Query(kp_dev, false, kp_host, kp_off, V, 1, true, group_off, G),
              Output::table_dev(out_DxG_dev, peer_rows, n_peers), out_idx);
    EAST_API_END
}

int east_table_texts_groups_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device, const uint32_t *kp,
                                 const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G, double *out_DxG,
                                 int64_t *doc_off_out, int32_t *doc_m_out, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::TEXTS, utf8, 1, text_off, nullptr, n_texts, device, 0, doc_off_out, doc_m_out},
              Query(kp, true, nullptr, kp_off, V, 1, true, group_off, G), Output::table_host(out_DxG), out_idx);
    EAST_API_END
}

// ---- keyphrase graphs in one call: build, score and count co-occurrences, no score table ------------------------------
// (group_off NULL: plain keyphrases)
int east_graph_host(const void *text, int32_t text_width, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs,
                    int device, const uint32_t *kp, const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G,
                    int normalized, double threshold, int32_t *C_host, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::HOST, text, text_width, doc_off, doc_m, n_docs, device},
              Query(kp, true, nullptr, kp_off, V, normalized, group_off != nullptr, group_off, G),
              Output::counts(threshold, nullptr, C_host), out_idx);
    EAST_API_END
}

int east_graph_dev(const uint32_t *text_dev, const int64_t *doc_off, const int32_t *doc_m, int32_t n_docs, int device,
                   const uint32_t *kp_dev, const uint32_t *kp_host, const int64_t *kp_off, int32_t V, const int64_t *group_off,
                   int32_t G, int normalized, double threshold, int32_t *C_dev, void *stream, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::DEVICE, text_dev, 4, doc_off, doc_m, n_docs, device, (cudaStream_t)stream},
              Query(kp_dev, false, kp_host, kp_off, V, normalized, group_off != nullptr, group_off, G),
              Output::counts(threshold, C_dev, nullptr), out_idx);
    EAST_API_END
}

int east_graph_texts_host(const uint8_t *utf8, const int64_t *text_off, int32_t n_texts, int device, const uint32_t *kp,
                          const int64_t *kp_off, int32_t V, const int64_t *group_off, int32_t G, int normalized, double threshold,
                          int32_t *C_host, int64_t *doc_off_out, int32_t *doc_m_out, east_index **out_idx) {
    EAST_API_BEGIN
    run_table({Source::TEXTS, utf8, 1, text_off, nullptr, n_texts, device, 0, doc_off_out, doc_m_out},
              Query(kp, true, nullptr, kp_off, V, normalized, group_off != nullptr, group_off, G),
              Output::counts(threshold, nullptr, C_host), out_idx);
    EAST_API_END
}

// ---- graph ------------------------------------------------------------------------------
int east_cooc_dev(const double *S_DxK_dev, int64_t D, int32_t K, double threshold, int32_t *C_KxK_dev, int device,
                  void *stream) {
    EAST_API_BEGIN
    if (!S_DxK_dev || !C_KxK_dev || D <= 0 || K <= 0) throw Error(EAST_ERR_INVALID, "bad argument");
    use_device(device);
    cudaStream_t s = (cudaStream_t)stream;
    StageTimer tm(s);
    tm.mark("cooc");
    if (get_option("cooc_variant", 0) == 1) cooc_counts(S_DxK_dev, D, K, threshold, C_KxK_dev, s);
    else cooc_counts_tc(S_DxK_dev, D, K, threshold, C_KxK_dev, s, cooc_tc_kernel());
    tm.finish();
    EAST_CUDA(cudaStreamSynchronize(s));
    tm.collect();
    EAST_API_END
}

int east_cooc_host(const double *S_DxK, int64_t D, int32_t K, double threshold, int32_t *C_KxK, int device) {
    EAST_API_BEGIN
    if (!S_DxK || !C_KxK || D <= 0 || K <= 0) throw Error(EAST_ERR_INVALID, "bad argument");
    use_device(device);
    cudaStream_t s = 0;
    DevBuf<double> d_S((size_t)D * K, s);
    DevBuf<int32_t> d_C((size_t)K * K, s);
    EAST_CUDA(cudaMemcpyAsync(d_S.p, S_DxK, sizeof(double) * (size_t)D * K, cudaMemcpyHostToDevice, s));
    if (get_option("cooc_variant", 0) == 1) cooc_counts(d_S.p, D, K, threshold, d_C.p, s);
    else cooc_counts_tc(d_S.p, D, K, threshold, d_C.p, s, cooc_tc_kernel());
    EAST_CUDA(cudaMemcpy(C_KxK, d_C.p, sizeof(int32_t) * (size_t)K * K, cudaMemcpyDeviceToHost));
    EAST_API_END
}

// ---- persistence --------------------------------------------------------------------------
// One file per index (= one device batch of documents): header, then the arrays in a fixed order.  The reference
// rebuilds every AST on every run (relevance.py:38-47); a saved index is loaded at PCIe speed instead.
namespace {
struct IndexFileHeader {
    char magic[8];
    int32_t version, n_docs;
    int64_t n, m_total;
    int32_t sym_bits, term_code, fast_path, doc_sorted, rounds, key_chars, key_bits, tables_fused;
    int32_t has_t8, has_bkt, has_sk, reserved;
    uint8_t code_table[EAST_TERM_BASE];
};
const char INDEX_MAGIC[8] = {'E', 'A', 'S', 'T', 'I', 'D', 'X', '1'};

struct FileCloser { FILE *f; ~FileCloser() { if (f) fclose(f); } };

void write_dev_array(FILE *f, const void *dev, size_t bytes, std::vector<uint8_t> &stage) {
    const uint8_t *src = static_cast<const uint8_t *>(dev);
    for (size_t done = 0; done < bytes;) {
        const size_t part = std::min(stage.size(), bytes - done);
        EAST_CUDA(cudaMemcpy(stage.data(), src + done, part, cudaMemcpyDeviceToHost));
        if (fwrite(stage.data(), 1, part, f) != part) throw Error(EAST_ERR_INVALID, "index file: short write");
        done += part;
    }
}
void read_dev_array(FILE *f, void *dev, size_t bytes, std::vector<uint8_t> &stage) {
    uint8_t *dst = static_cast<uint8_t *>(dev);
    for (size_t done = 0; done < bytes;) {
        const size_t part = std::min(stage.size(), bytes - done);
        if (fread(stage.data(), 1, part, f) != part) throw Error(EAST_ERR_INVALID, "index file: truncated");
        EAST_CUDA(cudaMemcpy(dst + done, stage.data(), part, cudaMemcpyHostToDevice));
        done += part;
    }
}
}  // namespace

int east_index_save(const east_index *idx, const char *path) {
    EAST_API_BEGIN
    if (!idx || !path) throw Error(EAST_ERR_INVALID, "NULL argument");
    EAST_CUDA(cudaSetDevice(idx->device));
    wait_tables(idx);
    ensure_suffix_keys(idx, 0);
    EAST_CUDA(cudaDeviceSynchronize());
    FileCloser fc{fopen(path, "wb")};
    if (!fc.f) throw Error(EAST_ERR_INVALID, std::string("cannot open ") + path + " for writing");
    IndexFileHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, INDEX_MAGIC, 8);
    h.version = 1; h.n_docs = idx->n_docs; h.n = idx->n; h.m_total = idx->m_total;
    h.sym_bits = idx->sym_bits; h.term_code = idx->term_code; h.fast_path = idx->fast_path; h.doc_sorted = idx->doc_sorted;
    h.rounds = idx->rounds; h.key_chars = idx->key_chars; h.key_bits = idx->key_bits; h.tables_fused = idx->tables_fused;
    h.has_t8 = idx->t8 != nullptr; h.has_bkt = idx->bkt != nullptr; h.has_sk = idx->sk != nullptr;
    if (idx->code_table.size() == EAST_TERM_BASE) memcpy(h.code_table, idx->code_table.data(), EAST_TERM_BASE);
    if (fwrite(&h, sizeof(h), 1, fc.f) != 1) throw Error(EAST_ERR_INVALID, "index file: short write");
    if (fwrite(idx->doc_off.data(), sizeof(int32_t), (size_t)idx->n_docs + 1, fc.f) != (size_t)idx->n_docs + 1 ||
        fwrite(idx->doc_m.data(), sizeof(int32_t), (size_t)idx->n_docs, fc.f) != (size_t)idx->n_docs)
        throw Error(EAST_ERR_INVALID, "index file: short write");
    std::vector<uint8_t> stage((size_t)64 << 20);
    const size_t words = sizeof(int32_t) * (size_t)idx->n;
    write_dev_array(fc.f, idx->text, words, stage);
    for (const int32_t *a : {idx->sa, idx->lcp, idx->up, idx->down, idx->next, idx->ann}) write_dev_array(fc.f, a, words, stage);
    if (h.has_t8) write_dev_array(fc.f, idx->t8, (size_t)idx->n + 128, stage);
    if (h.has_bkt) write_dev_array(fc.f, idx->bkt, sizeof(uint32_t) * (((size_t)idx->n_docs << (2 * idx->sym_bits)) + 1), stage);
    if (h.has_sk) write_dev_array(fc.f, idx->sk, words, stage);
    EAST_API_END
}

int east_index_load(const char *path, int device, east_index **out) {
    EAST_API_BEGIN
    if (!path || !out) throw Error(EAST_ERR_INVALID, "NULL argument");
    use_device(device);
    FileCloser fc{fopen(path, "rb")};
    if (!fc.f) throw Error(EAST_ERR_INVALID, std::string("cannot open ") + path);
    IndexFileHeader h;
    if (fread(&h, sizeof(h), 1, fc.f) != 1 || memcmp(h.magic, INDEX_MAGIC, 8) != 0 || h.version != 1)
        throw Error(EAST_ERR_INVALID, "not an east_b200 index file (or another version)");
    if (h.n_docs <= 0 || h.n <= 0 || h.n >= (1ll << 30) || h.sym_bits < 0 || h.sym_bits > 7) throw Error(EAST_ERR_INVALID, "index file: bad header");
    std::unique_ptr<east_index, void (*)(east_index *)> idx(new east_index(), free_index);
    idx->device = device; idx->n_docs = h.n_docs; idx->n = (int32_t)h.n; idx->m_total = h.m_total;
    idx->sym_bits = h.sym_bits; idx->term_code = h.term_code; idx->fast_path = h.fast_path; idx->doc_sorted = h.doc_sorted;
    idx->rounds = h.rounds; idx->key_chars = h.key_chars; idx->key_bits = h.key_bits; idx->tables_fused = h.tables_fused;
    idx->code_table.assign(h.code_table, h.code_table + EAST_TERM_BASE);
    idx->doc_off.resize((size_t)h.n_docs + 1);
    idx->doc_m.resize((size_t)h.n_docs);
    if (fread(idx->doc_off.data(), sizeof(int32_t), idx->doc_off.size(), fc.f) != idx->doc_off.size() ||
        fread(idx->doc_m.data(), sizeof(int32_t), idx->doc_m.size(), fc.f) != idx->doc_m.size())
        throw Error(EAST_ERR_INVALID, "index file: truncated");
    if (idx->doc_off.front() != 0 || idx->doc_off.back() != idx->n) throw Error(EAST_ERR_INVALID, "index file: bad document offsets");
    const size_t words = sizeof(int32_t) * (size_t)idx->n;
    const size_t bkt_entries = ((size_t)h.n_docs << (2 * h.sym_bits)) + 1;
    size_t need = Arena::padded(sizeof(int32_t) * ((size_t)h.n_docs + 1)) + Arena::padded(sizeof(int32_t) * (size_t)h.n_docs) +
                  (7 + (h.has_sk ? 1 : 0)) * Arena::padded(words) + (h.has_t8 ? Arena::padded((size_t)idx->n + 128) : 0) +
                  (h.has_bkt ? Arena::padded(sizeof(uint32_t) * bkt_entries) : 0);
    cudaStream_t s = 0;
    idx->arena.base = (uint8_t *)dev_alloc(need, s, true);
    idx->arena.cap = need;
    auto take32 = [&](size_t count) { DevBuf<int32_t> b = idx->arena.take<int32_t>(count, s); int32_t *p = b.p; b.p = nullptr; return p; };
    idx->d_doc_off = take32((size_t)h.n_docs + 1);
    idx->d_doc_m = take32((size_t)h.n_docs);
    idx->text = (uint32_t *)take32((size_t)idx->n);   // inside the arena: owns_text stays false
    idx->sa = take32((size_t)idx->n); idx->lcp = take32((size_t)idx->n); idx->up = take32((size_t)idx->n);
    idx->down = take32((size_t)idx->n); idx->next = take32((size_t)idx->n); idx->ann = take32((size_t)idx->n);
    EAST_CUDA(cudaMemcpy(idx->d_doc_off, idx->doc_off.data(), sizeof(int32_t) * idx->doc_off.size(), cudaMemcpyHostToDevice));
    EAST_CUDA(cudaMemcpy(idx->d_doc_m, idx->doc_m.data(), sizeof(int32_t) * idx->doc_m.size(), cudaMemcpyHostToDevice));
    std::vector<uint8_t> stage((size_t)64 << 20);
    read_dev_array(fc.f, idx->text, words, stage);
    for (int32_t *a : {idx->sa, idx->lcp, idx->up, idx->down, idx->next, idx->ann}) read_dev_array(fc.f, a, words, stage);
    if (h.has_t8) {
        DevBuf<uint8_t> b = idx->arena.take<uint8_t>((size_t)idx->n + 128, s);
        idx->t8 = b.p; b.p = nullptr;
        read_dev_array(fc.f, idx->t8, (size_t)idx->n + 128, stage);
    }
    if (h.has_bkt) {
        idx->bkt = (uint32_t *)take32(bkt_entries);
        read_dev_array(fc.f, idx->bkt, sizeof(uint32_t) * bkt_entries, stage);
    }
    if (h.has_sk) {
        idx->sk = (uint32_t *)take32((size_t)idx->n);
        read_dev_array(fc.f, idx->sk, words, stage);
    }
    *out = idx.release();
    EAST_API_END
}

int east_trim(int device) {
    EAST_API_BEGIN
    use_device(device);
    EAST_CUDA(cudaDeviceSynchronize());
    g_kp_cache.reset();
    alphabet_guess_forget();
    big_cache_drop(device);
    EAST_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> g(g_pool_mutex);
    auto it = g_pools.find(device);
    if (it != g_pools.end())
        for (cudaMemPool_t pool : it->second) EAST_CUDA(cudaMemPoolTrimTo(pool, 0));
    EAST_API_END
}

}  // extern "C"
