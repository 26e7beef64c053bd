// sa_build.cu -- generalized suffix array of a batch of packed documents by prefix doubling.
//
// Replaces east/asts/easa.py:141-245 (_compute_suftab: DC3 in the reference).  The suffix
// array under code point order is unique, so a different construction gives the same array.
//
// One global problem for the whole batch: the document id is the most significant part of
// every sort key, so the result is doc-major and rank r of the batch is rank r - doc_off[d]
// of document d.
//
// Round 0  sorts all suffixes by a packed window of `kc` symbols (b bits each) under the
//          document id.  On the fast path (every code point >= 0x0A00 is one of the unique,
//          position-ordered terminators 0x0A00+i, east/asts/utils.py:25-40) symbols are dense
//          8-bit codes, all terminators share the top code and the window is cut after the
//          first terminator: two suffixes with equal windows that contain a terminator differ
//          only in WHICH terminator, i.e. in string index == text position, and the stable LSD
//          sort has already left them in position order.  They are final after round 0.
//          On the general path (text code points collide or interleave with the terminator
//          range, a reference quirk) symbols are raw code points and nothing is special-cased.
// Round r  (h = kc, 2kc, ...) re-sorts only the suffixes that still share their rank with
//          another one, by (own rank, rank[i+h]), and re-ranks; the active set shrinks fast.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include "radix_sort.cuh"
#include "sa_build.h"

namespace east {

// ------------------------------------------------------------------------------------------
// radix sort host driver
// ------------------------------------------------------------------------------------------
template <int THREADS, int ITEMS, int MINB>
static void launch_onesweep(const uint64_t *kin, uint64_t *kout, const uint32_t *vin, uint32_t *vout, int32_t n,
                            int shift, const uint32_t *hist_excl, uint32_t *status, uint32_t *ticket,
                            cudaStream_t s) {
    using Cfg = RsCfg<THREADS, ITEMS>;
    auto kern = k_rs_onesweep<THREADS, ITEMS, MINB>;
    ensure_dynamic_smem((const void *)kern, Cfg::SMEM);
    const int tiles = rs_num_tiles(n, Cfg::TILE);
    EAST_BYTES(24.0 * n);  // read + write of an 8-byte key and a 4-byte value per element
    if (g_time_kernels) ktime_begin("k_rs_onesweep", s);
    kern<<<tiles, THREADS, Cfg::SMEM, s>>>(kin, kout, vin, vout, n, shift, hist_excl, status, ticket,
                                           (const RsTileDesc *)nullptr, 0);
    if (g_time_kernels) ktime_end(s);
    ++g_launches;
    g_next_bytes = 0.0;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) throw Error(-2, std::string("k_rs_onesweep launch: ") + cudaGetErrorString(e));
}

int radix_sort_pairs(uint64_t *ka, uint64_t *kb, uint32_t *va, uint32_t *vb, int32_t n, int nbits,
                     uint32_t *hist, bool hist_ready, void *scratch, cudaStream_t s, int variant) {
    if (n <= 0) return 0;
    int passes = rs_num_passes(nbits);
    if (passes < 1) passes = 1;
    if (passes > RS_MAX_PASSES) throw Error(-1, "radix_sort_pairs: too many key bits");
    const int tiles = rs_num_tiles(n);  // scratch stride: the smallest tile of any variant
    if (!hist_ready) {
        EAST_CUDA(cudaMemsetAsync(hist, 0, sizeof(uint32_t) * 256 * passes, s));
        EAST_LAUNCH(k_rs_hist, grid_for(n, 256 * 8, 4), 256, 0, s, ka, n, passes, hist);
    }
    EAST_LAUNCH(k_rs_scan_hist, passes, 256, 0, s, hist);
    EAST_CUDA(cudaMemsetAsync(scratch, 0, rs_scratch_bytes(n, passes), s));
    uint32_t *status = (uint32_t *)scratch;
    uint32_t *tickets = status + (size_t)tiles * 256 * passes;
    int cur = 0;
    for (int p = 0; p < passes; ++p) {
        const uint64_t *kin = cur ? kb : ka;
        uint64_t *kout = cur ? ka : kb;
        const uint32_t *vin = cur ? vb : va;
        uint32_t *vout = cur ? va : vb;
        uint32_t *st = status + (size_t)tiles * 256 * p;
#define RS_CASE(id, T, I, B) case id: launch_onesweep<T, I, B>(kin, kout, vin, vout, n, 8 * p, hist + 256 * p, st, tickets + p, s); break;
        switch (variant) {
            RS_CASE(1, 256, 16, 2)
            RS_CASE(2, 256, 12, 4)
            RS_CASE(3, 256, 8, 5)
            RS_CASE(4, 384, 12, 2)
            RS_CASE(5, 512, 8, 2)
            RS_CASE(6, 512, 12, 1)
            RS_CASE(7, 384, 16, 2)
            RS_CASE(8, 256, 20, 2)
            RS_CASE(9, 512, 16, 1)
            default: launch_onesweep<256, 16, 3>(kin, kout, vin, vout, n, 8 * p, hist + 256 * p, st, tickets + p, s); break;
        }
#undef RS_CASE
        cur ^= 1;
    }
    return cur;
}

int radix_sort_pairs_segmented(uint64_t *ka, uint64_t *kb, uint32_t *va, uint32_t *vb, int nbits,
                               const RsTileDesc *descs, int num_tiles, int64_t n_total, uint32_t *hist, int n_seg,
                               void *scratch, cudaStream_t s) {
    if (num_tiles <= 0) return 0;
    int passes = rs_num_passes(nbits);
    if (passes < 1) passes = 1;
    if (passes > RS_MAX_PASSES) throw Error(-1, "radix_sort_pairs_segmented: too many key bits");
    using Cfg = RsCfg<256, 16>;
    static_assert(Cfg::TILE == RS_SEG_TILE, "tile descriptors are built for the 256 x 16 kernel");
    auto kern = k_rs_onesweep<256, 16, 3>;
    ensure_dynamic_smem((const void *)kern, Cfg::SMEM);
    // exclusive scan of every (segment, pass) row of 256 bins
    EAST_LAUNCH(k_rs_scan_hist, n_seg * passes, 256, 0, s, hist);
    const size_t status_words = (size_t)num_tiles * 256;
    EAST_CUDA(cudaMemsetAsync(scratch, 0, (status_words * passes + 64) * sizeof(uint32_t), s));
    uint32_t *status = (uint32_t *)scratch;
    uint32_t *tickets = status + status_words * passes;
    int cur = 0;
    for (int p = 0; p < passes; ++p) {
        const uint64_t *kin = cur ? kb : ka;
        uint64_t *kout = cur ? ka : kb;
        const uint32_t *vin = cur ? vb : va;
        uint32_t *vout = cur ? va : vb;
        EAST_BYTES(24.0 * (double)n_total);  // read + write of an 8-byte key and a 4-byte value per element
        if (g_time_kernels) ktime_begin("k_rs_onesweep", s);
        kern<<<num_tiles, 256, Cfg::SMEM, s>>>(kin, kout, vin, vout, 0, 8 * p, hist + 256 * p, status + status_words * p,
                                               tickets + p, descs, passes * 256);
        if (g_time_kernels) ktime_end(s);
        ++g_launches;
        g_next_bytes = 0.0;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) throw Error(-2, std::string("k_rs_onesweep (segmented) launch: ") + cudaGetErrorString(e));
        cur ^= 1;
    }
    return cur;
}

// ------------------------------------------------------------------------------------------
// text scan: alphabet, maximum code point, validation of the terminator layout
// ------------------------------------------------------------------------------------------
struct ScanResult {
    uint32_t present[EAST_TERM_BASE / 32];  // bitmap of code points < 0x0A00
    uint32_t max_code;
    uint32_t n_term;   // positions with code >= 0x0A00
    uint32_t bad;      // terminator layout violated
};

constexpr int ST_TILE = 4096;
constexpr int ST_HALO = 256;
constexpr int ST_NONE = -2;   // scan state: nothing seen
constexpr int ST_RESET = -1;  // scan state: a document started, no terminator since

// One streaming pass over the packed text, staged through shared memory: alphabet bitmap of the
// code points below 0x0A00, maximum code point, and validation that the code points >= 0x0A00
// are exactly the terminators 0x0A00+i of string i of each document, in order.
// "The previous terminator of my document" is a prefix scan with the operator "take the right
// operand unless it is empty" over (document start -> RESET, terminator -> its value): each warp
// scans its 512 consecutive code points 32 at a time with shuffles, warps are chained through
// shared-memory summaries, and the state before the tile comes from the 256-code-point halo
// (one ballot per 32 code points; global memory only for strings longer than the halo).
__global__ void __launch_bounds__(256)
k_scan_text(const uint32_t *__restrict__ T, int32_t n, const int32_t *__restrict__ doc_off,
            const int32_t *__restrict__ doc_m, int D, ScanResult *res, int tile_begin, int tile_end, int check_doc_ends) {
    __shared__ uint32_t s_present[EAST_TERM_BASE / 32];
    __shared__ uint32_t s_max, s_nterm, s_bad;
    __shared__ __align__(16) uint32_t s_t[ST_HALO + ST_TILE];
    __shared__ uint32_t s_ds[ST_TILE / 32];  // document-start flags of the tile
    __shared__ int s_sum[8];
    __shared__ int s_carry;
    __shared__ int s_dlo, s_dhi;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    for (int i = t; i < EAST_TERM_BASE / 32; i += 256) s_present[i] = 0;
    if (t == 0) { s_max = 0; s_nterm = 0; s_bad = 0; }
    uint32_t mx = 0, nt = 0, bad = 0;
    // tiles [tile_begin, tile_end) of the text (a pipelined build scans what has arrived so far; a tile only
    // looks backwards, at its halo)
    for (int tile = tile_begin + blockIdx.x; tile < tile_end; tile += gridDim.x) {
        const int64_t base = (int64_t)tile * ST_TILE;
        const int64_t win = base - ST_HALO;  // global position of s_t[0]
        const int tile_n = (int)min((int64_t)ST_TILE, (int64_t)n - base);
        __syncthreads();
        for (int o = t * 4; o < ST_HALO + ST_TILE; o += 256 * 4) {
            const int64_t g = win + o;
            if (g >= 0 && g + 4 <= n) {
                *reinterpret_cast<uint4 *>(s_t + o) = *reinterpret_cast<const uint4 *>(T + g);  // 128-bit
            } else {
                for (int q = 0; q < 4; ++q) s_t[o + q] = (g + q >= 0 && g + q < n) ? T[g + q] : 0u;
            }
        }
        if (t < ST_TILE / 32) s_ds[t] = 0;
        if (t == 0) s_dlo = doc_of(doc_off, D, (int32_t)base);
        if (t == 32) s_dhi = doc_of(doc_off, D, (int32_t)(base + tile_n - 1));
        __syncthreads();
        const int dlo = s_dlo, dhi = s_dhi;
        for (int d = dlo + t; d <= dhi; d += 256) {
            const int64_t off = (int64_t)__ldg(doc_off + d) - base;
            if (off >= 0) atomicOr(&s_ds[off >> 5], 1u << (off & 31));
        }
        // ---- state before the tile (warp 0): last terminator of the halo that belongs to document dlo
        if (w == 0) {
            const int64_t dstart = __ldg(doc_off + dlo);
            int carry = ST_NONE;
            if (dstart >= base) carry = ST_RESET;  // the tile starts a document
            else {
                const int64_t lower = max(dstart, max(win, (int64_t)0));
                for (int64_t hi = base - 1; hi >= lower && carry == ST_NONE; hi -= 32) {
                    const int64_t p = hi - (31 - lane);  // lanes cover [hi-31, hi]
                    const bool is_t = p >= lower && s_t[p - win] >= EAST_TERM_BASE;
                    const unsigned m = __ballot_sync(0xffffffffu, is_t);
                    if (m) {
                        const int hl = 31 - __clz(m);
                        carry = (int)__shfl_sync(0xffffffffu, is_t ? s_t[p - win] : 0u, hl);
                    }
                }
                if (carry == ST_NONE) {
                    if (lower == dstart) carry = ST_RESET;
                    else {  // a string longer than the halo: walk global memory (lane 0)
                        int64_t j = lower - 1;
                        if (lane == 0) {
                            while (j >= dstart && T[j] < EAST_TERM_BASE) --j;
                            carry = (j >= dstart) ? (int)T[j] : ST_RESET;
                        }
                        carry = __shfl_sync(0xffffffffu, carry, 0);
                    }
                }
            }
            if (lane == 0) s_carry = carry;
        }
        __syncthreads();
        // ---- phase 1: what each warp's 512 code points leave behind
        {
            int summary = ST_NONE;
            for (int r = 15; r >= 0 && summary == ST_NONE; --r) {
                const int o = w * 512 + r * 32 + lane;
                const uint32_t c = s_t[ST_HALO + o];
                const bool is_t = o < tile_n && c >= EAST_TERM_BASE;
                const bool is_d = o < tile_n && ((s_ds[o >> 5] >> (o & 31)) & 1u);
                const unsigned m = __ballot_sync(0xffffffffu, is_t || is_d);
                if (m) {
                    const int hl = 31 - __clz(m);
                    summary = __shfl_sync(0xffffffffu, is_t ? (int)c : ST_RESET, hl);
                }
            }
            if (lane == 0) s_sum[w] = summary;
        }
        __syncthreads();
        int state = s_carry;  // state before this warp's first code point
        for (int i = 0; i < w; ++i) if (s_sum[i] != ST_NONE) state = s_sum[i];
        // ---- phase 2: scan the rows, check every terminator against the state in front of it
#pragma unroll 4
        for (int r = 0; r < 16; ++r) {
            const int o = w * 512 + r * 32 + lane;
            const int64_t i = base + o;
            const bool in = o < tile_n;
            const uint32_t c = s_t[ST_HALO + o];
            const bool is_t = in && c >= EAST_TERM_BASE;
            const bool is_d = in && ((s_ds[o >> 5] >> (o & 31)) & 1u);
            int x = is_t ? (int)c : (is_d ? ST_RESET : ST_NONE);  // what this code point leaves behind
#pragma unroll
            for (int sh = 1; sh < 32; sh <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, x, sh);
                if (lane >= sh && x == ST_NONE) x = y;
            }
            int before = __shfl_up_sync(0xffffffffu, x, 1);   // inclusive state of the lane to the left
            if (lane == 0 || before == ST_NONE) before = (lane == 0) ? state : before;
            // lanes whose left neighbours saw nothing inherit the row's incoming state
            if (before == ST_NONE) before = state;
            if (is_d) before = ST_RESET;
            if (in) {
                mx = max(mx, c);
                if (!is_t) {
                    if (c < EAST_TERM_BASE && !(((volatile uint32_t *)s_present)[c >> 5] & (1u << (c & 31))))
                        atomicOr(&s_present[c >> 5], 1u << (c & 31));
                } else {
                    ++nt;
                    const uint32_t expect = (before >= 0) ? (uint32_t)before + 1u : EAST_TERM_BASE;
                    if (c != expect) bad = 1;
                    // the last code point of a document must be its last terminator
                    const bool doc_end = (i + 1 == n) || (o + 1 < tile_n ? ((s_ds[(o + 1) >> 5] >> ((o + 1) & 31)) & 1u) : false);
                    if (doc_end || o + 1 == tile_n) {
                        int lo = dlo, hi = dhi;
                        while (lo < hi) {
                            int mid = (lo + hi + 1) >> 1;
                            if (__ldg(doc_off + mid) <= i) lo = mid; else hi = mid - 1;
                        }
                        if (i == __ldg(doc_off + lo + 1) - 1 && c != EAST_TERM_BASE + (uint32_t)__ldg(doc_m + lo) - 1u) bad = 1;
                    }
                }
            }
            const int last = __shfl_sync(0xffffffffu, x, 31);
            if (last != ST_NONE) state = last;
        }
    }
    // every document must end with a terminator
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; check_doc_ends && d < D; d += stride) {
        int32_t e = doc_off[d + 1];
        if (e <= doc_off[d] || T[e - 1] < EAST_TERM_BASE) bad = 1;
    }
    __syncthreads();
    atomicMax(&s_max, mx);
    atomicAdd(&s_nterm, nt);
    if (bad) atomicOr(&s_bad, 1u);
    __syncthreads();
    for (int i = t; i < EAST_TERM_BASE / 32; i += 256)
        if (s_present[i]) atomicOr(&res->present[i], s_present[i]);
    if (t == 0) {
        atomicMax(&res->max_code, s_max);
        atomicAdd(&res->n_term, s_nterm);
        if (s_bad) atomicOr(&res->bad, 1u);
    }
}

// Four code points T[i .. i+3] (i a multiple of 4) as one 128-bit load when they all lie in [lo, hi),
// else element by element with `fill` outside the range
__device__ __forceinline__ uint4 load4_guarded(const uint32_t *__restrict__ T, int64_t i, int64_t lo, int64_t hi, uint32_t fill) {
    if (i >= lo && i + 3 < hi) return *reinterpret_cast<const uint4 *>(T + i);
    uint4 v;
    v.x = (i >= lo && i < hi) ? T[i] : fill;
    v.y = (i + 1 >= lo && i + 1 < hi) ? T[i + 1] : fill;
    v.z = (i + 2 >= lo && i + 2 < hi) ? T[i + 2] : fill;
    v.w = (i + 3 >= lo && i + 3 < hi) ? T[i + 3] : fill;
    return v;
}

// dense byte codes: 1..sigma for present code points < 0x0A00, sigma+1 for every terminator.
// Encodes [begin, end) (begin a multiple of 4 or a document start handled by the scalar edges);
// *miss is set when a code point below 0x0A00 has no code (speculative alphabet, see below).
__global__ void __launch_bounds__(256)
k_encode_text(const uint32_t *__restrict__ T, int32_t begin, int32_t end, const uint8_t *__restrict__ code_table,
              uint8_t term_code, uint8_t *__restrict__ T8, uint32_t *miss) {
    __shared__ uint8_t s_code[EAST_TERM_BASE];
    for (int i = threadIdx.x; i < (int)EAST_TERM_BASE; i += blockDim.x) s_code[i] = code_table[i];
    __syncthreads();
    const int32_t a0 = begin & ~3;   // groups of 4 aligned code points; the edges are masked
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    bool missed = false;
    constexpr int U = 4;   // independent 128-bit loads in flight per thread (one alone left HBM at ~40 %)
    for (int64_t i0 = a0 + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < end; i0 += U * stride) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = load4_guarded(T, i0 + u * stride, begin, end, EAST_TERM_BASE);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i >= end) break;
            const uint32_t c[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
            uint32_t packed = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t e = (c[q] < EAST_TERM_BASE) ? s_code[c[q]] : term_code;
                missed = missed || e == 0u;
                packed |= e << (8 * q);
            }
            if (i >= begin && i + 3 < end) *reinterpret_cast<uint32_t *>(T8 + i) = packed;
            else for (int q = 0; q < 4; ++q) if (i + q >= begin && i + q < end) T8[i + q] = (uint8_t)(packed >> (8 * q));
        }
    }
    if (missed && miss) atomicOr(miss, 1u);
}

// The dense-code table (code point < 0x0A00 -> 1..sigma in code point order, 0 = absent) from the scan's
// presence bitmap, on the device: the host derives the same table for itself, and a host-to-device upload here
// would queue behind the bulk text copies of a pipelined build (one copy engine per direction).
__device__ __forceinline__ void code_table_from_bits(uint32_t *s_bits, uint32_t *s_before, uint8_t *__restrict__ table) {
    constexpr int W = EAST_TERM_BASE / 32;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int w = 0; w < W; ++w) { s_before[w] = run; run += __popc(s_bits[w]); }
    }
    __syncthreads();
    for (int w = threadIdx.x; w < W; w += blockDim.x) {
        const uint32_t bits = s_bits[w];
        uint32_t code = s_before[w];
        for (int k = 0; k < 32; ++k) {
            const bool on = (bits >> k) & 1u;
            if (on) ++code;
            table[32 * w + k] = on ? (uint8_t)(code & 0xffu) : (uint8_t)0;
        }
    }
}

__global__ void __launch_bounds__(128)
k_code_table(const ScanResult *__restrict__ res, uint8_t *__restrict__ table, uint4 extra) {
    // extra: code points below 128 that get a code although the scan did not meet them (pipelined build)
    constexpr int W = EAST_TERM_BASE / 32;
    __shared__ uint32_t s_bits[W];
    __shared__ uint32_t s_before[W];
    const uint32_t ex[4] = {extra.x, extra.y, extra.z, extra.w};
    for (int w = threadIdx.x; w < W; w += blockDim.x) s_bits[w] = res->present[w] | (w < 4 ? ex[w] : 0u);
    code_table_from_bits(s_bits, s_before, table);
}

__global__ void k_store_u32(uint32_t *dst, uint32_t value) { *dst = value; }

// Everything a batch of per-document kernels needs before its first wave, in ONE launch: the code table (from the scan
// result, or from a bitmap handed over by value when the alphabet is a guess), the cleared flag words, the closing entries of
// the bucket tables.  Every launch of a dependent chain costs its latency; with the text of a pipelined build on the host
// link that is 30-50 us apiece (the command fetch shares the link with the copies), and the chain used to be five long.
struct PresentBits { uint32_t w[EAST_TERM_BASE / 32]; };

__global__ void __launch_bounds__(128)
k_doc_sort_prologue(const ScanResult *__restrict__ res /* or NULL: bits */, PresentBits bits, uint4 extra, uint8_t *__restrict__ table,
                    uint32_t *flags2, uint32_t *end0, uint32_t *end1, uint32_t n) {
    constexpr int W = EAST_TERM_BASE / 32;
    __shared__ uint32_t s_bits[W];
    __shared__ uint32_t s_before[W];
    const uint32_t ex[4] = {extra.x, extra.y, extra.z, extra.w};
    for (int w = threadIdx.x; w < W; w += blockDim.x) s_bits[w] = (res ? res->present[w] : bits.w[w]) | (w < 4 ? ex[w] : 0u);
    code_table_from_bits(s_bits, s_before, table);
    if (threadIdx.x == 0) {
        if (flags2) { flags2[0] = 0u; flags2[1] = 0u; }
        if (end0) *end0 = n;
        if (end1) *end1 = n;
    }
}

// Light text scan: bitmap of the code points below 0x0A00 that occur in T[0, n), number of code points
// >= 0x0A00 and the maximum code point -- everything k_scan_text reports except the validation of the
// terminator layout, which the per-document kernel does itself.  Streams at HBM speed.
__global__ void __launch_bounds__(256)
k_alphabet(const uint32_t *__restrict__ T, int32_t n, ScanResult *res) {
    __shared__ uint32_t s_present[EAST_TERM_BASE / 32];
    for (int i = threadIdx.x; i < (int)(EAST_TERM_BASE / 32); i += blockDim.x) s_present[i] = 0;
    __syncthreads();
    uint32_t mx = 0, nt = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    constexpr int U = 4;   // independent 128-bit loads in flight per thread
    for (int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < n; i0 += U * stride) {
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = load4_guarded(T, i0 + u * stride, 0, n, 0u);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t i = i0 + u * stride;
            if (i >= n) break;
            const uint32_t c[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                mx = max(mx, c[q]);
                if (c[q] >= EAST_TERM_BASE) ++nt;
                else if (i + q < n && !(((volatile uint32_t *)s_present)[c[q] >> 5] & (1u << (c[q] & 31))))
                    atomicOr(&s_present[c[q] >> 5], 1u << (c[q] & 31));
            }
        }
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    nt = __reduce_add_sync(0xffffffffu, nt);
    if ((threadIdx.x & 31) == 0) { atomicMax(&res->max_code, mx); if (nt) atomicAdd(&res->n_term, nt); }
    __syncthreads();
    for (int i = threadIdx.x; i < (int)(EAST_TERM_BASE / 32); i += blockDim.x)
        if (s_present[i]) atomicOr(&res->present[i], s_present[i]);
}

// The same for a text that arrives as one byte per code point (east_*_host_u8): bytes below 0xFF are code points,
// 0xFF ends a string.
__global__ void __launch_bounds__(256)
k_alphabet8(const uint8_t *__restrict__ T8, int32_t n, ScanResult *res) {
    __shared__ uint32_t s_present[8];
    if (threadIdx.x < 8) s_present[threadIdx.x] = 0;
    __syncthreads();
    // a code point costs one look at the CTA's bitmap in shared memory; the atomic only follows for the first few
    // occurrences of a symbol (a per-thread bitmap in registers cost ~25 instructions per byte)
    volatile uint32_t *seen = s_present;
    uint32_t nt = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 16;
    for (int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; i0 < n; i0 += stride) {
        uint4 v = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
        if (i0 + 15 < n) v = *reinterpret_cast<const uint4 *>(T8 + i0);   // the buffer starts 256-byte aligned
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            uint32_t c = (w[j >> 2] >> (8 * (j & 3))) & 0xffu;
            if (i0 + 15 >= n) { if (i0 + j >= n) continue; c = T8[i0 + j]; }
            if (c == 0xffu) ++nt;
            else {
                const uint32_t bit = 1u << (c & 31);
                if (!(seen[c >> 5] & bit)) atomicOr(&s_present[c >> 5], bit);
            }
        }
    }
    nt = __reduce_add_sync(0xffffffffu, nt);
    if ((threadIdx.x & 31) == 0 && nt) atomicAdd(&res->n_term, nt);
    __syncthreads();
    if (threadIdx.x < 8 && s_present[threadIdx.x]) atomicOr(&res->present[threadIdx.x], s_present[threadIdx.x]);
    if (threadIdx.x == 0) atomicMax(&res->max_code, 0xfeu);
}

// one byte per code point -> code points: CTA d expands document d, the k-th 0xFF of the document becomes the terminator
// 0x0A00 + k (east/asts/utils.py:35-39).  *bad is set when a document does not hold exactly doc_m terminators or does not
// end with one.  (Batches that do not take the pipelined per-document path.)
__global__ void __launch_bounds__(256)
k_expand_text8(const uint8_t *__restrict__ T8, const int32_t *__restrict__ doc_off, const int32_t *__restrict__ doc_m,
               uint32_t *__restrict__ T, uint32_t *bad) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_run;
    const int d = blockIdx.x;
    const int32_t b = doc_off[d], e = doc_off[d + 1];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) s_run = 0;
    __syncthreads();
    for (int32_t i0 = b; i0 < e; i0 += 256 * 8) {
        // thread t owns 8 consecutive bytes of the tile
        const int32_t p0 = i0 + t * 8;
        uint32_t c[8], cnt = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { c[j] = (p0 + j < e) ? T8[p0 + j] : 0u; cnt += (p0 + j < e && c[j] == 0xffu) ? 1u : 0u; }
        uint32_t x = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) s_warp[w] = x;
        __syncthreads();
        uint32_t k = s_run + x - cnt;
        for (int i = 0; i < w; ++i) k += s_warp[i];
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (p0 + j < e) T[p0 + j] = (c[j] == 0xffu) ? EAST_TERM_BASE + k++ : c[j];
        __syncthreads();
        if (t == 255) s_run = k;
        __syncthreads();
    }
    if (t == 0 && (s_run != (uint32_t)doc_m[d] || T8[e - 1] != 0xffu)) atomicOr(bad, 1u);
}

void expand_text8(const uint8_t *text8, const int32_t *doc_off, const int32_t *doc_m, int n_docs, uint32_t *text, uint32_t *bad,
                  cudaStream_t s) {
    EAST_LAUNCH(k_expand_text8, n_docs, 256, 0, s, text8, doc_off, doc_m, text, bad);
}

// ------------------------------------------------------------------------------------------
// round 0 key generation (+ fused digit histograms of all passes)
// ------------------------------------------------------------------------------------------
constexpr int KG_THREADS = 256;
constexpr int KG_ITEMS = 8;
constexpr int KG_TILE = KG_THREADS * KG_ITEMS;
constexpr int KG_HALO = 32;

struct KeyParams {
    int kc;          // symbols per window
    int b;           // bits per symbol
    int passes;      // radix passes over the key
    uint32_t term;   // fast path: terminator class code; general: 0xffffffff
};

// 8 consecutive byte codes (first symbol in the lowest byte) -> one field of 8*b bits with the
// first symbol most significant: three SWAR merge steps instead of eight shift-or steps.
__device__ __forceinline__ uint64_t pack8(uint64_t x, int b) {
    x = ((x & 0x00ff00ff00ff00ffull) << b) | ((x >> 8) & 0x00ff00ff00ff00ffull);
    x = ((x & 0x0000ffff0000ffffull) << (2 * b)) | ((x >> 16) & 0x0000ffff0000ffffull);
    return ((x & 0x00000000ffffffffull) << (4 * b)) | (x >> 32);
}

// 8 bytes of shared memory starting at an arbitrary byte offset (two aligned 64-bit loads)
__device__ __forceinline__ uint64_t lds8(const uint8_t *base, int o) {
    const uint64_t *q = reinterpret_cast<const uint64_t *>(base + (o & ~7));
    const int sh = (o & 7) * 8;
    const uint64_t lo = q[0];
    if (sh == 0) return lo;
    return (lo >> sh) | (q[1] << (64 - sh));
}

// fast path: byte codes.  The window of kc symbols is packed 8 symbols at a time; everything
// after the first terminator of the window is cleared (SWAR zero-byte search for its position).
__global__ void __launch_bounds__(KG_THREADS)
k_keygen0_fast(const uint8_t *__restrict__ T8, int32_t n, int32_t begin, int32_t end,
               const int32_t *__restrict__ doc_off, int D,
               KeyParams kp, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
               uint32_t *g_hist) {
    __shared__ uint32_t s_hist[RS_MAX_PASSES * 256];
    __shared__ __align__(16) uint8_t s_t[KG_TILE + KG_HALO + 16];
    __shared__ int s_dlo, s_dhi;
    for (int i = threadIdx.x; i < kp.passes * 256; i += blockDim.x) s_hist[i] = 0;
    // tiles of the global tile grid that overlap [begin, end) (tile bases stay 16-byte aligned)
    const int tile_lo = begin / KG_TILE, tile_hi = (end + KG_TILE - 1) / KG_TILE;
    const int b = kp.b, kc = kp.kc;
    const int groups = (kc + 7) >> 3, rem = kc - 8 * (groups - 1);  // symbols taken from the last group
    const uint64_t term8 = 0x0101010101010101ull * (uint64_t)kp.term;
    for (int tile = tile_lo + blockIdx.x; tile < tile_hi; tile += gridDim.x) {
        const int32_t base = tile * KG_TILE;
        __syncthreads();
        // stage the tile (+halo) of byte codes; 128-bit loads where fully in range
        for (int o = threadIdx.x * 16; o < KG_TILE + KG_HALO + 16; o += blockDim.x * 16) {
            int64_t g = (int64_t)base + o;
            if (g + 16 <= n) {
                *reinterpret_cast<uint4 *>(s_t + o) = *reinterpret_cast<const uint4 *>(T8 + g);
            } else {
                for (int q = 0; q < 16; ++q) s_t[o + q] = (g + q < n) ? T8[g + q] : 0;
            }
        }
        if (threadIdx.x == 0) s_dlo = doc_of(doc_off, D, max(base, begin));
        if (threadIdx.x == 32) s_dhi = doc_of(doc_off, D, min(base + KG_TILE, end) - 1);
        __syncthreads();
        const int dlo = s_dlo, dhi = s_dhi;
#pragma unroll 2
        for (int it = 0; it < KG_ITEMS; ++it) {
            const int o = it * KG_THREADS + threadIdx.x;
            const int32_t i = base + o;
            const bool valid = i >= begin && i < end;
            uint64_t key = 0;
            if (valid) {
                int lo = dlo, hi = dhi;  // document of position i (tile spans [dlo, dhi])
                while (lo < hi) {
                    int mid = (lo + hi + 1) >> 1;
                    if (__ldg(doc_off + mid) <= i) lo = mid; else hi = mid - 1;
                }
                int tpos = kc;  // window offset of the first terminator (kc = none)
                for (int gq = 0; gq < groups; ++gq) {
                    const uint64_t x = lds8(s_t, o + 8 * gq);
                    if (tpos == kc) {
                        const uint64_t t = x ^ term8;
                        const uint64_t z = (t - 0x0101010101010101ull) & ~t & 0x8080808080808080ull;
                        if (z) tpos = min(kc, 8 * gq + ((__ffsll((long long)z) - 1) >> 3));
                    }
                    const uint64_t f = pack8(x, b);
                    if (gq + 1 < groups) key = (key << (8 * b)) | f;
                    else key = (key << (rem * b)) | (f >> ((8 - rem) * b));
                }
                if (tpos < kc - 1) key &= ~((1ull << (b * (kc - 1 - tpos))) - 1ull);
                if (kc * b < 64) key |= (uint64_t)lo << (kc * b);
                keys[i] = key;
                vals[i] = (uint32_t)i;
            }
            rs_hist_add(s_hist, key, kp.passes, valid, (kc * b) >> 3);
        }
    }
    __syncthreads();
    rs_hist_flush(s_hist, g_hist, kp.passes);
}

// Segmented variant of the fast-path key generator: works on the sort's tile descriptors (a tile
// never crosses a document, so the document id is a per-tile constant) and accumulates the digit
// histograms PER DOCUMENT (hist[seg][pass][256]).  A block owns a contiguous run of tiles and
// flushes its shared-memory histogram only when the document changes.
__global__ void __launch_bounds__(KG_THREADS)
k_keygen0_fast_seg(const uint8_t *__restrict__ T8, int32_t n, const RsTileDesc *__restrict__ descs, int num_tiles,
                   int tiles_per_block, KeyParams kp, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                   uint32_t *g_hist) {
    __shared__ uint32_t s_hist[RS_MAX_PASSES * 256];
    __shared__ __align__(16) uint8_t s_t[KG_TILE + KG_HALO + 32];
    const int b = kp.b, kc = kp.kc;
    const int groups = (kc + 7) >> 3, rem = kc - 8 * (groups - 1);
    const uint64_t term8 = 0x0101010101010101ull * (uint64_t)kp.term;
    const int t_lo = blockIdx.x * tiles_per_block, t_hi = min(num_tiles, t_lo + tiles_per_block);
    int cur_seg = -1;
    for (int i = threadIdx.x; i < kp.passes * 256; i += blockDim.x) s_hist[i] = 0;
    for (int ti = t_lo; ti < t_hi; ++ti) {
        const RsTileDesc d = descs[ti];
        if (d.seg != cur_seg) {
            __syncthreads();
            if (cur_seg >= 0) {
                rs_hist_flush(s_hist, g_hist + (size_t)cur_seg * kp.passes * 256, kp.passes);
                __syncthreads();
                for (int i = threadIdx.x; i < kp.passes * 256; i += blockDim.x) s_hist[i] = 0;
            }
            cur_seg = d.seg;
        }
        for (int half = 0; half < d.n; half += KG_TILE) {
            const int32_t base = d.start + half;
            const int32_t a0 = base & ~15;            // 16-byte aligned staging window
            const int shift = base - a0;
            const int cnt = min(KG_TILE, d.n - half);
            __syncthreads();
            for (int o = threadIdx.x * 16; o < KG_TILE + KG_HALO + 32; o += blockDim.x * 16) {
                const int64_t g = (int64_t)a0 + o;
                if (g + 16 <= n) *reinterpret_cast<uint4 *>(s_t + o) = *reinterpret_cast<const uint4 *>(T8 + g);
                else for (int q = 0; q < 16; ++q) s_t[o + q] = (g + q < n) ? T8[g + q] : 0;
            }
            __syncthreads();
#pragma unroll 2
            for (int it = 0; it < KG_ITEMS; ++it) {
                const int o = it * KG_THREADS + threadIdx.x;
                const bool valid = o < cnt;
                uint64_t key = 0;
                if (valid) {
                    int tpos = kc;
                    for (int gq = 0; gq < groups; ++gq) {
                        const uint64_t x = lds8(s_t, o + shift + 8 * gq);
                        if (tpos == kc) {
                            const uint64_t tt = x ^ term8;
                            const uint64_t z = (tt - 0x0101010101010101ull) & ~tt & 0x8080808080808080ull;
                            if (z) tpos = min(kc, 8 * gq + ((__ffsll((long long)z) - 1) >> 3));
                        }
                        const uint64_t f = pack8(x, b);
                        if (gq + 1 < groups) key = (key << (8 * b)) | f;
                        else key = (key << (rem * b)) | (f >> ((8 - rem) * b));
                    }
                    if (tpos < kc - 1) key &= ~((1ull << (b * (kc - 1 - tpos))) - 1ull);
                    if (kc * b < 64) key |= (uint64_t)d.seg << (kc * b);
                    keys[base + o] = key;
                    vals[base + o] = (uint32_t)(base + o);
                }
                rs_hist_add(s_hist, key, kp.passes, valid, kp.passes);  // text symbols only: plain atomics
            }
        }
    }
    __syncthreads();
    if (cur_seg >= 0) rs_hist_flush(s_hist, g_hist + (size_t)cur_seg * kp.passes * 256, kp.passes);
}

// general path: raw code points + 1, window cut at the end of the document (pad 0)
__global__ void __launch_bounds__(KG_THREADS)
k_keygen0_general(const uint32_t *__restrict__ T, int32_t begin, int32_t end_, const int32_t *__restrict__ doc_off,
                  int D, KeyParams kp, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                  uint32_t *g_hist) {
    __shared__ uint32_t s_hist[RS_MAX_PASSES * 256];
    for (int i = threadIdx.x; i < kp.passes * 256; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_round = (((int64_t)end_ - begin) + 31) & ~31ll;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_round; j += stride) {
        const int64_t i = begin + j;
        const bool valid = i < end_;
        uint64_t key = 0;
        if (valid) {
            int d = doc_of(doc_off, D, (int32_t)i);
            int32_t end = doc_off[d + 1];
            key = (uint64_t)d;
            for (int c = 0; c < kp.kc; ++c) {
                uint64_t sym = (i + c < end) ? (uint64_t)T[i + c] + 1ull : 0ull;
                key = (key << kp.b) | sym;
            }
            keys[i] = key;
            vals[i] = (uint32_t)i;
        }
        rs_hist_add(s_hist, key, kp.passes, valid);
    }
    __syncthreads();
    rs_hist_flush(s_hist, g_hist, kp.passes);
}

// ------------------------------------------------------------------------------------------
// doubling-round key generation: key = own rank (primary) . rank[i+h] (secondary)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_keygen_h(const uint32_t *__restrict__ vals, const uint32_t *__restrict__ prim, int32_t n_act,
           const uint32_t *__restrict__ rank, int32_t h, int sb, int passes, int general,
           const int32_t *__restrict__ doc_off, int D, uint64_t *__restrict__ keys, uint32_t *g_hist) {
    __shared__ uint32_t s_hist[RS_MAX_PASSES * 256];
    for (int i = threadIdx.x; i < passes * 256; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_round = ((int64_t)n_act + 31) & ~31ll;
    for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_round; a += stride) {
        const bool valid = a < n_act;
        uint64_t key = 0;
        if (valid) {
            uint32_t i = vals[a];
            uint32_t sec;
            if (general) {
                int d = doc_of(doc_off, D, (int32_t)i);
                int64_t j = (int64_t)i + h;
                sec = (j < doc_off[d + 1]) ? rank[j] + 1u : 0u;
            } else {
                sec = rank[i + h];  // stays inside the string: the group shares h terminator-free symbols
            }
            key = ((uint64_t)prim[a] << sb) | sec;
            keys[a] = key;
        }
        if (passes > 0) rs_hist_add(s_hist, key, passes, valid);
    }
    __syncthreads();
    rs_hist_flush(s_hist, g_hist, passes);
}

// ------------------------------------------------------------------------------------------
// doubling rounds, common case: the groups that are still ambiguous are SMALL (a few to a few
// hundred suffixes sharing a repeated phrase), so instead of seven global radix passes every
// element ranks itself inside its own group: it finds the group's extent in the active list
// (equal primary = equal upper key bits), counts the members with a smaller (secondary, index)
// pair and writes its key/value to group_start + count.  Reads are contiguous and shared by the
// threads of the group.  A group larger than GS_MAX sets *overflow and the host redoes the round
// with the radix sort (deep-LCP inputs: many identical strings).
// ------------------------------------------------------------------------------------------
constexpr int GS_MAX = 1024;

__global__ void __launch_bounds__(256)
k_group_sort(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals, int32_t n_act, int sb,
             uint64_t *__restrict__ keys_out, uint32_t *__restrict__ vals_out, uint32_t *overflow) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < n_act; a += stride) {
        const uint64_t key = keys[a];
        const uint64_t prim = key >> sb;
        int64_t gs = a, ge = a + 1;
        int steps = 0;
        while (gs > 0 && (keys[gs - 1] >> sb) == prim && steps < GS_MAX) { --gs; ++steps; }
        while (ge < n_act && (keys[ge] >> sb) == prim && steps < GS_MAX) { ++ge; ++steps; }
        if (steps >= GS_MAX) { *overflow = 1u; continue; }
        uint32_t below = 0;
        for (int64_t b = gs; b < ge; ++b) {
            const uint64_t kb = keys[b];
            below += (kb < key || (kb == key && b < a)) ? 1u : 0u;
        }
        keys_out[gs + below] = key;
        vals_out[gs + below] = vals[a];
    }
}

// ------------------------------------------------------------------------------------------
// re-rank + compaction after a sort: single pass, decoupled look-back over the pair
// (index of the last group head, number of elements kept so far).
// ------------------------------------------------------------------------------------------
constexpr int RR_THREADS = 256;
constexpr int RR_ITEMS = 8;
constexpr int RR_TILE = RR_THREADS * RR_ITEMS;
constexpr uint64_t RR_FLAG_AGG = 1ull << 62;
constexpr uint64_t RR_FLAG_PREFIX = 2ull << 62;
constexpr uint64_t RR_FIELD = (1ull << 31) - 1;

struct RRState { uint32_t mx, sum; };
__device__ __forceinline__ RRState rr_op(RRState a, RRState b) { return RRState{max(a.mx, b.mx), a.sum + b.sum}; }
__device__ __forceinline__ uint64_t rr_pack(RRState s, uint64_t flag) { return flag | ((uint64_t)s.mx << 31) | s.sum; }
__device__ __forceinline__ RRState rr_unpack(uint64_t w) { return RRState{(uint32_t)((w >> 31) & RR_FIELD), (uint32_t)(w & RR_FIELD)}; }

template <bool ROUND0>
__global__ void __launch_bounds__(RR_THREADS)
k_rerank(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals,
         const uint32_t *__restrict__ slots, int32_t n_act, uint64_t sym_mask, uint64_t term,
         int32_t *__restrict__ sa, uint32_t *__restrict__ rank, uint32_t *__restrict__ new_vals,
         uint32_t *__restrict__ new_slots, uint32_t *__restrict__ new_prim,
         volatile uint64_t *status, uint32_t *ticket, uint32_t *out_counts /*[0]=kept*/,
         uint32_t *__restrict__ bkt, int bkt_shift, const uint32_t *__restrict__ abort_flag) {
    if (abort_flag != nullptr && *abort_flag != 0u) return;  // the local group sort gave up: host redoes the round
    __shared__ RRState s_warp[RR_THREADS / 32];
    __shared__ RRState s_prefix;
    __shared__ uint32_t s_tile;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t base = (int64_t)tile * RR_TILE + (int64_t)t * RR_ITEMS;

    uint64_t k[RR_ITEMS + 2];  // k[0] = predecessor, k[RR_ITEMS+1] = successor
    bool head[RR_ITEMS + 1];
    if (base + RR_ITEMS <= n_act) {
        // full thread chunk: 128-bit loads of the 8 own keys; the neighbours' edge keys come from
        // the adjacent lanes (only warp-edge lanes touch global memory again)
#pragma unroll
        for (int j = 0; j < RR_ITEMS; j += 2) {
            const ulonglong2 kk = *reinterpret_cast<const ulonglong2 *>(keys + base + j);
            k[j + 1] = kk.x; k[j + 2] = kk.y;
        }
    } else {
#pragma unroll
        for (int j = 1; j <= RR_ITEMS; ++j) {
            int64_t a = base + j - 1;
            k[j] = (a < n_act) ? keys[a] : 0ull;
        }
    }
    {
        const uint64_t from_prev = __shfl_up_sync(0xffffffffu, k[RR_ITEMS], 1);
        const uint64_t from_next = __shfl_down_sync(0xffffffffu, k[1], 1);
        k[0] = (lane > 0) ? from_prev : ((base - 1 >= 0 && base - 1 < n_act) ? keys[base - 1] : 0ull);
        k[RR_ITEMS + 1] = (lane < 31) ? from_next : ((base + RR_ITEMS < n_act) ? keys[base + RR_ITEMS] : 0ull);
    }
    // head[j] describes element base+j (j = RR_ITEMS: the successor, for singleton detection)
#pragma unroll
    for (int j = 0; j <= RR_ITEMS; ++j) {
        int64_t a = base + j;
        bool hd = (a == 0) || (a >= n_act) || (k[j + 1] != k[j]);
        if (ROUND0) {
            uint64_t f = k[j + 1] & sym_mask;  // last symbol of the window: 0 = cut, term = terminator
            hd = hd || (f == 0ull) || (f == term);
        }
        head[j] = hd;
        // 2-gram bucket table of the scorer: first rank of every (document, symbol 0, symbol 1)
        if (ROUND0 && bkt != nullptr && j < RR_ITEMS && a < n_act) {
            const uint64_t pre = k[j + 1] >> bkt_shift;
            if (a == 0 || pre != (k[j] >> bkt_shift)) bkt[pre] = (uint32_t)a;
        }
    }
    RRState loc[RR_ITEMS];
    RRState run{0u, 0u};
#pragma unroll
    for (int j = 0; j < RR_ITEMS; ++j) {
        int64_t a = base + j;
        bool valid = a < n_act;
        bool keep = valid && !(head[j] && head[j + 1]);
        RRState e{(valid && head[j]) ? (uint32_t)a : 0u, keep ? 1u : 0u};
        run = rr_op(run, e);
        loc[j] = run;  // inclusive within the thread
    }
    // warp inclusive scan of thread totals
    RRState x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        RRState y{__shfl_up_sync(0xffffffffu, x.mx, o), __shfl_up_sync(0xffffffffu, x.sum, o)};
        if (lane >= o) x = rr_op(y, x);
    }
    if (lane == 31) s_warp[w] = x;
    __syncthreads();
    RRState wbase{0u, 0u};
    for (int i = 0; i < w; ++i) wbase = rr_op(wbase, s_warp[i]);
    RRState thread_excl{__shfl_up_sync(0xffffffffu, x.mx, 1), __shfl_up_sync(0xffffffffu, x.sum, 1)};
    if (lane == 0) thread_excl = RRState{0u, 0u};
    thread_excl = rr_op(wbase, thread_excl);

    // ---- decoupled look-back by the LAST WARP: each lane inspects one predecessor tile, so a
    // window of 32 status words costs one round trip (a single thread walking them one by one was
    // 45 % of this kernel's stall samples)
    if (w == RR_THREADS / 32 - 1) {
        const RRState mine = rr_op(wbase, x);  // lane 31: the tile aggregate
        const RRState agg{__shfl_sync(0xffffffffu, mine.mx, 31), __shfl_sync(0xffffffffu, mine.sum, 31)};
        RRState excl{0u, 0u};
        if (tile == 0) {
            if (lane == 31) status[0] = rr_pack(agg, RR_FLAG_PREFIX);
        } else {
            if (lane == 31) status[tile] = rr_pack(agg, RR_FLAG_AGG);
            int64_t win = (int64_t)tile - 1;
            while (true) {
                const int64_t idx = win - lane;
                uint64_t sv = 2ull << 62;  // before tile 0: an empty inclusive prefix
                if (idx >= 0) sv = status[idx];
                const unsigned flag = (unsigned)(sv >> 62);
                const unsigned ready = __ballot_sync(0xffffffffu, flag != 0u);
                const unsigned pref = __ballot_sync(0xffffffffu, flag == 2u);
                const int first_pref = pref ? (__ffs(pref) - 1) : 31;
                const unsigned need = (first_pref == 31) ? 0xffffffffu : ((2u << first_pref) - 1u);
                if ((ready & need) != need) continue;  // a needed predecessor has not published yet
                RRState r = (lane <= first_pref) ? rr_unpack(sv) : RRState{0u, 0u};
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    RRState y{__shfl_xor_sync(0xffffffffu, r.mx, o), __shfl_xor_sync(0xffffffffu, r.sum, o)};
                    r = rr_op(r, y);
                }
                excl = rr_op(excl, r);
                if (pref) break;
                win -= 32;
            }
            if (lane == 31) status[tile] = rr_pack(rr_op(excl, agg), RR_FLAG_PREFIX);
        }
        if (lane == 31) {
            s_prefix = excl;
            if ((int64_t)(tile + 1) * RR_TILE >= n_act) out_counts[0] = excl.sum + agg.sum;
        }
    }
    __syncthreads();
    const RRState pre = rr_op(s_prefix, thread_excl);
    uint32_t vv[RR_ITEMS], ss[RR_ITEMS];
    const bool full = base + RR_ITEMS <= n_act;
    if (full) {
#pragma unroll
        for (int j = 0; j < RR_ITEMS; j += 4) {
            const uint4 q4 = *reinterpret_cast<const uint4 *>(vals + base + j);
            vv[j] = q4.x; vv[j + 1] = q4.y; vv[j + 2] = q4.z; vv[j + 3] = q4.w;
            if (!ROUND0) {
                const uint4 s4 = *reinterpret_cast<const uint4 *>(slots + base + j);
                ss[j] = s4.x; ss[j + 1] = s4.y; ss[j + 2] = s4.z; ss[j + 3] = s4.w;
            }
        }
        if (ROUND0) {  // SA slot == position in the sorted order: two 128-bit stores per thread
#pragma unroll
            for (int j = 0; j < RR_ITEMS; j += 4)
                *reinterpret_cast<int4 *>(sa + base + j) = make_int4((int)vv[j], (int)vv[j + 1], (int)vv[j + 2], (int)vv[j + 3]);
        }
    }
#pragma unroll
    for (int j = 0; j < RR_ITEMS; ++j) {
        int64_t a = base + j;
        if (a >= n_act) break;
        RRState inc = rr_op(pre, loc[j]);
        uint32_t v = full ? vv[j] : vals[a];
        uint32_t slot = ROUND0 ? (uint32_t)a : (full ? ss[j] : slots[a]);
        uint32_t r = ROUND0 ? inc.mx : slots[inc.mx];
        if (!(ROUND0 && full)) sa[slot] = (int32_t)v;
        rank[v] = r;
        bool keep = !(head[j] && head[j + 1]);
        if (keep) {
            uint32_t dst = inc.sum - 1u;
            new_vals[dst] = v;
            new_slots[dst] = slot;
            new_prim[dst] = r;
        }
    }
}

// Buckets that do not occur keep 0xffffffff after the re-rank; give every entry the first rank of
// the next existing bucket (suffix minimum), so that [bkt[x], bkt[x+1]) is the SA interval of
// 2-gram x and [bkt[c << b], bkt[(c+1) << b]) that of first symbol c.  One CTA per document.
__global__ void __launch_bounds__(256)
k_bucket_fill(uint32_t *__restrict__ bkt, int entries, const int32_t *__restrict__ doc_off) {
    __shared__ uint32_t s_carry;
    uint32_t *row = bkt + (size_t)blockIdx.x * entries;
    if (threadIdx.x == 0) s_carry = (uint32_t)doc_off[blockIdx.x + 1];
    __syncthreads();
    for (int hi = entries; hi > 0; hi -= 256) {  // chunks of 256 from the end
        const int x = hi - 256 + (int)threadIdx.x;
        uint32_t v = (x >= 0) ? row[x] : 0xffffffffu;
        // suffix-min within the chunk (thread t needs min over t..255)
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        uint32_t m = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_down_sync(0xffffffffu, m, o);
            if (lane + o < 32) m = min(m, y);
        }
        __shared__ uint32_t s_w[8];
        if (lane == 0) s_w[w] = m;
        __syncthreads();
        uint32_t tail = s_carry;
        for (int i = w + 1; i < 8; ++i) tail = min(tail, s_w[i]);
        m = min(m, tail);
        if (x >= 0) row[x] = m;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = m;  // minimum of this chunk and everything after it
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------
// Pipelined host build (east_build_host on a large batch of small documents): the text arrives chunk
// by chunk on a copy stream.  The alphabet is taken from chunk 0 (speculation: later chunks use no
// other code point below 0x0A00), every chunk is encoded and sorted by the per-document kernel as soon
// as it is resident.  Two flags confirm the speculation at the end, with no further pass over the text: the
// encoder reports a code point below 0x0A00 that the alphabet of chunk 0 lacks (the only way the alphabets can
// differ: chunk 0 is part of the text), and the per-document kernel validates the terminator layout of its
// document (count, values, order, last position).  If either is set, nothing is kept and the ordinary build
// runs on the resident text.
// arrays that stay with the index come from its arena (one allocation per index), scratch from the pool
template <typename T>
static DevBuf<T> take(const SaInput &in, size_t count, cudaStream_t s) {
    return in.arena ? in.arena->take<T>(count, s) : DevBuf<T>(count, s);
}

// An alphabet taken from PART of the text (run 0 of a pipelined build, the sampled prefix of a device-resident one) may
// lack a rare letter or digit that the rest uses, and a miss costs a second build.  A code that the text never uses costs
// nothing as long as the symbol width stays the same: a class of ASCII symbols (A-Z, a-z, 0-9) that the part has met at all
// is completed when that fits.  present: bitmap of the code points seen (updated); extra: what was added (code points < 128).
static void complete_symbol_classes(uint32_t *present, uint32_t extra[4]) {
    int seen = 0;
    for (int w = 0; w < (int)(EAST_TERM_BASE / 32); ++w) seen += __builtin_popcount(present[w]);
    const int width = bits_for((uint64_t)seen + 1);
    int room = (1 << width) - 1 - (seen + 1);   // codes 1..sigma and sigma + 1 for the terminators must fit `width` bits
    const int classes[3][2] = {{'A', 'Z'}, {'a', 'z'}, {'0', '9'}};
    for (auto &cl : classes) {
        int have = 0, lack = 0;
        for (int c = cl[0]; c <= cl[1]; ++c) (present[c >> 5] & (1u << (c & 31))) ? ++have : ++lack;
        if (have == 0 || lack == 0 || lack > room) continue;
        for (int c = cl[0]; c <= cl[1]; ++c)
            if (!(present[c >> 5] & (1u << (c & 31)))) extra[c >> 5] |= 1u << (c & 31);
        room -= lack;
    }
    for (int w = 0; w < 4; ++w) present[w] |= extra[w];
}

// The alphabet a thread's last batch of small documents was indexed with, as a guess for its next batch on the same
// device (collections come in batches of one language).  It is the same speculation as the alphabet of run 0 / of a
// sampled prefix -- phase 1 of the per-document kernel reports every code point the table lacks, and the batch is then
// redone from a scan -- but it needs no scan kernel and, above all, no host round trip before the first wave: with the
// text of the later runs in flight the answer of the scan took 0.1-0.2 ms to reach the host.
struct AlphabetGuess {
    bool valid = false;
    int device = -1;
    uint32_t present[EAST_TERM_BASE / 32];
};
static thread_local AlphabetGuess g_alphabet_guess;

__global__ void __launch_bounds__(128)
k_set_present(ScanResult *res, PresentBits bits) {
    for (int i = threadIdx.x; i < (int)(EAST_TERM_BASE / 32); i += blockDim.x) res->present[i] = bits.w[i];
}

static bool alphabet_guess_for(const SaInput &in, PresentBits &bits) {
    int dev = -1;
    if (!in.alphabet_guess || !g_alphabet_guess.valid || cudaGetDevice(&dev) != cudaSuccess || dev != g_alphabet_guess.device) return false;
    memcpy(bits.w, g_alphabet_guess.present, sizeof(bits.w));
    return true;
}

static void alphabet_guess_keep(const uint32_t *present) {
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    g_alphabet_guess.valid = true;
    g_alphabet_guess.device = dev;
    memcpy(g_alphabet_guess.present, present, sizeof(g_alphabet_guess.present));
    uint32_t extra[4] = {0u, 0u, 0u, 0u};   // kept with its ASCII classes completed (idempotent): what a build makes of it
    complete_symbol_classes(g_alphabet_guess.present, extra);
}

void alphabet_guess_forget() { g_alphabet_guess.valid = false; }

// The code table a build on this thread and device would derive from the guess (codes 1..sigma in code point order), for
// callers that prepare something for that table before the build runs (the keyphrases' dense codes); false: no guess.
bool alphabet_guess_code_table(uint8_t *table /* EAST_TERM_BASE entries */) {
    int dev = -1;
    if (!g_alphabet_guess.valid || cudaGetDevice(&dev) != cudaSuccess || dev != g_alphabet_guess.device) return false;
    int sigma = 0;
    for (uint32_t c = 0; c < EAST_TERM_BASE; ++c) {
        const bool on = (g_alphabet_guess.present[c >> 5] >> (c & 31)) & 1u;
        if (on) ++sigma;
        table[c] = on ? (uint8_t)(sigma & 0xff) : (uint8_t)0;
    }
    return sigma <= 253;
}

static bool build_pipelined(const SaInput &in, SaOutput &out, StageTimer &tm, cudaStream_t s, uint32_t &doc_sort_flags) {
    const int32_t n = in.n;
    const int D = in.n_docs;
    int32_t max_doc_n = 0;
    for (int d = 0; d < D; ++d) max_doc_n = std::max(max_doc_n, in.doc_off_host[d + 1] - in.doc_off_host[d]);
    tm.mark("alphabet");
    DevBuf<ScanResult> d_first(1, s);
    const int32_t n0 = in.doc_off_host[in.chunk_doc[1]];
    ScanResult first;
    PresentBits guess;
    const bool guessed = alphabet_guess_for(in, guess);
    if (guessed) {
        memset(&first, 0, sizeof(first));
        memcpy(first.present, guess.w, sizeof(guess.w));
    } else {
        EAST_CUDA(cudaMemsetAsync(d_first.p, 0, sizeof(ScanResult), s));
        EAST_CUDA(cudaStreamWaitEvent(s, in.chunk_ready[0], 0));
        if (in.text8) EAST_LAUNCH(k_alphabet8, grid_for(n0, 256 * 16, 4), 256, 0, s, in.text8, n0, d_first.p);
        else EAST_LAUNCH(k_alphabet, grid_for(n0, 256 * 4 * 4, 4), 256, 0, s, in.text, n0, d_first.p);
        EAST_CUDA(cudaMemcpyAsync(&first, d_first.p, sizeof(ScanResult), cudaMemcpyDeviceToHost, s));
        EAST_CUDA(cudaStreamSynchronize(s));
        host_debug_mark("scan back");
    }
    // the alphabet of run 0 (a few dozen documents), with the ASCII classes it has met completed
    uint32_t *present = first.present;
    uint32_t extra[4] = {0u, 0u, 0u, 0u};
    complete_symbol_classes(present, extra);
    int sigma = 0;
    std::vector<uint8_t> table(EAST_TERM_BASE, 0);
    for (uint32_t c = 0; c < EAST_TERM_BASE; ++c)
        if (present[c >> 5] & (1u << (c & 31))) { ++sigma; table[c] = (uint8_t)(sigma & 0xff); }
    DocSortPlan plan;
    const bool eligible = sigma <= 253 && doc_sort_plan(sigma, max_doc_n, plan);
    const uint32_t term = (uint32_t)sigma + 1;

    DevBuf<uint8_t> t8;
    DevBuf<uint32_t> flags(2, s);   // [0] doc_sort overflow, [1] encode miss
    if (eligible) {
        tm.mark("doc_sort");
        DevBuf<uint8_t> d_table(EAST_TERM_BASE, s);
        t8 = take<uint8_t>(in, (size_t)n + 128, s);
        uint32_t *end0 = nullptr, *end1 = nullptr;
        if (((size_t)D << (2 * plan.b)) <= (size_t)2 * n + 4096) {
            const size_t entries = ((size_t)D << (2 * plan.b)) + 1;
            out.bkt = take<uint32_t>(in, entries, s);
            end0 = out.bkt.p + entries - 1;
            out.sym_bits = plan.b;
            if (in.want_bkt3 && plan.G == 3 && ((size_t)D << (3 * plan.b)) * sizeof(uint32_t) <= ((size_t)8 << 30)) {
                // the kernel's buckets ARE the 3-grams: their first ranks cost one more coalesced store and turn
                // the scorer's depth-2 narrowing (a binary search over the largest intervals) into a lookup
                const size_t e3 = ((size_t)D << (3 * plan.b)) + 1;
                out.bkt3 = take<uint32_t>(in, e3, s);
                end1 = out.bkt3.p + e3 - 1;
            }
        }
        {   // code table, cleared flags, closing entries of the bucket tables: one launch
            PresentBits bits;
            memcpy(bits.w, present, sizeof(bits.w));   // (completed; only read when the alphabet is a guess)
            EAST_LAUNCH(k_doc_sort_prologue, 1, 128, 0, s, guessed ? (const ScanResult *)nullptr : d_first.p, bits,
                        make_uint4(extra[0], extra[1], extra[2], extra[3]), d_table.p, flags.p, end0, end1, (uint32_t)n);
            if (guessed) EAST_CUDA(cudaStreamWaitEvent(s, in.chunk_ready[0], 0));   // (a scan has waited for the lead run already)
        }
        DocSortTables tables{in.lcp, in.up, in.down, in.next, in.ann};
        const bool fuse = in.lcp != nullptr && plan.tables_fit;
        // runs alternate between the main stream and a helper stream: a run is one wave of per-document CTAs,
        // and on one stream the next wave could not start before the slowest CTA of the previous one ended
        cudaStream_t lanes[2] = {s, in.helper_stream ? in.helper_stream : s};
        // By default the per-document kernel byte-codes its documents itself (in.fused_encode).  A separate byte-coding
        // kernel (option no_fused_encode) needs a few microseconds of the machine, but a per-document CTA owns its SM:
        // even on a high-priority stream of its own (prep) it only starts when a wave drains, and the kernel of the
        // run waits for it -- measured: consecutive waves then do not overlap (4.54 vs 4.23 ms end to end).
        cudaStream_t prep = (in.prep_stream && lanes[1] != s && !in.fused_encode) ? in.prep_stream : nullptr;
        cudaEvent_t ready_to_sort = nullptr, helper_done = nullptr;
        if (lanes[1] != s) {
            EAST_CUDA(cudaEventCreateWithFlags(&ready_to_sort, cudaEventDisableTiming));
            EAST_CUDA(cudaEventCreateWithFlags(&helper_done, cudaEventDisableTiming));
            EAST_CUDA(cudaEventRecord(ready_to_sort, s));           // code table, flag reset, allocations
            EAST_CUDA(cudaStreamWaitEvent(lanes[1], ready_to_sort, 0));
            if (prep) EAST_CUDA(cudaStreamWaitEvent(prep, ready_to_sort, 0));
        }
        for (int c = 0; c < in.n_chunks; ++c) {
            const int d0 = in.chunk_doc[c], d1 = in.chunk_doc[c + 1];
            const int32_t e0 = in.doc_off_host[d0], e1 = in.doc_off_host[d1];
            cudaStream_t ls = lanes[c & 1];
            cudaStream_t es = prep ? prep : ls;
            if (c > 0) EAST_CUDA(cudaStreamWaitEvent(es, in.chunk_ready[c], 0));
            if (!in.fused_encode) {
                EAST_BYTES(5.0 * (e1 - e0));
                EAST_LAUNCH(k_encode_text, grid_for(e1 - e0, 256 * 4 * 4, 4), 256, 0, es, in.text, e0, e1, d_table.p,
                            (uint8_t)term, t8.p, flags.p + 1);
            }
            if (prep) {
                cudaEvent_t coded;
                EAST_CUDA(cudaEventCreateWithFlags(&coded, cudaEventDisableTiming));
                EAST_CUDA(cudaEventRecord(coded, prep));
                EAST_CUDA(cudaStreamWaitEvent(ls, coded, 0));
                EAST_CUDA(cudaEventDestroy(coded));   // released once it has fired
            }
            const bool hooks = out.bkt.p != nullptr;
            const RunReady run{d0, d1 - d0, ls, t8.p, out.bkt.p, out.bkt3.p, out.sym_bits, &table, 1};
            DocScore score;
            host_debug_mark("run begin");
            if (hooks && in.run_begin) in.run_begin(in.run_ctx, run, score);
            host_debug_mark("run launch");
            doc_sort_launch(plan, t8.p, in.text, in.doc_off, in.doc_m, d0, d1 - d0, e1 - e0, term, out.sa, out.bkt.p,
                            out.bkt3.p, flags.p, ls, nullptr, fuse ? &tables : nullptr, in.sk, &score,
                            in.fused_encode ? d_table.p : nullptr, flags.p + 1, n, in.text8);
            if (hooks && in.run_hook) in.run_hook(in.run_ctx, run, score.recs != nullptr ? 1 : 0);
            if (score.recs && score.skip_suffix_keys) out.sk_skipped = 1;
        }
        if (lanes[1] != s) {
            EAST_CUDA(cudaEventRecord(helper_done, lanes[1]));
            EAST_CUDA(cudaStreamWaitEvent(s, helper_done, 0));
            EAST_CUDA(cudaEventDestroy(ready_to_sort));
            EAST_CUDA(cudaEventDestroy(helper_done));
        }
        out.tables_done = fuse ? 1 : 0;
    } else {
        for (int c = guessed ? 0 : 1; c < in.n_chunks; ++c) EAST_CUDA(cudaStreamWaitEvent(s, in.chunk_ready[c], 0));
    }
    tm.mark("validate");
    uint32_t h_flags[2] = {0u, 0u};
    if (eligible) EAST_CUDA(cudaMemcpyAsync(h_flags, flags.p, sizeof(h_flags), cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaStreamSynchronize(s));
    const bool ok = eligible && !h_flags[0] && !h_flags[1];
    doc_sort_flags = h_flags[0];
    out.alphabet_guessed = guessed ? 1 : 0;
    if (!ok) {
        if (guessed) g_alphabet_guess.valid = false;   // whatever went wrong: the next batch starts from a scan
        out.pipeline_miss = eligible ? 1 : 0;
        out.doc_sort_overflow = (h_flags[0] & 1u) ? 1 : 0;
        out.tables_done = 0;
        out.bkt = DevBuf<uint32_t>();
        out.bkt3 = DevBuf<uint32_t>();
        out.sym_bits = 0;
        return false;
    }
    alphabet_guess_keep(present);
    out.pipelined = 1;
    out.sk_done = in.sk ? 1 : 0;
    out.fast_path = 1;
    out.sigma = sigma;
    out.doc_sorted = 1;
    out.rounds = 1;
    out.key_chars = plan.G + 8;
    out.key_bits = plan.b * plan.G + 64;
    out.code_table = table;
    out.term_code = (int)term;
    out.t8 = std::move(t8);
    return true;
}

void build_suffix_array(const SaInput &in, SaOutput &out, StageTimer &tm, cudaStream_t s) {
    const int32_t n = in.n;
    const int D = in.n_docs;
    DevBuf<ScanResult> d_scan(1, s);
    ScanResult scan;
    bool allow_doc_sort = in.doc_sort != 0;
    const size_t arena_mark = in.arena ? in.arena->used : 0;   // a pass that fails gives its slices back
    if (in.n_chunks > 0) {
        uint32_t refused = 0;   // what the per-document kernel reported: bit 0 a bucket too large, bit 1 a bad layout
        if (build_pipelined(in, out, tm, s, refused)) return;
        if (in.arena) in.arena->used = arena_mark;
        if (refused) allow_doc_sort = false;  // it would refuse again: full scan, global sort
        if (in.text8) {
            // the runs were byte-coded from the one-byte text; what follows reads code points: expand the whole batch
            // (every run has arrived: build_pipelined ended on a host sync after the last one)
            DevBuf<uint32_t> bad(1, s);
            EAST_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(uint32_t), s));
            expand_text8(in.text8, in.doc_off, in.doc_m, D, const_cast<uint32_t *>(in.text), bad.p, s);
            uint32_t h_bad = 0;
            EAST_CUDA(cudaMemcpyAsync(&h_bad, bad.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            EAST_CUDA(cudaStreamSynchronize(s));
            if (h_bad) throw Error(-1, "one-byte text: a document does not hold exactly doc_m string ends (0xFF) or does not end with one");
        }
    }
    int32_t max_doc_n = 0;
    for (int d = 0; d < D; ++d) max_doc_n = std::max(max_doc_n, in.doc_off_host[d + 1] - in.doc_off_host[d]);
    // Batches of small documents start with the LIGHT scan (alphabet, counts): the per-document kernel
    // validates the terminator layout of its document itself.  Whatever it cannot take (bad layout, a
    // bucket too large, an alphabet too wide) is redone below with the validating scan.
    const bool light = allow_doc_sort && in.light_scan && !in.force_general && max_doc_n <= 65535;
    tm.mark("scan_text");
    EAST_CUDA(cudaMemsetAsync(d_scan.p, 0, sizeof(ScanResult), s));
    EAST_BYTES(4.0 * n);
    // Device-resident batches of small documents: the alphabet comes from a PREFIX of the text (speculation, as in the
    // pipelined host build: the rest uses no other code point below 0x0A00); the per-document kernel reports a code point
    // the table lacks and the batch is then redone with the alphabet of the whole text.  Saves the pass over the text.
    const int32_t n_scan = (light && in.fused_encode && in.alphabet_sample > 0 && in.alphabet_sample < n) ? (int32_t)in.alphabet_sample : n;
    const bool sampled = n_scan < n;
    // ... or, where a sample would do, from the alphabet of this thread's previous batch (g_alphabet_guess): no scan, no wait
    PresentBits guess;
    const bool guessed = sampled && alphabet_guess_for(in, guess);
    if (guessed) {
        memset(&scan, 0, sizeof(scan));
        memcpy(scan.present, guess.w, sizeof(guess.w));
        if (in.scan_queued) in.scan_queued(in.run_ctx);
    } else {
        if (light) {
            EAST_LAUNCH(k_alphabet, grid_for(n_scan, 256 * 4 * 4, 4), 256, 0, s, in.text, n_scan, d_scan.p);
        } else {
            EAST_LAUNCH(k_scan_text, grid_for(n, ST_TILE, 4), 256, 0, s, in.text, n, in.doc_off, in.doc_m, D, d_scan.p, 0,
                        (n + ST_TILE - 1) / ST_TILE, 1);
        }
        EAST_CUDA(cudaMemcpyAsync(&scan, d_scan.p, sizeof(ScanResult), cudaMemcpyDeviceToHost, s));
        if (in.scan_queued) in.scan_queued(in.run_ctx);
        EAST_CUDA(cudaStreamSynchronize(s));
    }
    out.alphabet_guessed = guessed ? 1 : 0;

    uint32_t extra[4] = {0u, 0u, 0u, 0u};
    if (sampled) complete_symbol_classes(scan.present, extra);
    int sigma = 0;
    std::vector<uint8_t> table(EAST_TERM_BASE, 0);
    for (uint32_t c = 0; c < EAST_TERM_BASE; ++c)
        if (scan.present[c >> 5] & (1u << (c & 31))) {
            ++sigma;
            table[c] = (uint8_t)(sigma & 0xff);
        }
    // (a sampled scan has not counted the terminators of the whole text: the per-document kernel validates the layout)
    bool fast = !scan.bad && (sampled || scan.n_term == (uint32_t)in.m_total) && sigma <= 253 && !in.force_general;
    out.fast_path = fast ? 1 : 0;
    out.sigma = sigma;

    const int dbits = bits_for((uint64_t)(D > 0 ? D - 1 : 0));
    KeyParams kp;
    if (fast) {
        kp.b = bits_for((uint64_t)sigma + 1);
        kp.term = (uint32_t)sigma + 1;
    } else {
        kp.b = bits_for((uint64_t)scan.max_code + 1);
        kp.term = 0xffffffffu;
    }
    if (dbits + kp.b > 64) throw Error(-5, "document count x alphabet does not fit a 64-bit sort key");
    int kc = (64 - dbits) / kp.b;
    if (kc > KG_HALO) kc = KG_HALO;
    // one symbol less when that saves a whole radix pass over all N suffixes and still leaves a
    // window of >= 8 symbols (measured on the Zipf workload: 55-bit keys / 7 passes beat 60 / 8)
    {
        // bits that actually get sorted: without the document id when the per-document sort applies
        const bool seg_like = fast && in.segmented_sort && (int64_t)n / D >= 2 * RS_SEG_TILE && in.sort_batch_elems == 0;
        const int extra = seg_like ? 0 : dbits;
        if (kc > 8 && rs_num_passes(extra + (kc - 1) * kp.b) < rs_num_passes(extra + kc * kp.b)) --kc;
    }
    if (in.key_chars > 0 && in.key_chars < kc) kc = in.key_chars;
    kp.kc = kc;
    const int key_bits = dbits + kc * kp.b;
    kp.passes = rs_num_passes(key_bits);
    out.key_chars = kc;
    out.key_bits = key_bits;

    tm.mark("encode");
    DevBuf<uint8_t> t8, d_table;
    size_t arena_after_t8 = arena_mark;
    // the per-document kernel byte-codes its document itself: the separate pass only runs for the global sort
    DocSortPlan doc_plan;
    const bool try_doc_sort = fast && allow_doc_sort && doc_sort_plan(sigma, max_doc_n, doc_plan);
    bool coded = false;
    auto encode_all = [&]() {
        EAST_BYTES(5.0 * n);
        EAST_LAUNCH(k_encode_text, grid_for(n, 256 * 4 * 4, 4), 256, 0, s, in.text, 0, n, d_table.p,
                    (uint8_t)kp.term, t8.p, (uint32_t *)nullptr);
        coded = true;
    };
    // the per-document kernel that byte-codes its documents itself gets the code table from its one-launch prologue below
    const bool table_in_prologue = try_doc_sort && in.fused_encode;
    if (fast) {
        d_table = DevBuf<uint8_t>(EAST_TERM_BASE, s);
        if (!table_in_prologue) {
            if (guessed) {   // (the bitmap only exists on the host so far)
                PresentBits bits;
                memcpy(bits.w, scan.present, sizeof(bits.w));
                EAST_LAUNCH(k_set_present, 1, 128, 0, s, d_scan.p, bits);
            }
            EAST_LAUNCH(k_code_table, 1, 128, 0, s, d_scan.p, d_table.p, make_uint4(extra[0], extra[1], extra[2], extra[3]));
        }
        t8 = take<uint8_t>(in, (size_t)n + 128, s);
        arena_after_t8 = in.arena ? in.arena->used : 0;
        if (!table_in_prologue) encode_all();
    }
    out.code_table = table;
    out.term_code = fast ? (int)kp.term : 0;

    if (sampled && !try_doc_sort) {   // the sample does not lead to the per-document kernel: decide on the whole text
        if (guessed) g_alphabet_guess.valid = false;
        t8.release();
        if (in.arena) in.arena->used = arena_mark;
        SaInput again = in;
        again.alphabet_sample = 0;
        build_suffix_array(again, out, tm, s);
        return;
    }
    // ---- small documents: one CTA per document, everything in shared memory (doc_sort.cu)
    uint32_t doc_sort_flags = 0;   // bit 0: a bucket too large, bit 1: bad terminator layout
    if (try_doc_sort) {
        const DocSortPlan &plan = doc_plan;
        {
            tm.mark("doc_sort");
            DevBuf<uint32_t> flag(2, s);   // [0] the kernel's flags, [1] encoder miss (a sampled or guessed alphabet lacks a code point)
            uint32_t *end0 = nullptr, *end1 = nullptr;
            if (((size_t)D << (2 * plan.b)) <= (size_t)2 * n + 4096) {
                const size_t entries = ((size_t)D << (2 * plan.b)) + 1;
                out.bkt = take<uint32_t>(in, entries, s);
                end0 = out.bkt.p + entries - 1;
                out.sym_bits = plan.b;
                if (in.want_bkt3 && plan.G == 3 && ((size_t)D << (3 * plan.b)) * sizeof(uint32_t) <= ((size_t)8 << 30)) {
                    // the kernel's buckets ARE the 3-grams: their first ranks cost one more coalesced store and turn
                    // the scorer's depth-2 narrowing (a binary search over the largest intervals) into a lookup
                    const size_t e3 = ((size_t)D << (3 * plan.b)) + 1;
                    out.bkt3 = take<uint32_t>(in, e3, s);
                    end1 = out.bkt3.p + e3 - 1;
                }
            }
            if (table_in_prologue) {   // code table, cleared flags, closing entries of the bucket tables: one launch
                PresentBits bits;
                memcpy(bits.w, scan.present, sizeof(bits.w));
                EAST_LAUNCH(k_doc_sort_prologue, 1, 128, 0, s, guessed ? (const ScanResult *)nullptr : d_scan.p, bits,
                            make_uint4(extra[0], extra[1], extra[2], extra[3]), d_table.p, flag.p, end0, end1, (uint32_t)n);
            } else {
                EAST_CUDA(cudaMemsetAsync(flag.p, 0, 2 * sizeof(uint32_t), s));
                if (end0) EAST_LAUNCH(k_store_u32, 1, 1, 0, s, end0, (uint32_t)n);
                if (end1) EAST_LAUNCH(k_store_u32, 1, 1, 0, s, end1, (uint32_t)n);
            }
            static const bool profile = getenv("EAST_DOC_SORT_PROFILE") != nullptr;
            DevBuf<unsigned long long> clk;
            if (profile) {
                clk = DevBuf<unsigned long long>(17, s);
                EAST_CUDA(cudaMemsetAsync(clk.p, 0, 17 * sizeof(unsigned long long), s));
            }
            DocSortTables tables{in.lcp, in.up, in.down, in.next, in.ann};
            const bool fuse = in.lcp != nullptr && plan.tables_fit;
            const bool hooks = out.bkt.p != nullptr;
            const RunReady run{0, D, s, t8.p, out.bkt.p, out.bkt3.p, out.sym_bits, &table, 0};
            DocScore score;
            if (hooks && in.run_begin) in.run_begin(in.run_ctx, run, score);
            doc_sort_launch(plan, t8.p, in.text, in.doc_off, in.doc_m, 0, D, n, kp.term, out.sa, out.bkt.p, out.bkt3.p, flag.p, s, clk.p,
                            fuse ? &tables : nullptr, in.sk, &score, coded ? nullptr : d_table.p, flag.p + 1, n);
            uint32_t h_flag[2] = {0u, 0u};
            EAST_CUDA(cudaMemcpyAsync(h_flag, flag.p, sizeof(h_flag), cudaMemcpyDeviceToHost, s));
            EAST_CUDA(cudaStreamSynchronize(s));
            const uint32_t overflow = h_flag[0];
            const bool missed = sampled && h_flag[1] != 0u;   // the sampled alphabet lacks a code point of the text
            if (profile) {
                unsigned long long h[17];
                EAST_CUDA(cudaMemcpy(h, clk.p, sizeof(h), cudaMemcpyDeviceToHost));
                // phase 8: "child" = stack walk or tiles, "child_outside" = outside-chunk searches or redone tiles
                static const char *names[10] = {"load", "hist", "scan", "scatter", "refine", "windows", "lcp", "child", "child_outside", "score"};
                fprintf(stderr, "[east] doc_sort phases, kilo-cycles per document:");
                for (int k = 0; k < 10; ++k) fprintf(stderr, " %s %.1f", names[k], (double)h[k] / D / 1e3);
                fprintf(stderr, "\n");
                // tile path of phase 8 only (zero for the stack walk): queries that leave their tile, by the pyramid level
                // that answers them, the stores into other warps' ranges queued for after the barrier and the tiles redone
                // because that queue was full
                fprintf(stderr, "[east] doc_sort phase 8 per document: queries answered by the next tile %.1f, at level 1 %.1f, "
                        "level 2 %.1f, level 3 %.1f, none %.1f; stores queued %.1f, tiles redone %.1f\n", (double)h[10] / D,
                        (double)h[11] / D, (double)h[12] / D, (double)h[13] / D, (double)h[14] / D, (double)h[16] / D, (double)h[15] / D);
            }
            if (missed) {
                // nothing of this pass is kept: the same build with the alphabet of the whole text
                if (guessed) g_alphabet_guess.valid = false;
                out.bkt = DevBuf<uint32_t>();
                out.bkt3 = DevBuf<uint32_t>();
                out.sym_bits = 0;
                t8.release();
                if (in.arena) in.arena->used = arena_mark;
                SaInput again = in;
                again.alphabet_sample = 0;
                build_suffix_array(again, out, tm, s);
                out.alphabet_miss = 1;
                out.alphabet_guessed = guessed ? 1 : 0;
                return;
            }
            if (!overflow) {
                alphabet_guess_keep(scan.present);
                if (hooks && in.run_hook) in.run_hook(in.run_ctx, run, score.recs != nullptr ? 1 : 0);
                if (score.recs && score.skip_suffix_keys) out.sk_skipped = 1;
                out.doc_sorted = 1;
                out.tables_done = fuse ? 1 : 0;
                out.sk_done = in.sk ? 1 : 0;
                out.rounds = 1;
                out.key_chars = plan.G + 8;
                out.key_bits = plan.b * plan.G + 64;
                out.t8 = std::move(t8);
                return;
            }
            doc_sort_flags = overflow;
            out.doc_sort_overflow = (overflow & 1u) ? 1 : 0;   // a bucket of > 4096 suffixes: the global sort redoes the batch
            out.bkt = DevBuf<uint32_t>();
            out.bkt3 = DevBuf<uint32_t>();
            out.sym_bits = 0;
            if (in.arena) in.arena->used = arena_after_t8;   // the byte text stays
        }
    }
    if (fast && !coded && !light) encode_all();   // the global sort reads the whole byte text
    if (light) {
        // the global sort relies on the validated layout: start over with the full scan
        SaInput again = in;
        again.light_scan = 0;
        again.alphabet_sample = 0;
        if (doc_sort_flags & 1u) again.doc_sort = 0;
        t8.release();
        if (in.arena) in.arena->used = arena_mark;
        build_suffix_array(again, out, tm, s);
        if (doc_sort_flags & 1u) out.doc_sort_overflow = 1;
        return;
    }

    // buffers: ping-pong keys/values, active-list side arrays, histogram + look-back scratch
    DevBuf<uint64_t> keys_a(n, s), keys_b(n, s);
    DevBuf<uint32_t> vals_a(n, s), vals_b(n, s);
    DevBuf<uint32_t> hist(256 * RS_MAX_PASSES, s);
    DevBuf<uint8_t> scratch(rs_scratch_bytes(n, RS_MAX_PASSES), s);
    const int rr_tiles_max = (n + RR_TILE - 1) / RR_TILE;
    DevBuf<uint64_t> rr_status((size_t)rr_tiles_max + 2, s);
    DevBuf<uint32_t> rr_misc(8, s);  // [0] ticket, [1] kept count
    DevBuf<uint32_t> rank_buf(n, s);   // inverse permutation while the doubling rounds run
    uint32_t *rank = rank_buf.p;

    tm.mark("keygen0+sort0");
    int cur = 0;
    std::vector<RsTileDesc> descs;  // lives until the function's next host sync: source of an async copy
    const bool segmented = fast && in.segmented_sort && (int64_t)n / D >= 2 * RS_SEG_TILE && in.sort_batch_elems == 0;
    out.segmented = segmented ? 1 : 0;
    if (segmented) {
        // ---- per-document (segmented) sort: every tile belongs to one document, digit offsets and
        // look-back chains are per document, the document id is not part of the sorted bits
        const int sort_bits = kc * kp.b;
        kp.passes = rs_num_passes(sort_bits);
        out.key_bits = sort_bits;
        descs.reserve((size_t)n / RS_SEG_TILE + D + 1);
        for (int d = 0; d < D; ++d) {
            const int32_t e0 = in.doc_off_host[d], e1 = in.doc_off_host[d + 1];
            for (int32_t st = e0; st < e1; st += RS_SEG_TILE)
                descs.push_back(RsTileDesc{st, std::min<int32_t>(RS_SEG_TILE, e1 - st), d, e0});
        }
        const int num_tiles = (int)descs.size();
        DevBuf<RsTileDesc> d_descs(descs.size(), s);
        EAST_CUDA(cudaMemcpyAsync(d_descs.p, descs.data(), sizeof(RsTileDesc) * descs.size(), cudaMemcpyHostToDevice, s));
        DevBuf<uint32_t> hist_seg((size_t)D * kp.passes * 256, s);
        EAST_CUDA(cudaMemsetAsync(hist_seg.p, 0, sizeof(uint32_t) * (size_t)D * kp.passes * 256, s));
        const int blocks = std::min(num_tiles, EAST_NUM_SMS * 4);
        const int per_block = (num_tiles + blocks - 1) / blocks;
        EAST_BYTES(13.0 * n);
        EAST_LAUNCH(k_keygen0_fast_seg, (num_tiles + per_block - 1) / per_block, KG_THREADS, 0, s, t8.p, n, d_descs.p,
                    num_tiles, per_block, kp, keys_a.p, vals_a.p, hist_seg.p);
        DevBuf<uint8_t> seg_scratch(((size_t)num_tiles * 256 * kp.passes + 64) * sizeof(uint32_t), s);
        cur = radix_sort_pairs_segmented(keys_a.p, keys_b.p, vals_a.p, vals_b.p, sort_bits, d_descs.p, num_tiles, n,
                                         hist_seg.p, D, seg_scratch.p, s);
    } else {
    // Global sort (document id on top of the key).  It may be cut into batches of 2^g whole
    // documents (option sort_batch_elems): inside a batch only the low g bits of the id vary.
    // Measured on B200: batching is a LOSS (every launch pays ~13 us of ramp-up/tail and the kernel
    // is latency- not bandwidth-bound), so the default sorts the whole batch at once.
    int g = dbits;
    {
        const int64_t target = in.sort_batch_elems > 0 ? in.sort_batch_elems : (int64_t)n;
        const int64_t avg = std::max<int64_t>(1, (int64_t)n / D);
        int want = 0;
        while (want < dbits && (avg << (want + 1)) <= target) ++want;
        g = (target >= (int64_t)n) ? dbits : std::min(dbits, want);
    }
    const int sort_bits = kc * kp.b + g;
    kp.passes = rs_num_passes(sort_bits);
    out.key_bits = sort_bits;
    for (int d0 = 0; d0 < D; d0 += (1 << g)) {
        const int d1 = std::min(D, d0 + (1 << g));
        const int32_t e0 = in.doc_off_host[d0], e1 = in.doc_off_host[d1];
        const int32_t nb = e1 - e0;
        EAST_CUDA(cudaMemsetAsync(hist.p, 0, sizeof(uint32_t) * 256 * RS_MAX_PASSES, s));
        if (fast) {
            EAST_BYTES(13.0 * nb);
            EAST_LAUNCH(k_keygen0_fast, grid_for(nb, KG_TILE, 4), KG_THREADS, 0, s, t8.p, n, e0, e1, in.doc_off, D, kp,
                        keys_a.p, vals_a.p, hist.p);
        } else {
            EAST_BYTES(16.0 * nb);
            EAST_LAUNCH(k_keygen0_general, grid_for(nb, 256 * 8, 4), 256, 0, s, in.text, e0, e1, in.doc_off, D, kp,
                        keys_a.p, vals_a.p, hist.p);
        }
        cur = radix_sort_pairs(keys_a.p + e0, keys_b.p + e0, vals_a.p + e0, vals_b.p + e0, nb, sort_bits, hist.p, true,
                               scratch.p, s, in.rs_variant);
    }
    }

    // scorer acceleration (fast path): first ranks of all (document, 2-gram) buckets
    if (fast && kc >= 2 && ((size_t)D << (2 * kp.b)) <= (size_t)2 * n + 4096) {
        const size_t entries = ((size_t)D << (2 * kp.b)) + 1;
        out.bkt = take<uint32_t>(in, entries, s);
        EAST_CUDA(cudaMemsetAsync(out.bkt.p, 0xff, sizeof(uint32_t) * (entries - 1), s));
        EAST_LAUNCH(k_store_u32, 1, 1, 0, s, out.bkt.p + entries - 1, (uint32_t)n);
        out.sym_bits = kp.b;
    }
    tm.mark("rerank0");
    DevBuf<uint32_t> act_vals(n, s), act_slots(n, s), act_prim(n, s);
    DevBuf<uint32_t> nxt_vals, nxt_slots, nxt_prim;
    EAST_CUDA(cudaMemsetAsync(rr_status.p, 0, sizeof(uint64_t) * ((size_t)rr_tiles_max + 2), s));
    EAST_CUDA(cudaMemsetAsync(rr_misc.p, 0, sizeof(uint32_t) * 8, s));
    {
        const uint64_t sym_mask = (kp.b >= 64) ? ~0ull : ((1ull << kp.b) - 1ull);
        const uint64_t term = fast ? (uint64_t)kp.term : ~0ull;
        EAST_BYTES(20.0 * n);  // keys + values in, SA + rank out (active-list output is data dependent)
        EAST_LAUNCH(k_rerank<true>, rr_tiles_max, RR_THREADS, 0, s, cur ? keys_b.p : keys_a.p,
                    cur ? vals_b.p : vals_a.p, (const uint32_t *)nullptr, n, sym_mask, term, out.sa, rank,
                    act_vals.p, act_slots.p, act_prim.p, rr_status.p, rr_misc.p, rr_misc.p + 1, out.bkt.p,
                    (kc - 2) * kp.b, (const uint32_t *)nullptr);
        if (out.bkt.p) {
            EAST_LAUNCH(k_bucket_fill, D, 256, 0, s, out.bkt.p, 1 << (2 * kp.b), in.doc_off);
        }
    }
    uint32_t n_act = 0;
    EAST_CUDA(cudaMemcpyAsync(&n_act, rr_misc.p + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaStreamSynchronize(s));
    out.active_after_round0 = n_act;

    const int sb = bits_for((uint64_t)n);          // secondary: rank (+1 on the general path) <= n
    const int pbits = bits_for((uint64_t)n - 1);   // primary: a rank
    int rounds = 1;
    int64_t h = kc;
    tm.mark("doubling");
    if (n_act > 0) {
        nxt_vals = DevBuf<uint32_t>(n_act, s);
        nxt_slots = DevBuf<uint32_t>(n_act, s);
        nxt_prim = DevBuf<uint32_t>(n_act, s);
    }
    while (n_act > 0) {
        if (rounds > 64) throw Error(-2, "prefix doubling did not converge");
        if (h >= n) throw Error(-2, "prefix doubling ran past the text (malformed input?)");
        const int nbits = sb + pbits;
        const int passes = rs_num_passes(nbits);
        const int rr_tiles = ((int)n_act + RR_TILE - 1) / RR_TILE;
        // rank-in-group costs O(g) reads per element: a win for the late rounds (tiny groups, and each
        // avoided radix launch saves ~13 us of fixed cost), a loss for the first doubling round of
        // Zipf text, where the occurrences of frequent words still form groups of several hundred
        bool local = in.local_group_sort != 0 && n_act <= (1u << 20);
        while (true) {
            EAST_CUDA(cudaMemsetAsync(hist.p, 0, sizeof(uint32_t) * 256 * RS_MAX_PASSES, s));
            EAST_CUDA(cudaMemsetAsync(rr_status.p, 0, sizeof(uint64_t) * ((size_t)rr_tiles + 2), s));
            EAST_CUDA(cudaMemsetAsync(rr_misc.p, 0, sizeof(uint32_t) * 8, s));
            EAST_BYTES(20.0 * n_act);  // value + primary in, one rank gather, key out
            EAST_LAUNCH(k_keygen_h, grid_for(n_act, 256 * 4, 8), 256, 0, s, act_vals.p, act_prim.p, (int32_t)n_act,
                        rank, (int32_t)h, sb, local ? 0 : passes, fast ? 0 : 1, in.doc_off, D, keys_a.p, hist.p);
            const uint64_t *sk;
            const uint32_t *sv;
            if (local) {
                EAST_BYTES(24.0 * n_act);
                EAST_LAUNCH(k_group_sort, grid_for(n_act, 256, 16), 256, 0, s, keys_a.p, act_vals.p, (int32_t)n_act, sb,
                            keys_b.p, vals_b.p, rr_misc.p + 2);
                sk = keys_b.p; sv = vals_b.p;
            } else {
                // values to sort along: the suffix index
                int c2 = radix_sort_pairs(keys_a.p, keys_b.p, act_vals.p, vals_b.p, (int32_t)n_act, nbits, hist.p, true,
                                          scratch.p, s, in.rs_variant);
                sk = c2 ? keys_b.p : keys_a.p;
                sv = c2 ? vals_b.p : act_vals.p;
            }
            EAST_BYTES(24.0 * n_act);
            EAST_LAUNCH(k_rerank<false>, rr_tiles, RR_THREADS, 0, s, sk, sv, act_slots.p, (int32_t)n_act, 0ull, 0ull,
                        out.sa, rank, nxt_vals.p, nxt_slots.p, nxt_prim.p, rr_status.p, rr_misc.p, rr_misc.p + 1,
                        (uint32_t *)nullptr, 0, local ? rr_misc.p + 2 : (const uint32_t *)nullptr);
            uint32_t res[2] = {0u, 0u};  // kept count, overflow flag
            EAST_CUDA(cudaMemcpyAsync(res, rr_misc.p + 1, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
            EAST_CUDA(cudaStreamSynchronize(s));
            if (local && res[1] != 0u) { local = false; ++out.radix_fallback_rounds; continue; }  // a huge group: radix this round
            n_act = res[0];
            break;
        }
        std::swap(act_vals, nxt_vals);
        std::swap(act_slots, nxt_slots);
        std::swap(act_prim, nxt_prim);
        h *= 2;
        ++rounds;
    }
    out.rounds = rounds;
    out.t8 = std::move(t8);
}

}  // namespace east
