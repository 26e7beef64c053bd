// doc_sort.cu -- suffix array, LCP, child table, annotation (and keyphrase scores) of every SMALL document by one CTA that keeps
// the document in shared memory (B200: 227 KB per CTA hold the text, the bucket counters and the scratch).
//
// Replaces east/asts/easa.py:141-331 (_compute_suftab, _compute_lcptab, _compute_childtab,
// _compute_childtab_next_l_index, _compute_anntab) for batches whose documents have at most 65 535 code
// points each (BASELINE configs 1, 2, 4, 5: 10-50 KB texts) on the terminator-class fast path.  Larger
// documents keep the global prefix-doubling sort of sa_build.cu and the table kernels of tables.cu.
//
// Order being computed (equal to the code point order of the reference because dense codes are
// monotone and every terminator 0x0A00+i sorts above all text): compare symbol by symbol, all
// terminators share the top code `term`; two suffixes that agree up to and including their first
// terminator differ only in WHICH terminator they reach = string index = text position.
//
// Phases of one CTA (document of n code points, b bits per symbol, G = symbols per bucket id):
//   1  stage the byte-coded text in shared memory (128-bit loads); the suffixes that ARE a terminator form
//      the last bucket and are placed at once (rank = string index); the terminator layout the later phases
//      rely on is validated here (a bad one raises flag bit 1: the host takes the general path)
//   2  histogram of the G-gram bucket ids (window cut after the first terminator): packed 16-bit
//      shared-memory counters, 8 consecutive suffixes per 16-byte window
//   3  warp-cooperative exclusive scan -> bucket starts; bitmap of the ranks where a bucket starts; work
//      list of the buckets larger than a warp; the scorer's 2-gram and 3-gram tables (first ranks)
//   4  scatter every suffix into its bucket (shared-memory cursor atomics, 4-byte global stores
//      that stay in L2)
//   5  refine the buckets of more than 32 suffixes level by level: a warp takes a bucket (<= 1024; larger
//      ones a group of 4 warps) from a shared work counter, skips the prefix all members share (SWAR compare
//      against the first member), counting-sorts the members on the first symbol that differs, marks the new
//      bucket starts and queues what is still larger than a warp; a bucket whose members are identical up to
//      their terminator is sorted by position (register bitonic network)
//   6  buckets of <= 32 suffixes: a warp takes a window of 32 ranks and every suffix ranks itself inside its
//      own bucket by counting the smaller members; keys are the next 8 symbols (raw bytes, byte-reversed),
//      ties go to a byte-wise SWAR comparison of the shared-memory text (or to the position)
//   7  LCP of neighbouring suffixes (SWAR on the staged text), 16-bit copy + min-pyramid in the freed scratch,
//      per-rank key bytes for the scorer
//   8  child table and annotation from PSE / NSV (previous smaller-or-equal, next smaller LCP value) in closed form: a
//      warp takes tiles of 32 ranks, one lane per rank; bit-plane ballots resolve PSE and NSV inside the tile, the
//      neighbouring tiles (in registers) or the min-pyramid (one ballot per level) the rest, one query at a time.  Every
//      warp zero-fills up / down / next of its range right before its tiles store sparsely into it (the lines reach HBM
//      once) and stores ann densely; stores into other warps' ranges are queued and made after a barrier.
//      (EAST_DOC_SORT_STACK_WALK=1: per-thread chunks walked with the reference's stack discipline, what lies outside a
//      chunk searched in the pyramid afterwards, farthest first)
//   9  (optional: east_table_host / east_table_dev) score every distinct query suffix against the document
//      (easa.py:91-139; walks of score_walk.cuh) from a copy of text + suffix array in the freed shared memory,
//      then add the results up per keyphrase: the CTA writes its row of the score table (k_doc_suffix_sort_groups: the
//      best variant of each group of synonym variants); k_doc_suffix_sort_graph / _groups_graph store the document's
//      column of relevance bytes (score >= threshold) of a keyphrase graph instead of the row.
// A bucket of more than 4096 suffixes raises flag bit 0: the host redoes the batch with the global sort.  A
// document the kernel gives up on gets empty bucket rows (and, for a bad layout, an in-range suffix array), so
// that a caller that scores speculatively stays inside the arrays.
#include <cstdlib>
#include "sa_build.h"
#include "score_walk.cuh"

namespace east {

constexpr int DS_THREADS = 1024;
constexpr int DS_WARPS = DS_THREADS / 32;
constexpr int DS_GROUP = 128;                       // threads of a bucket-refining group
constexpr int DS_GWARPS = DS_GROUP / 32;
constexpr int DS_NGROUPS = DS_THREADS / DS_GROUP;   // 8
constexpr int DS_REFINE_MAX = 4096;                 // largest bucket a group refines
constexpr int DS_SUB_BINS = 1024;                   // bins of one refinement level (S2 * b <= 10 bits)
constexpr int DS_GRP_BYTES = DS_REFINE_MAX * 2 + DS_SUB_BINS * 4;   // staged positions + bin counters: 12 KB
constexpr int DS_SCR_BYTES = DS_NGROUPS * DS_GRP_BYTES;             // 96 KB (>= 64 KB of phase-2 counters)
constexpr int DS_WARP_MAX = 1024;                   // largest bucket one warp refines (one symbol per level)
constexpr int DS_WARP_BYTES = DS_WARP_MAX * 2 + 128 * 4;   // per-warp scratch: staged positions + <= 128 bin counters
constexpr int DS_LIST_CAP = 2048;                   // >= 65535 / 33 buckets can be larger than a warp
constexpr int DS_WIN_BYTES = 64 * 8 + 64 * 4;       // per-warp window scratch: 64 keys + 64 positions
constexpr int DS_INF = 0x7fffffff;
static_assert(DS_WARPS * DS_WARP_BYTES <= DS_SCR_BYTES && DS_WARPS * DS_WIN_BYTES <= DS_SCR_BYTES, "scratch");
static_assert(8 * DocScore::MAX_GROUPS <= DS_SCR_BYTES, "phase 9 keeps the groups' maxima in shared memory");

struct DocSortParams {
    const uint8_t *t8;        // byte-coded text of the batch (n + 128 bytes allocated)
    const uint32_t *text;     // code points of the batch (only the terminators are read: string index)
    const int32_t *doc_off;
    const int32_t *doc_m;     // strings (= terminators) per document
    int32_t *sa;              // out: global text positions in suffix order, doc-major
    uint32_t *bkt;            // out (optional): first global rank of every (document, 2-gram)
    uint32_t *bkt3;           // out (optional, G == 3): first global rank of every (document, 3-gram) = bucket
    uint32_t *overflow;       // out: set when a bucket exceeds DS_REFINE_MAX
    int b, G, S2;             // bits per symbol, symbols per bucket id, symbols per refinement level
    uint32_t term;            // terminator class code
    int text_cap;             // bytes reserved for the staged text
    int bits_words;           // words of the bucket-start bitmap
    int doc_begin;            // first document of this launch (CTA x sorts document doc_begin + x)
    unsigned long long *phase_clk;  // optional (profiling, 17 counters): SM cycles per phase, summed over the CTAs; phase-8 counts
    // optional fused tables (all or none): LCP (easa.py:247-266), child table (:268-304), annotation (:306-331);
    // every entry of the documents of the launch is written (the kernel zero-fills what phase 8 does not set)
    int32_t *lcp, *up, *down, *next, *ann;
    uint32_t *sk;             // optional: the 4 text bytes at offsets 2..5 of every suffix, in rank order (scorer)
    DocScore score;           // optional (recs != nullptr; needs bkt and sk): score the keyphrases against the document
    // optional (code_table != nullptr): the kernel byte-codes its document itself from the code points (phase 1)
    // and writes the codes to t8_out = t8; *miss is set when a code point below 0x0A00 has no code
    const uint8_t *code_table;
    uint8_t *t8_out;
    uint32_t *miss;
    int64_t text_len;         // code points of the whole batch (bound of the 128-bit loads)
    // optional (with code_table): the text arrives as ONE BYTE per code point (east_*_host_u8: code points < 0xFF as
    // themselves, 0xFF = end of a string); the kernel byte-codes from it and writes the code points -- the k-th 0xFF of
    // the document becomes the terminator 0x0A00 + k -- to text_out (= text) for the later readers of the index
    const uint8_t *text8;
    uint32_t *text_out;
    int fill_early;           // tuning / A-B: zero-fill the child and annotation slices at the start of phase 7 (round 1)
    int stack_walk;           // A-B / tests: phase 8 by per-thread stack walks over chunks (round 2) instead of tiles of 32 ranks
};

// 8 bytes of shared memory at an arbitrary byte offset from a 16-byte aligned base: three aligned
// 32-bit loads and two funnel shifts (64-bit variable shifts cost several instructions each)
__device__ __forceinline__ uint64_t ds_lds8(const uint8_t *base, int o) {
    const uint32_t *q = reinterpret_cast<const uint32_t *>(base + (o & ~3));
    const uint32_t sh = (uint32_t)(o & 3) * 8u;
    const uint32_t w0 = q[0], w1 = q[1], w2 = q[2];
    return ((uint64_t)__funnelshift_r(w1, w2, sh) << 32) | __funnelshift_r(w0, w1, sh);
}
__device__ __forceinline__ uint32_t ds_lds4(const uint8_t *base, int o) {
    const uint32_t *q = reinterpret_cast<const uint32_t *>(base + (o & ~3));
    return __funnelshift_r(q[0], q[1], (uint32_t)(o & 3) * 8u);
}

// 0x80 in every zero byte of v (exact for every byte, unlike the borrow trick below)
__device__ __forceinline__ uint32_t ds_zero4(uint32_t v) {
    return ~(((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v | 0x7f7f7f7fu);
}

__device__ __forceinline__ uint64_t ds_haszero(uint64_t v) {
    return (v - 0x0101010101010101ull) & ~v & 0x8080808080808080ull;
}

// bucket id from the first nsym <= 4 symbols held in the low bytes of w, cut after the first terminator
__device__ __forceinline__ uint32_t ds_id_from_word(uint32_t w, uint32_t term4, int b, int nsym) {
    const uint32_t z = ds_zero4(w ^ term4) & (0xffffffffu >> (8 * (4 - nsym)));
    if (z) w &= 0xffffffffu >> (8 * (3 - ((__ffs(z) - 1) >> 3)));
    const uint32_t s0 = w & 0xffu, s1 = (w >> 8) & 0xffu, s2 = (w >> 16) & 0xffu, s3 = w >> 24;
    switch (nsym) {   // uniform: no variable-shift loop
        case 1: return s0;
        case 2: return (s0 << b) | s1;
        case 3: return (((s0 << b) | s1) << b) | s2;
        default: return (((((s0 << b) | s1) << b) | s2) << b) | s3;
    }
}

// bucket id of the suffix at byte offset o: its first nsym symbols, cut after the first terminator
__device__ __forceinline__ uint32_t ds_bucket(const uint8_t *s_raw, int o, uint64_t term8, int b, int nsym) {
    if (nsym <= 4) return ds_id_from_word(ds_lds4(s_raw, o), (uint32_t)term8, b, nsym);
    uint64_t x = ds_lds8(s_raw, o);
    const uint64_t z = ds_haszero(x ^ term8);
    if (z) {
        const int k = (__ffsll((long long)z) - 1) >> 3;  // byte index of the first terminator
        if (k < 7) x &= (1ull << (8 * (k + 1))) - 1ull;
    }
    uint32_t id = 0;
    for (int g = 0; g < nsym; ++g) id = (id << b) | (uint32_t)((x >> (8 * g)) & 0xffull);
    return id;
}

// bucket ids of 8 consecutive suffixes starting at byte offset o (one 16-byte window, shared loads)
struct Ids8 { uint32_t id[8]; };
__device__ __forceinline__ Ids8 ds_bucket8(const uint8_t *s_raw, int o, uint64_t term8, int b, int nsym) {
    Ids8 r;
    if (nsym <= 4) {
        const uint64_t x0 = ds_lds8(s_raw, o), x1 = ds_lds8(s_raw, o + 8);
        const uint32_t W[4] = {(uint32_t)x0, (uint32_t)(x0 >> 32), (uint32_t)x1, (uint32_t)(x1 >> 32)};
#pragma unroll
        for (int j = 0; j < 8; ++j)
            r.id[j] = ds_id_from_word(__funnelshift_r(W[j >> 2], W[(j >> 2) + 1], (uint32_t)(j & 3) * 8u), (uint32_t)term8, b, nsym);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) r.id[j] = ds_bucket(s_raw, o + j, term8, b, nsym);
    }
    return r;
}

// does a bucket id of nsym symbols contain the terminator (then all its members are identical)
__device__ __forceinline__ bool ds_id_has_term(uint32_t id, int nsym, int b, uint32_t term) {
    const uint32_t mask = (1u << b) - 1u;
    bool t = false;
    for (int g = 0; g < nsym; ++g) t = t || (((id >> (g * b)) & mask) == term);
    return t;
}

// window key of the suffix at byte offset o: symbols [G, G+8) of its cut window as raw bytes, first
// symbol in the top byte.  0 when the terminator is among the first G symbols.
__device__ __forceinline__ uint64_t ds_key8(const uint8_t *s_raw, int o, uint64_t term8, int G) {
    const uint64_t x0 = ds_lds8(s_raw, o), x1 = ds_lds8(s_raw, o + 8);
    if (ds_haszero(x0 ^ term8) & ((1ull << (8 * G)) - 1ull)) return 0ull;
    uint64_t y = (x0 >> (8 * G)) | (x1 << (64 - 8 * G));   // 1 <= G <= 7
    const uint64_t z = ds_haszero(y ^ term8);
    if (z) {
        const int k = (__ffsll((long long)z) - 1) >> 3;
        if (k < 7) y &= (1ull << (8 * (k + 1))) - 1ull;
    }
    const uint32_t hi = __byte_perm((uint32_t)y, 0u, 0x0123), lo = __byte_perm((uint32_t)(y >> 32), 0u, 0x0123);
    return ((uint64_t)hi << 32) | lo;
}

// suffixes at byte offsets oi, oj agree on [0, from) and have no terminator there: is i < j ?
__device__ __forceinline__ bool ds_deep_less(const uint8_t *s_raw, int oi, int oj, int from, uint64_t term8) {
    int o = from;
    while (true) {
        const uint64_t x = ds_lds8(s_raw, oi + o), y = ds_lds8(s_raw, oj + o);
        const uint64_t stop = (x ^ y) | ds_haszero(x ^ term8);
        if (stop) {
            const int sh = (__ffsll((long long)stop) - 1) & ~7;
            const uint32_t bx = (uint32_t)(x >> sh) & 0xffu, by = (uint32_t)(y >> sh) & 0xffu;
            if (bx != by) return bx < by;
            return oi < oj;  // both reach their terminator here: the earlier string comes first
        }
        o += 8;
    }
}

__device__ __forceinline__ void ds_group_sync(int id) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(DS_GROUP) : "memory");
}


struct DocCtx {
    const uint8_t *s_raw;
    int shift;
    uint64_t term8;
    uint32_t term;
    int b, S2;
    int32_t base;
    int32_t *sa_doc;
    uint32_t *s_bits;
    uint32_t *overflow;
};

// rank the members of a bucket whose suffixes are identical up to their terminator by position:
// every member counts the members that start earlier (positions staged as 16-bit values)
__device__ __forceinline__ void ds_rank_by_position(const DocCtx &c, const uint16_t *pos, int start, int size, int t, int nthr) {
    const uint32_t *p2 = reinterpret_cast<const uint32_t *>(pos);
    for (int e = t; e < size; e += nthr) {
        const uint32_t pe = pos[e];
        int below = 0;
        for (int q = 0; q < (size >> 1); ++q) {
            const uint32_t v = p2[q];
            below += ((v & 0xffffu) < pe ? 1 : 0) + ((v >> 16) < pe ? 1 : 0);
        }
        if ((size & 1) && pos[size - 1] < pe) ++below;
        c.sa_doc[start + below] = c.base + (int32_t)pe;
    }
}

// The same for buckets of <= 32 E members by ONE warp without the quadratic count: a bitonic sorting network
// over E registers per lane (element e = r * 32 + lane; partners 32 or more apart are registers of the same
// lane, closer ones come by shuffle).  Sorted positions leave as coalesced stores.
template <int E>
__device__ __forceinline__ void ds_sort_by_position(const DocCtx &c, const uint16_t *pos, int start, int size, int lane) {
    uint32_t v[E];
#pragma unroll
    for (int r = 0; r < E; ++r) { const int e = r * 32 + lane; v[r] = e < size ? (uint32_t)pos[e] : 0xffffffffu; }
#pragma unroll
    for (int k = 2; k <= 32 * E; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int jr = j >> 5;
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    if ((r & jr) == 0) {
                        const bool up = ((r * 32) & k) == 0;
                        const uint32_t a = v[r], b = v[r | jr];
                        v[r] = up ? min(a, b) : max(a, b);
                        v[r | jr] = up ? max(a, b) : min(a, b);
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < E; ++r) {
                    const uint32_t o = __shfl_xor_sync(0xffffffffu, v[r], j);
                    const bool up = (((r * 32) | lane) & k) == 0;
                    const bool lower = (lane & j) == 0;
                    v[r] = (up == lower) ? min(v[r], o) : max(v[r], o);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < E; ++r) { const int e = r * 32 + lane; if (e < size) c.sa_doc[start + e] = c.base + (int32_t)v[r]; }
}

// symbols the members share beyond `depth` (DS_INF: all members are the same string tail), as seen
// by this thread's members e = t, t + nthr, ...: compare everybody with member 0
__device__ __forceinline__ int ds_common_prefix(const DocCtx &c, const uint16_t *pos, int size, int depth, int t, int nthr) {
    const int o0 = c.shift + (int)pos[0] + depth;
    int cp = DS_INF;
    for (int e = t; e < size; e += nthr) {
        const int oi = c.shift + (int)pos[e] + depth;
        int k = 0;
        while (k < cp) {
            const uint64_t x = ds_lds8(c.s_raw, oi + k), y = ds_lds8(c.s_raw, o0 + k);
            const uint64_t stop = (x ^ y) | ds_haszero(y ^ c.term8);
            if (stop) {
                const int j = (__ffsll((long long)stop) - 1) >> 3;
                if (((x >> (8 * j)) & 0xffull) != ((y >> (8 * j)) & 0xffull)) cp = min(cp, k + j);
                break;  // else: identical up to and including the terminator
            }
            k += 8;
        }
    }
    return cp;
}

// One refinement step of one bucket of <= DS_WARP_MAX suffixes by ONE warp: skip the shared prefix,
// counting-sort on the first symbol that differs (2^b <= 128 bins), no block-level barrier.
__device__ void ds_refine_warp(const DocCtx &c, uint2 entry, int lane, uint8_t *wscr, uint2 *next_list, uint32_t *next_n) {
    const int start = (int)(entry.x & 0xffffu), size = (int)(entry.x >> 16);
    const int depth = (int)(entry.y & 0xffffu);
    bool terminal = (entry.y >> 16) != 0u;
    uint16_t *wpos = reinterpret_cast<uint16_t *>(wscr);
    uint32_t *whist = reinterpret_cast<uint32_t *>(wscr + DS_WARP_MAX * 2);
    const int NB1 = 1 << c.b;

    for (int e = lane; e < size; e += 32) wpos[e] = (uint16_t)(c.sa_doc[start + e] - c.base);
    for (int i = lane; i < NB1; i += 32) whist[i] = 0;
    __syncwarp();
    int d2 = depth;
    if (!terminal) {
        const int cp = __reduce_min_sync(0xffffffffu, ds_common_prefix(c, wpos, size, depth, lane, 32));
        if (cp == DS_INF) terminal = true;
        else d2 = depth + cp;
    }
    if (terminal) {
        if (size <= 64) ds_sort_by_position<2>(c, wpos, start, size, lane);
        else if (size <= 128) ds_sort_by_position<4>(c, wpos, start, size, lane);
        else if (size <= 256) ds_sort_by_position<8>(c, wpos, start, size, lane);
        else ds_rank_by_position(c, wpos, start, size, lane, 32);
        __syncwarp();
        return;
    }
    for (int e = lane; e < size; e += 32) atomicAdd(&whist[c.s_raw[c.shift + (int)wpos[e] + d2]], 1u);
    __syncwarp();
    uint32_t run = 0;
    for (int i0 = 0; i0 < NB1; i0 += 32) {
        const int i = i0 + lane;
        const uint32_t cnt = (i < NB1) ? whist[i] : 0u;
        uint32_t x = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        const uint32_t excl = run + x - cnt;
        if (i < NB1) whist[i] = excl;  // scatter cursor
        if (cnt) {
            const uint32_t r = (uint32_t)start + excl;
            if (excl) atomicOr(&c.s_bits[r >> 5], 1u << (r & 31));
            if (cnt > 32u) {
                const uint32_t slot = atomicAdd(next_n, 1u);
                if (slot < (uint32_t)DS_LIST_CAP)
                    next_list[slot] = make_uint2(r | (cnt << 16), (uint32_t)(d2 + 1) | (((uint32_t)i == c.term ? 1u : 0u) << 16));
            }
        }
        run += __shfl_sync(0xffffffffu, x, 31);
    }
    __syncwarp();
    for (int e = lane; e < size; e += 32) {
        const uint32_t pe = wpos[e];
        const uint32_t r = atomicAdd(&whist[c.s_raw[c.shift + (int)pe + d2]], 1u);
        c.sa_doc[start + (int)r] = c.base + (int32_t)pe;
    }
    __syncwarp();
}

// One refinement step of one bucket by one group of DS_GROUP threads (gt = thread index in the group,
// g = group index).  entry: x = start | size << 16, y = depth | terminal << 16.
__device__ void ds_refine(const DocCtx &c, uint2 entry, int g, int gt, uint8_t *gscr, int *s_gmin, uint32_t *s_gw,
                          uint2 *next_list, uint32_t *next_n) {
    const int start = (int)(entry.x & 0xffffu), size = (int)(entry.x >> 16);
    const int depth = (int)(entry.y & 0xffffu);
    bool terminal = (entry.y >> 16) != 0u;
    uint16_t *gpos = reinterpret_cast<uint16_t *>(gscr);
    uint32_t *ghist = reinterpret_cast<uint32_t *>(gscr + DS_REFINE_MAX * 2);
    const int lane = gt & 31, gw = gt >> 5;
    const int NB2 = 1 << (c.S2 * c.b);

    for (int e = gt; e < size; e += DS_GROUP) gpos[e] = (uint16_t)(c.sa_doc[start + e] - c.base);
    if (!terminal) for (int i = gt; i < NB2; i += DS_GROUP) ghist[i] = 0;
    if (gt == 0) s_gmin[g] = DS_INF;
    ds_group_sync(1 + g);

    int d2 = depth;
    if (!terminal) {
        const int mycp = __reduce_min_sync(0xffffffffu, ds_common_prefix(c, gpos, size, depth, gt, DS_GROUP));
        if (lane == 0 && mycp != DS_INF) atomicMin(&s_gmin[g], mycp);
        ds_group_sync(1 + g);
        const int cp = s_gmin[g];
        if (cp == DS_INF) terminal = true;  // every member is the same string tail: order by position
        else d2 = depth + cp;
    }

    if (terminal) {
        ds_rank_by_position(c, gpos, start, size, gt, DS_GROUP);
        ds_group_sync(1 + g);
        return;
    }

    // counting sort on the S2 symbols at offset d2
    for (int e = gt; e < size; e += DS_GROUP)
        atomicAdd(&ghist[ds_bucket(c.s_raw, c.shift + (int)gpos[e] + d2, c.term8, c.b, c.S2)], 1u);
    ds_group_sync(1 + g);
    {
        const int PB = (NB2 + DS_GROUP - 1) / DS_GROUP;
        const int b0 = min(NB2, gt * PB), b1 = min(NB2, b0 + PB);
        uint32_t sum = 0;
        for (int i = b0; i < b1; ++i) sum += ghist[i];
        uint32_t x = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_gw[g * DS_GWARPS + gw] = x;
        ds_group_sync(1 + g);
        uint32_t run = x - sum;
        for (int i = 0; i < gw; ++i) run += s_gw[g * DS_GWARPS + i];
        for (int i = b0; i < b1; ++i) {
            const uint32_t cnt = ghist[i];
            ghist[i] = run;  // scatter cursor
            if (cnt) {
                const uint32_t r = (uint32_t)start + run;
                if (run) atomicOr(&c.s_bits[r >> 5], 1u << (r & 31));
                if (cnt > 32u) {
                    const uint32_t slot = atomicAdd(next_n, 1u);
                    const uint32_t term_flag = ds_id_has_term((uint32_t)i, c.S2, c.b, c.term) ? 1u : 0u;
                    if (slot < (uint32_t)DS_LIST_CAP)
                        next_list[slot] = make_uint2(r | (cnt << 16), (uint32_t)(d2 + c.S2) | (term_flag << 16));
                }
            }
            run += cnt;
        }
    }
    ds_group_sync(1 + g);
    for (int e = gt; e < size; e += DS_GROUP) {
        const uint32_t pe = gpos[e];
        const uint32_t r = atomicAdd(&ghist[ds_bucket(c.s_raw, c.shift + (int)pe + d2, c.term8, c.b, c.S2)], 1u);
        c.sa_doc[start + (int)r] = c.base + (int32_t)pe;
    }
    ds_group_sync(1 + g);
}

// min-pyramid over the document's LCP values in shared memory (16-bit: lcp < n <= 65535):
// lv[0] = lcp, lv[k+1][i] = min(lv[k][32 i .. 32 i + 31])
struct SPyr {
    const uint16_t *lcp;    // level 0
    const int *off;         // shared memory: element offset of level k from lcp
    const int *size_;       // shared memory: entries of level k
    int levels;
    __device__ __forceinline__ const uint16_t *lv(int k) const { return lcp + off[k]; }
    __device__ __forceinline__ int size(int k) const { return size_[k]; }
};

// largest q < p with lcp[q] <= l (exists: lcp[0] = 0)
__device__ __forceinline__ int ds_prev_le(const SPyr &M, int p, uint32_t l) {
    int idx = p, level = 0, j;
    while (true) {
        const int gs = idx & ~31;
        const uint16_t *a = M.lv(level);
        for (j = idx - 1; j >= gs; --j)
            if (a[j] <= l) goto found;
        idx >>= 5;
        ++level;
        if (level >= M.levels) return 0;
    }
found:
    while (level > 0) {
        --level;
        const uint16_t *a = M.lv(level);
        int c = min(j * 32 + 31, M.size(level) - 1);
        while (a[c] > l) --c;
        j = c;
    }
    return j;
}

// smallest e > p with lcp[e] < l, or n
__device__ __forceinline__ int ds_next_lt(const SPyr &M, int p, uint32_t l, int n) {
    int idx = p, level = 0, j;
    while (true) {
        const int ge = min((idx | 31) + 1, M.size(level));
        const uint16_t *a = M.lv(level);
        for (j = idx + 1; j < ge; ++j)
            if (a[j] < l) goto found;
        idx >>= 5;
        ++level;
        if (level >= M.levels) return n;
    }
found:
    while (level > 0) {
        --level;
        const uint16_t *a = M.lv(level);
        int c = j * 32;
        while (a[c] >= l) ++c;
        j = c;
    }
    return j;
}

// The same two searches by a whole warp for the lane-per-rank path of phase 8 (level, idx and l uniform): every level,
// on the way up and on the way down, is one coalesced load of 32 entries and one ballot instead of a scan by one lane.
// They start above level 0 (the tile itself is resolved by the caller).  cnt (profiling, else nullptr): queries
// counted by the level at which they found their block, cnt[levels] = not found.
// largest q with lcp[q] <= l before entry idx of `level` (0 if none)
__device__ __forceinline__ int ds_warp_prev_le(const SPyr &M, int level, int idx, uint32_t l, int lane, uint32_t *cnt) {
    int j;
    while (true) {
        const int g0 = idx & ~31;
        const uint32_t v = lane < (idx & 31) ? M.lv(level)[g0 + lane] : 0xffffffffu;
        const uint32_t B = __ballot_sync(0xffffffffu, v <= l);
        if (B) { j = g0 + 31 - __clz(B); break; }
        idx >>= 5;
        if (++level >= M.levels) { if (cnt && lane == 0) atomicAdd(&cnt[level], 1u); return 0; }
    }
    if (cnt && lane == 0) atomicAdd(&cnt[level], 1u);
    while (level > 0) {   // the block holds such an entry: the last one of its 32 children that does
        --level;
        const int i = j * 32 + lane;
        const uint32_t v = i < M.size(level) ? M.lv(level)[i] : 0xffffffffu;
        j = j * 32 + 31 - __clz(__ballot_sync(0xffffffffu, v <= l));
    }
    return j;
}

// smallest e with lcp[e] < l after entry idx of `level`, or n
__device__ __forceinline__ int ds_warp_next_lt(const SPyr &M, int level, int idx, uint32_t l, int n, int lane, uint32_t *cnt) {
    int j;
    while (true) {
        const int g0 = idx & ~31, i = g0 + lane;
        const uint32_t v = (lane > (idx & 31) && i < M.size(level)) ? M.lv(level)[i] : 0xffffffffu;
        const uint32_t B = __ballot_sync(0xffffffffu, v < l);
        if (B) { j = g0 + __ffs(B) - 1; break; }
        idx >>= 5;
        if (++level >= M.levels) { if (cnt && lane == 0) atomicAdd(&cnt[level], 1u); return n; }
    }
    if (cnt && lane == 0) atomicAdd(&cnt[level], 1u);
    while (level > 0) {   // the first of the block's children that holds such an entry
        --level;
        const int i = j * 32 + lane;
        const uint32_t v = i < M.size(level) ? M.lv(level)[i] : 0xffffffffu;
        j = j * 32 + __ffs(__ballot_sync(0xffffffffu, v < l)) - 1;
    }
    return j;
}

// empty 2-gram / 3-gram bucket tables of a document the kernel gives up on
__device__ __forceinline__ void ds_clear_tables(const DocSortParams &p, int doc, int b, int tid) {
    if (p.bkt) {
        uint32_t *row = p.bkt + ((size_t)doc << (2 * b));
        for (int i = tid; i < (1 << (2 * b)); i += DS_THREADS) row[i] = 0u;
    }
    if (p.bkt3) {
        uint32_t *row = p.bkt3 + ((size_t)doc << (3 * b));
        for (int i = tid; i < (1 << (3 * b)); i += DS_THREADS) row[i] = 0u;
    }
}

// Phase 9 of a synonym-expanded table: the variants' sums are taken as for a plain row, one thread per VARIANT (groups
// are 1-64 variants: a thread per group would leave most lanes idle), and each is folded into its group's maximum with
// a 64-bit shared-memory atomicMax on the bits of the double.  Scores are >= +0.0 and never NaN, so their bit patterns
// order as the values do and the maximum has the bits k_score_combine_max finds, whatever the order of the atomics.
// `smem` (the staged text, no longer read) holds the G running maxima.  GRAPH: the group's relevance byte instead.
template <bool GRAPH>
__device__ __forceinline__ void ds_store_group_maxima(const DocSortParams &p, uint8_t *smem, int doc, const double *out, int tid) {
    unsigned long long *s_best = reinterpret_cast<unsigned long long *>(smem);
    const int32_t G = p.score.G;
    for (int g = tid; g < G; g += DS_THREADS) s_best[g] = 0ull;
    __syncthreads();
    for (int v = tid; v < p.score.K; v += DS_THREADS) {
        const int32_t sb = __ldg(p.score.kp_off + v), se = __ldg(p.score.kp_off + v + 1);
        double result = 0.0;
        for (int32_t x = sb; x < se; ++x) result = result + __ldcg(out + __ldg(p.score.uniq_of + x));
        const double score = result / (double)(se - sb);
        atomicMax(s_best + doc_of(p.score.group_off, G, v), (unsigned long long)__double_as_longlong(score));
    }
    __syncthreads();
    if (GRAPH) {
        uint8_t *col = p.score.graph + p.score.graph_col0 + (doc - p.doc_begin);
        for (int g = tid; g < G; g += DS_THREADS)
            col[(size_t)g * (size_t)p.score.graph_pitch] = __longlong_as_double((long long)s_best[g]) >= p.score.threshold ? 1 : 0;
        return;
    }
    double *table_row = p.score.out + (size_t)(doc - p.doc_begin) * (size_t)G;
    for (int g = tid; g < G; g += DS_THREADS) {
        const double v = __longlong_as_double((long long)s_best[g]);
        table_row[g] = v;
        const size_t cell = (size_t)(doc - p.doc_begin) * (size_t)G + (size_t)g;
        for (int pi = 0; pi < p.score.n_peers; ++pi) p.score.peer_out[pi][cell] = v;
    }
    if (p.score.n_peers > 0) __threadfence_system();
}

// ---- phase 9 (optional): score the keyphrases against the document this CTA has just indexed
// (EnhancedAnnotatedSuffixArray._score, easa.py:91-139, for every distinct query suffix; score_walk.cuh).
// The CTA's shared memory is free again: the byte text and the suffix array (16-bit local positions) of the
// document are staged there, so every probe of a walk -- the binary searches over (rank -> symbol at depth d)
// -- is two shared-memory loads instead of dependent L2 / HBM round trips.  Only the bucket-table lookups that
// open a walk (one batch of loads per suffix) and the suffix records go to global memory.
// GRAPH: the CTA stores its document's column of relevance bytes instead of its row of the table (DocScore::graph).
template <bool GROUPS, bool GRAPH>
__device__ __forceinline__ void ds_score_document(const DocSortParams &p, uint8_t *smem, int smem_bytes, int doc, int32_t base, int n, int tid) {
    if (p.score.recs == nullptr) return;
    __syncthreads();   // every rank of sa and every bucket start of this document is in place; shared memory is free
    const int b = p.b;
    const uint32_t *row = p.bkt + ((size_t)doc << (2 * b));
    const uint32_t *row3 = p.bkt3 ? p.bkt3 + ((size_t)doc << (3 * b)) : nullptr;
    const int32_t m = p.doc_m[doc];
    double *out = p.score.tmp + (size_t)(doc - p.doc_begin) * (size_t)p.score.n_uniq;
    const int32_t a0 = base & ~15;
    const int shift = base - a0;
    const int text_bytes = (shift + n + 48 + 15) & ~15;   // as staged in phase 1: the walks read 8 bytes at a time
    const bool staged = text_bytes + 2 * n <= smem_bytes;
    const uint8_t *s_text = smem + shift;
    uint16_t *s_sa = reinterpret_cast<uint16_t *>(smem + text_bytes);
    if (staged) {
        for (int o = tid * 16; o < text_bytes; o += DS_THREADS * 16)
            *reinterpret_cast<uint4 *>(smem + o) = *reinterpret_cast<const uint4 *>(p.t8 + a0 + o);
        const int32_t *sa_doc = p.sa + base;
        for (int r = tid; r < n; r += DS_THREADS) s_sa[r] = (uint16_t)(sa_doc[r] - base);
        __syncthreads();
    }
    unsigned long long probes = 0;
    for (int u = tid; u < p.score.n_uniq; u += DS_THREADS) {
        const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(p.score.recs) + u);
        const uint64_t qw = ((uint64_t)raw.y << 32) | raw.x;
        const int32_t sidx = (int32_t)raw.z;
        const int32_t len = (int32_t)(raw.w & 0xffffu);
        const bool generic = ((raw.w >> 16) & 0xffu) != 0u;
        double r;
        if (generic)
            r = score_one_suffix<false, false>(p.text, p.sa, base, base + n, m, p.score.kp + sidx, len, p.score.normalized, probes);
        else if (staged)
            r = score_one_suffix_fast<false, false, uint16_t>(s_text, s_sa, nullptr, row, row3, b, base, base + n, m,
                                                              p.score.q8 + sidx, qw, len, p.score.normalized, probes, base);
        else
            r = score_one_suffix_fast<false, false>(p.t8, p.sa, p.sk, row, row3, b, base, base + n, m, p.score.q8 + sidx, qw, len,
                                                    p.score.normalized, probes);
        out[u] = r;
    }
    // the keyphrase sums: the results of the keyphrase's suffixes IN SUFFIX ORDER (the reference's fp64 order,
    // easa.py:127-134), each fetched through the position of its distinct twin -- k_score_combine's arithmetic
    __syncthreads();
    if (GROUPS) {
        ds_store_group_maxima<GRAPH>(p, smem, doc, out, tid);
        return;
    }
    if (GRAPH) {
        // the same sums; one byte per keyphrase, Dp apart (the threshold compare of k_threshold_bytes)
        uint8_t *col = p.score.graph + p.score.graph_col0 + (doc - p.doc_begin);
        for (int k = tid; k < p.score.K; k += DS_THREADS) {
            const int32_t sb = __ldg(p.score.kp_off + k), se = __ldg(p.score.kp_off + k + 1);
            double result = 0.0;
            for (int32_t x = sb; x < se; ++x) result = result + __ldcg(out + __ldg(p.score.uniq_of + x));
            col[(size_t)k * (size_t)p.score.graph_pitch] = result / (double)(se - sb) >= p.score.threshold ? 1 : 0;
        }
        return;
    }
    double *table_row = p.score.out + (size_t)(doc - p.doc_begin) * (size_t)p.score.K;
    for (int k = tid; k < p.score.K; k += DS_THREADS) {
        const int32_t sb = __ldg(p.score.kp_off + k), se = __ldg(p.score.kp_off + k + 1);
        double result = 0.0;
        for (int32_t x = sb; x < se; ++x) result = result + __ldcg(out + __ldg(p.score.uniq_of + x));
        const double v = result / (double)(se - sb);
        table_row[k] = v;
        // sharded table: the row goes to the other ranks' gathered tables as well (peer memory over NVLink) -- the
        // all-gather happens here, row by row, under the indexing of the documents still to come
        const size_t cell = (size_t)(doc - p.doc_begin) * (size_t)p.score.K + (size_t)k;
        for (int pi = 0; pi < p.score.n_peers; ++pi) p.score.peer_out[pi][cell] = v;
    }
    if (p.score.n_peers > 0) __threadfence_system();
}

// The per-document kernel; GROUPS: phase 9 writes synonym-expanded rows (G wide); GRAPH: phase 9 writes relevance bytes
// instead of rows.  Four kernels instead of a kernel template, so that the plain one keeps its name (kernel timings,
// profiles) and its register allocation.
template <bool GROUPS, bool GRAPH>
__device__ __forceinline__ void doc_suffix_sort(const DocSortParams &p) {
    extern __shared__ __align__(16) uint8_t ds_smem[];
    uint8_t *s_raw = ds_smem;                                                    // staged text
    uint32_t *s_scr = reinterpret_cast<uint32_t *>(ds_smem + p.text_cap);        // counters, later sort scratch
    uint32_t *s_bits = reinterpret_cast<uint32_t *>(ds_smem + p.text_cap + DS_SCR_BYTES);
    uint2 *s_list0 = reinterpret_cast<uint2 *>(s_bits + p.bits_words);           // bits_words is even
    uint2 *s_list1 = s_list0 + DS_LIST_CAP;
    __shared__ uint32_t s_warp_sum[DS_WARPS];
    __shared__ uint32_t s_nlist[2];
    __shared__ uint32_t s_work;
    __shared__ uint32_t s_fail;   // this document cannot be sorted here (a bucket too large)
    __shared__ uint8_t s_code[EAST_TERM_BASE];   // code point -> dense code (only when the kernel byte-codes its document)
    __shared__ int s_gmin[DS_NGROUPS];
    __shared__ uint32_t s_gw[DS_NGROUPS * DS_GWARPS];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int doc = p.doc_begin + (int)blockIdx.x;
    const int32_t base = p.doc_off[doc];
    const int n = p.doc_off[doc + 1] - base;
    const int b = p.b, G = p.G;
    const uint64_t term8 = 0x0101010101010101ull * (uint64_t)p.term;
    const int NB = 1 << (G * b);      // bucket ids
    const int NW = NB >> 1;           // counter words (two 16-bit counters each)
    const uint32_t term_bucket = p.term << ((G - 1) * b);   // the suffixes that ARE a terminator
    int32_t *sa_doc = p.sa + base;    // plain pointer: written and re-read by this CTA

    uint32_t t_prev = (uint32_t)clock();   // 32 bits (one register for the whole kernel): a phase takes < 2^32 cycles
#define DS_STAMP(k)                                                                     \
    do {                                                                                \
        if (p.phase_clk && tid == 0) {                                                  \
            const uint32_t t_now = (uint32_t)clock();                                   \
            atomicAdd(&p.phase_clk[k], (unsigned long long)(t_now - t_prev));           \
            t_prev = t_now;                                                             \
        }                                                                               \
    } while (0)

    // ---- phase 1: stage the text, clear counters / bitmap; place and VALIDATE the terminators
    const int32_t a0 = base & ~15;
    const int shift = base - a0;
    {
        const int nbytes = (shift + n + 48 + 15) & ~15;
        const int m = p.doc_m[doc];
        const uint32_t term4 = (uint32_t)term8;
        for (int k = tid; k < m; k += DS_THREADS) sa_doc[n - m + k] = -1;
        for (int i = tid; i < NW; i += DS_THREADS) s_scr[i] = 0;
        for (int i = tid; i < p.bits_words; i += DS_THREADS) s_bits[i] = 0;
        if (tid < 2) s_nlist[tid] = 0;
        if (tid == 0) { s_work = 0; s_fail = 0; }   // s_work here: number of terminator codes seen
        const bool encode = p.code_table != nullptr;
        const bool from8 = encode && p.text8 != nullptr;
        // from8: terminators of the document inside every 16-byte chunk, then their exclusive prefix (the work lists
        // are not in use yet)
        uint16_t *s_tc = reinterpret_cast<uint16_t *>(s_list0);
        if (encode)
            for (int i = tid; i < (int)EAST_TERM_BASE; i += DS_THREADS) s_code[i] = p.code_table[i];
        __syncthreads();
        int bad = 0, missed = 0;
        for (int o = tid * 16; o < nbytes; o += DS_THREADS * 16) {
            uint4 v;
            if (!encode) {
                v = *reinterpret_cast<const uint4 *>(p.t8 + a0 + o);
            } else if (from8) {
                const uint4 raw = *reinterpret_cast<const uint4 *>(p.text8 + a0 + o);   // 16 code points in one load
                const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
                uint32_t w[4];
                uint32_t cnt = 0;
#pragma unroll
                for (int wi = 0; wi < 4; ++wi) {
                    uint32_t packed = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t c = (rw[wi] >> (8 * j)) & 0xffu;
                        const uint32_t e = c == 0xffu ? p.term : (uint32_t)s_code[c];
                        const int i = o + 4 * wi + j - shift;
                        const bool inside = i >= 0 && i < n;
                        if (e == 0u && inside) missed = 1;
                        if (c == 0xffu && inside) ++cnt;
                        packed |= e << (8 * j);
                    }
                    w[wi] = packed;
                }
                s_tc[o >> 4] = (uint16_t)cnt;
                v = make_uint4(w[0], w[1], w[2], w[3]);
                const int i0 = o - shift;
                if (i0 >= 0 && i0 + 15 < n) {
                    *reinterpret_cast<uint4 *>(p.t8_out + a0 + o) = v;
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (i0 + j >= 0 && i0 + j < n) p.t8_out[base + i0 + j] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
                }
            } else {
                // 16 code points -> 16 byte codes (k_encode_text's mapping); only the document's own positions
                // count for the miss flag and are written back: its neighbours may not even be resident yet
                uint32_t w[4];
#pragma unroll
                for (int wi = 0; wi < 4; ++wi) {
                    const int64_t g = (int64_t)a0 + o + 4 * wi;
                    uint4 c4;
                    if (g + 3 < p.text_len) c4 = *reinterpret_cast<const uint4 *>(p.text + g);
                    else {
                        c4.x = g < p.text_len ? p.text[g] : EAST_TERM_BASE;
                        c4.y = g + 1 < p.text_len ? p.text[g + 1] : EAST_TERM_BASE;
                        c4.z = g + 2 < p.text_len ? p.text[g + 2] : EAST_TERM_BASE;
                        c4.w = EAST_TERM_BASE;
                    }
                    const uint32_t c[4] = {c4.x, c4.y, c4.z, c4.w};
                    uint32_t packed = 0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t e = c[j] < EAST_TERM_BASE ? (uint32_t)s_code[c[j]] : p.term;
                        const int i = o + 4 * wi + j - shift;
                        if (e == 0u && i >= 0 && i < n) missed = 1;
                        packed |= e << (8 * j);
                    }
                    w[wi] = packed;
                }
                v = make_uint4(w[0], w[1], w[2], w[3]);
                const int i0 = o - shift;
                if (i0 >= 0 && i0 + 15 < n) {
                    *reinterpret_cast<uint4 *>(p.t8_out + a0 + o) = v;
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (i0 + j >= 0 && i0 + j < n) p.t8_out[base + i0 + j] = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
                }
            }
            *reinterpret_cast<uint4 *>(s_raw + o) = v;
            // the suffixes that ARE a terminator form the last bucket (term is the top code) and are
            // ordered by string index = terminator value - 0x0A00: final right here, while the
            // loads of the code points overlap the staging
            const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
            if (from8) continue;   // placed below, once the string index of every terminator is known
#pragma unroll
            for (int wi = 0; wi < 4; ++wi) {
                uint32_t z = ds_zero4(wv[wi] ^ term4);
                while (z) {
                    const int i = o + 4 * wi + ((__ffs(z) - 1) >> 3) - shift;
                    z &= z - 1u;
                    if (i >= 0 && i < n) {
                        const uint32_t k = p.text[base + i] - EAST_TERM_BASE;
                        if (k < (uint32_t)m) sa_doc[n - m + (int)k] = base + i; else bad = 1;
                        atomicAdd(&s_work, 1u);
                    }
                }
            }
        }
        if (missed) atomicOr(p.miss, 1u);
        __syncthreads();
        if (from8) {
            // string index of a terminator = number of terminators of the document before it: block-wide exclusive
            // scan of the per-chunk counts, then a second pass places the terminators (rank = string index) and
            // writes the code points of the document
            const int nch = nbytes >> 4;
            const int per = (nch + DS_THREADS - 1) / DS_THREADS;
            const int c0 = min(nch, tid * per), c1 = min(nch, c0 + per);
            uint32_t sum = 0;
            for (int c = c0; c < c1; ++c) sum += s_tc[c];
            uint32_t x = sum;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            if (lane == 31) s_warp_sum[warp] = x;
            __syncthreads();
            uint32_t run = x - sum;
            for (int i = 0; i < warp; ++i) run += s_warp_sum[i];
            for (int c = c0; c < c1; ++c) { const uint32_t cv = s_tc[c]; s_tc[c] = (uint16_t)run; run += cv; }
            if (tid == DS_THREADS - 1) s_work = run;
            __syncthreads();
            for (int o = tid * 16; o < nbytes; o += DS_THREADS * 16) {
                const uint4 raw = *reinterpret_cast<const uint4 *>(p.text8 + a0 + o);
                const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
                uint32_t k = s_tc[o >> 4];
                uint32_t cp[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const uint32_t c = (rw[j >> 2] >> (8 * (j & 3))) & 0xffu;
                    const int i = o + j - shift;
                    cp[j] = c;
                    if (c == 0xffu && i >= 0 && i < n) {
                        if (k < (uint32_t)m) sa_doc[n - m + (int)k] = base + i; else bad = 1;
                        cp[j] = EAST_TERM_BASE + k;
                        ++k;
                    }
                }
                const int i0 = o - shift;
                if (i0 >= 0 && i0 + 15 < n) {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        *reinterpret_cast<uint4 *>(p.text_out + a0 + o + 4 * q) = make_uint4(cp[4 * q], cp[4 * q + 1], cp[4 * q + 2], cp[4 * q + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (i0 + j >= 0 && i0 + j < n) p.text_out[base + i0 + j] = cp[j];
                }
            }
            __syncthreads();
        }
        // The layout every later phase relies on (east/asts/utils.py:25-40): exactly m terminator codes,
        // string k ends with 0x0A00 + k, the document ends with its last terminator.  A build that
        // runs ahead of the validating text scan (pipelined host build) finds out here.
        if (s_work != (uint32_t)m) bad = 1;
        for (int k = tid; k < m; k += DS_THREADS) {
            const int32_t v = sa_doc[n - m + k];
            if (v < 0 || (k > 0 && sa_doc[n - m + k - 1] >= v) || (k == m - 1 && v != base + n - 1)) bad = 1;
        }
        if (__syncthreads_or(bad)) {
            if (tid == 0) atomicOr(p.overflow, 2u);
            // Nothing of this document is usable.  A caller that scores speculatively (east_table_host scores a
            // run before the host has seen the flag) must still stay inside the arrays: empty bucket tables end
            // every fast walk before its first suffix-array read, an in-range suffix array bounds the generic walk.
            for (int r = tid; r < n; r += DS_THREADS) sa_doc[r] = base + r;
            ds_clear_tables(p, doc, b, tid);
            return;
        }
    }
    __syncthreads();
    DS_STAMP(0);

    // ---- phase 2: bucket histogram
    for (int c0 = tid * 8; c0 < n; c0 += DS_THREADS * 8) {
        const Ids8 ids = ds_bucket8(s_raw, shift + c0, term8, b, G);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (c0 + j < n) atomicAdd(&s_scr[ids.id[j] >> 1], (ids.id[j] & 1u) ? 0x10000u : 1u);
    }
    __syncthreads();
    DS_STAMP(1);

    // ---- phase 3: exclusive scan of the counters.  Warp w owns WPW consecutive counter words and
    // walks them 32 at a time (lane-contiguous: no bank conflicts), carrying the running rank.
    {
        const int WPW = max(32, NW / DS_WARPS);
        const int w0 = min(NW, warp * WPW), w1 = min(NW, w0 + WPW);
        uint32_t sum = 0;
        for (int w = w0 + lane; w < w1; w += 32) { const uint32_t v = s_scr[w]; sum += (v & 0xffffu) + (v >> 16); }
        sum = __reduce_add_sync(0xffffffffu, sum);
        if (lane == 0) s_warp_sum[warp] = sum;
        __syncthreads();
        uint32_t run = 0;
        for (int i = 0; i < warp; ++i) run += s_warp_sum[i];
        const int sub = (G - 2) * b;                 // a 2-gram owns 2^sub consecutive bucket ids
        const uint32_t sub_mask = (1u << sub) - 1u;
        uint32_t *bkt_row = p.bkt ? p.bkt + ((size_t)doc << (2 * b)) : nullptr;
        uint32_t *bkt3_row = p.bkt3 ? p.bkt3 + ((size_t)doc << (3 * b)) : nullptr;
        for (int wb = w0; wb < w1; wb += 32) {
            const int w = wb + lane;
            const uint32_t v = (w < w1) ? s_scr[w] : 0u;
            const uint32_t c0 = v & 0xffffu, c1 = v >> 16;
            uint32_t x = c0 + c1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            const uint32_t st0 = run + x - (c0 + c1), st1 = st0 + c0;   // first ranks of buckets 2w, 2w+1
            run += __shfl_sync(0xffffffffu, x, 31);
            if (w < w1) {
                const uint32_t id0 = 2u * (uint32_t)w;
                if (bkt_row) {
                    if ((id0 & sub_mask) == 0u) bkt_row[id0 >> sub] = (uint32_t)base + st0;
                    if (sub == 0) bkt_row[id0 + 1u] = (uint32_t)base + st1;
                }
                if (bkt3_row) *reinterpret_cast<uint2 *>(bkt3_row + id0) = make_uint2((uint32_t)base + st0, (uint32_t)base + st1);
                s_scr[w] = (st0 & 0xffffu) | (st1 << 16);  // bucket starts, used as the scatter cursors
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t id = id0 + (uint32_t)h, cnt = h ? c1 : c0, st = h ? st1 : st0;
                    if (cnt) {
                        atomicOr(&s_bits[st >> 5], 1u << (st & 31));
                        if (cnt > 32u && id != term_bucket) {
                            if (cnt > (uint32_t)DS_REFINE_MAX) { atomicOr(p.overflow, 1u); s_fail = 1u; }
                            else {
                                const uint32_t slot = atomicAdd(&s_nlist[0], 1u);
                                const uint32_t term_flag = ds_id_has_term(id, G, b, p.term) ? 1u : 0u;
                                if (slot < (uint32_t)DS_LIST_CAP)
                                    s_list0[slot] = make_uint2(st | (cnt << 16), (uint32_t)G | (term_flag << 16));
                            }
                        }
                    }
                }
            }
        }
        if (tid == 0) atomicOr(&s_bits[n >> 5], 1u << (n & 31));  // sentinel: "a bucket starts at rank n"
    }
    __syncthreads();
    if (s_fail) ds_clear_tables(p, doc, b, tid);   // the suffix array stays a permutation, but not a sorted one: see phase 1
    DS_STAMP(2);

    // ---- phase 4: scatter the suffixes into their buckets (arbitrary order inside a bucket)
    for (int c0 = tid * 8; c0 < n; c0 += DS_THREADS * 8) {
        const Ids8 ids = ds_bucket8(s_raw, shift + c0, term8, b, G);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t id = ids.id[j];
            if (c0 + j < n && id != term_bucket) {   // bare terminators were placed in phase 1
                const uint32_t old = atomicAdd(&s_scr[id >> 1], (id & 1u) ? 0x10000u : 1u);
                sa_doc[(id & 1u) ? (old >> 16) : (old & 0xffffu)] = base + c0 + j;
            }
        }
    }
    __syncthreads();
    DS_STAMP(3);

    // ---- phase 5: refine the buckets of more than 32 suffixes, level by level
    {
        DocCtx c;
        c.s_raw = s_raw; c.shift = shift; c.term8 = term8; c.term = p.term; c.b = b; c.S2 = p.S2;
        c.base = base; c.sa_doc = sa_doc; c.s_bits = s_bits; c.overflow = p.overflow;
        const int g = tid / DS_GROUP, gt = tid % DS_GROUP;
        uint8_t *gscr = reinterpret_cast<uint8_t *>(s_scr) + g * DS_GRP_BYTES;
        uint8_t *wscr = reinterpret_cast<uint8_t *>(s_scr) + warp * DS_WARP_BYTES;
        int cur = 0;
        while (true) {
            const int cnt = min((int)s_nlist[cur], DS_LIST_CAP);
            __syncthreads();
            if (cnt == 0) { if (tid == 0) s_work = 0; __syncthreads(); break; }   // s_work: the window counter of phase 6
            if (tid == 0) { s_nlist[cur ^ 1] = 0; s_work = 0; }
            __syncthreads();
            uint2 *list = cur ? s_list1 : s_list0, *next = cur ? s_list0 : s_list1;
            // buckets of <= DS_WARP_MAX suffixes: one warp each, taken from a shared work counter
            bool any_big = false;
            while (true) {
                int e = 0;
                if (lane == 0) e = (int)atomicAdd(&s_work, 1u);
                e = __shfl_sync(0xffffffffu, e, 0);
                if (e >= cnt) break;
                const uint2 entry = list[e];
                if ((entry.x >> 16) > (uint32_t)DS_WARP_MAX) { any_big = true; continue; }
                ds_refine_warp(c, entry, lane, wscr, next, &s_nlist[cur ^ 1]);
            }
            // larger ones (rare): groups of 4 warps
            if (__syncthreads_or(any_big ? 1 : 0)) {
                for (int e = g; e < cnt; e += DS_NGROUPS) {
                    const uint2 entry = list[e];
                    if ((entry.x >> 16) <= (uint32_t)DS_WARP_MAX) continue;
                    ds_refine(c, entry, g, gt, gscr, s_gmin, s_gw, next, &s_nlist[cur ^ 1]);
                }
                __syncthreads();
            }
            cur ^= 1;
        }
    }
    DS_STAMP(4);

    // ---- phase 6: windows of 32 ranks; every bucket of <= 32 suffixes that STARTS in the window
    {
        uint64_t *wkeys = reinterpret_cast<uint64_t *>(reinterpret_cast<uint8_t *>(s_scr) + warp * DS_WIN_BYTES);
        uint32_t *wpos = reinterpret_cast<uint32_t *>(wkeys + 64);
        const int nwin = (n + 31) >> 5;
        while (true) {
            // windows are handed out from a shared counter (static striding left warps idle for ~15 % of
            // this phase: window cost varies with the bucket sizes)
            int w = 0;
            if (lane == 0) w = (int)atomicAdd(&s_work, 1u);
            w = __shfl_sync(0xffffffffu, w, 0);
            if (w >= nwin) break;
            uint32_t word = s_bits[w];
            const bool last_win = w == (n >> 5);              // the window that holds the sentinel bit of rank n
            if (last_win) word &= (1u << (n & 31)) - 1u;
            if (word == 0u) continue;
            const int r0 = 32 * w + (__ffs(word) - 1);
            int r1 = n;   // first bucket start at or after the end of the window (the sentinel at the latest)
            if (!last_win) {
                int ww = w + 1;
                uint32_t x;
                while ((x = s_bits[ww]) == 0u) ++ww;
                r1 = 32 * ww + (__ffs(x) - 1);
            }
            const int last_start = 32 * w + (31 - __clz(word));
            int nseg = __popc(word);
            if (r1 - last_start > 32) { r1 = last_start; --nseg; }  // a bucket of > 32 identical tails: already in position order
            const int len = r1 - r0;   // <= 63
            if (len <= nseg) continue; // only singletons
            // per slot (lane, lane + 32): bucket [sb, se) of the member, packed -- what else the ranking needs (key,
            // position) is re-read from the window scratch instead of being kept in registers across the loops
            uint32_t seg[2];
            const int nslots = len > 32 ? 2 : 1;   // warp-uniform: the second slot only exists for ranges of 33..63
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int x = lane + 32 * s;
                seg[s] = 0;
                if (s < nslots && x < len) {
                    const int r = r0 + x;
                    const int li = sa_doc[r] - base;
                    const int wp = r - 32 * w;  // 0..63
                    const uint32_t le = (wp < 32) ? (word & (0xffffffffu >> (31 - wp))) : word;
                    const int sb = 32 * w + (31 - __clz(le)) - r0;
                    const uint32_t gt = (wp < 31) ? (word & (0xfffffffeu << wp)) : 0u;
                    int se = gt ? (32 * w + (__ffs(gt) - 1) - r0) : len;
                    if (se > len) se = len;
                    if (se - sb > 1) {
                        wkeys[x] = ds_key8(s_raw, shift + li, term8, G);
                        seg[s] = (uint32_t)sb | ((uint32_t)se << 8);
                    }
                    wpos[x] = (uint32_t)li;
                }
            }
            __syncwarp();
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int x = lane + 32 * s;
                if (s < nslots && seg[s] != 0u) {
                    const int q0 = (int)(seg[s] & 0xffu), q1 = (int)(seg[s] >> 8);
                    const uint64_t key = wkeys[x];
                    const uint32_t li = wpos[x];
                    int below = 0;
                    const uint32_t last = (uint32_t)key & 0xffu;
                    const bool by_pos = last == 0u || last == p.term;   // the window reaches the terminator
                    // members with a smaller key are counted in a branch-free loop; the members with an EQUAL key
                    // are only noted (a bucket has at most 32 members: one bit each) and resolved afterwards, so
                    // that the expensive comparison runs as often as the lane with the most ties needs it, not
                    // in every iteration in which some lane of the warp meets one
                    uint32_t ties = 0;
#pragma unroll 4
                    for (int q = q0; q < q1; ++q) {
                        const uint64_t kq = wkeys[q];
                        below += (kq < key) ? 1 : 0;
                        ties |= (kq == key ? 1u : 0u) << (q - q0);
                    }
                    ties &= ~(1u << (x - q0));
                    while (ties) {
                        const uint32_t pq = wpos[q0 + __ffs(ties) - 1];
                        ties &= ties - 1u;
                        const bool less = by_pos ? (pq < li) : ds_deep_less(s_raw, shift + (int)pq, shift + (int)li, G + 8, term8);
                        below += less ? 1 : 0;
                    }
                    seg[s] = (uint32_t)(q0 + below) | 0x100u;   // final offset in the range (< 64), bit 8 = "moved"
                }
            }
            __syncwarp();
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const int x = lane + 32 * s;
                if (s < nslots && seg[s] != 0u) sa_doc[r0 + (int)(seg[s] & 0xffu)] = base + (int32_t)wpos[x];
            }
            __syncwarp();
        }
    }
    DS_STAMP(5);
    if (p.lcp == nullptr) {
        if (p.sk) {   // suffix array only: the scorer's per-rank key bytes still come from the staged text
            __syncthreads();
            for (int r = tid; r < n; r += DS_THREADS) p.sk[base + r] = ds_lds4(s_raw, shift + (sa_doc[r] - base) + 2);
        }
        ds_score_document<GROUPS, GRAPH>(p, ds_smem, p.text_cap + DS_SCR_BYTES + 4 * p.bits_words + 2 * (int)sizeof(uint2) * DS_LIST_CAP, doc, base, n, tid);
        return;
    }

    // ---- phase 7: LCP of neighbouring suffixes from the staged text; 16-bit copy + min-pyramid in the
    // (now free) scratch, which continues into the bitmap and the work lists
    __syncthreads();
    uint16_t *s_lcp = reinterpret_cast<uint16_t *>(s_scr);
    __shared__ int s_pyr_off[4], s_pyr_size[4], s_pyr_levels;
    __shared__ uint32_t s_qcnt[7];   // profiling: phase-8 queries by the level that answers them (0: the neighbouring tile,
                                     // 4: none), 5: tiles redone, 6: stores queued
    if (tid < 7) s_qcnt[tid] = 0u;
    if (tid == 0) {
        int off = 0, sz = n, levels = 1;
        s_pyr_off[0] = 0; s_pyr_size[0] = n;
        for (int k = 1; k < 4; ++k) {
            off += (sz + 1) & ~1;
            sz = (sz + 31) >> 5;
            s_pyr_off[k] = off; s_pyr_size[k] = sz;
            levels = k + 1;
            if (sz <= 1) break;
        }
        s_pyr_levels = levels;
    }
    __syncthreads();
    // child table and annotation are stored sparsely in phase 8: their slices of this document are zero-filled
    // here, by the CTA itself -- the stores drain under the LCP computation and the sparse stores that follow find
    // the lines in L2 (host-side fills of the whole batch made the kernel wait for them and went to HBM twice)
    // (option fill_early, round 1: here, for the whole document -- 120 k cycles before the walk dirties the lines again, with
    // 108 MB of such lines in flight over the 148 CTAs most of them were written back twice.  Default: every warp fills the
    // slices of its own 32 chunks right before it walks them, see phase 8.)
    if (p.fill_early) {
        int32_t *const up_doc = p.up + base, *const down_doc = p.down + base, *const next_doc = p.next + base, *const ann_doc = p.ann + base;
        for (int r = tid; r < n; r += DS_THREADS) { up_doc[r] = 0; down_doc[r] = 0; next_doc[r] = 0; ann_doc[r] = 0; }
    }
    SPyr M;
    M.lcp = s_lcp; M.off = s_pyr_off; M.size_ = s_pyr_size; M.levels = s_pyr_levels;
    uint16_t *s_lv1 = s_lcp + s_pyr_off[1];
    constexpr int LU = 4;   // ranks per thread and round: their suffix-array loads (L2 latency) are issued together
    for (int r0 = 0; r0 < n; r0 += LU * DS_THREADS) {
        int pi[LU], pj[LU];
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int r = r0 + u * DS_THREADS + tid;
            pi[u] = (r > 0 && r < n) ? sa_doc[r - 1] : 0;
            pj[u] = (r > 0 && r < n) ? sa_doc[r] : 0;
        }
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int r = r0 + u * DS_THREADS + tid;
            uint32_t h = 0xffffu;
            if (r < n) {
                h = 0;
                if (r > 0) {
                    const int oi = shift + (pi[u] - base), oj = shift + (pj[u] - base);
                    while (true) {
                        const uint64_t x = ds_lds8(s_raw, oi + (int)h), y = ds_lds8(s_raw, oj + (int)h);
                        const uint64_t stop = (x ^ y) | ds_haszero(x ^ term8);   // distinct terminators differ
                        if (stop) { h += (uint32_t)((__ffsll((long long)stop) - 1) >> 3); break; }
                        h += 8;
                    }
                }
                p.lcp[base + r] = (int32_t)h;
                s_lcp[r] = (uint16_t)h;
                if (p.sk) p.sk[base + r] = ds_lds4(s_raw, shift + ((r > 0 ? pj[u] : sa_doc[0]) - base) + 2);
            }
            const uint32_t wmin = __reduce_min_sync(0xffffffffu, h);
            if (lane == 0 && (r - lane) < n) s_lv1[r >> 5] = (uint16_t)wmin;
        }
    }
    __syncthreads();
    for (int k = 2; k < M.levels; ++k) {
        for (int c = warp; c < M.size(k); c += DS_WARPS) {
            const int i = c * 32 + lane;
            const uint32_t v = (i < M.size(k - 1)) ? M.lv(k - 1)[i] : 0xffffu;
            const uint32_t wmin = __reduce_min_sync(0xffffffffu, v);
            if (lane == 0) s_lcp[s_pyr_off[k] + c] = (uint16_t)wmin;
        }
        __syncthreads();
    }
    DS_STAMP(6);

    // ---- phase 8: child table and annotation in closed form (as in tables.cu): for rank r with l = lcp[r],
    // q = PSE(r) = largest q < r with lcp[q] <= l, e = NSV(r) = smallest e > r with lcp[e] < l (or n).
    // lcp[q] == l -> next[q] = r; else r is the first l-index of [q .. e-1]: ann[r] = e - q, up[e] = r if
    // lcp[q] <= lcp[e], down[q] = r if lcp[e] <= lcp[q] (e inside the document); ann[0] = n - m (easa.py:329).
    // Values are ranks local to the document, 0 = none.
    // A warp takes a tile of 32 ranks, one lane per rank: bit-plane ballots give every lane the masks of the lanes with
    // a smaller and with an equal LCP value, and from them PSE and NSV inside the tile.  What the tile does not resolve
    // (its prefix and suffix minima) the whole warp answers one query at a time: first from the neighbouring tile (its
    // LCP values are in registers: the warp walks its tiles in order and carries them), then from the min-pyramid,
    // whose level 1 is the tiles' minima: one load and one ballot per level, up and down.  NSV is only searched for
    // first l-indices.  Ranks past the end count as LCP 0, so that the first of them is NSV = n.
    // The tiles of a warp are contiguous; the warp zero-fills up / down / next of its range right before its tiles store
    // into it (the lines are still in L2 and reach HBM once), ann is stored for every rank.  A store into another warp's
    // range would race with that warp's fill: such stores (only prefix and suffix minima of the warp's range have them,
    // a handful per warp) are queued as (target, rank) in the warp's share of the free text area and made after a block
    // barrier.  Should the queue be full, the tile is noted in a 64-bit mask and its outside stores are computed again
    // after the barrier.  (EAST_DOC_SORT_STACK_WALK=1: the stack walk below; both measured in DESIGN section 4.)
    if (!p.stack_walk) {
        const int T = (n + 31) >> 5, TW = (T + DS_WARPS - 1) / DS_WARPS;   // T <= 2048: TW <= 64
        const int t0 = min(T, warp * TW), t1 = min(T, t0 + TW);
        const int w0 = 32 * t0, w1 = min(n, 32 * t1);
        const int cap = p.text_cap / (4 * DS_WARPS);   // queue entries per warp: target << 16 | rank (both < 65 535)
        uint32_t *const queue = reinterpret_cast<uint32_t *>(s_raw) + warp * cap;
        int queued = 0;   // warp-uniform; > cap: the queue overflowed
        if (!p.fill_early) {
            for (int x = w0 + lane; x < w1; x += 32) { p.up[base + x] = 0; p.down[base + x] = 0; p.next[base + x] = 0; }
            __syncwarp();
        }
        auto lcp_at = [&](int r) -> uint32_t { return r < n ? (uint32_t)s_lcp[r] : 0u; };
        // tile t with the LCP values lp / l / ln of the tiles t - 1 / t / t + 1 (lp unused for t = 0: lane 0 has LCP 0).
        // outside == false: every store inside [w0, w1), the others queued; returns whether the queue overflowed.
        // outside == true: only the stores outside [w0, w1)
        auto tile = [&](int t, uint32_t lp, uint32_t l, uint32_t ln, bool outside) -> bool {
            const int r = 32 * t + lane;
            const bool valid = r < n;
            uint32_t lt = 0u, eq = 0xffffffffu;
            const uint32_t mx = __reduce_max_sync(0xffffffffu, l);   // 16 bits at most (deep-LCP inputs reach 65 534)
            for (int k = 31 - __clz(mx); k >= 0; --k) {
                const bool bit = (l >> k) & 1u;
                const uint32_t B = __ballot_sync(0xffffffffu, bit);
                if (bit) { lt |= eq & ~B; eq &= B; } else eq &= ~B;
            }
            const uint32_t below = (1u << lane) - 1u, above = ~((2u << lane) - 1u);
            const uint32_t pb = (lt | eq) & below;
            int q = pb ? 32 * t + 31 - __clz(pb) : -1;
            // PSE before the tile: the lanes smaller than every lane below them (strictly decreasing values)
            uint32_t U = __ballot_sync(0xffffffffu, q < 0 && valid && r > 0);
            while (U) {
                const int x = __ffs(U) - 1;
                U &= U - 1u;
                const uint32_t lx = __shfl_sync(0xffffffffu, l, x);
                const uint32_t B = __ballot_sync(0xffffffffu, lp <= lx);
                int f;
                if (B) { f = 32 * (t - 1) + 31 - __clz(B); if (p.phase_clk && lane == 0) atomicAdd(&s_qcnt[0], 1u); }
                else f = ds_warp_prev_le(M, 1, t - 1, lx, lane, p.phase_clk ? s_qcnt : nullptr);
                if (lane == x) q = f;
            }
            const bool inner = valid && r > 0;   // rank 0 has neither PSE nor NSV
            const uint32_t lq = inner ? (uint32_t)s_lcp[q] : 0u;
            const bool first = inner && lq != l;   // first l-index of [q .. e-1]
            const uint32_t na = lt & above;
            int e = na ? 32 * t + __ffs(na) - 1 : -1;
            U = __ballot_sync(0xffffffffu, e < 0 && first);
            while (U) {
                const int x = __ffs(U) - 1;
                U &= U - 1u;
                const uint32_t lx = __shfl_sync(0xffffffffu, l, x);
                const uint32_t B = __ballot_sync(0xffffffffu, ln < lx);   // lx > 0: a rank past the end stops it
                int f;
                if (B) { f = 32 * (t + 1) + __ffs(B) - 1; if (p.phase_clk && lane == 0) atomicAdd(&s_qcnt[0], 1u); }
                else f = ds_warp_next_lt(M, 1, t + 1, lx, n, lane, p.phase_clk ? s_qcnt : nullptr);
                if (lane == x) e = f;
            }
            bool dq = false, de = false;   // the store into down / next [q], into up[e] lies outside [w0, w1)
            if (inner) {
                if (!first) {
                    dq = q < w0;
                    if (dq == outside) p.next[base + q] = r;
                } else if (e < n) {
                    const uint32_t le = s_lcp[e];
                    if (lq <= le) { de = e >= w1; if (de == outside) p.up[base + e] = r; }
                    if (le <= lq) { dq = q < w0; if (dq == outside) p.down[base + q] = r; }
                }
            }
            if (outside) return false;
            if (valid) p.ann[base + r] = r == 0 ? n - p.doc_m[doc] : (first ? e - q : 0);
            const uint32_t mq = __ballot_sync(0xffffffffu, dq), me = __ballot_sync(0xffffffffu, de);
            if ((mq | me) == 0u) return false;
            const int iq = queued + __popc(mq & below), ie = queued + __popc(mq) + __popc(me & below);
            if (dq && iq < cap) queue[iq] = ((uint32_t)q << 16) | (uint32_t)r;
            if (de && ie < cap) queue[ie] = ((uint32_t)e << 16) | (uint32_t)r;
            queued += __popc(mq) + __popc(me);
            return queued > cap;   // what did fit is stored twice: the same values
        };
        uint64_t redo = 0ull;
        uint32_t lp = t0 > 0 ? lcp_at(32 * t0 - 32 + lane) : 0u, l = lcp_at(32 * t0 + lane);
        for (int t = t0; t < t1; ++t) {
            const uint32_t ln = lcp_at(32 * t + 32 + lane);
            if (tile(t, lp, l, ln, false)) redo |= 1ull << (t - t0);
            lp = l;
            l = ln;
        }
        __syncthreads();   // every warp has filled its range: from here on the stores may land in other warps' ranges
        DS_STAMP(7);
        if (p.phase_clk && lane == 0) { atomicAdd(&s_qcnt[5], (uint32_t)__popcll(redo)); atomicAdd(&s_qcnt[6], (uint32_t)queued); }
        for (int i = lane; i < min(queued, cap); i += 32) {
            const uint32_t ent = queue[i];
            const int x = (int)(ent >> 16), r = (int)(ent & 0xffffu);
            if (x > r) p.up[base + x] = r;                          // NSV side
            else if (s_lcp[x] == s_lcp[r]) p.next[base + x] = r;    // PSE side
            else p.down[base + x] = r;
        }
        while (redo) {
            const int t = t0 + __ffsll((long long)redo) - 1;
            redo &= redo - 1ull;
            tile(t, t > 0 ? lcp_at(32 * t - 32 + lane) : 0u, lcp_at(32 * t + lane), lcp_at(32 * t + 32 + lane), true);
        }
    } else
    // ---- phase 8, stack walk (EAST_DOC_SORT_STACK_WALK=1).  Thread t walks C consecutive ranks with the reference's
    // own stack discipline (easa.py:268-331): the stack holds the ranks whose next smaller LCP value
    // has not been met yet, LCP values non-decreasing from bottom to top.  Pushing rank r: the top is
    // q = PSE(r) (largest q < r with lcp[q] <= lcp[r]); popping t because of r: r = NSV(t) (smallest
    // e > t with lcp[e] < lcp[t]).  What lies outside the chunk -- q of a rank pushed on an empty
    // stack, e of the ranks still stacked at the end -- comes from the min-pyramid.  Closed forms as
    // in tables.cu: lcp[q] == l -> next[q] = r; else r is the first l-index of [q .. e-1]:
    // ann[r] = e - q, up[e] = r if lcp[q] <= lcp[e], down[q] = r if lcp[e] <= lcp[q] (e inside the
    // document).  Values are ranks local to the document, 0 = none (every warp zero-fills the slices of its 32 chunks right before it walks them).
    // The stacks (one byte per entry: offset in the chunk | 0x80 = first l-index) reuse the text area.
    {
        const int m = p.doc_m[doc];
        const int C = max(8, (n + DS_THREADS - 1) / DS_THREADS);   // <= 64
        const int c0 = tid * C, c1 = min(n, c0 + C);
        uint8_t *stk = s_raw + tid * C;
        // (rank, popping rank) records of the ranks pushed on an empty stack: 2 bytes each, in what is
        // left of the scratch after the LCP copy and its pyramid
        const int used = 2 * (s_pyr_off[M.levels - 1] + ((s_pyr_size[M.levels - 1] + 1) & ~1));
        const int avail = DS_SCR_BYTES + 4 * p.bits_words + 2 * (int)sizeof(uint2) * DS_LIST_CAP - used;
        const int R = max(0, min(24, avail / (2 * DS_THREADS)));
        uint8_t *rec = reinterpret_cast<uint8_t *>(s_scr) + used + tid * 2 * R;
        int nrec = 0;
        int depth = 0;
        auto close_interval = [&](int t, int q, int e, uint32_t le) {   // t: first l-index of [q .. e-1]
            p.ann[base + t] = e - q;
            if (e < n) {
                const uint32_t lq = s_lcp[q];
                if (lq <= le) p.up[base + e] = t;
                if (le <= lq) p.down[base + q] = t;
            }
        };
        // a rank that was pushed on an empty stack: its PSE lies before the chunk (every rank of
        // [c0, t) is larger); e = its NSV if it was met inside the chunk, else -1
        auto resolve_outside = [&](int t, int e) {
            const uint32_t l = s_lcp[t];
            const int q = ds_prev_le(M, c0, l);
            if (s_lcp[q] == l) { p.next[base + q] = t; return; }
            if (e < 0) e = ds_next_lt(M, c1 - 1, l, n);
            close_interval(t, q, e, e < n ? s_lcp[e] : 0u);
        };
        // ---- the walk never leaves the chunk.  One action per iteration and lane -- pop the top (it is
        // larger than lcp[r]: r is its NSV) or push r and advance -- so the lanes of a warp stay together:
        // at most 2 C iterations ("pop everything, then push" waited for the longest pop run of the 32
        // lanes at every rank).  Stack byte: offset in the chunk | 0x80 first l-index | 0x40 pushed on an
        // empty stack (PSE unknown).
        // The top entry and its LCP value live in registers: shared memory is read only when a pop
        // uncovers the entry below (which is also the popped rank's PSE).
        if (!p.fill_early) {
            // zero-fill, warp by warp: the 32 chunks of a warp are 32 C consecutive ranks -- coalesced stores --, and the walk
            // that follows at once stores into these very lines (it never leaves its chunk): they are still in L2, so they
            // reach HBM once.  What is stored outside a chunk comes after the block-wide barrier below.
            const int w0 = min(n, warp * 32 * C), w1 = min(n, w0 + 32 * C);
            int32_t *const up_w = p.up + base, *const down_w = p.down + base, *const next_w = p.next + base, *const ann_w = p.ann + base;
            for (int x = w0 + lane; x < w1; x += 32) { up_w[x] = 0; down_w[x] = 0; next_w[x] = 0; ann_w[x] = 0; }
            __syncwarp();
        }
        uint64_t lost = 0ull;   // chunk offsets of the ranks pushed on an empty stack whose record did not fit
        int r = c0;
        uint32_t l = (r < c1) ? s_lcp[r] : 0u;
        uint32_t top = 0, top_l = 0;   // valid while depth > 0
        int32_t *const ann_doc = p.ann + base, *const up_doc = p.up + base, *const down_doc = p.down + base,
                *const next_doc = p.next + base;
        while (r < c1) {
            if (depth > 0 && top_l > l) {
                // pop: r is the NSV of the top
                const uint32_t popped = top;
                const int t = c0 + (int)(popped & 0x3fu);
                --depth;
                uint32_t below = 0, below_l = 0;
                if (depth > 0) { below = stk[depth - 1]; below_l = s_lcp[c0 + (int)(below & 0x3fu)]; }
                if (popped & 0x40u) {
                    if (nrec < R) { rec[2 * nrec] = (uint8_t)(popped & 0x3fu); rec[2 * nrec + 1] = (uint8_t)(r - c0); ++nrec; }
                    else lost |= 1ull << (popped & 0x3fu);   // no room for the record: both neighbours are searched for later
                } else if (popped & 0x80u) {   // first l-index of [q .. r-1], q = the entry below (not the bottom: it exists)
                    const int q = c0 + (int)(below & 0x3fu);
                    ann_doc[t] = r - q;
                    if (below_l <= l) up_doc[r] = t;      // r < c1 <= n: inside the document
                    if (l <= below_l) down_doc[q] = t;
                }
                top = below; top_l = below_l;
            } else {
                uint32_t flag = 0;
                if (r == 0) {
                    ann_doc[0] = n - m;   // easa.py:329; rank 0 is nobody's first l-index and is never popped
                } else if (depth > 0) {
                    if (top_l == l) next_doc[c0 + (int)(top & 0x3fu)] = r;
                    else flag = 0x80u;
                } else {
                    flag = 0x40u;
                }
                top = (uint32_t)(r - c0) | flag;
                top_l = l;
                stk[depth++] = (uint8_t)top;
                ++r;
                if (r < c1) l = s_lcp[r];
            }
        }
        __syncthreads();   // every slice is filled and walked: from here on the stores may land in other threads' chunks
        DS_STAMP(7);
        // ---- what lies outside the chunk, from the min-pyramid.  Farthest first in every lane: the
        // bottom of the stack and the LAST record have the smallest LCP values, whose neighbours are
        // thousands of ranks away (the ends of a first-letter block); met in the same iterations by all
        // lanes they cost one long search per warp instead of one per iteration.
        for (int i = 0; i < depth; ++i) {
            const uint32_t ent = stk[i];
            const int t = c0 + (int)(ent & 0x3fu);
            if (ent & 0x40u) resolve_outside(t, -1);
            else if (ent & 0x80u) {
                const int e = ds_next_lt(M, c1 - 1, s_lcp[t], n);   // everything in (t, c1) is >= lcp[t]
                close_interval(t, c0 + (int)(stk[i - 1] & 0x3fu), e, e < n ? s_lcp[e] : 0u);
            }
        }
        for (int i = nrec - 1; i >= 0; --i) resolve_outside(c0 + (int)rec[2 * i], c0 + (int)rec[2 * i + 1]);
        while (lost) {   // (rare) popped inside the chunk, record dropped: its next smaller value is searched for from the rank itself
            const int t = c0 + (__ffsll((long long)lost) - 1);
            lost &= lost - 1ull;
            resolve_outside(t, ds_next_lt(M, t, s_lcp[t], n));
        }
    }
    if (p.phase_clk) __syncthreads();
    DS_STAMP(8);
    if (p.phase_clk && tid < 7) atomicAdd(&p.phase_clk[10 + tid], (unsigned long long)s_qcnt[tid]);
    ds_score_document<GROUPS, GRAPH>(p, ds_smem, p.text_cap + DS_SCR_BYTES + 4 * p.bits_words + 2 * (int)sizeof(uint2) * DS_LIST_CAP, doc, base, n, tid);
    if (p.phase_clk) __syncthreads();
    DS_STAMP(9);
#undef DS_STAMP
}

__global__ void __launch_bounds__(DS_THREADS, 1)
k_doc_suffix_sort(DocSortParams p) { doc_suffix_sort<false, false>(p); }

__global__ void __launch_bounds__(DS_THREADS, 1)
k_doc_suffix_sort_groups(DocSortParams p) { doc_suffix_sort<true, false>(p); }

__global__ void __launch_bounds__(DS_THREADS, 1)
k_doc_suffix_sort_graph(DocSortParams p) { doc_suffix_sort<false, true>(p); }

__global__ void __launch_bounds__(DS_THREADS, 1)
k_doc_suffix_sort_groups_graph(DocSortParams p) { doc_suffix_sort<true, true>(p); }

// Host side: can the batch take the per-document path, and with which parameters
bool doc_sort_plan(int sigma, int32_t max_doc_n, DocSortPlan &plan) {
    const int b = bits_for((uint64_t)sigma + 1);
    if (b < 1 || b > 7) return false;
    if (max_doc_n > 65535) return false;
    int G = 15 / b;
    if (G > 7) G = 7;
    if (G < 2) return false;
    int S2 = 10 / b;
    if (S2 < 1) S2 = 1;
    if (S2 > 7) S2 = 7;
    plan.b = b; plan.G = G; plan.S2 = S2;
    plan.text_cap = (max_doc_n + 15 + 48 + 16 + 15) & ~15;
    plan.bits_words = ((max_doc_n >> 5) + 3 + 1) & ~1;
    const size_t after_text = DS_SCR_BYTES + sizeof(uint32_t) * (size_t)plan.bits_words + 2 * sizeof(uint2) * (size_t)DS_LIST_CAP;
    plan.smem = (size_t)plan.text_cap + after_text;
    // fused LCP / child / annotation phases: 16-bit LCP copy + pyramid levels overlay everything after the text
    size_t need = 0;
    for (int sz = max_doc_n, k = 0; k < 4; ++k) { need += 2 * (((size_t)sz + 1) & ~(size_t)1); if (sz <= 1) break; sz = (sz + 31) >> 5; }
    plan.tables_fit = need <= after_text ? 1 : 0;
    return plan.smem <= (size_t)220 * 1024;
}

void doc_sort_launch(const DocSortPlan &plan, const uint8_t *t8, const uint32_t *text, const int32_t *doc_off,
                     const int32_t *doc_m, int doc_begin, int n_docs,
                     int64_t n_total, uint32_t term, int32_t *sa, uint32_t *bkt, uint32_t *bkt3, uint32_t *overflow, cudaStream_t s,
                     unsigned long long *phase_clk, const DocSortTables *tables, uint32_t *sk, const DocScore *score,
                     const uint8_t *code_table, uint32_t *miss, int64_t text_len, const uint8_t *text8) {
    const bool groups = score && score->recs && bkt && score->group_off;
    const bool graph = score && score->recs && bkt && score->graph;
    const void *kernel = graph ? (groups ? (const void *)k_doc_suffix_sort_groups_graph : (const void *)k_doc_suffix_sort_graph)
                               : (groups ? (const void *)k_doc_suffix_sort_groups : (const void *)k_doc_suffix_sort);
    ensure_dynamic_smem(kernel, 220 * 1024);
    DocSortParams p;
    p.t8 = t8; p.text = text; p.doc_off = doc_off; p.doc_m = doc_m; p.sa = sa; p.bkt = bkt; p.bkt3 = (plan.G == 3) ? bkt3 : nullptr; p.overflow = overflow;
    p.b = plan.b; p.G = plan.G; p.S2 = plan.S2; p.term = term;
    p.text_cap = plan.text_cap; p.bits_words = plan.bits_words;
    p.phase_clk = phase_clk;
    p.doc_begin = doc_begin;
    p.sk = sk;
    if (score && score->recs && bkt) p.score = *score;
    if (p.score.recs && p.score.skip_suffix_keys) p.sk = nullptr;
    p.code_table = (code_table && miss) ? code_table : nullptr;
    p.t8_out = const_cast<uint8_t *>(t8); p.miss = miss; p.text_len = text_len;
    p.text8 = p.code_table ? text8 : nullptr; p.text_out = const_cast<uint32_t *>(text);
    static const bool fill_early = getenv("EAST_DOC_SORT_FILL_EARLY") != nullptr;
    p.fill_early = fill_early ? 1 : 0;
    static const bool stack_walk = getenv("EAST_DOC_SORT_STACK_WALK") != nullptr;
    p.stack_walk = stack_walk ? 1 : 0;
    p.lcp = p.up = p.down = p.next = p.ann = nullptr;
    if (tables && plan.tables_fit) { p.lcp = tables->lcp; p.up = tables->up; p.down = tables->down; p.next = tables->next; p.ann = tables->ann; }
    // algorithmic bytes per code point: 1 (byte text in) + 4 (suffix array out), with the fused tables + 5 x 4
    // (LCP, up, down, next, annotation out), + 4 when the kernel byte-codes the text itself (code points in);
    // with the scorer inside, plus the bytes of its walks (counted by the
    // instrumented scorer, option score_bytes)
    EAST_BYTES(((p.lcp ? 25.0 : 5.0) + (p.code_table ? (p.text8 ? 5.0 : 4.0) : 0.0)) * (double)n_total + (p.score.recs ? p.score.algorithmic_bytes : 0.0));
    if (graph && groups) EAST_LAUNCH(k_doc_suffix_sort_groups_graph, n_docs, DS_THREADS, plan.smem, s, p);
    else if (graph) EAST_LAUNCH(k_doc_suffix_sort_graph, n_docs, DS_THREADS, plan.smem, s, p);
    else if (groups) EAST_LAUNCH(k_doc_suffix_sort_groups, n_docs, DS_THREADS, plan.smem, s, p);
    else EAST_LAUNCH(k_doc_suffix_sort, n_docs, DS_THREADS, plan.smem, s, p);
}

}  // namespace east
