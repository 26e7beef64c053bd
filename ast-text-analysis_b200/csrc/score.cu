// score.cu -- batched keyphrase x document scorer.
//
// Replaces EnhancedAnnotatedSuffixArray._score (east/asts/easa.py:91-139) together with
// _get_child_interval (:379-400), _lcp_value (:349-356) and _annotation (:340-344) for every
// (document, keyphrase) pair of applications.keyphrases_table (applications.py:43-52).
//
// The reference walks the child table; the set of suffixes below the node reached after
// matching d characters is exactly the SA interval of suffixes that start with those d
// characters, and the node frequency is the interval size (root: n - m).  So one query suffix
// is scored by narrowing an SA interval one character at a time:
//     entering a NEW node (d == 0, or the interval got smaller)   frac += |child| / |parent|
// and the suffix result is ((frac + d) - nodes) [/ d], accumulated in the reference's order
// in IEEE fp64 (only +, -, / : nothing can be contracted into an FMA).
//
//   k_score_suffixes  one thread per (document, query suffix)   -> tmp[doc][suffix]
//   k_score_combine   one thread per (document, keyphrase)      -> out[doc][k] = (sum in suffix order) / len
//   k_score_combine_max  one thread per (document, group of variants) -> out[doc][g] = best variant of the group
#include "sa_build.h"
#include "score_walk.cuh"

namespace east {

constexpr int SC_THREADS = 128;


template <bool PROBES>
__global__ void __launch_bounds__(SC_THREADS)
k_score_suffixes(ScoreInput in, double *__restrict__ tmp, unsigned long long *probe_count) {
    unsigned long long probes = 0;
    const int64_t total = (int64_t)in.n_docs * in.n_uniq;
    const int64_t stride = (int64_t)gridDim.x * SC_THREADS;
    for (int64_t idx = (int64_t)blockIdx.x * SC_THREADS + threadIdx.x; idx < total; idx += stride) {
        const int32_t doc = (int32_t)(idx / in.n_uniq);
        const int32_t u = (int32_t)(idx - (int64_t)doc * in.n_uniq);   // position in visiting order
        // one coalesced 16-byte load: where the suffix is, how long, its first 8 symbols
        const uint4 raw = __ldg(reinterpret_cast<const uint4 *>(in.recs) + u);
        const uint64_t qw = ((uint64_t)raw.y << 32) | raw.x;
        const int32_t sidx = (int32_t)raw.z;
        const int32_t len = (int32_t)(raw.w & 0xffffu);
        const bool generic = ((raw.w >> 16) & 0xffu) != 0u;
        const int32_t start = __ldg(in.doc_off + doc), end = __ldg(in.doc_off + doc + 1);
        double r;
        if (in.bkt != nullptr && !generic) {
            r = score_one_suffix_fast<PROBES, true>(in.t8, in.sa, in.sk, in.bkt + ((size_t)doc << (2 * in.sym_bits)),
                                              in.bkt3 ? in.bkt3 + ((size_t)doc << (3 * in.sym_bits)) : nullptr, in.sym_bits, start, end,
                                              __ldg(in.doc_m + doc), in.q8 + sidx, qw, len, in.normalized, probes);
        } else {
            r = score_one_suffix<PROBES, true>(in.text, in.sa, start, end, __ldg(in.doc_m + doc), in.kp + sidx, len,
                                         in.normalized, probes);
        }
        tmp[(int64_t)doc * in.n_uniq + u] = r;   // coalesced: results are stored in visiting order
    }
    if (PROBES) {
        for (int o = 16; o > 0; o >>= 1) probes += __shfl_down_sync(0xffffffffu, probes, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(probe_count, probes);
    }
}

// One thread per (document, keyphrase): adds up the results of the keyphrase's suffixes IN SUFFIX ORDER
// (the reference's fp64 order, easa.py:127-134), each fetched through the position of its distinct twin from the
// document's row of tmp (L2-resident: the row was just written).  Adjacent threads own adjacent
// keyphrases, so the id loads are contiguous across the warp.
__global__ void __launch_bounds__(SC_THREADS)
k_score_combine(ScoreInput in, const double *__restrict__ tmp, double *__restrict__ out) {
    const int64_t total = (int64_t)in.n_docs * in.K;
    const int64_t stride = (int64_t)gridDim.x * SC_THREADS;
    for (int64_t idx = (int64_t)blockIdx.x * SC_THREADS + threadIdx.x; idx < total; idx += stride) {
        const int32_t doc = (int32_t)(idx / in.K);
        const int32_t k = (int32_t)(idx - (int64_t)doc * in.K);
        const int32_t b = __ldg(in.kp_off + k), e = __ldg(in.kp_off + k + 1);
        const double *row = tmp + (int64_t)doc * in.n_uniq;
        double result = 0.0;
        for (int32_t s = b; s < e; ++s) result = result + row[__ldg(in.uniq_of + s)];
        const double v = result / (double)(e - b);
        out[idx] = v;
        for (int pi = 0; pi < in.n_peers; ++pi) in.peer_out[pi][idx] = v;   // NVLink peer stores: the fused all-gather
    }
    if (in.n_peers > 0) __threadfence_system();
}

// One thread per (document, group of variants) -- the synonym substitutions of one keyphrase (easa.py:27-34): every
// variant's score is taken as k_score_combine takes it (suffix results in suffix order, divided by the variant's
// length) and the best of the group is stored, so the document x variant table never exists.  The maximum starts from
// the first variant's score: scores are >= 0 and never NaN, so it is one of the scores, bit for bit.
__global__ void __launch_bounds__(SC_THREADS)
k_score_combine_max(ScoreInput in, const double *__restrict__ tmp, double *__restrict__ out) {
    const int64_t total = (int64_t)in.n_docs * in.G;
    const int64_t stride = (int64_t)gridDim.x * SC_THREADS;
    for (int64_t idx = (int64_t)blockIdx.x * SC_THREADS + threadIdx.x; idx < total; idx += stride) {
        const int32_t doc = (int32_t)(idx / in.G);
        const int32_t g = (int32_t)(idx - (int64_t)doc * in.G);
        const int32_t v0 = __ldg(in.group_off + g), v1 = __ldg(in.group_off + g + 1);
        const double *row = tmp + (int64_t)doc * in.n_uniq;
        double best = 0.0;
        for (int32_t v = v0; v < v1; ++v) {
            const int32_t b = __ldg(in.kp_off + v), e = __ldg(in.kp_off + v + 1);
            double result = 0.0;
            for (int32_t s = b; s < e; ++s) result = result + row[__ldg(in.uniq_of + s)];
            const double score = result / (double)(e - b);
            if (v == v0 || score > best) best = score;
        }
        out[idx] = best;
        for (int pi = 0; pi < in.n_peers; ++pi) in.peer_out[pi][idx] = best;   // as k_score_combine: the fused all-gather
    }
    if (in.n_peers > 0) __threadfence_system();
}

__global__ void __launch_bounds__(256)
k_fill_suffix_keys(const uint8_t *__restrict__ t8, const int32_t *__restrict__ sa, int32_t n, uint32_t *__restrict__ sk) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
        const uint8_t *p = t8 + sa[r] + 2;   // the byte text carries 128 bytes of slack
        sk[r] = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    }
}

void fill_suffix_keys(const uint8_t *t8, const int32_t *sa, int32_t n, uint32_t *sk, cudaStream_t s) {
    EAST_BYTES(12.0 * n);
    EAST_LAUNCH(k_fill_suffix_keys, grid_for(n, 256, 16), 256, 0, s, t8, sa, n, sk);
}

void score_combine(const ScoreInput &in, const double *suffix_tmp, double *out_DxK, cudaStream_t s) {
    if (in.group_off) {
        const int64_t cells = (int64_t)in.n_docs * in.G;
        if (cells > 0)
            EAST_LAUNCH(k_score_combine_max, grid_for(cells, SC_THREADS, 64), SC_THREADS, 0, s, in, suffix_tmp, out_DxK);
        return;
    }
    const int64_t cells = (int64_t)in.n_docs * in.K;
    if (cells > 0)
        EAST_LAUNCH(k_score_combine, grid_for(cells, SC_THREADS, 64), SC_THREADS, 0, s, in, suffix_tmp, out_DxK);
}

void score_table(const ScoreInput &in, double *suffix_tmp, double *out_DxK, cudaStream_t s) {
    score_suffixes(in, suffix_tmp, s);
    score_combine(in, suffix_tmp, out_DxK, s);
}

void score_suffixes(const ScoreInput &in, double *suffix_tmp, cudaStream_t s) {
    const int64_t work = (int64_t)in.n_docs * in.n_uniq;
    if (work > 0) {
        if (in.probe_count) {
            EAST_LAUNCH(k_score_suffixes<true>, grid_for(work, SC_THREADS, 64), SC_THREADS, 0, s, in, suffix_tmp,
                        in.probe_count);
        } else {
            EAST_BYTES(in.algorithmic_bytes);
            EAST_LAUNCH(k_score_suffixes<false>, grid_for(work, SC_THREADS, 64), SC_THREADS, 0, s, in, suffix_tmp,
                        (unsigned long long *)nullptr);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Co-occurrence counts of the keyphrase graph (applications.py:111-113, 136-147):
//   B[k][d] = S[d][k] >= threshold, C = B * B^T.  First version: bit-packed rows, AND + POPC.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_threshold_pack(const double *__restrict__ S, int64_t D, int32_t K, double thr, uint32_t *__restrict__ bits,
                 int64_t words) {
    // bits[k][w]: bit j of word w = (S[(32 w + j)][k] >= thr).  thread per (w, k), k fastest (coalesced S rows)
    const int64_t total = words * K;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t w = idx / K;
        const int32_t k = (int32_t)(idx - w * K);
        uint32_t v = 0;
        for (int j = 0; j < 32; ++j) {
            int64_t d = w * 32 + j;
            if (d < D && S[d * K + k] >= thr) v |= 1u << j;
        }
        bits[(int64_t)k * words + w] = v;
    }
}

__global__ void __launch_bounds__(256)
k_cooc_popc(const uint32_t *__restrict__ bits, int32_t K, int64_t words, int32_t *__restrict__ C) {
    // 16x16 output tile per CTA, words streamed through shared memory
    __shared__ uint32_t sa_[16][33], sb_[16][33];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i = blockIdx.y * 16 + ty, j = blockIdx.x * 16 + tx;
    int32_t acc = 0;
    for (int64_t w0 = 0; w0 < words; w0 += 32) {
        for (int e = threadIdx.x; e < 16 * 32; e += 256) {
            int r = e >> 5, c = e & 31;
            int64_t w = w0 + c;
            int ri = blockIdx.y * 16 + r, rj = blockIdx.x * 16 + r;
            sa_[r][c] = (ri < K && w < words) ? bits[(int64_t)ri * words + w] : 0u;
            sb_[r][c] = (rj < K && w < words) ? bits[(int64_t)rj * words + w] : 0u;
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < 32; ++c) acc += __popc(sa_[ty][c] & sb_[tx][c]);
        __syncthreads();
    }
    if (i < K && j < K) C[(int64_t)i * K + j] = acc;
}

void cooc_counts(const double *S_DxK, int64_t D, int32_t K, double threshold, int32_t *C, cudaStream_t s) {
    const int64_t words = (D + 31) / 32;
    DevBuf<uint32_t> bits((size_t)words * K, s);
    EAST_LAUNCH(k_threshold_pack, grid_for(words * K, 256, 32), 256, 0, s, S_DxK, D, K, threshold, bits.p, words);
    dim3 grid((K + 15) / 16, (K + 15) / 16);
    EAST_LAUNCH(k_cooc_popc, grid, 256, 0, s, bits.p, K, words, C);
}

}  // namespace east
