// graph_edges.cu -- the keyphrase graph assembled where its co-occurrence counts are (applications.py:115-149): the
// supports and the edges of every threshold plane come back to the host, the cols x cols counts stay on the device.
//
// Node n (the n-th keyphrase, duplicates included) reads column node_col[n].  Per plane t:
//   support[t][n] = C[t][col_n][col_n]; n is kept iff (double)support >= p (exact for int32; NaN keeps nothing);
//   for kept i1 != i2 (positions, not columns), in row-major order over the kept positions, conf =
//   (double)C[t][col_i1][col_i2] / (double)max(support_i1, 1) -- an IEEE division, as the host's numpy divide -- and
//   (i1, i2) is an edge iff conf >= c.
// Three passes: the supports (gathered, copied to the host, which picks the kept nodes of every plane); a count pass,
// one warp per kept row over the row's kept columns with __ballot_sync / __popc; an int64 exclusive scan of the row
// counts of all planes on the host (N (N - 1) edges can pass 2^31); an emit pass in the same order.  A row's edges go
// to [first[row], first[row + 1]) whatever the launch configuration, so the output does not depend on it.
#include <algorithm>
#include <cstdint>
#include <vector>

#include "../../include/east_b200.h"
#include "sa_build.h"

namespace east {
namespace {

// the kept entries of all planes, plane-major, ascending positions inside a plane
struct KeptRows {
    const int32_t *C;          // T x cols x cols
    int64_t cols;
    const int32_t *node;       // [R] node position of kept entry r
    const int32_t *col;        // [R] its column
    const int32_t *sup;        // [R] its support
    int32_t plane_off[MAX_THRESHOLDS + 1];   // entries of plane t: [plane_off[t], plane_off[t + 1])
    double c;
    int32_t *count;            // count pass: [R] edges of row r
    const int64_t *first;      // emit pass: [R] where row r's edges start
    int32_t *src, *dst;
    double *conf;
};

__global__ void __launch_bounds__(256) k_graph_supports(const int32_t *__restrict__ C, int64_t cols, int32_t T,
                                                        const int32_t *__restrict__ node_col, int32_t N,
                                                        int32_t *__restrict__ support) {
    const int64_t total = (int64_t)T * N;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = i / N, col = __ldg(node_col + (i - t * N));
        support[i] = __ldg(C + (t * cols + col) * cols + col);
    }
}

constexpr int EDGE_UNROLL = 4;   // chunks of 32 columns whose counts are loaded before any is compared

// one warp per kept row (grid-stride); Emit = false: count the row's edges, true: write them
template <bool Emit>
__global__ void __launch_bounds__(256) k_graph_edges(KeptRows k, int32_t R) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < R; r += warps) {
        // the plane of row r, with constant indices into the parameter (a variable one would copy it to local memory)
        int t = 0;
        int32_t b = 0, e = k.plane_off[1];
#pragma unroll
        for (int q = 1; q < MAX_THRESHOLDS; ++q)
            if (r >= k.plane_off[q]) { t = q; b = k.plane_off[q]; e = k.plane_off[q + 1]; }
        const int32_t n = e - b, self = (int32_t)r - b;
        const int32_t *row = k.C + ((int64_t)t * k.cols + __ldg(k.col + r)) * k.cols;
        const double sup = (double)max(__ldg(k.sup + r), 1);
        const int32_t src = __ldg(k.node + r);
        int64_t out = Emit ? k.first[r] : 0;
        int32_t cnt = 0;
        for (int32_t j0 = 0; j0 < n; j0 += 32 * EDGE_UNROLL) {
            int32_t v[EDGE_UNROLL];
#pragma unroll
            for (int u = 0; u < EDGE_UNROLL; ++u) {
                const int32_t j = j0 + 32 * u + lane;
                v[u] = j < n ? __ldg(row + __ldg(k.col + b + j)) : 0;
            }
#pragma unroll
            for (int u = 0; u < EDGE_UNROLL; ++u) {
                const int32_t j = j0 + 32 * u + lane;
                // 0 / sup is +0.0 exactly: only a non-zero count needs the division
                const double conf = v[u] == 0 ? 0.0 : (double)v[u] / sup;
                const bool edge = j < n && j != self && conf >= k.c;
                const unsigned m = __ballot_sync(0xffffffffu, edge);
                if (Emit) {
                    if (edge) {
                        const int64_t o = out + __popc(m & lanemask_lt());
                        k.src[o] = src;
                        k.dst[o] = __ldg(k.node + b + j);
                        k.conf[o] = conf;
                    }
                    out += __popc(m);
                } else {
                    cnt += __popc(m);
                }
            }
        }
        if (!Emit && lane == 0) k.count[r] = cnt;
    }
}

int grid_for_rows(int64_t rows) { return grid_for(rows, 8); }   // 8 warps of 256 threads, one row each

}  // namespace

int64_t graph_edges(const int32_t *C, int64_t cols, int32_t T, const int32_t *node_col_host, int32_t N, double c, double p,
                    cudaStream_t s, int32_t *support_host, int64_t *n_edges_host, int64_t edge_cap, int32_t *src_host,
                    int32_t *dst_host, double *conf_host) {
    std::fill(n_edges_host, n_edges_host + T, (int64_t)0);
    if (N == 0) return 0;
    // supports
    {
        DevBuf<int32_t> d_col((size_t)N, s), d_sup((size_t)T * N, s);
        EAST_CUDA(cudaMemcpyAsync(d_col.p, node_col_host, sizeof(int32_t) * N, cudaMemcpyHostToDevice, s));
        EAST_BYTES(12.0 * T * N);
        EAST_LAUNCH(k_graph_supports, grid_for((int64_t)T * N, 256), 256, 0, s, C, cols, T, d_col.p, N, d_sup.p);
        EAST_CUDA(cudaMemcpyAsync(support_host, d_sup.p, sizeof(int32_t) * T * N, cudaMemcpyDeviceToHost, s));
        EAST_CUDA(cudaStreamSynchronize(s));
    }
    // kept entries: [node | col | sup], plane after plane
    KeptRows k{};
    std::vector<int32_t> node, col, sup;
    for (int32_t t = 0; t < T; ++t) {
        k.plane_off[t] = (int32_t)node.size();
        for (int32_t n = 0; n < N; ++n) {
            const int32_t v = support_host[(size_t)t * N + n];
            if ((double)v >= p) { node.push_back(n); col.push_back(node_col_host[n]); sup.push_back(v); }
        }
        if (node.size() > (size_t)INT32_MAX) throw Error(EAST_ERR_RANGE, "more than 2^31 - 1 kept nodes over all planes");
    }
    const int32_t R = (int32_t)node.size();
    k.plane_off[T] = R;
    for (int32_t t = T + 1; t <= MAX_THRESHOLDS; ++t) k.plane_off[t] = R;
    if (R == 0) return 0;
    std::vector<int32_t> kept(node);
    kept.insert(kept.end(), col.begin(), col.end());
    kept.insert(kept.end(), sup.begin(), sup.end());
    DevBuf<int32_t> d_kept(kept.size(), s), d_count((size_t)R, s);
    EAST_CUDA(cudaMemcpyAsync(d_kept.p, kept.data(), sizeof(int32_t) * kept.size(), cudaMemcpyHostToDevice, s));
    k.C = C;
    k.cols = cols;
    k.node = d_kept.p;
    k.col = d_kept.p + R;
    k.sup = d_kept.p + 2 * (size_t)R;
    k.c = c;
    k.count = d_count.p;
    double cells = 0.0;   // counts read per pass (+ the column of each)
    for (int32_t t = 0; t < T; ++t) {
        const double n = (double)(k.plane_off[t + 1] - k.plane_off[t]);
        cells += n * n;
    }
    // count pass
    EAST_BYTES(8.0 * cells + 16.0 * R);
    EAST_LAUNCH_AS("k_graph_edge_count", k_graph_edges<false>, grid_for_rows(R), 256, 0, s, k, R);
    std::vector<int32_t> count((size_t)R);
    EAST_CUDA(cudaMemcpyAsync(count.data(), d_count.p, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaStreamSynchronize(s));
    // int64 exclusive scan over the rows of all planes
    std::vector<int64_t> first((size_t)R);
    int64_t total = 0;
    for (int32_t t = 0; t < T; ++t) {
        const int64_t before = total;
        for (int32_t r = k.plane_off[t]; r < k.plane_off[t + 1]; ++r) { first[r] = total; total += count[r]; }
        n_edges_host[t] = total - before;
    }
    if (total > edge_cap || total == 0) return total;
    // emit pass
    DevBuf<int64_t> d_first((size_t)R, s);
    DevBuf<int32_t> d_src((size_t)total, s), d_dst((size_t)total, s);
    DevBuf<double> d_conf((size_t)total, s);
    EAST_CUDA(cudaMemcpyAsync(d_first.p, first.data(), sizeof(int64_t) * R, cudaMemcpyHostToDevice, s));
    k.count = nullptr;
    k.first = d_first.p;
    k.src = d_src.p;
    k.dst = d_dst.p;
    k.conf = d_conf.p;
    EAST_BYTES(8.0 * cells + 20.0 * R + 16.0 * (double)total);
    EAST_LAUNCH_AS("k_graph_edge_emit", k_graph_edges<true>, grid_for_rows(R), 256, 0, s, k, R);
    EAST_CUDA(cudaMemcpyAsync(src_host, d_src.p, sizeof(int32_t) * total, cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaMemcpyAsync(dst_host, d_dst.p, sizeof(int32_t) * total, cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaMemcpyAsync(conf_host, d_conf.p, sizeof(double) * total, cudaMemcpyDeviceToHost, s));
    EAST_CUDA(cudaStreamSynchronize(s));
    return total;
}

}  // namespace east
