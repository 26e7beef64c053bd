// cooc_tc.cu -- keyphrase co-occurrence counts C = B * B^T on the 5th-generation tensor cores.
//
// Replaces the K^2 Python set intersections of applications.keyphrases_graph
// (east/applications.py:111-113, 136-147):  B[k][d] = (S[d][k] >= threshold) in {0,1},
// C[i][j] = sum_d B[i][d] * B[j][d] = |T_i & T_j|, support[k] = C[k][k].
//
// The one GEMM-shaped piece of the hot path (north_star).  Hand-written tcgen05:
//   * k_threshold_bytes  : S (fp64, doc-major) -> B as uint8 0/1, keyphrase-major (K-major operand
//                          for both sides of B * B^T), padded to multiples of 128 with zeros;
//   * k_cooc_umma        : one CTA per 128 x 128 tile of C.  Per 128-byte slice of the document
//                          dimension the CTA stages the two 128 x 128-byte operand tiles in shared
//                          memory in the canonical K-major / no-swizzle core-matrix layout
//                          (8 rows x 16 bytes = 128 contiguous bytes; LBO = 128 B between core matrices
//                          along K, SBO = 1024 B between 8-row groups), one elected thread issues
//                          four tcgen05.mma.kind::i8 (M=128, N=128, K=32, u8 x u8 -> s32) that
//                          accumulate in TMEM, and tcgen05.commit signals an mbarrier so the
//                          two-stage shared-memory ring can be refilled while the MMAs run.
//                          Epilogue: tcgen05.ld (32 lanes x 32 columns per warp) -> int32 stores.
// C = B * B^T is symmetric: the CTAs below the diagonal exit at once, the others store their tile and its transpose.
// Counts are exact: u8 products accumulated in int32 (D < 2^31).
#include <cuda.h>   // CUtensorMap and the enums of cuTensorMapEncodeTiled (types only: libcuda is not linked)
#include "sa_build.h"

namespace east {

constexpr int CT_TILE = 128;      // M = N = 128
constexpr int CT_BK = 128;        // bytes of the reduction dimension per stage
constexpr int CT_THREADS = 128;
constexpr int CT_STAGE_BYTES = 2 * CT_TILE * CT_BK;  // A tile + B tile = 32 KB

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4)        // start address, 16-byte units
           | ((uint64_t)(128 >> 4) << 16)              // leading byte offset: next core matrix along K
           | ((uint64_t)(1024 >> 4) << 32)             // stride byte offset: next 8-row group
           | (1ull << 46);                             // descriptor version 1 (sm_100)
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}

// S[d][k] >= thr  ->  Bm[k][col0 + d] (uint8): 128 (documents) x 32 (keyphrases) transposing tiles through shared memory.
// Reads: a warp takes 32 consecutive doubles of a row of S (256 bytes), four rows in flight per thread; writes: every
// keyphrase row of the tile leaves as 128 contiguous bytes (eight 16-byte stores).  HBM-bound: 8 D K bytes in, D K out.
// Only the columns [col0, col0 + D) are written, so that document tiles scored one after another (possibly on two
// streams) fill their own columns of one matrix; a piece that is not a whole aligned 16 bytes inside them is stored
// byte by byte.
constexpr int TB_D = 128, TB_K = 32;
__global__ void __launch_bounds__(256)
k_threshold_bytes(const double *__restrict__ S, int64_t D, int32_t K, double thr, uint8_t *__restrict__ Bm,
                  int64_t Dp, int64_t col0) {
    __shared__ __align__(16) uint8_t tile[TB_K][TB_D + 16];    // [k][d]: the store phase reads 16 consecutive d of one k
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const int64_t d0 = (int64_t)blockIdx.x * TB_D;
    const int32_t k0 = blockIdx.y * TB_K;
    const int32_t k = k0 + tx;
#pragma unroll
    for (int r0 = 0; r0 < TB_D; r0 += 32) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t d = d0 + r0 + ty + 8 * u;
            v[u] = (d < D && k < K) ? __ldcs(S + d * K + k) : -1.0;   // streamed: S is read once
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t d = d0 + r0 + ty + 8 * u;
            tile[tx][r0 + ty + 8 * u] = (d < D && k < K && v[u] >= thr) ? 1 : 0;
        }
    }
    __syncthreads();
    // thread t: keyphrase row t >> 3 of the tile, 16-byte piece t & 7 of its 128 bytes
    const int kr = threadIdx.x >> 3, piece = threadIdx.x & 7;
    const int32_t ko = k0 + kr;
    const int64_t dd = d0 + 16 * piece;
    if (ko < K && dd < D) {
        uint8_t *dst = Bm + (int64_t)ko * Dp + col0 + dd;
        if (dd + 16 <= D && (col0 & 15) == 0) {
            *reinterpret_cast<uint4 *>(dst) = *reinterpret_cast<const uint4 *>(&tile[kr][16 * piece]);
        } else {
            for (int i = 0; i < 16 && dd + i < D; ++i) dst[i] = tile[kr][16 * piece + i];
        }
    }
}

__global__ void __launch_bounds__(CT_THREADS, 1)
k_cooc_umma(const uint8_t *__restrict__ Bm, int64_t Dp, int32_t Kp, int32_t K, int32_t *__restrict__ C) {
    extern __shared__ __align__(1024) uint8_t ct_smem[];
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ uint32_t s_tmem;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    // C is symmetric: only the tiles on and above the diagonal are computed, each is stored twice
    if (blockIdx.x < blockIdx.y) return;
    const int32_t i0 = blockIdx.y * CT_TILE, j0 = blockIdx.x * CT_TILE;
    const bool mirror = blockIdx.x != blockIdx.y;

    if (warp == 0) {
        // 128 TMEM columns x 128 lanes of 32-bit accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "n"(128));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (t == 32) {
        mbar_init(smem_u32(&s_bar[0]), 1);
        mbar_init(smem_u32(&s_bar[1]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = s_tmem;

    // instruction descriptor (cute::UMMA::InstrDescriptor): D = s32, A = B = u8, K-major, N = 128, M = 128
    const uint32_t idesc = (2u << 4) | ((uint32_t)(CT_TILE >> 3) << 17) | ((uint32_t)(CT_TILE >> 4) << 24);
    const int chunks = (int)(Dp / CT_BK);

    for (int c = 0; c < chunks; ++c) {
        const int s = c & 1;
        uint8_t *sa = ct_smem + s * CT_STAGE_BYTES;
        uint8_t *sb = sa + CT_TILE * CT_BK;
        if (c >= 2) {  // the MMAs that read this stage two chunks ago must have finished
            mbar_wait(smem_u32(&s_bar[s]), (uint32_t)(((c >> 1) - 1) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;");
        }
        // stage A (rows i0..) and B (rows j0..): 16-byte pieces into the core-matrix layout
        const int64_t col = (int64_t)c * CT_BK;
#pragma unroll
        for (int q = 0; q < (CT_TILE * CT_BK / 16) / CT_THREADS; ++q) {
            const int piece = q * CT_THREADS + t;   // 0 .. 1023
            const int r = piece >> 3, kc = piece & 7;  // row, 16-byte chunk along K
            const uint32_t off = (uint32_t)((r >> 3) * 1024 + kc * 128 + (r & 7) * 16);
            const uint4 va = *reinterpret_cast<const uint4 *>(Bm + (int64_t)(i0 + r) * Dp + col + kc * 16);
            const uint4 vb = *reinterpret_cast<const uint4 *>(Bm + (int64_t)(j0 + r) * Dp + col + kc * 16);
            *reinterpret_cast<uint4 *>(sa + off) = va;
            *reinterpret_cast<uint4 *>(sb + off) = vb;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
        __syncthreads();
        if (warp == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;");
            if (lane == 0) {
                const uint32_t a_base = smem_u32(sa), b_base = smem_u32(sb);
#pragma unroll
                for (int k = 0; k < CT_BK / 32; ++k) {  // K = 32 bytes per instruction = 2 core matrices
                    const uint64_t da = umma_desc(a_base + k * 256), db = umma_desc(b_base + k * 256);
                    const uint32_t accumulate = (c > 0 || k > 0) ? 1u : 0u;
                    asm volatile(
                        "{\n\t"
                        ".reg .pred p;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
                        "}\n" ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
                        : "memory");
                }
                // arrives on the stage's mbarrier when every MMA issued so far has completed
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&s_bar[s]))
                             : "memory");
            }
            __syncwarp();
        }
    }
    // all MMAs complete in order: wait for the commit of the last chunk
    mbar_wait(smem_u32(&s_bar[(chunks - 1) & 1]), (uint32_t)(((chunks - 1) >> 1) & 1));
    asm volatile("tcgen05.fence::after_thread_sync;");

    // ---- epilogue: warp w owns TMEM lanes 32w..32w+31 = rows i0+32w.. of the tile
    const int32_t row = i0 + warp * 32 + lane;
#pragma unroll 1
    for (int cb = 0; cb < CT_TILE; cb += 32) {
        uint32_t v[32];
        const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
              "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
              "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (row < K) {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
                const int32_t colj = j0 + cb + q;
                if (colj < K) C[(int64_t)row * K + colj] = (int32_t)v[q];
            }
            if (mirror) {   // the transposed tile: for a fixed q the 32 lanes write 32 consecutive ints
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const int32_t colj = j0 + cb + q;
                    if (colj < K) C[(int64_t)colj * K + row] = (int32_t)v[q];
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(128));
}

// ------------------------------------------------------------------------------------------
// Pipelined version (default): 128 x 256 tile of C per CTA, warp-specialised.
//   warps 0-3  producers: 16-byte cp.async copies of the A (128 rows) and B (256 rows) slices straight
//              into the core-matrix layout of a 4-stage ring (48 KB per stage); completion is signalled
//              with cp.async.mbarrier.arrive.noinc on the stage's "full" barrier.  Afterwards the same
//              warps run the epilogue (TMEM lanes 32w..32w+31).
//   warp 4     one elected thread waits for "full", issues four tcgen05.mma.kind::i8 (M = 128, N = 256,
//              K = 32) per stage and commits to the stage's "empty" barrier, which releases the slot.
// Operand traffic per output element is 0.75x that of the 128 x 128 kernel and the loads of stage
// s+1..s+3 overlap the MMAs of stage s (the simple kernel serialised them with a block barrier).
// ------------------------------------------------------------------------------------------
constexpr int CP_TM = 128, CP_TN = 256, CP_BK = 128, CP_STAGES = 4;
constexpr int CP_A_BYTES = CP_TM * CP_BK, CP_B_BYTES = CP_TN * CP_BK;
constexpr int CP_STAGE_BYTES = CP_A_BYTES + CP_B_BYTES;   // 48 KB
constexpr int CP_THREADS = 160;                            // 4 producer/epilogue warps + 1 MMA warp

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

__global__ void __launch_bounds__(CP_THREADS, 1)
k_cooc_umma_pipe(const uint8_t *__restrict__ Bm, int64_t Dp, int32_t K, int32_t *__restrict__ C) {
    extern __shared__ __align__(1024) uint8_t cp_smem[];
    __shared__ __align__(8) uint64_t s_full[CP_STAGES], s_empty[CP_STAGES], s_done;
    __shared__ uint32_t s_tmem;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const int32_t i0 = blockIdx.y * CP_TM, j0 = blockIdx.x * CP_TN;
    // symmetric result: a tile whose columns all lie left of its rows is covered by the transposed stores of another tile
    if (j0 + CP_TN <= i0) return;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "n"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (t == 32) {
        for (int i = 0; i < CP_STAGES; ++i) {
            mbar_init(smem_u32(&s_full[i]), 128);   // one (non-incrementing) arrival per producer thread
            mbar_init(smem_u32(&s_empty[i]), 1);    // one tcgen05.commit
        }
        mbar_init(smem_u32(&s_done), 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = s_tmem;
    const int chunks = (int)(Dp / CP_BK);

    if (warp < 4) {
        // ---- producers
        for (int c = 0; c < chunks; ++c) {
            const int st = c % CP_STAGES, round = c / CP_STAGES;
            if (round > 0) mbar_wait(smem_u32(&s_empty[st]), (uint32_t)((round - 1) & 1));
            const uint32_t sa = smem_u32(cp_smem + st * CP_STAGE_BYTES), sb = sa + CP_A_BYTES;
            const int64_t col = (int64_t)c * CP_BK;
#pragma unroll
            for (int q = 0; q < (CP_TM * CP_BK / 16) / 128; ++q) {     // 8 pieces of A per thread
                const int piece = q * 128 + t;
                const int r = piece >> 3, kc = piece & 7;
                cp_async16(sa + (uint32_t)((r >> 3) * 1024 + kc * 128 + (r & 7) * 16), Bm + (int64_t)(i0 + r) * Dp + col + kc * 16);
            }
#pragma unroll
            for (int q = 0; q < (CP_TN * CP_BK / 16) / 128; ++q) {     // 16 pieces of B per thread
                const int piece = q * 128 + t;
                const int r = piece >> 3, kc = piece & 7;
                cp_async16(sb + (uint32_t)((r >> 3) * 1024 + kc * 128 + (r & 7) * 16), Bm + (int64_t)(j0 + r) * Dp + col + kc * 16);
            }
            // arrives on "full" once all cp.async of this thread have landed
            asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(&s_full[st])) : "memory");
        }
    } else if (lane == 0) {
        // ---- MMA issuer
        const uint32_t idesc = (2u << 4) | ((uint32_t)(CP_TN >> 3) << 17) | ((uint32_t)(CP_TM >> 4) << 24);
        for (int c = 0; c < chunks; ++c) {
            const int st = c % CP_STAGES, round = c / CP_STAGES;
            mbar_wait(smem_u32(&s_full[st]), (uint32_t)(round & 1));
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // cp.async (generic proxy) writes -> tensor-core reads
            asm volatile("tcgen05.fence::after_thread_sync;");
            const uint32_t a_base = smem_u32(cp_smem + st * CP_STAGE_BYTES), b_base = a_base + CP_A_BYTES;
#pragma unroll
            for (int k = 0; k < CP_BK / 32; ++k) {
                const uint64_t da = umma_desc(a_base + k * 256), db = umma_desc(b_base + k * 256);
                const uint32_t accumulate = (c > 0 || k > 0) ? 1u : 0u;
                asm volatile(
                    "{\n\t"
                    ".reg .pred p;\n\t"
                    "setp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
                    "}\n" ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
                    : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&s_empty[st]))
                         : "memory");
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&s_done)) : "memory");
    }

    // ---- epilogue (warps 0-3): warp w owns TMEM lanes 32w..32w+31 = rows i0+32w.. of the tile
    if (warp < 4) {
        mbar_wait(smem_u32(&s_done), 0u);
        asm volatile("tcgen05.fence::after_thread_sync;");
        const int32_t row = i0 + warp * 32 + lane;
#pragma unroll 1
        for (int cb = 0; cb < CP_TN; cb += 32) {
            uint32_t v[32];
            const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)cb;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (row < K) {
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const int32_t colj = j0 + cb + q;
                    if (colj < K) {
                        C[(int64_t)row * K + colj] = (int32_t)v[q];
                        C[(int64_t)colj * K + row] = (int32_t)v[q];   // the transposed element (same value where tiles overlap)
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(256));
}

// ------------------------------------------------------------------------------------------
// TMA-fed cluster version (default): the same 128 x 256 tile per CTA, but
//   * the operands arrive by TMA (cp.async.bulk.tensor.2d, SASS UTMALDG) as 128-row x 128-byte boxes in the 128-byte
//     swizzled K-major layout the tensor cores read directly (UMMA descriptors with SWIZZLE_128B, 32-byte steps
//     along K inside the swizzle atom): ONE thread issues the loads, nobody computes addresses;
//   * two CTAs that own vertically adjacent tiles (same 256 columns of C = the same rows of B as their N-side operand)
//     form a thread-block cluster: each loads ONE half of that operand and multicasts it into both CTAs' shared
//     memory, so the pair pulls 512 operand rows per K-slab out of L2 instead of 768.  The profile of the cp.async
//     kernel (profiles/r2): tensor pipe 15 % active, L2 -> SM traffic 126 GB per launch at 8.2 TB/s -- operand feed
//     from L2 is the limit, not the tensor cores;
//   * a stage is released to BOTH producers by the tcgen05.commit of both consumers (multicast commit on the
//     stage's "empty" barriers, arrival count 2), since each producer writes into both CTAs.
// Warps: 0 = TMA producer (one lane), 1 = MMA issuer (one lane), 2-5 = epilogue (TMEM quarter = warp & 3).
// ------------------------------------------------------------------------------------------
constexpr int CQ_TM = 128, CQ_TN = 256, CQ_BK = 128, CQ_STAGES = 4;
constexpr int CQ_BOX_BYTES = 128 * CQ_BK;                          // one TMA box: 128 rows x 128 bytes = 16 KB
constexpr int CQ_STAGE_BYTES = (CQ_TM + CQ_TN) * CQ_BK;            // A box + two B boxes = 48 KB
constexpr int CQ_THREADS = 192;

// K-major SWIZZLE_128B shared-memory matrix descriptor: 8-row x 128-byte atoms, 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4)        // start address, 16-byte units
           | ((uint64_t)1 << 16)                       // leading byte offset: unused for swizzled K-major layouts
           | ((uint64_t)(1024 >> 4) << 32)             // stride byte offset: next 8-row group
           | (1ull << 46)                              // descriptor version 1 (sm_100)
           | (2ull << 61);                             // layout type SWIZZLE_128B
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__global__ void __cluster_dims__(1, 2, 1) __launch_bounds__(CQ_THREADS, 1)
k_cooc_umma_tma(const __grid_constant__ CUtensorMap tmap, int64_t Dp, int32_t K, int32_t *__restrict__ C) {
    extern __shared__ __align__(1024) uint8_t cq_smem_raw[];
    __shared__ __align__(8) uint64_t s_full[CQ_STAGES], s_empty[CQ_STAGES], s_done;
    __shared__ uint32_t s_tmem;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
    const uint32_t rank = cluster_ctarank();                 // 0 / 1: upper / lower tile of the pair
    const int32_t i0 = blockIdx.y * CQ_TM, j0 = blockIdx.x * CQ_TN;
    const int32_t pair_i0 = (int32_t)(blockIdx.y & ~1u) * CQ_TM;
    // symmetric result: a PAIR whose columns all lie left of its rows is covered by the transposed stores of other tiles
    // (the decision must be the same for both CTAs of a cluster: they synchronise with each other)
    if (j0 + CQ_TN <= pair_i0) return;
    // dynamic shared memory: the swizzle atoms need 1024-byte alignment
    uint8_t *cq_smem = reinterpret_cast<uint8_t *>(((uintptr_t)cq_smem_raw + 1023) & ~(uintptr_t)1023);

    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "n"(256));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (t == 0) {
        for (int i = 0; i < CQ_STAGES; ++i) {
            mbar_init(smem_u32(&s_full[i]), 1);     // the producer's arrive.expect_tx; the bytes of both CTAs' loads complete it
            mbar_init(smem_u32(&s_empty[i]), 2);    // one tcgen05.commit from each CTA of the pair
        }
        mbar_init(smem_u32(&s_done), 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    cluster_sync_all();     // the peer's barriers exist before anything of ours can land there
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = s_tmem;
    const int chunks = (int)(Dp / CQ_BK);

    if (warp == 0) {
        if (lane == 0) {
            // ---- TMA producer
            const uint64_t tm = reinterpret_cast<uint64_t>(&tmap);
            for (int c = 0; c < chunks; ++c) {
                const int st = c % CQ_STAGES, round = c / CQ_STAGES;
                if (round > 0) mbar_wait(smem_u32(&s_empty[st]), (uint32_t)((round - 1) & 1));
                const uint32_t full = smem_u32(&s_full[st]);
                const uint32_t sa = smem_u32(cq_smem + st * CQ_STAGE_BYTES), sb = sa + CQ_BOX_BYTES;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(full), "r"((uint32_t)CQ_STAGE_BYTES) : "memory");
                const int32_t x = c * CQ_BK;
                // own M-side operand: rows i0 .. i0 + 127
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                             ::"r"(sa), "l"(tm), "r"(x), "r"(i0), "r"(full) : "memory");
                // this CTA's half of the shared N-side operand (rows j0 + 128 rank ..), into both CTAs of the pair
                asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster "
                             "[%0], [%1, {%2, %3}], [%4], %5;"
                             ::"r"(sb + rank * CQ_BOX_BYTES), "l"(tm), "r"(x), "r"(j0 + (int32_t)rank * 128), "r"(full), "h"((uint16_t)3)
                             : "memory");
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ---- MMA issuer
            const uint32_t idesc = (2u << 4) | ((uint32_t)(CQ_TN >> 3) << 17) | ((uint32_t)(CQ_TM >> 4) << 24);
            for (int c = 0; c < chunks; ++c) {
                const int st = c % CQ_STAGES, round = c / CQ_STAGES;
                mbar_wait(smem_u32(&s_full[st]), (uint32_t)(round & 1));
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t a_base = smem_u32(cq_smem + st * CQ_STAGE_BYTES), b_base = a_base + CQ_BOX_BYTES;
#pragma unroll
                for (int k = 0; k < CQ_BK / 32; ++k) {
                    const uint64_t da = umma_desc_sw128(a_base + k * 32), db = umma_desc_sw128(b_base + k * 32);
                    const uint32_t accumulate = (c > 0 || k > 0) ? 1u : 0u;
                    asm volatile(
                        "{\n\t"
                        ".reg .pred p;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
                        "}\n" ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
                        : "memory");
                }
                // the slot goes back to BOTH producers: each of them writes into both CTAs
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                             ::"r"(smem_u32(&s_empty[st])), "h"((uint16_t)3) : "memory");
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(&s_done)) : "memory");
        }
    } else {
        // ---- epilogue (warps 2-5): TMEM lanes 32 q .. 32 q + 31 = rows i0 + 32 q .. of the tile, q = warp & 3
        const int q4 = warp & 3;
        mbar_wait(smem_u32(&s_done), 0u);
        asm volatile("tcgen05.fence::after_thread_sync;");
        const int32_t row = i0 + q4 * 32 + lane;
#pragma unroll 1
        for (int cb = 0; cb < CQ_TN; cb += 32) {
            uint32_t v[32];
            const uint32_t taddr = tmem + ((uint32_t)(q4 * 32) << 16) + (uint32_t)cb;
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (row < K) {
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const int32_t colj = j0 + cb + q;
                    if (colj < K) {
                        C[(int64_t)row * K + colj] = (int32_t)v[q];
                        C[(int64_t)colj * K + row] = (int32_t)v[q];   // the transposed element (same value where tiles overlap)
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    cluster_sync_all();     // nobody leaves while the peer may still signal its barriers
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(256));
}

// the tensor map of B (uint8 [Kp][Dp], 128-row x 128-byte boxes, 128-byte swizzle) through the driver entry point
// (libcuda is not linked: the runtime hands the function out); false = no TMA on this driver, use the cp.async kernel
static bool make_b_tensor_map(const uint8_t *Bm, int64_t Dp, int32_t Kp, CUtensorMap *out) {
    typedef CUresult (*EncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeTiled encode = nullptr;
    static bool looked = false;
    if (!looked) {
        looked = true;
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            encode = (EncodeTiled)fn;
        else
            cudaGetLastError();
    }
    if (!encode) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)Dp, (cuuint64_t)Kp};
    const cuuint64_t gstride[1] = {(cuuint64_t)Dp};
    const cuuint32_t box[2] = {(cuuint32_t)CQ_BK, 128u};
    const cuuint32_t estride[2] = {1u, 1u};
    return encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t *>(Bm), gdim, gstride, box, estride,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

void cooc_padding(int64_t D, int32_t K, int64_t *Dp, int32_t *Kp) {
    *Dp = (D + CT_BK - 1) / CT_BK * CT_BK;
    *Kp = (K + CP_TN - 1) / CP_TN * CP_TN;   // rows padded to the larger tile edge (256)
}

void threshold_bytes(const double *S_DxK, int64_t D, int32_t K, double threshold, uint8_t *Bm, int64_t Dp, int64_t col0,
                     cudaStream_t s) {
    dim3 tg((unsigned)((D + TB_D - 1) / TB_D), (unsigned)((K + TB_K - 1) / TB_K));
    EAST_BYTES(8.0 * (double)D * K + (double)K * D);
    EAST_LAUNCH(k_threshold_bytes, tg, 256, 0, s, S_DxK, D, K, threshold, Bm, Dp, col0);
}

void cooc_counts_tc(const double *S_DxK, int64_t D, int32_t K, double threshold, int32_t *C, cudaStream_t s, int simple) {
    int64_t Dp;
    int32_t Kp;
    cooc_padding(D, K, &Dp, &Kp);
    DevBuf<uint8_t> Bm((size_t)Kp * (size_t)Dp, s);
    EAST_CUDA(cudaMemsetAsync(Bm.p, 0, (size_t)Kp * (size_t)Dp, s));  // padding rows / columns are zero
    threshold_bytes(S_DxK, D, K, threshold, Bm.p, Dp, 0, s);
    cooc_counts_bytes(Bm.p, Dp, Kp, K, C, s, simple);
}

void cooc_counts_bytes(const uint8_t *Bm, int64_t Dp, int32_t Kp, int32_t K, int32_t *C, cudaStream_t s, int simple) {
    const int smem = 2 * CT_STAGE_BYTES + 1024, smem_pipe = CP_STAGES * CP_STAGE_BYTES + 1024;
    ensure_dynamic_smem((const void *)k_cooc_umma, smem);
    ensure_dynamic_smem((const void *)k_cooc_umma_pipe, smem_pipe);
    CUtensorMap tmap;
    if (simple == 0 && make_b_tensor_map(Bm, Dp, Kp, &tmap)) {
        const int smem_tma = CQ_STAGES * CQ_STAGE_BYTES + 1024;
        ensure_dynamic_smem((const void *)k_cooc_umma_tma, smem_tma);
        dim3 grid(Kp / CQ_TN, Kp / CQ_TM);   // Kp is a multiple of 256: an even number of tile rows, clusters of (1, 2)
        EAST_LAUNCH(k_cooc_umma_tma, grid, CQ_THREADS, smem_tma, s, tmap, Dp, K, C);
    } else if (simple == 1) {
        dim3 grid(Kp / CT_TILE, Kp / CT_TILE);
        EAST_LAUNCH(k_cooc_umma, grid, CT_THREADS, smem, s, Bm, Dp, Kp, K, C);
    } else {
        dim3 grid(Kp / CP_TN, Kp / CP_TM);
        EAST_LAUNCH(k_cooc_umma_pipe, grid, CP_THREADS, smem_pipe, s, Bm, Dp, K, C);
    }
}

}  // namespace east
