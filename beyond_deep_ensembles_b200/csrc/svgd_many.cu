// svgd_many.cu — SVGD with 33 to 64 particles (runtime n): particle-tiled K1 (+K1b) and K2 on FP32 CUDA cores.
//
//   K1  svgd_pairdist_many_kernel : one persistent CTA per SM; a producer lane streams [n x 256] tensor-map boxes of X
//       into a shared-memory ring.  The rows are cut into blocks of 8 (the last one zero-padded) and every thread
//       owns one block pair (I <= J) of the upper triangle: 8 x 8 = 64 packed-fp32 accumulators over a column pair,
//       direct differences (x_i - x_j)^2 with FADD2 / FFMA2.  Every kManyFlushTiles tiles the S threads of a block
//       pair sum their partials in fp32 (fixed shuffle tree) and one of them adds the sum to the CTA's fp64
//       accumulator; the CTA partials then go through grid_reduce_fp64 like every other K1 form.
//   K1b bandwidth_sorted with its 64^2-entry sort buffers in dynamic shared memory (the ring area in K1's tail).
//   K2  svgd_apply_many_kernel    : X and G as [n x 128] tensor-map boxes through the same kind of ring; K^T and A^T
//       in shared memory; a warp owns 16 output rows of a 128-column tile, a thread one column quad of them.
//
// Results are bit-identical from run to run: every sum has one fixed order for a given grid.
#include "svgd_kernels.cuh"

namespace bde {

constexpr int kManyMaxN = BDE_MAX_PARTICLES;   // 64
constexpr int kManyRB = 8;                     // K1 rows per register block
constexpr int kManyMaxBlockPairs = (kManyMaxN / kManyRB) * (kManyMaxN / kManyRB + 1) / 2;   // 36
constexpr int kManyPdTC = kTmaBoxCols;         // K1 tile columns (one box)
constexpr int kManyPdStageFloats = kManyMaxN * kManyPdTC;   // a stage always has 64 row slots; rows >= n stay zero
constexpr int kManyPdStages = 3;               // 3 x 64 KB
// fp32 window: the S threads of a block pair together see 256 columns per tile, i.e. 256 * kManyFlushTiles columns
// (8192) go into one fp32 sum before it is flushed to fp64 — the same bound as the staged K1's 32 lanes x 4 columns x
// kFlushTiles (tests/test_svgd_matrix.py:value_range).
constexpr int kManyFlushTiles = 32;
constexpr int kManyPdMaxThreads = 256;         // consumers + a producer warp

constexpr int kManyApTC = 128;                 // K2 tile columns
constexpr int kManyApRB = 16;                  // K2 output rows per warp
constexpr int kManyApSets = 2;                 // tile sets: set c consumes the tiles it = c (mod 2) of the ring
constexpr int kManyApRingBytes = 192 * 1024;
constexpr int kManyApMaxThreads = kManyApSets * (kManyMaxN / kManyApRB) * 32 + 32;

struct ManyPdGeom {
    int nb, nbp, S, consumers;
};
__host__ __device__ inline ManyPdGeom many_pd_geom(int n) {
    ManyPdGeom g;
    g.nb = (n + kManyRB - 1) / kManyRB;
    g.nbp = g.nb * (g.nb + 1) / 2;
    // threads per block pair: the largest power of two that keeps the CTA at 8 warps (at most two per SM
    // sub-partition, so the 128 accumulator registers fit the 255-register budget): 4 to 7 consumer warps
    g.S = 16;
    while (g.nbp * g.S > kManyPdMaxThreads - 32) g.S >>= 1;
    g.consumers = (g.nbp * g.S + 31) & ~31;
    return g;
}
// shared memory of K1b at n particles: sd, sk [n*n fp64], then the sort buffers s_key [fp64] and s_ord [int32] of
// pow2_ceil(n*n) entries each
__host__ __device__ constexpr size_t many_bw_bytes(int n) {
    return 2 * sizeof(double) * n * n + (sizeof(double) + sizeof(int)) * pow2_ceil(n * n);
}
__device__ __forceinline__ void many_bandwidth(const double* dist, int n, const BandwidthParams& bp, double* sd) {
    double* sk = sd + n * n;
    double* key = sk + n * n;
    bandwidth_sorted(dist, n, bp, sd, sk, key, reinterpret_cast<int*>(key + pow2_ceil(n * n)));
}

__global__ void __launch_bounds__(kManyPdMaxThreads, 1)
svgd_pairdist_many_kernel(const __grid_constant__ CUtensorMap mapX, int n, int64_t D, double* __restrict__ dist,
                          int accumulate, void* ws, int fuse_bandwidth, BandwidthParams bp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* ring = reinterpret_cast<float*>(smem_raw);   // [kManyPdStages][64][256]
    __shared__ double wacc[kManyMaxBlockPairs][kManyRB * kManyRB];
    __shared__ __align__(8) uint64_t full_bar[kManyPdStages];
    __shared__ __align__(8) uint64_t empty_bar[kManyPdStages];

    const ManyPdGeom geo = many_pd_geom(n);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int P = pair_count(n);
    const int rows = geo.nb * kManyRB;
    for (int k = tid; k < geo.nbp * kManyRB * kManyRB; k += nthreads) (&wacc[0][0])[k] = 0.0;
    for (int e = tid; e < kManyPdStages * (rows - n) * kManyPdTC; e += nthreads) {   // padding rows: zero once
        const int s = e / ((rows - n) * kManyPdTC), r = e - s * (rows - n) * kManyPdTC;
        ring[s * kManyPdStageFloats + n * kManyPdTC + r] = 0.0f;
    }
    if (tid == 0) {
        for (int s = 0; s < kManyPdStages; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], geo.consumers / 32);
        }
        mbar_fence_init();
        tma_prefetch_map(&mapX);
    }
    __syncthreads();

    const int64_t ntiles = (D + kManyPdTC - 1) / kManyPdTC;
    if (tid >= geo.consumers) {
        if (tid == geo.consumers) {
            int it = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
                const int s = it % kManyPdStages;
                const uint32_t use = static_cast<uint32_t>(it / kManyPdStages);
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                // the box always delivers (and counts) n x 256 floats: columns beyond D arrive as zeros
                mbar_arrive_expect_tx(&full_bar[s], static_cast<uint32_t>(n) * kManyPdTC * 4u);
                tma_load_2d(ring + s * kManyPdStageFloats, &mapX, static_cast<int>(t * kManyPdTC), 0, &full_bar[s]);
            }
        }
    } else {
        const int lane = tid & 31;
        const int S = geo.S, M = (kManyPdTC / 2) / S;   // column pairs of a tile per thread (16 or 32)
        const int bpi = tid / S, k = tid - bpi * S;
        const bool active = bpi < geo.nbp;
        int I = 0, r = active ? bpi : 0;
        while (r >= geo.nb - I) {
            r -= geo.nb - I;
            ++I;
        }
        const int J = I + r;
        f32x2 acc[kManyRB * kManyRB];
#pragma unroll
        for (int q = 0; q < kManyRB * kManyRB; ++q) acc[q] = 0ull;
        int it = 0;
        int64_t t = blockIdx.x;
        bool more = true;
        while (more) {   // one flush site: every kManyFlushTiles tiles (uniform over the CTA: shuffles stay convergent)
            for (int f = 0; f < kManyFlushTiles && t < ntiles; ++f, t += gridDim.x, ++it) {
                const int s = it % kManyPdStages;
                mbar_wait(&full_bar[s], static_cast<uint32_t>(it / kManyPdStages) & 1u);
                if (active) {
                    const float* sI = ring + s * kManyPdStageFloats + I * kManyRB * kManyPdTC;
                    const float* sJ = ring + s * kManyPdStageFloats + J * kManyRB * kManyPdTC;
#pragma unroll 1
                    for (int m = 0; m < M; ++m) {
                        // staggered by block pair: the lanes of a half-warp read 16 distinct column pairs (no bank conflict)
                        const int cp = k + S * ((m + bpi) & (M - 1));
                        f32x2 xi[kManyRB];
#pragma unroll
                        for (int a = 0; a < kManyRB; ++a) {
                            const float2 v = *reinterpret_cast<const float2*>(sI + a * kManyPdTC + 2 * cp);
                            xi[a] = pack2(v.x, v.y);
                        }
#pragma unroll
                        for (int b = 0; b < kManyRB; ++b) {
                            const float2 v = *reinterpret_cast<const float2*>(sJ + b * kManyPdTC + 2 * cp);
                            const f32x2 xj = pack2(v.x, v.y);
#pragma unroll
                            for (int a = 0; a < kManyRB; ++a) {
                                const f32x2 d = sub2(xi[a], xj);
                                acc[a * kManyRB + b] = fma2(d, d, acc[a * kManyRB + b]);
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);
            }
            more = t < ntiles;
#pragma unroll
            for (int q = 0; q < kManyRB * kManyRB; ++q) {
                float lo, hi;
                unpack2(acc[q], lo, hi);
                acc[q] = 0ull;
                float v = lo + hi;
                for (int off = S >> 1; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
                if (active && k == 0) wacc[bpi][q] += static_cast<double>(v);
            }
        }
    }
    __syncthreads();   // every issued box has been consumed: the ring is free for the tail
    griddep_launch();   // streaming done: a dependent K2 may become resident during the tail

    double* cta_vals = reinterpret_cast<double*>(smem_raw);
    double* total = cta_vals + P;
    for (int p = tid; p < P; p += nthreads) {
        const int i = pair_row(p, n), j = p - pair_index(i, i + 1, n) + i + 1;
        const int I = i / kManyRB, J = j / kManyRB;
        const int bpi = I * geo.nb - I * (I - 1) / 2 + (J - I);
        cta_vals[p] = wacc[bpi][(i % kManyRB) * kManyRB + (j % kManyRB)];
    }
    __syncthreads();
    if (!grid_reduce_fp64(cta_vals, P, ws, total)) return;
    for (int e = tid; e < n * n; e += nthreads) {
        const int i = e / n, j = e - i * n;
        double v = 0.0;
        if (i != j) v = total[i < j ? pair_index(i, j, n) : pair_index(j, i, n)];
        if (accumulate) v += dist[e];
        dist[e] = v;
    }
    if (fuse_bandwidth && !peer_exchange_failed(ws)) {
        __syncthreads();
        many_bandwidth(dist, n, bp, total + P);
    }
}

__global__ void __launch_bounds__(256) svgd_bandwidth_many_kernel(const double* __restrict__ dist, int n, BandwidthParams bp) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    many_bandwidth(dist, n, bp, reinterpret_cast<double*>(smem_raw));
}

// out_i = sum_j K_ij g_j + A_ij x_j.  FMA order of every output element: j = 0, 1, ..., n-1, and for each j first
// K_ij g_j, then A_ij x_j, starting from 0 (the order of the generic and the register-resident kernels).
__global__ void __launch_bounds__(kManyApMaxThreads, 1)
svgd_apply_many_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapG,
                       float* __restrict__ out, const float* __restrict__ K, const float* __restrict__ A, int n,
                       int64_t D, int64_t ldo, int nst) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* ring = reinterpret_cast<float*>(smem_raw);   // [nst]{X box [n][128], G box [n][128]}
    // transposed, zero-padded coefficients: sKT[j][i] = K[i][j]
    __shared__ __align__(16) float sKT[kManyMaxN][kManyMaxN];
    __shared__ __align__(16) float sAT[kManyMaxN][kManyMaxN];
    __shared__ __align__(8) uint64_t full_bar[8];
    __shared__ __align__(8) uint64_t empty_bar[8];

    const int nrb = (n + kManyApRB - 1) / kManyApRB;   // warps per tile set
    const int consumers = kManyApSets * nrb * 32;
    const int stage_floats = 2 * n * kManyApTC;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < nst; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], nrb);   // released by the warps of the one set that consumed it
        }
        mbar_fence_init();
        tma_prefetch_map(&mapX);
        tma_prefetch_map(&mapG);
    }
    __syncthreads();
    // the producer streams X / G at once (no K1 writes them); the consumers wait for K1 before they read K / A
    const int64_t ntiles = (D + kManyApTC - 1) / kManyApTC;
    if (tid >= consumers) {
        if (tid == consumers) {
            int s = 0;
            uint32_t use = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, s = (s + 1 == nst) ? 0 : s + 1, use += (s == 0)) {
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                mbar_arrive_expect_tx(&full_bar[s], static_cast<uint32_t>(stage_floats) * 4u);
                float* sx = ring + static_cast<size_t>(s) * stage_floats;
                tma_load_2d(sx, &mapX, static_cast<int>(t * kManyApTC), 0, &full_bar[s]);
                tma_load_2d(sx + n * kManyApTC, &mapG, static_cast<int>(t * kManyApTC), 0, &full_bar[s]);
            }
        }
        griddep_wait();
        return;
    }
    griddep_wait();   // K / A come from the preceding K1 launch
    for (int e = tid; e < kManyMaxN * kManyMaxN; e += consumers) {
        const int j = e / kManyMaxN, i = e - j * kManyMaxN;
        const bool in = i < n && j < n;
        sKT[j][i] = in ? K[i * n + j] : 0.0f;
        sAT[j][i] = in ? A[i * n + j] : 0.0f;
    }
    asm volatile("bar.sync 1, %0;" ::"r"(consumers) : "memory");   // consumers only: the producer lane is in its loop
    const int lane = tid & 31, warp = tid >> 5;
    const int set = warp / nrb, rb = warp - set * nrb;
    const int row0 = rb * kManyApRB;
    int s = set;
    uint32_t use = 0;
    for (int64_t t = blockIdx.x + static_cast<int64_t>(set) * gridDim.x; t < ntiles;
         t += static_cast<int64_t>(kManyApSets) * gridDim.x, s += kManyApSets, use += (s >= nst), s -= (s >= nst) ? nst : 0) {
        // the other set consumed this stage's previous use: once that release is visible the full barrier can only be
        // in phase `use`, so the parity wait below cannot alias an older phase
        if (use > 0) mbar_wait(&empty_bar[s], (use - 1u) & 1u);
        mbar_wait(&full_bar[s], use & 1u);
        const float* sx = ring + static_cast<size_t>(s) * stage_floats + 4 * lane;
        const float* sg = sx + n * kManyApTC;
        f32x2 acc[kManyApRB][2];
#pragma unroll
        for (int i = 0; i < kManyApRB; ++i) acc[i][0] = acc[i][1] = 0ull;
#pragma unroll 2
        for (int j = 0; j < n; ++j) {
            const V4 g = lds_v4(sg + j * kManyApTC);
            const V4 x = lds_v4(sx + j * kManyApTC);
            apply_row<kManyApRB, true>(acc, g, x, &sKT[j][row0], &sAT[j][row0]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
        const int64_t c = t * kManyApTC + 4 * lane;
#pragma unroll
        for (int i = 0; i < kManyApRB; ++i) {
            if (row0 + i < n) {
                float* op = out + (row0 + i) * ldo + c;
                if (c + 4 <= D) {
                    V4 v;
                    v.lo = acc[i][0];
                    v.hi = acc[i][1];
                    stg_stream_v4(op, v);
                } else if (c < D) {   // ragged last quad: only the columns that exist
                    float v0, v1, v2, v3;
                    unpack2(acc[i][0], v0, v1);
                    unpack2(acc[i][1], v2, v3);
                    op[0] = v0;
                    if (c + 1 < D) op[1] = v1;
                    if (c + 2 < D) op[2] = v2;
                }
            }
        }
    }
}

int pairdist_many(const float* X, int n, int64_t D, int64_t ld, double* dist, int accumulate, void* ws, int fuse,
                  const BandwidthParams& bp, cudaStream_t st) {
    if (D == 0) {   // no columns: the distances are zero (or unchanged)
        if (!accumulate) BDE_RETURN_IF_CUDA(cudaMemsetAsync(dist, 0, sizeof(double) * n * n, st));
        return fuse ? bandwidth_many(dist, n, bp, st) : BDE_OK;
    }
    CUtensorMap mapX;
    int rc = encode_rows_tensor_map(&mapX, X, n, D, ld, kManyPdTC);
    if (rc != BDE_OK) return rc;
    constexpr int smem = kManyPdStages * kManyPdStageFloats * 4;
    static_assert(2 * sizeof(double) * pair_count(kManyMaxN) + many_bw_bytes(kManyMaxN) <= smem,
                  "K1's tail reuses the ring");
    static bool configured = false;
    if (!configured) {
        BDE_RETURN_IF_CUDA(cudaFuncSetAttribute(svgd_pairdist_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
    const int64_t ntiles = (D + kManyPdTC - 1) / kManyPdTC;
    int64_t grid = sm_count_cached();
    if (grid > kManyMaxCtas) grid = kManyMaxCtas;
    if (grid > ntiles) grid = ntiles;
    svgd_pairdist_many_kernel<<<static_cast<unsigned>(grid), many_pd_geom(n).consumers + 32, smem, st>>>(
        mapX, n, D, dist, accumulate, ws, fuse, bp);
    BDE_CHECK_LAUNCH();
    return BDE_OK;
}

int bandwidth_many(const double* dist, int n, const BandwidthParams& bp, cudaStream_t st) {
    constexpr int smem = static_cast<int>(many_bw_bytes(kManyMaxN));
    static bool configured = false;
    if (!configured) {
        BDE_RETURN_IF_CUDA(cudaFuncSetAttribute(svgd_bandwidth_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
    svgd_bandwidth_many_kernel<<<1, 256, many_bw_bytes(n), st>>>(dist, n, bp);
    BDE_CHECK_LAUNCH();
    return BDE_OK;
}

int apply_many(const float* X, const float* G, float* out, const float* K, const float* A, int n, int64_t D,
               int64_t ldx, int64_t ldg, int64_t ldo, cudaStream_t st) {
    CUtensorMap mapX, mapG;
    int rc = encode_rows_tensor_map(&mapX, X, n, D, ldx, kManyApTC);
    if (rc == BDE_OK) rc = encode_rows_tensor_map(&mapG, G, n, D, ldg, kManyApTC);
    if (rc != BDE_OK) return rc;
    static bool configured = false;
    if (!configured) {
        BDE_RETURN_IF_CUDA(cudaFuncSetAttribute(svgd_apply_many_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kManyApRingBytes));
        configured = true;
    }
    const int stage_bytes = 2 * n * kManyApTC * 4;
    int nst = kManyApRingBytes / stage_bytes;
    if (nst > 8) nst = 8;
    const int64_t ntiles = (D + kManyApTC - 1) / kManyApTC;
    int64_t grid = sm_count_cached();
    if (grid > ntiles) grid = ntiles;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(kManyApSets * ((n + kManyApRB - 1) / kManyApRB) * 32 + 32);
    cfg.dynamicSmemBytes = static_cast<size_t>(nst) * stage_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_for_this_apply() ? 1 : 0;   // only when the caller vouched that K1 is the preceding launch
    pdl_for_this_apply() = false;
    BDE_RETURN_IF_CUDA(cudaLaunchKernelEx(&cfg, svgd_apply_many_kernel, mapX, mapG, out, K, A, n, D, ldo, nst));
    return BDE_OK;
}

}  // namespace bde
