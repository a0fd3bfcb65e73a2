// svgd_kernels.cuh — SVGD posterior update on sm_100a (kernel templates).
//
//   K1  svgd_pairdist : one streaming pass over X[n, D]; all n(n-1)/2 squared pair
//                       distances accumulated in packed-fp32 registers (FADD2/FFMA2),
//                       flushed to fp64 per warp, combined over CTAs in fixed order.
//   K1b svgd_bandwidth: n*n fp64 epilogue — median heuristic, RBF kernel K and the
//                       fused coefficient matrix A.
//   K2  svgd_apply    : out = K·G + A·X in one pass (FFMA2 with scalar-broadcast
//                       coefficients from shared memory).
//
// Reference arithmetic: src/algos/svgd.py:14-32 (rbf) and :83-97 (step).
#pragma once
#include "common.cuh"
#include "svgd_internal.h"

namespace bde {

constexpr int kPairTarget = 48;    // pair accumulators (x2 registers) per thread
constexpr int kFlushIters = 128;   // fp32 -> fp64 flush period (columns*4 per thread)
constexpr int kMaxCtasPairdist = 148 * 8 * 2;

__host__ __device__ constexpr int pair_count(int n) { return n * (n - 1) / 2; }
__host__ __device__ __forceinline__ constexpr int pair_index(int i, int j, int n) {  // i < j
    return i * (2 * n - i - 1) / 2 + (j - i - 1);
}
__host__ __device__ constexpr int pair_row(int p, int n) {  // row i of pair p in the row-major upper triangle
    int i = 0;
    while (p >= n - 1 - i) {
        p -= n - 1 - i;
        ++i;
    }
    return i;
}
// How the n(n-1)/2 pairs are shared between the thread groups of a CTA (one group keeps <= ~50 pair accumulators):
//  * contiguous: group g owns pairs [g*PG, (g+1)*PG) of the row-major upper triangle (n = 11, 12: two groups);
//  * blocked (n = 20; rows in four blocks A B C D of n/4): group 0 = all pairs inside A+B, group 1 = all pairs inside
//    C+D, group 2 = AxC then BxD, group 3 = AxD then BxC.  A group then touches n/2 rows at a time instead of all n:
//    half the row registers (no spills under the 168-register cap of the 9-warp CTA) and 60 instead of 80 LDS.128
//    per column quad.
__host__ __device__ constexpr int pair_groups_contig(int n) {
    return pair_count(n) <= kPairTarget ? 1 : (pair_count(n) + kPairTarget - 1) / kPairTarget;
}
// measured on B200 (D = 5e7 / 6e7): n = 20 staged K1 1.155 -> 0.957 ms blocked; n = 16 is faster contiguous on 3 groups
// (7 warps, 255 registers: 0.886 ms vs 0.952 ms blocked on 4 groups / 9 warps), so only four-group shapes are blocked
__host__ __device__ constexpr bool pair_blocked(int n) { return n % 4 == 0 && pair_groups_contig(n) > 3; }
__host__ __device__ constexpr int pair_groups(int n) { return pair_blocked(n) ? 4 : pair_groups_contig(n); }
__host__ __device__ constexpr int pairs_per_group(int n) {
    if (pair_blocked(n)) return pair_count(n / 2) > 2 * (n / 4) * (n / 4) ? pair_count(n / 2) : 2 * (n / 4) * (n / 4);
    return pair_groups(n) == 0 ? 0 : (pair_count(n) + pair_groups(n) - 1) / pair_groups(n);
}
// (group, slot inside the group's accumulator array) of pair (i, j), i < j
__host__ __device__ constexpr int pair_group_of(int i, int j, int n) {
    if (!pair_blocked(n)) return pair_index(i, j, n) / pairs_per_group(n);
    const int bs = n / 4, bi = i / bs, bj = j / bs;
    if (bj <= 1) return 0;
    if (bi >= 2) return 1;
    return (bj - bi == 2) ? 2 : 3;   // AxC, BxD -> 2;  AxD, BxC -> 3
}
__host__ __device__ constexpr int pair_slot_of(int i, int j, int n) {
    if (!pair_blocked(n)) return pair_index(i, j, n) % pairs_per_group(n);
    const int bs = n / 4, h = n / 2, bi = i / bs, bj = j / bs;
    if (bj <= 1) return pair_index(i, j, h);
    if (bi >= 2) return pair_index(i - h, j - h, h);
    return (bi == 0 ? 0 : bs * bs) + (i - bi * bs) * bs + (j - bj * bs);
}
__host__ __device__ constexpr int pairdist_tpb(int n) {
    // threads along columns; total CTA threads = tpb * groups
    return pair_groups(n) <= 2 ? 128 : (pair_groups(n) <= 4 ? 64 : 32);
}

// ---------------------------------------------------------------------------------
// K1
// ---------------------------------------------------------------------------------
template <int N, int G>
__device__ __forceinline__ void pair_accumulate(const V4 (&v)[N], f32x2 (&acc)[pairs_per_group(N) > 0 ? pairs_per_group(N) : 1]) {
    constexpr int PG = pairs_per_group(N);
    constexpr int LO = G * PG;
    constexpr int HI = (LO + PG < pair_count(N)) ? LO + PG : pair_count(N);
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j) {
            const int p = pair_index(i, j, N);
            if (p >= LO && p < HI) {
                const f32x2 d0 = sub2(v[i].lo, v[j].lo);
                const f32x2 d1 = sub2(v[i].hi, v[j].hi);
                acc[p - LO] = fma2(d0, d0, acc[p - LO]);
                acc[p - LO] = fma2(d1, d1, acc[p - LO]);
            }
        }
    }
}

// all pairs among R rows held in registers: slot = pair_index(a, b, R) + BASE
template <int R, int BASE, int PGN>
__device__ __forceinline__ void pairs_within(const V4 (&v)[R], f32x2 (&acc)[PGN]) {
#pragma unroll
    for (int a = 0; a < R; ++a) {
#pragma unroll
        for (int b = a + 1; b < R; ++b) {
            const int k = BASE + pair_index(a, b, R);
            const f32x2 d0 = sub2(v[a].lo, v[b].lo);
            const f32x2 d1 = sub2(v[a].hi, v[b].hi);
            acc[k] = fma2(d0, d0, acc[k]);
            acc[k] = fma2(d1, d1, acc[k]);
        }
    }
}
// all BS x BS pairs between row block `u` (in registers) and the block starting at row WB, whose rows are pulled one
// at a time (5 + 1 rows live instead of 10): slot = BASE + a*BS + b.  `loaded()` runs after the very last row load.
template <int BS, int BASE, int WB, bool LAST, int PGN, typename Row, typename Loaded>
__device__ __forceinline__ void pairs_cross(const V4 (&u)[BS], Row&& row, Loaded&& loaded, f32x2 (&acc)[PGN]) {
#pragma unroll
    for (int b = 0; b < BS; ++b) {
        const V4 w = row(WB + b);
        if (LAST && b == BS - 1) loaded();
#pragma unroll
        for (int a = 0; a < BS; ++a) {
            const int k = BASE + a * BS + b;
            const f32x2 d0 = sub2(u[a].lo, w.lo);
            const f32x2 d1 = sub2(u[a].hi, w.hi);
            acc[k] = fma2(d0, d0, acc[k]);
            acc[k] = fma2(d1, d1, acc[k]);
        }
    }
}
// Blocked decomposition (pair_blocked(N)): group G pulls only the rows it needs through `row(r)` (shared memory,
// global memory or a ragged-tail column) — in two phases for the cross groups — and calls `loaded()` once its last row
// is in registers (the staged kernel releases the ring stage there).
template <int N, int G, typename Row, typename Loaded>
__device__ __forceinline__ void pair_accumulate_blocked(Row&& row, Loaded&& loaded, f32x2 (&acc)[pairs_per_group(N)]) {
    constexpr int BS = N / 4, H = N / 2, PGN = pairs_per_group(N);
    if constexpr (G <= 1) {
        V4 v[H];
#pragma unroll
        for (int r = 0; r < H; ++r) v[r] = row(G * H + r);
        loaded();
        pairs_within<H, 0, PGN>(v, acc);
    } else {
        constexpr int P1 = (G == 2) ? 2 : 3;   // partner block of A;  B pairs with the other one of C / D
        constexpr int P2 = (G == 2) ? 3 : 2;
        V4 u[BS];
#pragma unroll
        for (int r = 0; r < BS; ++r) u[r] = row(r);
        pairs_cross<BS, 0, P1 * BS, false, PGN>(u, row, loaded, acc);
#pragma unroll
        for (int r = 0; r < BS; ++r) u[r] = row(BS + r);
        pairs_cross<BS, BS * BS, P2 * BS, true, PGN>(u, row, loaded, acc);
    }
}

// fp32 lane pairs -> warp sums -> this warp's fp64 accumulators (lane k%32 owns pair k).
// Transposing butterfly: 32 values held by every lane are reduced with 31 shuffles (16 + 8 + 4 + 2 + 1)
// instead of 32 five-step trees; after the last step lane L holds the warp total of value L.
// The summation order is fixed by the lane ids -> deterministic.
template <int PG>
__device__ __forceinline__ void flush_pairs(f32x2 (&acc)[PG > 0 ? PG : 1], double* __restrict__ wacc, int lane) {
    constexpr int NB = (PG + 31) / 32;
#pragma unroll
    for (int blk = 0; blk < NB; ++blk) {
        float v[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const int k = blk * 32 + i;
            if (k < PG) {
                float lo, hi;
                unpack2(acc[k], lo, hi);
                v[i] = lo + hi;
                acc[k] = 0ull;
            } else {
                v[i] = 0.0f;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const bool upper = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
                const float send = upper ? v[i] : v[i + off];
                const float keep = upper ? v[i + off] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
        }
        const int k = blk * 32 + lane;
        if (k < PG) wacc[k] += static_cast<double>(v[0]);
    }
}

template <int N, int G>
__device__ __forceinline__ void pairdist_body(const float* __restrict__ X, int64_t D, int64_t ld,
                                              double* __restrict__ wacc /* this warp's PG doubles */) {
    constexpr int PG = pairs_per_group(N);
    constexpr int NG = pair_groups(N);
    constexpr int TPB = pairdist_tpb(N);
    f32x2 acc[PG > 0 ? PG : 1];
#pragma unroll
    for (int k = 0; k < PG; ++k) acc[k] = 0ull;
    const int lane = threadIdx.x & 31;


    const int64_t nquads = D >> 2;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * TPB;
    // block-uniform trip count so that the warp shuffles in flush() stay convergent; one flush site:
    // every kFlushIters column quads, and once more after the ragged tail
    int64_t q0 = static_cast<int64_t>(blockIdx.x) * TPB;
    bool more = true;
    while (more) {
        for (int iter = 0; iter < kFlushIters && q0 < nquads; ++iter, q0 += stride) {
            const int64_t q = q0 + threadIdx.x;
            if constexpr (pair_blocked(N)) {
                const float* p = X + 4 * q;
                const bool in = q < nquads;
                pair_accumulate_blocked<N, G>(
                    [&](int r) {
                        V4 z;
                        z.lo = z.hi = 0ull;
                        return in ? ldg_cached_v4(p + r * ld) : z;
                    },
                    [] {}, acc);
            } else {
                V4 v[N];
                if (q < nquads) {
                    const float* p = X + 4 * q;
#pragma unroll
                    for (int i = 0; i < N; ++i) v[i] = (NG > 1) ? ldg_cached_v4(p + i * ld) : ldg_stream_v4(p + i * ld);
                } else {
#pragma unroll
                    for (int i = 0; i < N; ++i) v[i].lo = v[i].hi = 0ull;
                }
                pair_accumulate<N, G>(v, acc);
            }
        }
        more = q0 < nquads;
        // ragged tail: columns 4*nquads .. D-1, one per thread of CTA 0
        if (!more && blockIdx.x == 0 && (D & 3)) {
            const int64_t c = 4 * nquads + threadIdx.x;
            const bool in = threadIdx.x < (D & 3);
            if constexpr (pair_blocked(N)) {
                pair_accumulate_blocked<N, G>(
                    [&](int r) {
                        V4 z;
                        z.lo = in ? pack2(__ldg(X + r * ld + c), 0.0f) : 0ull;
                        z.hi = 0ull;
                        return z;
                    },
                    [] {}, acc);
            } else {
                V4 v[N];
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    v[i].lo = in ? pack2(__ldg(X + i * ld + c), 0.0f) : 0ull;
                    v[i].hi = 0ull;
                }
                pair_accumulate<N, G>(v, acc);
            }
        }
        flush_pairs<PG>(acc, wacc, lane);
    }
}

template <int N, int G>
__device__ __forceinline__ void group_dispatch(int g, const float* X, int64_t D, int64_t ld, double* wacc) {
    if (g == G) {
        pairdist_body<N, G>(X, D, ld, wacc);
    } else {
        if constexpr (G + 1 < pair_groups(N)) group_dispatch<N, G + 1>(g, X, D, ld, wacc);
    }
}


// ---------------------------------------------------------------------------------
// K1b
// ---------------------------------------------------------------------------------
// Block-cooperative; sd/sk are n*n doubles of shared scratch.  Mirrors svgd.py:15-21:
// d = (sqrt(sum))^2 as torch.cdist(p=2)**2 does, torch.quantile(d, 0.5) over all n*n
// entries (order statistics of the (value, flat index)-sorted list + lerp),
// h = sqrt(0.5*med/ln(n+1)) + 1e-8, K = exp(-d / (2 h^2)); then
// A = (l2/2 + c) K - c diag(rowsum K), c = s/(N h^2).
// The n*n entries are sorted with a shared-memory bitonic network (padded with +inf to MAXPAD >= n*n,
// a power of two): ~45 compare-exchange stages at n = 20 instead of an O(n^4) rank count.
__host__ __device__ constexpr int pow2_ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

// s_key / s_ord: pow2_ceil(n*n) entries of shared scratch for the sort
__device__ __forceinline__ void bandwidth_sorted(const double* dist, int n, const BandwidthParams& bp, double* sd,
                                                 double* sk, double* s_key, int* s_ord) {
    const int tid = threadIdx.x + threadIdx.y * blockDim.x;
    const int nthreads = blockDim.x * blockDim.y;
    const int nn = n * n;
    __shared__ double s_sel[2];
    __shared__ int s_idx[2];
    __shared__ double s_h;
    int npad = 1;
    while (npad < nn) npad <<= 1;

    for (int e = tid; e < npad; e += nthreads) {
        double v = __longlong_as_double(0x7ff0000000000000LL);  // +inf padding sorts last
        if (e < nn) {
            const double r = sqrt(dist[e]);
            v = r * r;
            sd[e] = v;
        }
        s_key[e] = v;
        s_ord[e] = e;
    }
    __syncthreads();
    for (int k = 2; k <= npad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (npad >> 1); t += nthreads) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int l = i | j;
                const bool up = (i & k) == 0;
                const double a = s_key[i], b = s_key[l];
                const int ia = s_ord[i], ib = s_ord[l];
                const bool gt = (a > b) || (a == b && ia > ib);  // total order: value, then flat index
                if (gt == up) {
                    s_key[i] = b;
                    s_key[l] = a;
                    s_ord[i] = ib;
                    s_ord[l] = ia;
                }
            }
            // A 32-aligned block of compare-exchange indices t belongs to ONE warp in every pass (nthreads is a multiple of
            // 32), and with j <= 32 such a block only touches its own 64 elements: as long as this pass and the next both
            // have j <= 32, the hand-over is warp-local: 10 block-wide barriers instead of 45 at n = 20 (512 padded
            // entries), 3 instead of 28 at n = 10.  (Worth ~0.5 us only: K1b's 9 / 5 us at n = 20 / 10 are dependent fp64
            // chains — sqrt, log, exp, the division — not barriers and not instruction fetch: profiles/r02_tail_timing.jsonl.)
            const int j_next = j > 1 ? (j >> 1) : k;   // first pass of the next k runs with j = k
            if (j <= 32 && j_next <= 32 && !(k == npad && j == 1))
                __syncwarp();
            else
                __syncthreads();
        }
    }
    const int pos_lo = (nn - 1) / 2;
    const int pos_hi = nn / 2;
    if (tid < 2) {
        const int pos = tid == 0 ? pos_lo : pos_hi;
        const int e = s_ord[pos];
        const int i = e / n, j = e - i * n;
        s_sel[tid] = s_key[pos];
        s_idx[tid] = i <= j ? e : j * n + i;
    }
    __syncthreads();
    if (tid == 0) {
        const double a = s_sel[0], b = s_sel[1];
        const double w = 0.5 * (nn - 1) - pos_lo;
        // torch lerp: w < 0.5 ? a + w*(b-a) : b - (b-a)*(1-w)
        const double med = (w < 0.5) ? a + w * (b - a) : b - (b - a) * (1.0 - w);
        double h = sqrt(0.5 * med / log(static_cast<double>(n) + 1.0)) + 1e-8;
        if (bp.h_override > 0.0) h = bp.h_override;
        s_h = h;
        if (bp.info) {
            bp.info[0] = h;
            bp.info[1] = med;
            bp.info[2] = a;
            bp.info[3] = b;
        }
        if (bp.sel) {
            bp.sel[0] = s_idx[0];
            bp.sel[1] = s_idx[1];
        }
    }
    __syncthreads();
    const double h = s_h;
    const double inv2h2 = 1.0 / (2.0 * h * h);
    for (int e = tid; e < nn; e += nthreads) sk[e] = exp(-sd[e] * inv2h2);
    __syncthreads();
    const double c = bp.kernel_grad_scale / (bp.dataset_size * h * h);
    const double half_l2 = 0.5 * bp.l2_reg;
    for (int e = tid; e < nn; e += nthreads) {
        const int i = e / n, j = e - i * n;
        const double kij = sk[e];
        double a;
        if (i != j) {
            a = (half_l2 + c) * kij;
        } else {
            double off = 0.0;  // rowsum without the diagonal: (l2/2 + c) K_ii - c rowsum = l2/2 K_ii - c off
            for (int m = 0; m < n; ++m)
                if (m != i) off += sk[i * n + m];
            a = half_l2 * kij - c * off;
        }
        bp.K[e] = static_cast<float>(kij);
        bp.A[e] = static_cast<float>(a);
    }
}

template <int MAXPAD>
__device__ __forceinline__ void bandwidth_device(const double* dist, int n, const BandwidthParams& bp, double* sd, double* sk) {
    __shared__ double s_key[MAXPAD];
    __shared__ int s_ord[MAXPAD];
    bandwidth_sorted(dist, n, bp, sd, sk, s_key, s_ord);
}


template <int N>
__global__ void __launch_bounds__(pairdist_tpb(N) * pair_groups(N))
svgd_pairdist_kernel(const float* __restrict__ X, int64_t D, int64_t ld, double* __restrict__ dist, int accumulate,
                     void* ws, int fuse_bandwidth, BandwidthParams bp, int only_if_redo) {
    // enqueued behind the centred-Gram kernel: nothing to do unless its guard asked for exact distances
    if (only_if_redo && reinterpret_cast<const WsHeader*>(ws)->redo == 0) return;
    constexpr int P = pair_count(N);
    constexpr int PG = pairs_per_group(N);
    constexpr int NG = pair_groups(N);
    constexpr int TPB = pairdist_tpb(N);
    constexpr int WPG = TPB / 32;  // warps per group
    __shared__ double wacc[NG * WPG][PG];
    __shared__ double cta_vals[P];
    __shared__ double total[P];
    __shared__ double sd[N * N];
    __shared__ double sk[N * N];

    const int g = threadIdx.y;
    const int warp_in_group = threadIdx.x >> 5;
    const int tid = threadIdx.x + threadIdx.y * TPB;
    for (int k = tid; k < NG * WPG * PG; k += TPB * NG) (&wacc[0][0])[k] = 0.0;
    __syncthreads();

    group_dispatch<N, 0>(g, X, D, ld, wacc[g * WPG + warp_in_group]);
    __syncthreads();
    griddep_launch();   // streaming done: a dependent K2 may become resident during the tail

    for (int p = tid; p < P; p += TPB * NG) {
        const int i = pair_row(p, N), j = p - pair_index(i, i + 1, N) + i + 1;
        const int grp = pair_group_of(i, j, N), k = pair_slot_of(i, j, N);
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < WPG; ++w) s += wacc[grp * WPG + w][k];
        cta_vals[p] = s;
    }
    __syncthreads();

    if (!grid_reduce_fp64(cta_vals, P, ws, total)) return;

    // last CTA: symmetric n*n matrix, zero diagonal
    for (int e = tid; e < N * N; e += TPB * NG) {
        const int i = e / N, j = e - i * N;
        double v = 0.0;
        if (i != j) v = total[i < j ? pair_index(i, j, N) : pair_index(j, i, N)];
        if (accumulate) v += dist[e];
        dist[e] = v;
    }
    if (fuse_bandwidth && !peer_exchange_failed(ws)) {
        __syncthreads();
        bandwidth_device<pow2_ceil(N * N)>(dist, N, bp, sd, sk);
    }
}

// ---------------------------------------------------------------------------------
// K1, TMA-staged: one persistent CTA per SM; a producer warp streams [N x TC]-column tiles of X
// into a shared-memory ring with cp.async.bulk, consumer warps accumulate the pair distances of
// one column quad per thread per tile.  Besides keeping ~200 KB per SM in flight, this leaves
// only gridDim = #SMs partial sets for the deterministic last-CTA reduction.
// ---------------------------------------------------------------------------------
__host__ __device__ constexpr int pd_tile_cols(int n) {
    return pair_groups(n) == 1 ? 1024 : (pair_groups(n) == 2 ? 512 : (pair_groups(n) <= 4 ? 256 : 128));
}
__host__ __device__ constexpr int pd_stage_bytes(int n) { return n * pd_tile_cols(n) * 4; }
__host__ __device__ constexpr int pd_stages(int n) {
    return (200 * 1024) / pd_stage_bytes(n) > 8 ? 8 : (200 * 1024) / pd_stage_bytes(n);
}
// consumer threads: one column quad of the tile per thread and pair group (256; 192 at n = 16)
__host__ __device__ constexpr int pd_consumers(int n) { return pair_groups(n) * pd_tile_cols(n) / 4; }
constexpr int kFlushTiles = 64;

template <int N, int G>
__device__ __forceinline__ void pairdist_tma_consumer(const float* __restrict__ X, int64_t D, int64_t ld,
                                                      const float* __restrict__ tiles, uint64_t* full_bar,
                                                      uint64_t* empty_bar, double* __restrict__ wacc, int qi) {
    constexpr int PG = pairs_per_group(N);
    constexpr int TC = pd_tile_cols(N);
    constexpr int STAGES = pd_stages(N);
    f32x2 acc[PG > 0 ? PG : 1];
#pragma unroll
    for (int k = 0; k < PG; ++k) acc[k] = 0ull;
    const int lane = threadIdx.x & 31;
    const int64_t d4 = D & ~static_cast<int64_t>(3);
    const int64_t ntiles = (d4 + TC - 1) / TC;
    int it = 0;
    int64_t t = blockIdx.x;
    bool more = true;
    while (more) {  // one flush site: every kFlushTiles tiles, and once more after the ragged tail
        for (int f = 0; f < kFlushTiles && t < ntiles; ++f, t += gridDim.x, ++it) {
            const int s = it % STAGES;
            const uint32_t use = static_cast<uint32_t>(it / STAGES);
            const int64_t col0 = t * TC;
            const int64_t w = (d4 - col0 < TC) ? d4 - col0 : TC;
            mbar_wait(&full_bar[s], use & 1u);
            const float* sx = tiles + static_cast<size_t>(s) * N * TC + 4 * qi;
            if constexpr (pair_blocked(N)) {
                const bool in = 4 * qi < w;
                pair_accumulate_blocked<N, G>(
                    [&](int r) {
                        V4 z;
                        z.lo = z.hi = 0ull;
                        return in ? lds_v4(sx + r * TC) : z;
                    },
                    [&] {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty_bar[s]);  // last row is in registers: release the stage
                    },
                    acc);
            } else {
                V4 v[N];
                if (4 * qi < w) {
#pragma unroll
                    for (int i = 0; i < N; ++i) v[i] = lds_v4(sx + i * TC);
                } else {
#pragma unroll
                    for (int i = 0; i < N; ++i) v[i].lo = v[i].hi = 0ull;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);  // data is in registers: release the stage
                pair_accumulate<N, G>(v, acc);
            }
        }
        more = t < ntiles;
        if (!more && blockIdx.x == 0 && (D & 3)) {  // ragged tail columns (D % 4)
            const int64_t c = d4 + qi;
            const bool in = qi < (D & 3);
            if constexpr (pair_blocked(N)) {
                pair_accumulate_blocked<N, G>(
                    [&](int r) {
                        V4 z;
                        z.lo = in ? pack2(__ldg(X + r * ld + c), 0.0f) : 0ull;
                        z.hi = 0ull;
                        return z;
                    },
                    [] {}, acc);
            } else {
                V4 v[N];
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    v[i].lo = in ? pack2(__ldg(X + i * ld + c), 0.0f) : 0ull;
                    v[i].hi = 0ull;
                }
                pair_accumulate<N, G>(v, acc);
            }
        }
        flush_pairs<PG>(acc, wacc, lane);
    }
}

template <int N, int G>
__device__ __forceinline__ void pairdist_tma_dispatch(int g, const float* X, int64_t D, int64_t ld, const float* tiles,
                                                      uint64_t* full_bar, uint64_t* empty_bar, double* wacc, int qi) {
    if (g == G) {
        pairdist_tma_consumer<N, G>(X, D, ld, tiles, full_bar, empty_bar, wacc, qi);
    } else {
        if constexpr (G + 1 < pair_groups(N)) pairdist_tma_dispatch<N, G + 1>(g, X, D, ld, tiles, full_bar, empty_bar, wacc, qi);
    }
}

template <int N>
__global__ void __launch_bounds__(pd_consumers(N) + 32, 1)
svgd_pairdist_tma_kernel(const float* __restrict__ X, int64_t D, int64_t ld, double* __restrict__ dist, int accumulate,
                         void* ws, int fuse_bandwidth, BandwidthParams bp, int only_if_redo) {
    if (only_if_redo && reinterpret_cast<const WsHeader*>(ws)->redo == 0) return;
    constexpr int P = pair_count(N);
    constexpr int PG = pairs_per_group(N);
    constexpr int NG = pair_groups(N);
    constexpr int TC = pd_tile_cols(N);
    constexpr int QT = TC / 4;  // consumer threads per pair group
    constexpr int STAGES = pd_stages(N);
    constexpr int kPdConsumers = pd_consumers(N);
    constexpr int CWARPS = kPdConsumers / 32;
    static_assert(QT % 32 == 0 && kPdConsumers <= 992, "consumer layout");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tiles = reinterpret_cast<float*>(smem_raw);  // [STAGES][N][TC]
    __shared__ double wacc[CWARPS][PG];
    __shared__ double cta_vals[P];
    __shared__ double total[P];
    __shared__ double sd[N * N];
    __shared__ double sk[N * N];
    __shared__ __align__(8) uint64_t full_bar[STAGES];
    __shared__ __align__(8) uint64_t empty_bar[STAGES];

    const int tid = threadIdx.x;
    const int nthreads = kPdConsumers + 32;
    if (blockIdx.x == 0) BDE_TS(ws, 0);
    for (int k = tid; k < CWARPS * PG; k += nthreads) (&wacc[0][0])[k] = 0.0;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], CWARPS);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (tid >= kPdConsumers) {
        if (tid == kPdConsumers) {
            const int64_t d4 = D & ~static_cast<int64_t>(3);
            const int64_t ntiles = (d4 + TC - 1) / TC;
            int it = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
                const int s = it % STAGES;
                const uint32_t use = static_cast<uint32_t>(it / STAGES);
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                const int64_t col0 = t * TC;
                const int64_t w = (d4 - col0 < TC) ? d4 - col0 : TC;
                const uint32_t row_bytes = static_cast<uint32_t>(w) * 4u;
                mbar_arrive_expect_tx(&full_bar[s], N * row_bytes);
                float* sx = tiles + static_cast<size_t>(s) * N * TC;
#pragma unroll
                for (int r = 0; r < N; ++r) tma_load_1d(sx + r * TC, X + r * ld + col0, row_bytes, &full_bar[s]);
            }
        }
    } else {
        // pair group = warp % NG: warps w and w + 4 sit on the same SM sub-partition, and with NG = 2 or 4 they then
        // run the SAME unrolled pair loop (one copy in that scheduler's instruction cache instead of two)
        const int wid = tid >> 5;
        const int g = wid % NG, qi = (wid / NG) * 32 + (tid & 31);
        pairdist_tma_dispatch<N, 0>(g, X, D, ld, tiles, full_bar, empty_bar, wacc[wid], qi);
    }
    __syncthreads();
    BDE_TS_MAX(ws, 1);
    griddep_launch();   // streaming done: a dependent K2 may become resident during the tail

    // pair p of group grp is accumulated by that group's warps only
    for (int p = tid; p < P; p += nthreads) {
        const int i = pair_row(p, N), j = p - pair_index(i, i + 1, N) + i + 1;
        const int grp = pair_group_of(i, j, N), k = pair_slot_of(i, j, N);
        double sacc = 0.0;
        for (int wv = grp; wv < CWARPS; wv += NG) sacc += wacc[wv][k];
        cta_vals[p] = sacc;
    }
    __syncthreads();
    if (!grid_reduce_fp64(cta_vals, P, ws, total)) return;
    for (int e = tid; e < N * N; e += nthreads) {
        const int i = e / N, j = e - i * N;
        double v = 0.0;
        if (i != j) v = total[i < j ? pair_index(i, j, N) : pair_index(j, i, N)];
        if (accumulate) v += dist[e];
        dist[e] = v;
    }
    BDE_TS(ws, 4);
    if (fuse_bandwidth && !peer_exchange_failed(ws)) {
        __syncthreads();
        bandwidth_device<pow2_ceil(N * N)>(dist, N, bp, sd, sk);
    }
    __syncthreads();
    BDE_TS(ws, 5);
#ifdef BDE_TAIL_TIMING
    if (fuse_bandwidth && !peer_exchange_failed(ws)) {   // the same code again, now warm: what of K1b's time is instruction fetch?
        __syncthreads();
        bandwidth_device<pow2_ceil(N * N)>(dist, N, bp, sd, sk);
    }
    __syncthreads();
    BDE_TS(ws, 6);
#endif
}

// ---------------------------------------------------------------------------------
// K2 (+ optional fused base-optimizer step, f1)
// ---------------------------------------------------------------------------------
// n > 16: the j-loop of K2 stays rolled (see apply_row)
__host__ __device__ constexpr bool apply_rolled(int n) { return n > 16; }
// the staged kernel with a fused optimizer also rolls at n = 16: rolled it fits four tile sets into the 168-register
// budget of nine warps, and the serial chain of n shared-state optimizer steps needs the extra warps to hide behind
__host__ __device__ constexpr bool apply_rolled(int n, int opt) { return n > 16 || (n == 16 && opt != kOptNone); }
__host__ __device__ constexpr int apply_row_chunk(int n) { return n <= 12 ? n : (n <= 16 ? 8 : 4); }

// out_i += K_ij g_j + A_ij x_j for one source row j of a column quad.  n <= 12: fully unrolled over j by the
// callers (coefficients become immediates-offset LDS).  n > 12: the callers keep j as a ROLLED loop — the fully
// unrolled 4 n^2 FFMA2 body (26 KB of code at n = 20) thrashed the instruction cache ("no instruction" was the
// top warp stall in ncu) — and read the coefficient rows as 128-bit words.
#ifndef BDE_APPLY_J_UNROLL
#define BDE_APPLY_J_UNROLL 5   // source rows per iteration of the rolled j-loop (n = 20: 4 iterations of 400 FFMA2)
#endif
template <int N, bool ROLLED = apply_rolled(N)>
__device__ __forceinline__ void apply_row(f32x2 (&acc)[N][2], const V4& g, const V4& x, const float* __restrict__ kt,
                                          const float* __restrict__ at) {
    if constexpr (N % 4 == 0 && ROLLED) {
#pragma unroll
        for (int c = 0; c < N / 4; ++c) {
            const float4 k4 = *reinterpret_cast<const float4*>(kt + 4 * c);
            const float4 a4 = *reinterpret_cast<const float4*>(at + 4 * c);
            const float kk[4] = {k4.x, k4.y, k4.z, k4.w};
            const float aa[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = 4 * c + u;
                acc[i][0] = fma2s(kk[u], g.lo, acc[i][0]);
                acc[i][1] = fma2s(kk[u], g.hi, acc[i][1]);
                acc[i][0] = fma2s(aa[u], x.lo, acc[i][0]);
                acc[i][1] = fma2s(aa[u], x.hi, acc[i][1]);
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const float kij = kt[i];
            const float aij = at[i];
            acc[i][0] = fma2s(kij, g.lo, acc[i][0]);
            acc[i][1] = fma2s(kij, g.hi, acc[i][1]);
            acc[i][0] = fma2s(aij, x.lo, acc[i][0]);
            acc[i][1] = fma2s(aij, x.hi, acc[i][1]);
        }
    }
}

__device__ __forceinline__ f32x2 mul2s(float s, f32x2 b) {
    f32x2 r;
    const f32x2 a = pack2(s, s);
    asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ V4 ld_coherent_v4(const float* p) {
    V4 v;
    asm volatile("ld.global.v2.u64 {%0, %1}, [%2];" : "=l"(v.lo), "=l"(v.hi) : "l"(p));
    return v;
}

// torch.optim.SGD._single_tensor_sgd on two columns of particle `first`..: g is the new gradient
// (out_i), x the particle value, b the shared momentum buffer.
__device__ __forceinline__ void sgd_update2(const BaseOptParams& o, bool clone_buf, f32x2 g, f32x2& x, f32x2& b) {
    if (o.weight_decay != 0.0f) g = fma2s(o.weight_decay, x, g);           // grad.add(param, alpha=wd)
    if (o.momentum != 0.0f) {
        if (clone_buf)
            b = g;                                                          // buf = clone(grad)
        else
            b = fma2s(o.one_minus_dampening, g, mul2s(o.momentum, b));      // buf.mul_(m).add_(grad, alpha=1-damp)
        g = o.nesterov ? fma2s(o.momentum, b, g) : b;
    }
    x = fma2s(-o.lr, g, x);                                                 // param.add_(grad, alpha=-lr)
}

// torch.optim.Adam / AdamW (_single_tensor_adam, no amsgrad) for particle i = optimizer step step0+i+1.
// sqrt and the final division run on the SFU (MUFU.SQRT / MUFU.RCP, ~1 ulp each; the update is a small
// correction to x, so the result stays far inside rtol 1e-5 of eager PyTorch).
__device__ __forceinline__ float adam_update1(const BaseOptParams& o, int i, float g, float x, float& m, float& v) {
    if (o.weight_decay != 0.0f) {
        if (o.decoupled_wd)
            x = x * o.decay_factor;                                         // param.mul_(1 - lr*wd)
        else
            g = fmaf(o.weight_decay, x, g);
    }
    m = fmaf(o.one_minus_beta1, g - m, m);                                  // exp_avg.lerp_(grad, 1-beta1)
    v = fmaf(o.one_minus_beta2 * g, g, o.beta2 * v);                        // mul_(beta2).addcmul_(g, g, 1-beta2)
    const float denom = fmaf(sqrt_approx(v), o.inv_bc2_sqrt[i], o.eps);
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(denom));
    return fmaf(-o.step_size[i] * m, r, x);                                 // param.addcdiv_(m, denom, -step_size)
}
// two columns at once: the same operations as adam_update1, lane for lane, on the packed pipe (FADD2 / FMUL2 /
// FFMA2 are IEEE per lane, so the results are bit-identical to the scalar form); only sqrt and rcp stay scalar (SFU)
__device__ __forceinline__ void adam_update2(const BaseOptParams& o, int i, f32x2 g, f32x2& x, f32x2& m, f32x2& v) {
    if (o.weight_decay != 0.0f) {
        if (o.decoupled_wd)
            x = mul2s(o.decay_factor, x);
        else
            g = fma2s(o.weight_decay, x, g);
    }
    m = fma2s(o.one_minus_beta1, sub2(g, m), m);
    v = fma2(mul2s(o.one_minus_beta2, g), g, mul2s(o.beta2, v));
    float v0, v1, r0, r1;
    unpack2(v, v0, v1);
    const f32x2 denom = fma2s(o.inv_bc2_sqrt[i], pack2(sqrt_approx(v0), sqrt_approx(v1)), pack2(o.eps, o.eps));
    unpack2(denom, v0, v1);
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r0) : "f"(v0));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r1) : "f"(v1));
    x = fma2(mul2s(-o.step_size[i], m), pack2(r0, r1), x);
}

// one particle's optimizer step on a column quad; s0 / s1 are the shared state quads
template <int OPT>
__device__ __forceinline__ void opt_update_quad(const BaseOptParams& o, int i, f32x2 g_lo, f32x2 g_hi, V4& x, V4& s0, V4& s1) {
    if constexpr (OPT == kOptSgd) {
        const bool clone_buf = (i == 0) && !o.buf_initialized;
        sgd_update2(o, clone_buf, g_lo, x.lo, s0.lo);
        sgd_update2(o, clone_buf, g_hi, x.hi, s0.hi);
    } else if constexpr (OPT == kOptAdam) {
        adam_update2(o, i, g_lo, x.lo, s0.lo, s1.lo);
        adam_update2(o, i, g_hi, x.hi, s0.hi, s1.hi);
    }
}
__host__ __device__ constexpr int opt_state_rows(int opt) { return opt == kOptAdam ? 2 : (opt == kOptSgd ? 1 : 0); }

// scalar (one column) form for ragged tails and the generic kernels
template <int OPT>
__device__ __forceinline__ float opt_update_scalar(const BaseOptParams& o, int i, float g, float x, float& s0, float& s1) {
    if constexpr (OPT == kOptSgd) {
        if (o.weight_decay != 0.0f) g = fmaf(o.weight_decay, x, g);
        if (o.momentum != 0.0f) {
            if (i == 0 && !o.buf_initialized)
                s0 = g;
            else
                s0 = fmaf(o.one_minus_dampening, g, o.momentum * s0);
            g = o.nesterov ? fmaf(o.momentum, s0, g) : s0;
        }
        return fmaf(-o.lr, g, x);
    } else {
        return adam_update1(o, i, g, x, s0, s1);
    }
}

// tail columns (D % 4) of the fused / plain K2: one thread per column
template <int N, int OPT>
__device__ __forceinline__ void apply_tail_column(const float* X, const float* G, float* out, const float (*sKT)[(N + 3) & ~3],
                                                  const float (*sAT)[(N + 3) & ~3], int64_t c, int64_t ldx, int64_t ldg,
                                                  int64_t ldo, const BaseOptParams& o, float* xnew = nullptr) {
    float res[N];
    for (int i = 0; i < N; ++i) {
        float sacc = 0.0f;
        for (int j = 0; j < N; ++j) {
            sacc = fmaf(sKT[j][i], G[j * ldg + c], sacc);
            sacc = fmaf(sAT[j][i], X[j * ldx + c], sacc);
        }
        res[i] = sacc;
    }
    if constexpr (OPT == kOptNone) {
        for (int i = 0; i < N; ++i) out[i * ldo + c] = res[i];
    } else {
        float* Xw = const_cast<float*>(X);
        float s0 = 0.0f, s1 = 0.0f;
        const bool has_s0 = (OPT == kOptAdam) || (o.momentum != 0.0f && o.buf_initialized);
        if (has_s0) s0 = o.state0[c];
        if (OPT == kOptAdam) s1 = o.state1[c];
        if (o.out_last) o.out_last[c] = res[N - 1];
        for (int i = 0; i < N; ++i) {
            const float xv = opt_update_scalar<OPT>(o, i, res[i], X[i * ldx + c], s0, s1);
            Xw[i * ldx + c] = xv;
            if (xnew) xnew[i] = xv;
        }
        if (OPT == kOptAdam || o.momentum != 0.0f) o.state0[c] = s0;
        if (OPT == kOptAdam) o.state1[c] = s1;
    }
}

// Tail of the training-step kernels (NEXT): per-warp fp64 pair sums -> CTA sums -> deterministic grid
// reduction -> the last CTA writes the n*n distance matrix of the updated particles and (optionally) runs K1b.
template <int N, int WARPS>
__device__ __forceinline__ void next_dist_epilogue(double (*wacc)[pair_count(N) > 0 ? pair_count(N) : 1],
                                                   const NextDistParams& nd) {
    constexpr int P = pair_count(N);
    __shared__ double cta_vals[P > 0 ? P : 1];
    __shared__ double total[P > 0 ? P : 1];
    __shared__ double sd[N * N];
    __shared__ double sk[N * N];
    const int tid = threadIdx.x;
    const int nthreads = blockDim.x;
    __syncthreads();
    for (int p = tid; p < P; p += nthreads) {
        double sacc = 0.0;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) sacc += wacc[w][p];
        cta_vals[p] = sacc;
    }
    __syncthreads();
    if (!grid_reduce_fp64(cta_vals, P, nd.ws, total)) return;
    for (int e = tid; e < N * N; e += nthreads) {
        const int i = e / N, j = e - i * N;
        nd.dist[e] = (i != j) ? total[i < j ? pair_index(i, j, N) : pair_index(j, i, N)] : 0.0;
    }
    if (nd.fuse_bandwidth && !peer_exchange_failed(nd.ws)) {
        __syncthreads();
        bandwidth_device<pow2_ceil(N * N)>(nd.dist, N, nd.bp, sd, sk);
    }
}

template <int N, int OPT, bool NEXT = false>
__global__ void __launch_bounds__(128)
svgd_apply_kernel(const float* X, const float* __restrict__ G, float* out, const float* __restrict__ K,
                  const float* __restrict__ A, int64_t D, int64_t ldx, int64_t ldg, int64_t ldo,
                  const __grid_constant__ BaseOptParams o, const __grid_constant__ NextDistParams nd) {
    constexpr int NP = (N + 3) & ~3;
    constexpr int JC = apply_row_chunk(N);
    static_assert(!apply_rolled(N) || N % JC == 0, "the rolled chunk loop has no ragged last chunk");
    constexpr int PN = NEXT ? pair_count(N) : 1;  // pair accumulators of the updated particles
    static_assert(!NEXT || (OPT != kOptNone && pair_groups(N) == 1 && N >= 2), "NEXT needs a fused optimizer and n <= 10");
    // transposed coefficients: sKT[j][i] = K[i][j] so that the i-loop reads contiguous words
    __shared__ __align__(16) float sKT[N][NP];
    __shared__ __align__(16) float sAT[N][NP];
    __shared__ double wacc[NEXT ? 4 : 1][NEXT ? pair_count(N) : 1];
    griddep_wait();   // K / A come from the preceding K1 launch
    for (int e = threadIdx.x; e < N * NP; e += blockDim.x) {
        const int j = e / NP, i = e - j * NP;
        sKT[j][i] = (i < N) ? K[i * N + j] : 0.0f;
        sAT[j][i] = (i < N) ? A[i * N + j] : 0.0f;
    }
    if constexpr (NEXT) {
        for (int k = threadIdx.x; k < 4 * pair_count(N); k += blockDim.x) (&wacc[0][0])[k] = 0.0;
    }
    __syncthreads();
    f32x2 pacc[PN];
#pragma unroll
    for (int k = 0; k < PN; ++k) pacc[k] = 0ull;

    const int64_t nquads = D >> 2;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t q = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; q < nquads; q += stride) {
        f32x2 acc[N][2];
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i][0] = acc[i][1] = 0ull;
        const float* xp = X + 4 * q;
        const float* gp = G + 4 * q;
        auto row_chunk = [&](int jc) {  // JC source rows: all loads first, then the FFMA2 work
            V4 x[JC], g[JC];
#pragma unroll
            for (int jj = 0; jj < JC; ++jj) {
                if (jc + jj < N) {
                    g[jj] = ldg_stream_v4(gp + (jc + jj) * ldg);
                    // fused form: X is rewritten by this kernel -> coherent loads (and L1 keeps the rows for
                    // the re-read in the optimizer epilogue)
                    x[jj] = (OPT == kOptNone) ? ldg_stream_v4(xp + (jc + jj) * ldx) : ld_coherent_v4(xp + (jc + jj) * ldx);
                }
            }
#pragma unroll
            for (int jj = 0; jj < JC; ++jj)
                if (jc + jj < N) apply_row<N>(acc, g[jj], x[jj], sKT[jc + jj], sAT[jc + jj]);
        };
        if constexpr (apply_rolled(N)) {  // rolled over the chunks (N % JC == 0): keeps the loop body inside the instruction cache
#pragma unroll 1
            for (int jc = 0; jc < N; jc += JC) row_chunk(jc);
        } else {
#pragma unroll
            for (int jc = 0; jc < N; jc += JC) row_chunk(jc);
        }
        if constexpr (OPT == kOptNone) {
            float* op = out + 4 * q;
#pragma unroll
            for (int i = 0; i < N; ++i) {
                V4 v;
                v.lo = acc[i][0];
                v.hi = acc[i][1];
                stg_stream_v4(op + i * ldo, v);
            }
        } else {
            float* xw = const_cast<float*>(xp);
            V4 s0, s1;
            s0.lo = s0.hi = s1.lo = s1.hi = 0ull;
            const bool has_s0 = (OPT == kOptAdam) || (o.momentum != 0.0f && o.buf_initialized);
            if (has_s0) s0 = ld_coherent_v4(o.state0 + 4 * q);
            if (OPT == kOptAdam) s1 = ld_coherent_v4(o.state1 + 4 * q);
            if (o.out_last) {
                V4 v;
                v.lo = acc[N - 1][0];
                v.hi = acc[N - 1][1];
                stg_stream_v4(o.out_last + 4 * q, v);
            }
            V4 xn[NEXT ? N : 1];
#pragma unroll
            for (int i = 0; i < N; ++i) {
                V4 x = ld_coherent_v4(xp + i * ldx);
                opt_update_quad<OPT>(o, i, acc[i][0], acc[i][1], x, s0, s1);
                stg_stream_v4(xw + i * ldx, x);
                if constexpr (NEXT) xn[i] = x;
            }
            if (OPT == kOptAdam || o.momentum != 0.0f) stg_stream_v4(o.state0 + 4 * q, s0);
            if (OPT == kOptAdam) stg_stream_v4(o.state1 + 4 * q, s1);
            // this kernel only runs when every thread sees a handful of quads: fp32 partials until the end
            if constexpr (NEXT) pair_accumulate<N, 0>(xn, pacc);
        }
    }
    // ragged tail columns
    if constexpr (NEXT) {
        V4 xt[N];
#pragma unroll
        for (int i = 0; i < N; ++i) xt[i].lo = xt[i].hi = 0ull;
        if (blockIdx.x == 0 && threadIdx.x < (D & 3)) {
            float xnew[N];
            apply_tail_column<N, OPT>(X, G, out, sKT, sAT, 4 * nquads + threadIdx.x, ldx, ldg, ldo, o, xnew);
#pragma unroll
            for (int i = 0; i < N; ++i) xt[i].lo = pack2(xnew[i], 0.0f);
        }
        pair_accumulate<N, 0>(xt, pacc);
        flush_pairs<PN>(pacc, wacc[threadIdx.x >> 5], threadIdx.x & 31);
        next_dist_epilogue<N, 4>(wacc, nd);
    } else {
        if (blockIdx.x == 0 && threadIdx.x < (D & 3))
            apply_tail_column<N, OPT>(X, G, out, sKT, sAT, 4 * nquads + threadIdx.x, ldx, ldg, ldo, o);
    }
}

// ---------------------------------------------------------------------------------
// K2, TMA-staged: a producer warp streams [N x TC]-column tiles of X and G (and, in the fused form,
// the optimizer-state rows) into a ring of shared-memory stages with cp.async.bulk (completion on
// mbarriers); the consumer warps compute out = K G + A X for one column quad per thread straight
// from shared memory and stream the result to HBM.  The loads are decoupled from the FFMA2 work,
// so the bytes in flight per SM are set by the ring depth (~200 KB) instead of by register occupancy.
// Fused form (OPT != 0): the thread then walks its quad through the n optimizer steps (particle
// order, shared state in registers), re-reading x_i from the stage, and writes X in place — `out`
// never touches HBM.
// ---------------------------------------------------------------------------------
// Tile sets (TS): for n > 12 a thread's quad costs 4 n^2 FFMA2, so the 64 consumer threads of a 256-column tile
// cannot keep the FMA pipes of four SM sub-partitions busy.  The consumers are therefore split into TS sets of
// TC/4 threads and set c works on the tiles it = c (mod TS) of the ring: 2 TS consumer warps, every tile still read
// from shared memory exactly once, every thread still owns all n rows of its quad (the shared-state optimizer
// steps of the fused form stay thread-local).
// Training-step form (NEXT): the pair distances of the updated particles make the consumer FP32-latency-bound with
// one warp per scheduler (4 warps on a 512-column tile), so it runs 3 tile sets on 256-column tiles instead
// (6 consumer warps + producer = 7 warps: still two warps per sub-partition at most, i.e. the 255-register budget
// that its n(n-1)/2 extra accumulators need).  n > 12: 3 sets for the same reason — with 4 sets (9 warps) one
// sub-partition holds three warps and the kernel is capped at 168 registers.
// Measured on B200 (profiles/r01_tilesets_n16_n20.jsonl): plain K2 at n = 16 is fastest fully unrolled on 3 sets (its fused
// forms rolled on 4: profiles/r02_k2f_n16_ab.jsonl, -24..-29 %), n = 20 rolled
// (see apply_row) on 4 sets.  n <= 12: 3 x 256 wins for plain K2 at n >= 8 (+3..5 %) and for the training-step form
// at n >= 9, where a stage is large enough that the 8-stage ring still keeps ~150 KB in flight; the fused K2f forms
// and small n stay on 1 x 512 (at n = 5 it is 10-25 % faster).
constexpr int64_t kApplySmallTileMaxElems = 1500000000;  // n * row stride above which plain K2 goes back to 1 x 512
__host__ __device__ constexpr bool apply_small_tiles(int n, int opt, bool next) {
    return n > 12 || (next && n >= 9) || (opt == kOptNone && n >= 8);
}
__host__ __device__ constexpr int apply_tile_cols(int n, int opt, bool next) { return apply_small_tiles(n, opt, next) ? 256 : 512; }
__host__ __device__ constexpr int apply_default_tile_sets(int n, int opt, bool next) {
    return !apply_small_tiles(n, opt, next) ? 1 : (apply_rolled(n, opt) ? 4 : 3);
}
__host__ __device__ constexpr int apply_stage_bytes(int n, int opt, int tc) {
    return (2 * n + opt_state_rows(opt)) * tc * 4;
}
__host__ __device__ constexpr int apply_smem_budget(int n) { return (n <= 12 ? 200 : 212) * 1024; }
__host__ __device__ constexpr int apply_stages(int n, int opt, int tc) {
    return apply_smem_budget(n) / apply_stage_bytes(n, opt, tc) > 8 ? 8 : apply_smem_budget(n) / apply_stage_bytes(n, opt, tc);
}

template <int N, int OPT, bool NEXT = false, int TS = apply_default_tile_sets(N, OPT, NEXT), int TC = apply_tile_cols(N, OPT, NEXT)>
__global__ void __launch_bounds__(TS * TC / 4 + 32, 1)
svgd_apply_tma_kernel(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapG, const float* X,
                      const float* __restrict__ G, float* out, const float* __restrict__ K, const float* __restrict__ A,
                      int64_t D, int64_t ldx, int64_t ldg, int64_t ldo, const __grid_constant__ BaseOptParams o,
                      const __grid_constant__ NextDistParams nd, int nst /* ring stages in use, TS < nst <= STAGES */) {
    static_assert(!NEXT || (OPT != kOptNone && pair_groups(N) == 1 && N >= 2), "NEXT needs a fused optimizer and n <= 10");
    constexpr int PN = NEXT ? pair_count(N) : 1;
    constexpr int NP = (N + 3) & ~3;
    constexpr int STAGES = apply_stages(N, OPT, TC);
    constexpr bool kApplyRolled = apply_rolled(N, OPT);
    constexpr int kApplyJUnroll = N == 16 ? 4 : BDE_APPLY_J_UNROLL;
    constexpr int ROWS = 2 * N + opt_state_rows(OPT);
    constexpr int QT = TC / 4;              // threads of one tile set; one column quad each
    constexpr int BW = kTmaBoxCols;         // a stage holds X and G as TC / BW boxes of [N][BW] each, then the state rows [.][TC]
    constexpr int NB = TC / BW;
    static_assert(TC % BW == 0, "tile width must be a multiple of the TMA box width");
    constexpr int CONSUMERS = TS * QT;
    constexpr int CWARPS = CONSUMERS / 32;
    static_assert(STAGES > TS || TS == 1, "every set holds a stage while it computes: the ring must be deeper than TS");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tiles = reinterpret_cast<float*>(smem_raw);  // [STAGES]{X boxes [NB][N][BW], G boxes [NB][N][BW], state rows [.][TC]}
    __shared__ __align__(16) float sKT[N][NP];
    __shared__ __align__(16) float sAT[N][NP];
    __shared__ __align__(8) uint64_t full_bar[STAGES];
    __shared__ __align__(8) uint64_t empty_bar[STAGES];
    __shared__ double wacc[NEXT ? CWARPS : 1][NEXT ? pair_count(N) : 1];

    const int tid = threadIdx.x;
    if constexpr (NEXT) {
        for (int k = tid; k < CWARPS * pair_count(N); k += blockDim.x) (&wacc[0][0])[k] = 0.0;
    }
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], QT / 32);   // released by the warps of the one set that consumed it
        }
        mbar_fence_init();
        tma_prefetch_map(&mapX);
        tma_prefetch_map(&mapG);
    }
    __syncthreads();
    // From here the producer streams X / G tiles at once — neither is written by a K1 that may still be in its tail
    // (programmatic dependent launch) — while the consumers first wait for that K1 to complete, then fetch K and A.

    const int64_t d4 = D & ~static_cast<int64_t>(3);
    const int64_t ntiles = (d4 + TC - 1) / TC;
    const bool is_producer = tid >= CONSUMERS;
    const bool has_s0 = (OPT == kOptAdam) || (OPT == kOptSgd && o.momentum != 0.0f && o.buf_initialized);

    if (is_producer) {
        if (tid == CONSUMERS) {  // one elected lane drives the copy engine
            int s = 0;            // ring slot and how often it has been used before: advanced without div / mod
            uint32_t use = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, s = (s + 1 == nst) ? 0 : s + 1, use += (s == 0)) {
                mbar_wait(&empty_bar[s], (use & 1u) ^ 1u);
                const int64_t col0 = t * TC;
                const int64_t w = (d4 - col0 < TC) ? d4 - col0 : TC;
                const uint32_t row_bytes = static_cast<uint32_t>(w) * 4u;
                const uint32_t nstate = (has_s0 ? 1u : 0u) + (OPT == kOptAdam ? 1u : 0u);
                // the tensor-map boxes always deliver (and count) their full size: columns beyond d4 arrive as zeros
                mbar_arrive_expect_tx(&full_bar[s], 2u * N * TC * 4u + nstate * row_bytes);
                float* sx = tiles + static_cast<size_t>(s) * ROWS * TC;
                float* sg = sx + N * TC;
#pragma unroll
                for (int b = 0; b < NB; ++b) {   // one UTMALDG per box instead of one UBLKCP per row (2 N per tile before)
                    tma_load_2d(sx + b * N * BW, &mapX, static_cast<int>(col0) + b * BW, 0, &full_bar[s]);
                    tma_load_2d(sg + b * N * BW, &mapG, static_cast<int>(col0) + b * BW, 0, &full_bar[s]);
                }
                if constexpr (OPT != kOptNone) {
                    if (has_s0) tma_load_1d(sg + N * TC, o.state0 + col0, row_bytes, &full_bar[s]);
                    if (OPT == kOptAdam) tma_load_1d(sg + (N + 1) * TC, o.state1 + col0, row_bytes, &full_bar[s]);
                }
            }
        }
        griddep_wait();   // before the common tail (training-step form) touches the workspace
    } else {
        griddep_wait();
        for (int e = tid; e < N * NP; e += CONSUMERS) {   // transposed coefficients: sKT[j][i] = K[i][j]
            const int j = e / NP, i = e - j * NP;
            sKT[j][i] = (i < N) ? K[i * N + j] : 0.0f;
            sAT[j][i] = (i < N) ? A[i * N + j] : 0.0f;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(CONSUMERS) : "memory");   // consumers only: the producer lane is in its loop
        const int lane = tid & 31;
        const int set = tid / QT, q = tid - set * QT;   // tile set and quad within the tile
        f32x2 pacc[PN];
#pragma unroll
        for (int k = 0; k < PN; ++k) pacc[k] = 0ull;
        int it = set;
        int s = set;          // ring slot of tile `it` and its use count (nst > TS): advanced without div / mod
        uint32_t use = 0;
        for (int64_t t = blockIdx.x + static_cast<int64_t>(set) * gridDim.x; t < ntiles;
             t += static_cast<int64_t>(TS) * gridDim.x, it += TS, s += TS, use += (s >= nst), s -= (s >= nst) ? nst : 0) {
            const int64_t col0 = t * TC;
            const int64_t w = (d4 - col0 < TC) ? d4 - col0 : TC;
            const bool active = 4 * q < w;
            if constexpr (TS > 1) {
                // another set consumed this stage's previous use: once that release is visible the full barrier can
                // only be in phase `use`, so the parity wait below cannot alias an older phase
                if (use > 0) mbar_wait(&empty_bar[s], (use - 1u) & 1u);
            }
            mbar_wait(&full_bar[s], use & 1u);
            const float* stage = tiles + static_cast<size_t>(s) * ROWS * TC;
            const float* sx = stage + (q / (BW / 4)) * (N * BW) + 4 * (q % (BW / 4));   // row j of this quad: sx + j * BW
            const float* sg = sx + N * TC;
            const float* sst = stage + 2 * N * TC + 4 * q;                              // optimizer-state rows: sst + r * TC
            f32x2 acc[N][2];
#pragma unroll
            for (int i = 0; i < N; ++i) acc[i][0] = acc[i][1] = 0ull;
            if (active) {
                if constexpr (kApplyRolled) {
#pragma unroll(kApplyJUnroll)
                    for (int j = 0; j < N; ++j) apply_row<N, true>(acc, lds_v4(sg + j * BW), lds_v4(sx + j * BW), sKT[j], sAT[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < N; ++j) apply_row<N>(acc, lds_v4(sg + j * BW), lds_v4(sx + j * BW), sKT[j], sAT[j]);
                }
            }
            if constexpr (OPT == kOptNone) {
                // this warp is done reading the stage: hand it back to the producer, then store
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);
                if (active) {
                    float* op = out + col0 + 4 * q;
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        V4 v;
                        v.lo = acc[i][0];
                        v.hi = acc[i][1];
                        stg_stream_v4(op + i * ldo, v);
                    }
                }
            } else {
                V4 s0, s1;
                s0.lo = s0.hi = s1.lo = s1.hi = 0ull;
                V4 xn[NEXT ? N : 1];
                if constexpr (NEXT) {
#pragma unroll
                    for (int i = 0; i < N; ++i) xn[i].lo = xn[i].hi = 0ull;
                }
                if (active) {
                    float* xw = const_cast<float*>(X) + col0 + 4 * q;
                    if (has_s0) s0 = lds_v4(sst);
                    if (OPT == kOptAdam) s1 = lds_v4(sst + TC);
                    if (o.out_last) {
                        V4 v;
                        v.lo = acc[N - 1][0];
                        v.hi = acc[N - 1][1];
                        stg_stream_v4(o.out_last + col0 + 4 * q, v);
                    }
#pragma unroll
                    for (int i = 0; i < N; ++i) {
                        V4 x = lds_v4(sx + i * BW);
                        opt_update_quad<OPT>(o, i, acc[i][0], acc[i][1], x, s0, s1);
                        stg_stream_v4(xw + i * ldx, x);
                        if constexpr (NEXT) xn[i] = x;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty_bar[s]);
                if (active) {
                    if (OPT == kOptAdam || o.momentum != 0.0f) stg_stream_v4(o.state0 + col0 + 4 * q, s0);
                    if (OPT == kOptAdam) stg_stream_v4(o.state1 + col0 + 4 * q, s1);
                }
                if constexpr (NEXT) {
                    // the K1 of the next step, on the updated particles while they are still in registers
                    pair_accumulate<N, 0>(xn, pacc);
                    // `it` is uniform over the tile set (all of its warps walk the same tiles): warp-level flush
                    if (((it / TS) % kFlushTiles) == kFlushTiles - 1) flush_pairs<PN>(pacc, wacc[tid >> 5], lane);
                }
            }
        }
        // ragged tail columns (D % 4), CTA 0 only
        if constexpr (NEXT) {
            V4 xt[N];
#pragma unroll
            for (int i = 0; i < N; ++i) xt[i].lo = xt[i].hi = 0ull;
            if (blockIdx.x == 0 && tid < (D & 3)) {
                float xnew[N];
                apply_tail_column<N, OPT>(X, G, out, sKT, sAT, d4 + tid, ldx, ldg, ldo, o, xnew);
#pragma unroll
                for (int i = 0; i < N; ++i) xt[i].lo = pack2(xnew[i], 0.0f);
            }
            pair_accumulate<N, 0>(xt, pacc);
            flush_pairs<PN>(pacc, wacc[tid >> 5], lane);
        } else {
            if (blockIdx.x == 0 && tid < (D & 3)) apply_tail_column<N, OPT>(X, G, out, sKT, sAT, d4 + tid, ldx, ldg, ldo, o);
        }
    }
    if constexpr (NEXT) next_dist_epilogue<N, CWARPS>(wacc, nd);
}

// ---------------------------------------------------------------------------------
// host-side launchers
// ---------------------------------------------------------------------------------
template <int N>
int launch_pairdist(const float* X, int64_t D, int64_t ld, double* dist, int accumulate, void* ws, int fuse,
                    const BandwidthParams& bp, cudaStream_t st, int only_if_redo) {
    constexpr int TPB = pairdist_tpb(N);
    constexpr int NG = pair_groups(N);
    {
        constexpr int TC = pd_tile_cols(N);
        const int64_t ntiles = ((D & ~static_cast<int64_t>(3)) + TC - 1) / TC;
        int variant = tuning().pairdist_variant;
        if (variant == 0 || variant > 2) variant = (ntiles >= 2 * static_cast<int64_t>(sm_count_cached())) ? 2 : 1;
        if (variant == 2) {
            constexpr int smem = pd_stages(N) * pd_stage_bytes(N);
            static bool configured = false;
            if (!configured) {
                BDE_RETURN_IF_CUDA(cudaFuncSetAttribute(svgd_pairdist_tma_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                configured = true;
            }
            int64_t grid = sm_count_cached();
            if (grid > ntiles) grid = ntiles;
            if (grid < 1) grid = 1;
            svgd_pairdist_tma_kernel<N><<<static_cast<unsigned>(grid), pd_consumers(N) + 32, smem, st>>>(X, D, ld, dist, accumulate,
                                                                                                 ws, fuse, bp, only_if_redo);
            BDE_CHECK_LAUNCH();
            return BDE_OK;
        }
    }
    static int ctas_per_sm = 0;
    if (ctas_per_sm == 0) {
        int v = 0;
        BDE_RETURN_IF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, svgd_pairdist_kernel<N>, TPB * NG, 0));
        ctas_per_sm = v > 0 ? v : 1;
    }
    const int64_t nquads = D >> 2;
    int64_t want = (nquads + TPB - 1) / TPB;
    int per_sm = ctas_per_sm;
    if (tuning().pairdist_ctas_per_sm > 0 && tuning().pairdist_ctas_per_sm < per_sm) per_sm = tuning().pairdist_ctas_per_sm;
    int64_t cap = static_cast<int64_t>(sm_count_cached()) * per_sm;
    // small D: the deterministic last-CTA reduction costs O(grid * pairs); one CTA per SM keeps it short
    if (tuning().pairdist_ctas_per_sm == 0 && want <= 16 * static_cast<int64_t>(sm_count_cached())) cap = sm_count_cached();
    if (cap > kMaxCtasPairdist) cap = kMaxCtasPairdist;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    svgd_pairdist_kernel<N><<<dim3(static_cast<unsigned>(want)), dim3(TPB, NG), 0, st>>>(X, D, ld, dist, accumulate, ws,
                                                                                      fuse, bp, only_if_redo);
    BDE_CHECK_LAUNCH();
    return BDE_OK;
}

template <int N, int OPT, bool NEXT, int TS, int TC>
int launch_apply_tma(const float* X, const float* G, float* out, const float* K, const float* A, int64_t D, int64_t ldx,
                     int64_t ldg, int64_t ldo, const BaseOptParams& o, cudaStream_t st, const NextDistParams& nd) {
    constexpr int smem = apply_stages(N, OPT, TC) * apply_stage_bytes(N, OPT, TC);
    static_assert(apply_stages(N, OPT, TC) >= 2, "ring too shallow");
    const int64_t d4 = D & ~static_cast<int64_t>(3);
    const int64_t ntiles = (d4 + TC - 1) / TC;
    static bool configured = false;
    if (!configured) {
        BDE_RETURN_IF_CUDA(cudaFuncSetAttribute(svgd_apply_tma_kernel<N, OPT, NEXT, TS, TC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
    // tensor maps over the first d4 columns of X and G: columns of the last tile beyond d4 arrive as zeros
    CUtensorMap mapX, mapG;
    int rc = encode_rows_tensor_map(&mapX, X, N, d4, ldx, kTmaBoxCols);
    if (rc == BDE_OK) rc = encode_rows_tensor_map(&mapG, G, N, d4, ldg, kTmaBoxCols);
    if (rc != BDE_OK) return rc;
    int nst = apply_stages(N, OPT, TC);
    // Ring depth in use.  With tensor-map loads the producer is no longer the limit, and for the plain K2 at n <= 12 a
    // ~128 KB ring streams faster than the whole ~164-200 KB one (interleaved same-build A/B, profiles/r02_ring_ab.jsonl:
    // n = 10 -5.6 %, n = 5 -1.4 %, n = 8 +-0; n = 16 / 20 and the fused forms are best or mixed at full depth) — fewer
    // reads in flight leave the DRAM queues room for the write stream.  bde_tune("ring_kb") overrides (A/B runs).
    int ring_kb = tuning().ring_kb;
    if (ring_kb == 0 && OPT == kOptNone && !NEXT && N <= 12) ring_kb = 128;
    if (ring_kb > 0) {
        const int want = ring_kb * 1024 / apply_stage_bytes(N, OPT, TC);
        if (want < nst) nst = want > TS + 1 ? want : TS + 1;
    }
    int64_t grid = sm_count_cached();
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(TS * (TC / 4) + 32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_for_this_apply() ? 1 : 0;   // only when the caller vouched that K1 is the preceding launch
    pdl_for_this_apply() = false;
    BDE_RETURN_IF_CUDA(cudaLaunchKernelEx(&cfg, svgd_apply_tma_kernel<N, OPT, NEXT, TS, TC>, mapX, mapG, X, G, out, K, A, D, ldx,
                                          ldg, ldo, o, nd, nst));
    return BDE_OK;
}

template <int N, int OPT, bool NEXT = false>
int launch_apply_opt(const float* X, const float* G, float* out, const float* K, const float* A, int64_t D, int64_t ldx,
                     int64_t ldg, int64_t ldo, const BaseOptParams& o, cudaStream_t st,
                     const NextDistParams& nd = NextDistParams{}) {
    const int64_t nquads = D >> 2;
    constexpr int TC = apply_tile_cols(N, OPT, NEXT);
    constexpr int TS0 = apply_default_tile_sets(N, OPT, NEXT);
    const int64_t d4 = D & ~static_cast<int64_t>(3);
    const int64_t ntiles = (d4 + TC - 1) / TC;
    int variant = tuning().apply_variant;
    // auto: the staged kernel wins once every SM has a few tiles per tile set — and, for K2 / K2f, already from 64 K columns on:
    // the direct kernel at n = 20 loads its 40 row quads one j at a time (rolled loop, ~20 exposed latencies per thread), the
    // ring keeps them all in flight.  Measured with a flushed L2 (profiles/r02_apply_small.jsonl): n = 20, D = 273,664: K2 27.0 ->
    // 21.7 us, K2f 30.7 -> 23.9 us; n = 10, D = 65,536: 11.3 -> 8.9 us; never slower from 65,536 columns up at n = 5 ... 20.
    // (The training-step form keeps its own rule: it was not part of that measurement.)
    if (variant == 0) {
        variant = (ntiles >= 2 * TS0 * static_cast<int64_t>(sm_count_cached()) || (!NEXT && d4 >= 65536)) ? 2 : 1;
    }
    if (d4 == 0 || d4 > 0x7fffffffLL) variant = 1;   // the tensor maps need >= 1 column quad and int32 coordinates
    if (variant == 2) {
        // "apply_tile_sets" selects the alternative geometry (A/B runs and the parity tests of both)
        constexpr int TS_ALT = !apply_small_tiles(N, OPT, NEXT) ? 3 : (N > 12 ? 7 - TS0 : 1);
        constexpr int TC_ALT = N > 12 ? 256 : 768 - TC;
        if (tuning().apply_tile_sets == TS_ALT) return launch_apply_tma<N, OPT, NEXT, TS_ALT, TC_ALT>(X, G, out, K, A, D, ldx, ldg, ldo, o, st, nd);
        if constexpr (!NEXT && OPT == kOptNone && N <= 12 && apply_small_tiles(N, OPT, NEXT)) {
            // plain K2, same-box A/B at n = 10 (profiles/r01_geometry_vs_D.jsonl): 3 x 256 wins by 3-8 % up to D = 1e8 but
            // loses 3-6 % from D = 2e8 on (rows 0.8 GB apart: half as many bytes per touched page as 512-column tiles)
            if (tuning().apply_tile_sets == 0 && static_cast<int64_t>(N) * ldx > kApplySmallTileMaxElems)
                return launch_apply_tma<N, OPT, NEXT, TS_ALT, TC_ALT>(X, G, out, K, A, D, ldx, ldg, ldo, o, st, nd);
        }
        return launch_apply_tma<N, OPT, NEXT, TS0, TC>(X, G, out, K, A, D, ldx, ldg, ldo, o, st, nd);
    }
    static int ctas_per_sm = 0;
    if (ctas_per_sm == 0) {
        int v = 0;
        BDE_RETURN_IF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, svgd_apply_kernel<N, OPT, NEXT>, 128, 0));
        ctas_per_sm = v > 0 ? v : 1;
    }
    int64_t want = (nquads + 127) / 128;
    const int per_sm = tuning().apply_ctas_per_sm > 0 ? tuning().apply_ctas_per_sm : ctas_per_sm;
    int64_t cap = static_cast<int64_t>(sm_count_cached()) * per_sm;
    // training-step form: the deterministic last-CTA reduction costs O(grid * pairs) -> one CTA per SM at small D
    if (NEXT && tuning().apply_ctas_per_sm == 0 && want <= 16 * static_cast<int64_t>(sm_count_cached())) cap = sm_count_cached();
    if (NEXT && cap > kMaxCtasPairdist) cap = kMaxCtasPairdist;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    svgd_apply_kernel<N, OPT, NEXT><<<static_cast<unsigned>(want), 128, 0, st>>>(X, G, out, K, A, D, ldx, ldg, ldo, o, nd);
    BDE_CHECK_LAUNCH();
    return BDE_OK;
}

template <int N>
int launch_apply(const float* X, const float* G, float* out, const float* K, const float* A, int64_t D, int64_t ldx,
                 int64_t ldg, int64_t ldo, cudaStream_t st) {
    return launch_apply_opt<N, kOptNone>(X, G, out, K, A, D, ldx, ldg, ldo, BaseOptParams{}, st);
}

// fused K2 + base-optimizer step; X updated in place.  next != nullptr (n <= kNextDistMaxParticles): the
// training-step form that also produces the pair distances of the updated particles.
template <int N>
int launch_apply_fused(float* X, const float* G, const float* K, const float* A, int64_t D, int64_t ldx, int64_t ldg,
                       const BaseOptParams& o, cudaStream_t st, const NextDistParams* next) {
    if constexpr (N <= kNextDistMaxParticles) {
        if (next) {
            if (o.kind == kOptSgd) return launch_apply_opt<N, kOptSgd, true>(X, G, nullptr, K, A, D, ldx, ldg, 0, o, st, *next);
            return launch_apply_opt<N, kOptAdam, true>(X, G, nullptr, K, A, D, ldx, ldg, 0, o, st, *next);
        }
    } else {
        if (next) return BDE_ERR_UNSUPPORTED_N;
    }
    if (o.kind == kOptSgd) return launch_apply_opt<N, kOptSgd>(X, G, nullptr, K, A, D, ldx, ldg, 0, o, st);
    return launch_apply_opt<N, kOptAdam>(X, G, nullptr, K, A, D, ldx, ldg, 0, o, st);
}

}  // namespace bde
