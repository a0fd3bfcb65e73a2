// common.cuh — shared device helpers for the sm_100a posterior-update kernels.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

#include "bde_b200.h"

namespace bde {

// ----------------------------------------------------------------------------
// launch helpers
// ----------------------------------------------------------------------------
#define BDE_RETURN_IF_CUDA(expr)                       \
    do {                                               \
        cudaError_t _e = (expr);                       \
        if (_e != cudaSuccess) return static_cast<int>(_e); \
    } while (0)

#define BDE_CHECK_LAUNCH()                             \
    do {                                               \
        cudaError_t _e = cudaGetLastError();           \
        if (_e != cudaSuccess) return static_cast<int>(_e); \
    } while (0)

inline int sm_count_cached() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        cached[dev] = v;
    }
    return cached[dev];
}

// runtime launch-geometry overrides (0 = automatic); set through bde_tune(), used by the sweep tool
struct Tuning {
    int pairdist_ctas_per_sm = 0;
    int apply_ctas_per_sm = 0;
    int ew_ctas_per_sm = 0;
    int apply_variant = 0;     // 0 auto, 1 direct-LDG kernel, 2 TMA-staged kernel
    int pairdist_variant = 0;  // same for K1; 3 = centred-Gram kernel (n = 16 / 20), 4 = Gram + forced redo (tests)
    int ew_variant = 0;        // same for the elementwise family (ew_tma.cuh)
    int apply_tile_sets = 0;   // staged K2: alternative consumer geometry (0 = default; see launch_apply_opt)
    int swag_batch = 0;        // draws per pass of the batched SWAG sampler (0 = default 16; 2, 4, 8, 16; 1 = general kernels, SWAG and iVON)
    int batch_splits = 0;      // fast batched SWAG sampler: partner CTAs per pass (0 = default 1; 2, 4)
    int batch_prefetch = 0;    // fast batched samplers: L2 prefetch distance in grid-stride iterations (0 = default 1; 9 = off)
    int gram_pairing = 0;      // centred-Gram K1: warp -> pair-group mapping (svgd_gram.cuh:gram_warp_role)
    int gram_fold = 0;         // Gram K1 register budget: 0 auto, 1 producer warpgroup + setmaxnreg (SHIFT), 2 plain ninth warp
    int gram_l2_promotion = 0; // tensor-map L2 promotion of the Gram kernel's tile loads: 0 none, 1 64 B, 2 128 B, 3 256 B
    int ring_kb = 0;           // staged SVGD kernels: cap on the shared-memory ring in use, KB (0 = whole ring)
    int gram_guard_x1000 = 0;  // centred-Gram K1: acceptance bound (S_ii + S_jj) / d_ij in 1/1000 (0 = default 32.0; 1 forces the exact redo)
};
Tuning& tuning();

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ----------------------------------------------------------------------------
// packed FP32x2 (Blackwell FADD2 / FMUL2 / FFMA2): two fp32 lanes in one 64-bit reg
// ----------------------------------------------------------------------------
typedef unsigned long long f32x2;

__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// explicitly rounded packed add / mul: ptxas may contract the un-suffixed forms into an FFMA2, these it may not
__device__ __forceinline__ f32x2 mul2_rn(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2_rn(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// scalar-broadcast multiply-add: ptxas folds pack2(s, s) into the FFMA2 ".F32" operand form
__device__ __forceinline__ f32x2 fma2s(float s, f32x2 b, f32x2 c) { return fma2(pack2(s, s), b, c); }

// ----------------------------------------------------------------------------
// 128-bit streaming global access (read-once / write-once data: keep it out of L1)
// ----------------------------------------------------------------------------
struct __align__(16) V4 {
    f32x2 lo, hi;  // columns (0,1) and (2,3)
};

__device__ __forceinline__ V4 ldg_stream_v4(const float* p) {
    V4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(v.lo), "=l"(v.hi) : "l"(p));
    return v;
}
// cached variant (several warps of one CTA re-read the same lines)
__device__ __forceinline__ V4 ldg_cached_v4(const float* p) {
    V4 v;
    asm volatile("ld.global.nc.v2.u64 {%0, %1}, [%2];" : "=l"(v.lo), "=l"(v.hi) : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream_v4(float* p, V4 v) {
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(v.lo), "l"(v.hi) : "memory");
}
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
// plain (coherent) 128-bit load for buffers that the same kernel also writes
__device__ __forceinline__ float4 ld_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void stg_stream_f4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}

// ----------------------------------------------------------------------------
// TMA bulk copies (cp.async.bulk, SASS UBLKCP) completing on shared-memory mbarriers
// ----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy of `bytes` (multiple of 16, both sides 16-byte aligned)
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// non-blocking probe of an mbarrier phase
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred P1;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// TMA tensor-map load (SASS UTMALDG.2D): box [rows x box_cols] of a row-major fp32 matrix starting at column c0, row c1,
// lands densely ([rows][box_cols]) at smem_dst; columns / rows outside the tensor are zero-filled and still counted
// in the barrier's transaction bytes.  Measured on B200 (tools/microbench/tma_stream.cu): one elected lane issuing
// one cp.async.bulk per 1 KB row segment cannot stream more than ~3-4 TB/s (the copy instruction is the limit); one
// tensor-map load per [20 x 256] box streams 6.8-7.3 TB/s.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_map(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// host: tensor map over the rows of M[rows, cols] (row stride ld elements), box = box_cols x rows (svgd_gram.cu)
int encode_rows_tensor_map(CUtensorMap* map, const float* M, int rows, int64_t cols, int64_t ld, int box_cols,
                           int l2_promotion = 0);
constexpr int kTmaBoxCols = 256;   // widest box dimension the tensor map allows

__device__ __forceinline__ V4 lds_v4(const float* p) {
    V4 v;
    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(v.lo), "=l"(v.hi) : "r"(smem_u32(p)));
    return v;
}

// ----------------------------------------------------------------------------
// Programmatic dependent launch (K1 -> K2): K1 calls griddep_launch() once its streaming loop is done, so that a K2
// launched with cudaLaunchAttributeProgrammaticStreamSerialization becomes resident during K1's tail (grid reduction,
// cross-rank exchange, K1b) and fills its shared-memory ring; K2 calls griddep_wait() — which returns when the WHOLE
// preceding grid has completed and its writes are visible — before it reads K / A or writes anything.  Both are no-ops
// for ordinary launches.
// ----------------------------------------------------------------------------
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// host: did the caller declare (bde_svgd_chain_next) that the next apply launch on `st` directly follows this library's
// K1 launch, nothing else enqueued in between?  Consumed by the first apply launch that asks.
bool take_chain_hint(cudaStream_t st);
// set by apply_impl / apply_opt_impl from the hint for the launch they are about to make; read (and cleared) by the staged launcher
bool& pdl_for_this_apply();

// ----------------------------------------------------------------------------
// reductions
// ----------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ----------------------------------------------------------------------------
// Peer exchange over NVLink (D-sharded jobs, SURVEY.md §8e).  A reduction workspace that has been
// attached to a peer set (bde_peer_attach) makes the LAST CTA of a grid reduction finish the sum
// across the R ranks inside the same launch: it stores its `count` fp64 totals into slot [rank] of
// every peer's exchange buffer (plain P2P stores through NVLink / NVSwitch), publishes a per-rank
// epoch flag with release.sys semantics, waits for the R flags in its own buffer and adds the R
// slots in rank order — so every rank obtains the bit-identical global sums without a separate
// all-reduce launch.  Buffers are double-buffered by epoch parity: a rank can only reach epoch e+2
// after every peer has published e+1, i.e. after it finished reading e.
// ----------------------------------------------------------------------------
constexpr int kPeerMaxRanks = 16;
constexpr int kPeerMaxVals = 512;   // >= pair_count(32) = 496: the exchange covers n <= 32 (larger sums stay rank-local)
struct PeerBuf {                    // one per rank, cudaMalloc'ed (IPC-shareable), zero-filled
    unsigned long long epoch;       // exchanges completed on this rank (device-side counter)
    unsigned long long timeouts;    // exchanges abandoned after kPeerTimeoutNs (results poisoned with NaN)
    unsigned long long wait_ns_sum; // time the last CTA spent waiting for its slowest peer, summed over exchanges ...
    unsigned long long wait_ns_max; // ... and the longest single wait (rank skew; bde_peer_wait_stats)
    unsigned long long waits;       // exchanges counted in the two fields above
    unsigned long long pad[11];
    unsigned long long flags[2][kPeerMaxRanks][4];   // [parity][writer rank], one 32-byte sector each
    double slots[2][kPeerMaxRanks][kPeerMaxVals];    // [parity][writer rank][value]
};
struct WsHeader {                   // first kWsHeaderBytes of every reduction workspace
    unsigned int ticket;            // CTA arrival counter (left at zero by every launch)
    int peer_world;                 // 0 / 1: workspace not attached, plain single-GPU reduction
    int peer_rank;
    int redo;                       // set by the centred-Gram K1 (svgd_gram.cuh) when its cancellation guard fails: the
                                    // direct K1 enqueued behind it (only_if_redo) then recomputes exact distances
    PeerBuf* peer[kPeerMaxRanks];   // peer[r] = rank r's exchange buffer mapped into this process
    unsigned long long timeout_ns;  // how long the last CTA waits for its peers (0 = kPeerTimeoutNs)
    unsigned long long* host_status;   // pinned, device-mapped host word (may be null): receives the number of abandoned
                                       // exchanges, so the host can notice a failure without synchronising
    int peer_failed;                // sticky: an exchange on this workspace timed out — every later exchange is skipped
                                    // (sums poisoned, K1b not run) until the workspace is attached again
};
constexpr size_t kWsHeaderBytes = 256;
static_assert(sizeof(WsHeader) <= kWsHeaderBytes, "workspace header");
constexpr unsigned long long kPeerTimeoutNs = 120ull * 1000 * 1000 * 1000;   // default; bde_peer_attach sets the real one

__device__ __forceinline__ void st_relaxed_sys_f64(double* p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys_f64(const double* p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// Build-time instrumentation (-DBDE_TAIL_TIMING, tools/exp_tail_timing.py; never in the shipped library): %globaltimer stamps
// in the unused bytes 192.. of the workspace header — where K1's fixed cost goes at small D.
#ifdef BDE_TAIL_TIMING
#define BDE_TS_SLOT(ws_, i) (reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(ws_) + 192) + (i))
#define BDE_TS(ws_, i)                                                                       \
    do {                                                                                     \
        if (threadIdx.x == 0 && threadIdx.y == 0) *BDE_TS_SLOT(ws_, i) = globaltimer_ns();   \
    } while (0)
#define BDE_TS_MAX(ws_, i)                                                                             \
    do {                                                                                               \
        if (threadIdx.x == 0 && threadIdx.y == 0) atomicMax(BDE_TS_SLOT(ws_, i), globaltimer_ns());    \
    } while (0)
#else
#define BDE_TS(ws_, i) do { } while (0)
#define BDE_TS_MAX(ws_, i) do { } while (0)
#endif

// Called by every thread of the last CTA with the local sums in total[0..count): on return total holds
// the sums over all ranks (same bits on every rank).  No-op for an unattached workspace.
__device__ __forceinline__ void peer_allreduce_fp64(WsHeader* h, double* total, int count) {
    const int world = h->peer_world;
    if (world <= 1) return;
    const int rank = h->peer_rank;
    const int tid = threadIdx.x + threadIdx.y * blockDim.x;
    const int nthreads = blockDim.x * blockDim.y;
    const double poison = __longlong_as_double(0x7ff8000000000000LL);
    if (h->peer_failed) {   // an earlier exchange was abandoned: the ranks' epochs may no longer pair up
        for (int k = tid; k < count; k += nthreads) total[k] = poison;
        __syncthreads();
        return;
    }
    PeerBuf* me = h->peer[rank];
    __shared__ unsigned long long s_epoch;
    __shared__ unsigned long long s_wait_ns;
    __shared__ int s_timed_out;
    if (tid == 0) {
        s_epoch = *reinterpret_cast<volatile unsigned long long*>(&me->epoch) + 1ull;
        s_timed_out = 0;
        s_wait_ns = 0ull;
    }
    __syncthreads();
    const unsigned long long epoch = s_epoch;
    const unsigned long long limit = h->timeout_ns ? h->timeout_ns : kPeerTimeoutNs;
    const int b = static_cast<int>(epoch & 1ull);
    for (int idx = tid; idx < world * count; idx += nthreads) {
        const int r = idx / count, k = idx - r * count;
        st_relaxed_sys_f64(&h->peer[r]->slots[b][rank][k], total[k]);
    }
    __threadfence_system();
    __syncthreads();
    if (tid < world) {
        st_release_sys_u64(&h->peer[tid]->flags[b][rank][0], epoch);
        const unsigned long long t0 = globaltimer_ns();
        while (ld_acquire_sys_u64(&me->flags[b][tid][0]) < epoch) {
            if (globaltimer_ns() - t0 > limit) {  // a peer never arrived: give up instead of hanging the GPU
                s_timed_out = 1;
                break;
            }
        }
        atomicMax(&s_wait_ns, globaltimer_ns() - t0);   // the slowest peer sets the wait of this exchange
    }
    __syncthreads();
    const bool bad = s_timed_out != 0;
    for (int k = tid; k < count; k += nthreads) {
        double s = 0.0;
        for (int r = 0; r < world; ++r) s += ld_relaxed_sys_f64(&me->slots[b][r][k]);
        total[k] = bad ? poison : s;
    }
    if (tid == 0) {
        *reinterpret_cast<volatile unsigned long long*>(&me->epoch) = epoch;
        me->wait_ns_sum += s_wait_ns;
        if (s_wait_ns > me->wait_ns_max) me->wait_ns_max = s_wait_ns;
        me->waits += 1ull;
        if (bad) {
            const unsigned long long nbad = me->timeouts + 1ull;
            *reinterpret_cast<volatile unsigned long long*>(&me->timeouts) = nbad;
            h->peer_failed = 1;
            if (h->host_status) {
                *reinterpret_cast<volatile unsigned long long*>(h->host_status) = nbad;
                __threadfence_system();
            }
        }
    }
    __syncthreads();
}
// true (in the last CTA, after grid_reduce_fp64) when the cross-rank sum behind `ws` was abandoned: the callers
// then leave K / A as they are instead of running K1b on poisoned sums
__device__ __forceinline__ bool peer_exchange_failed(const void* ws) { return reinterpret_cast<const WsHeader*>(ws)->peer_failed != 0; }

// Deterministic grid-wide fp64 sum of `count` values per CTA.
//   cta_vals: this CTA's values in shared memory (count doubles), valid after __syncthreads.
//   ws layout: WsHeader (ticket + optional peer table, kWsHeaderBytes), then gridDim.x*count doubles.
// Returns true in every thread of the LAST CTA to arrive, after which total[k] = sum over all
// CTAs (and, for a workspace attached to a peer set, over all ranks) is available in `total`
// (shared, count doubles).  The order of the additions depends only
// on (gridDim, count): every warp of the last CTA owns groups of 4 consecutive values k, its lanes
// walk the CTA list with stride 32 (coalesced: the partials are stored value-major) keeping 4 x 8 independent loads in
// flight, and the 32 lane sums are combined by the fixed xor-shuffle tree.  The ticket is reset so
// the workspace can be reused by the next launch.
__device__ __forceinline__ bool grid_reduce_fp64(const double* cta_vals, int count, void* ws, double* total) {
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws);
    double* parts = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + kWsHeaderBytes);
    const int tid = threadIdx.x + threadIdx.y * blockDim.x;
    const int nthreads = blockDim.x * blockDim.y;
    __shared__ bool is_last;
    // value-major layout parts[k][cta]: the last CTA's lanes walk the CTA list, so consecutive lanes read consecutive
    // doubles — one 256-byte request per warp load.  (CTA-major, every lane touched its own 32-byte sector with four
    // separate 8-byte loads: 128 sector transactions per warp and group, 18.6 us for 148 x 190 values at n = 20 —
    // measured with the stamps below, profiles/r02_tail_timing.jsonl.  Same addends in the same order: same bits.)
    for (int k = tid; k < count; k += nthreads) parts[(size_t)k * gridDim.x + blockIdx.x] = cta_vals[k];
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        unsigned int prev = atomicAdd(ticket, 1u);
        is_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return false;
    __threadfence();
    BDE_TS(ws, 2);
    constexpr int KU = 4, BU = 8;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;  // CTA sizes are multiples of 32
    const unsigned int G = gridDim.x;
    for (int k0 = warp * KU; k0 < count; k0 += nwarps * KU) {
        double s[KU];
#pragma unroll
        for (int u = 0; u < KU; ++u) s[u] = 0.0;
        for (unsigned int b0 = lane; b0 < G; b0 += 32 * BU) {
            double v[BU][KU];
#pragma unroll
            for (int r = 0; r < BU; ++r) {
                const unsigned int b = b0 + 32u * r;
#pragma unroll
                for (int u = 0; u < KU; ++u)
                    v[r][u] = (b < G && k0 + u < count) ? __ldcg(&parts[(size_t)(k0 + u) * G + b]) : 0.0;
            }
#pragma unroll
            for (int r = 0; r < BU; ++r)
#pragma unroll
                for (int u = 0; u < KU; ++u) s[u] += v[r][u];
        }
#pragma unroll
        for (int u = 0; u < KU; ++u) {
            const double t = warp_sum(s[u]);
            if (lane == 0 && k0 + u < count) total[k0 + u] = t;
        }
    }
    if (tid == 0) *ticket = 0u;
    __syncthreads();
    BDE_TS(ws, 3);
    if (count <= kPeerMaxVals) peer_allreduce_fp64(reinterpret_cast<WsHeader*>(ws), total, count);
    return true;
}

inline size_t grid_reduce_ws_bytes(int max_ctas, int count) { return kWsHeaderBytes + sizeof(double) * (size_t)max_ctas * count; }

// ----------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011) + Box-Muller.  counter = (q_lo, q_hi, sid_lo, sid_hi)
// with q = global element index / 4; key = 64-bit seed.  One call -> 4 normals for
// elements 4q .. 4q+3.
// ----------------------------------------------------------------------------
// 32 x 32 -> 64-bit product as ONE IMAD.WIDE.U32 with both halves used.  (Written as a C++ 64-bit multiply, ptxas keeps a
// dead "+ 0" on the high word of every product — the zero-extended operand's upper half — one extra IADD3 per product,
// 20 per Philox call; seen in SASS.)
__device__ __forceinline__ void mul_wide_u32(unsigned int a, unsigned int b, unsigned int& hi, unsigned int& lo) {
    unsigned long long p;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(p) : "r"(a), "r"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(p));
}

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    constexpr unsigned int M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        // one IMAD.WIDE.U32 per product (hi and lo halves together); the key schedule is uniform
        unsigned int hi0, lo0, hi1, lo1;
        mul_wide_u32(M0, ctr.x, hi0, lo0);
        mul_wide_u32(M1, ctr.z, hi1, lo1);
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0;
        key.y += W1;
    }
    return ctr;
}

// The same function with the ten round keys precomputed (they depend on the seed only): kernels that draw many streams
// per thread (the batched samplers) build them once before their element loop instead of once per call.
struct PhiloxKeys {
    uint2 rk[10];
};
__device__ __forceinline__ PhiloxKeys philox_round_keys(uint64_t seed) {
    PhiloxKeys k;
    uint2 key = make_uint2(static_cast<unsigned int>(seed), static_cast<unsigned int>(seed >> 32));
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        k.rk[r] = key;
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return k;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, const PhiloxKeys& k) {
    constexpr unsigned int M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        unsigned int hi0, lo0, hi1, lo1;
        mul_wide_u32(M0, ctr.x, hi0, lo0);
        mul_wide_u32(M1, ctr.z, hi1, lo1);
        ctr = make_uint4(hi1 ^ ctr.y ^ k.rk[r].x, lo1, hi0 ^ ctr.w ^ k.rk[r].y, lo0);
    }
    return ctr;
}

// 23 random bits -> the float 2^23 + x, x in [0, 2^23): ONE logic op, exact.  (An int -> float conversion is an XU-pipe
// instruction like the MUFU transcendentals — quarter rate; four of them per normal quad made the XU pipe the co-limiter of
// the batched samplers: ncu, math-pipe-throttle / dispatch stalls.)
__device__ __forceinline__ float bits23_to_float(unsigned int r) {
    unsigned int d;   // (r & mask) | magic as one LOP3 (from C, ptxas emits an AND and an OR: two immediates do not fit one LOP3)
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(r), "r"(0x007FFFFFu), "r"(0x4B000000u));
    return __uint_as_float(d);
}

__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // MUFU.SQRT, ~1 ulp
    return r;
}
// Pull the 128-byte line of `p` into L2 without occupying a register or a scoreboard slot (no data returns to the SM).
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ float lg2_approx(float x) {
    // MUFU.LG2 alone.  __log2f() wraps it in a denormal-input path (FSETP, predicated FMUL by 2^24, predicated FADD -24: three
    // issue slots per call that never execute for our inputs, u >= 2^-25); for normal inputs the result is the same bits.
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));  // MUFU.RSQ, ~1 ulp
    return r;
}

// Box-Muller on the SFU: radius from MUFU.LG2 + MUFU.SQRT, angle uniform on [-pi, pi) where MUFU.SIN/COS are accurate to
// 2^-21.4 absolute.  Both uniforms come from the low 23 bits of a Philox word through bits23_to_float and one FMA each:
//   u   = (2 x0 + 1) 2^-24            in (0, 1), exact, symmetric, never 0 or 1   (|z| <= 5.77)
//   ang = (2^23 + x1) 2 pi 2^-23 - 3 pi   in [-pi, pi)
// (Noise quality, not reference parity: parity tests inject the reference's own noise.  oracle/bde_oracle.py:philox_normal
// restates this function.)
__device__ __forceinline__ void box_muller(unsigned int r0, unsigned int r1, float& z0, float& z1) {
    const float u = fmaf(bits23_to_float(r0), 1.1920928955078125e-07f, 5.9604644775390625e-08f - 1.0f);
    const float ang = fmaf(bits23_to_float(r1), 7.4901405658478572e-07f, -9.42477796076937972f);
    const float rad = sqrt_approx(fmaxf(-1.3862943611198906f * lg2_approx(u), 0.0f));  // sqrt(-2 ln u)
    z0 = rad * __cosf(ang);
    z1 = rad * __sinf(ang);
}

__device__ __forceinline__ float4 philox_normal4(uint64_t seed, uint64_t stream_id, uint64_t quad) {
    const uint4 ctr = make_uint4(static_cast<unsigned int>(quad), static_cast<unsigned int>(quad >> 32),
                                 static_cast<unsigned int>(stream_id), static_cast<unsigned int>(stream_id >> 32));
    const uint2 key = make_uint2(static_cast<unsigned int>(seed), static_cast<unsigned int>(seed >> 32));
    const uint4 r = philox4x32_10(ctr, key);
    float4 z;
    box_muller(r.x, r.y, z.x, z.y);
    box_muller(r.z, r.w, z.z, z.w);
    return z;
}

__device__ __forceinline__ float4 philox_normal4(const PhiloxKeys& k, uint64_t stream_id, uint64_t quad) {
    const uint4 ctr = make_uint4(static_cast<unsigned int>(quad), static_cast<unsigned int>(quad >> 32),
                                 static_cast<unsigned int>(stream_id), static_cast<unsigned int>(stream_id >> 32));
    const uint4 r = philox4x32_10(ctr, k);
    float4 z;
    box_muller(r.x, r.y, z.x, z.y);
    box_muller(r.z, r.w, z.z, z.w);
    return z;
}

// torch's softplus (beta=1, threshold=20) and its derivative factor, util.py:181-183
__device__ __forceinline__ float softplus_ref(float x) { return x > 20.0f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float softplus_grad_ref(float x) {
    if (x > 20.0f) return 1.0f;
    const float z = expf(x);
    return __fdiv_rn(z, __fadd_rn(z, 1.0f));
}

// ----------------------------------------------------------------------------
// elementwise launch geometry: each thread handles one float4 per pass, grid-stride
// ----------------------------------------------------------------------------
struct EwGrid {
    int blocks;
    int threads;
};
inline EwGrid ew_grid(int64_t n_elems, int threads, int ctas_per_sm) {
    const int64_t quads = (n_elems + 3) / 4;
    int64_t want = (quads + threads - 1) / threads;
    if (tuning().ew_ctas_per_sm > 0) ctas_per_sm = tuning().ew_ctas_per_sm;
    const int64_t cap = (int64_t)sm_count_cached() * ctas_per_sm;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    return EwGrid{static_cast<int>(want), threads};
}

}  // namespace bde
