// svgd.cu — SVGD posterior update on sm_100a: generic kernels, K1b, dispatch and C-ABI.
// Kernel templates live in svgd_kernels.cuh; reference arithmetic: src/algos/svgd.py:14-32, :83-97.
#include "svgd_kernels.cuh"
#include "svgd_gram.cuh"

namespace bde {

// unaligned / generic fallback: one column per thread, runtime n, fp64 accumulate per thread
__global__ void __launch_bounds__(256)
svgd_pairdist_scalar_kernel(const float* __restrict__ X, int n, int64_t D, int64_t ld, double* __restrict__ dist,
                            int accumulate, void* ws) {
    extern __shared__ double sm[];  // [P] cta_vals, [P] total
    const int P = pair_count(n);
    double* cta_vals = sm;
    double* total = sm + P;
    for (int p = threadIdx.x; p < P; p += blockDim.x) cta_vals[p] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    int p = 0;
    for (int i = 0; i < n; ++i) {
        for (int j = i + 1; j < n; ++j, ++p) {
            double s = 0.0;
            for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < D;
                 c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
                const float d = __ldg(X + i * ld + c) - __ldg(X + j * ld + c);
                s += static_cast<double>(d * d);
            }
            s = warp_sum(s);
            if (lane == 0) atomicAdd(&cta_vals[p], s);  // order within a CTA: fp64, <=8 warps
        }
    }
    __syncthreads();
    if (!grid_reduce_fp64(cta_vals, P, ws, total)) return;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e - i * n;
        double v = 0.0;
        if (i != j) v = total[i < j ? pair_index(i, j, n) : pair_index(j, i, n)];
        if (accumulate) v += dist[e];
        dist[e] = v;
    }
}

// ws (nullable): the reduction workspace that produced `dist` — K1b is skipped after an abandoned peer exchange
__global__ void __launch_bounds__(256) svgd_bandwidth_kernel(const double* __restrict__ dist, int n, BandwidthParams bp,
                                                             const void* ws) {
    if (ws && peer_exchange_failed(ws)) return;
    __shared__ double sd[kGenericMaxParticles * kGenericMaxParticles];
    __shared__ double sk[kGenericMaxParticles * kGenericMaxParticles];
    bandwidth_device<kGenericMaxParticles * kGenericMaxParticles>(dist, n, bp, sd, sk);
}

__global__ void __launch_bounds__(256)
svgd_apply_scalar_kernel(const float* __restrict__ X, const float* __restrict__ G, float* __restrict__ out,
                         const float* __restrict__ K, const float* __restrict__ A, int n, int64_t D, int64_t ldx,
                         int64_t ldg, int64_t ldo) {
    __shared__ float sK[kGenericMaxParticles * kGenericMaxParticles];
    __shared__ float sA[kGenericMaxParticles * kGenericMaxParticles];
    griddep_wait();
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        sK[e] = K[e];
        sA[e] = A[e];
    }
    __syncthreads();
    for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < D;
         c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float xs[kGenericMaxParticles], gs[kGenericMaxParticles];
        for (int j = 0; j < n; ++j) {
            xs[j] = __ldg(X + j * ldx + c);
            gs[j] = __ldg(G + j * ldg + c);
        }
        for (int i = 0; i < n; ++i) {
            float s = 0.0f;
            for (int j = 0; j < n; ++j) {
                s = fmaf(sK[i * n + j], gs[j], s);
                s = fmaf(sA[i * n + j], xs[j], s);
            }
            out[i * ldo + c] = s;
        }
    }
}

// fused K2 + base-optimizer step, generic form (runtime n, any alignment): one column per thread
template <int OPT>
__global__ void __launch_bounds__(256)
svgd_apply_opt_scalar_kernel(float* X, const float* __restrict__ G, const float* __restrict__ K,
                             const float* __restrict__ A, int n, int64_t D, int64_t ldx, int64_t ldg,
                             const __grid_constant__ BaseOptParams o) {
    __shared__ float sK[kGenericMaxParticles * kGenericMaxParticles];
    __shared__ float sA[kGenericMaxParticles * kGenericMaxParticles];
    griddep_wait();
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        sK[e] = K[e];
        sA[e] = A[e];
    }
    __syncthreads();
    const bool has_s0 = (OPT == kOptAdam) || (o.momentum != 0.0f && o.buf_initialized);
    for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < D;
         c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        float xs[kGenericMaxParticles], gs[kGenericMaxParticles];
        for (int j = 0; j < n; ++j) {
            xs[j] = X[j * ldx + c];
            gs[j] = __ldg(G + j * ldg + c);
        }
        float s0 = has_s0 ? o.state0[c] : 0.0f;
        float s1 = (OPT == kOptAdam) ? o.state1[c] : 0.0f;
        for (int i = 0; i < n; ++i) {
            float s = 0.0f;
            for (int j = 0; j < n; ++j) {
                s = fmaf(sK[i * n + j], gs[j], s);
                s = fmaf(sA[i * n + j], xs[j], s);
            }
            if (i == n - 1 && o.out_last) o.out_last[c] = s;
            X[i * ldx + c] = opt_update_scalar<OPT>(o, i, s, xs[i], s0, s1);
        }
        if (OPT == kOptAdam || o.momentum != 0.0f) o.state0[c] = s0;
        if (OPT == kOptAdam) o.state1[c] = s1;
    }
}

// particle counts with a register-resident fast path (explicitly instantiated in svgd_inst_*.cu);
// any other n <= kGenericMaxParticles runs the generic runtime-n kernels, n up to BDE_MAX_PARTICLES svgd_many.cu.
#define BDE_FOR_EACH_N(X_) X_(2) X_(3) X_(4) X_(5) X_(6) X_(7) X_(8) X_(9) X_(10) X_(11) X_(12) X_(16) X_(20)

#define X_(N_)                                                                                                     \
    extern template int launch_pairdist<N_>(const float*, int64_t, int64_t, double*, int, void*, int,              \
                                            const BandwidthParams&, cudaStream_t, int);                                 \
    extern template int launch_apply<N_>(const float*, const float*, float*, const float*, const float*, int64_t, \
                                         int64_t, int64_t, int64_t, cudaStream_t);                           \
    extern template int launch_apply_fused<N_>(float*, const float*, const float*, const float*, int64_t, int64_t, \
                                               int64_t, const BaseOptParams&, cudaStream_t, const NextDistParams*);
BDE_FOR_EACH_N(X_)
#undef X_
extern template int launch_pairgram<16>(const float*, int64_t, int64_t, double*, void*, int, const BandwidthParams&, cudaStream_t);
extern template int launch_pairgram<20>(const float*, int64_t, int64_t, double*, void*, int, const BandwidthParams&, cudaStream_t);

static bool has_fast_path(int n) {
    switch (n) {
#define X_(N_) case N_:
        BDE_FOR_EACH_N(X_)
#undef X_
        return true;
        default:
            return false;
    }
}

static bool overlaps(const void* a, size_t abytes, const void* b, size_t bbytes) {
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(a), b0 = reinterpret_cast<uintptr_t>(b);
    return a0 < b0 + bbytes && b0 < a0 + abytes;
}

int pairdist_impl(const float* X, int n, int64_t D, int64_t ld, double* dist, int accumulate, void* ws,
                  size_t ws_bytes, int fuse, const BandwidthParams& bp, cudaStream_t st) {
    if (!X || !dist || n < 1 || n > BDE_MAX_PARTICLES || D < 0 || ld < D) return BDE_ERR_INVALID_ARG;
    size_t need = 0;
    bde_svgd_workspace_bytes(n, &need);
    if (!ws || ws_bytes < need) return BDE_ERR_WORKSPACE;
    if (n > kGenericMaxParticles) {
        // the in-kernel exchange carries at most kPeerMaxVals sums: an attached workspace would yield rank-local sums
        if (peer_attached(ws)) return BDE_ERR_UNSUPPORTED_N;
        if (!aligned16(X) || ld % 4 != 0) return BDE_ERR_ALIGNMENT;
        return pairdist_many(X, n, D, ld, dist, accumulate, ws, fuse, bp, st);
    }
    if (n == 1) {
        if (!accumulate) BDE_RETURN_IF_CUDA(cudaMemsetAsync(dist, 0, sizeof(double), st));
        if (fuse) {
            svgd_bandwidth_kernel<<<1, 256, 0, st>>>(dist, n, bp, ws);
            BDE_CHECK_LAUNCH();
        }
        return BDE_OK;
    }
    const bool vec_ok = aligned16(X) && (ld % 4 == 0);
    if (!vec_ok || !has_fast_path(n)) {
        const int P = pair_count(n);
        int64_t want = (D + 255) / 256;
        const int64_t cap = static_cast<int64_t>(sm_count_cached()) * 4;
        if (want > cap) want = cap;
        if (want < 1) want = 1;
        svgd_pairdist_scalar_kernel<<<static_cast<unsigned>(want), 256, 2 * P * sizeof(double), st>>>(X, n, D, ld, dist,
                                                                                                  accumulate, ws);
        BDE_CHECK_LAUNCH();
        if (fuse) {
            svgd_bandwidth_kernel<<<1, 256, 0, st>>>(dist, n, bp, ws);
            BDE_CHECK_LAUNCH();
        }
        return BDE_OK;
    }
    // n = 16 / 20, large D, K1b fused: centred-Gram kernel, with the direct kernel enqueued behind it as the exact
    // recomputation that only runs when the Gram kernel's cancellation guard raised `redo` (svgd_gram.cuh)
    int only_if_redo = 0;
    if ((n == 16 || n == 20) && fuse && !accumulate && D <= 0x7fffffffLL &&
        (tuning().pairdist_variant == 3 ||
         (tuning().pairdist_variant == 0 && D >= kGramMinColumns))) {
        const int rc = n == 16 ? launch_pairgram<16>(X, D, ld, dist, ws, fuse, bp, st)
                               : launch_pairgram<20>(X, D, ld, dist, ws, fuse, bp, st);
        if (rc != BDE_OK) return rc;
        only_if_redo = 1;
    }
    switch (n) {
#define X_(N_) \
    case N_:   \
        return launch_pairdist<N_>(X, D, ld, dist, accumulate, ws, fuse, bp, st, only_if_redo);
        BDE_FOR_EACH_N(X_)
#undef X_
        default:
            return BDE_ERR_UNSUPPORTED_N;
    }
}

int apply_impl(const float* X, const float* G, float* out, const float* K, const float* A, int n, int64_t D,
               int64_t ldx, int64_t ldg, int64_t ldo, cudaStream_t st) {
    pdl_for_this_apply() = take_chain_hint(st);   // consumed by whichever apply launch comes first (only the staged kernel uses it)
    if (!X || !G || !out || !K || !A || n < 1 || n > BDE_MAX_PARTICLES || D < 0 || ldx < D || ldg < D || ldo < D)
        return BDE_ERR_INVALID_ARG;
    if (D == 0) return BDE_OK;
    const size_t span_x = sizeof(float) * (static_cast<size_t>(n - 1) * ldx + D);
    const size_t span_g = sizeof(float) * (static_cast<size_t>(n - 1) * ldg + D);
    const size_t span_o = sizeof(float) * (static_cast<size_t>(n - 1) * ldo + D);
    if (overlaps(out, span_o, X, span_x) || overlaps(out, span_o, G, span_g)) return BDE_ERR_INVALID_ARG;
    const bool vec_ok = aligned16(X) && aligned16(G) && aligned16(out) && (ldx % 4 == 0) && (ldg % 4 == 0) && (ldo % 4 == 0);
    if (n > kGenericMaxParticles) return vec_ok ? apply_many(X, G, out, K, A, n, D, ldx, ldg, ldo, st) : BDE_ERR_ALIGNMENT;
    if (!vec_ok || !has_fast_path(n)) {
        int64_t want = (D + 255) / 256;
        const int64_t cap = static_cast<int64_t>(sm_count_cached()) * 4;
        if (want > cap) want = cap;
        svgd_apply_scalar_kernel<<<static_cast<unsigned>(want), 256, 0, st>>>(X, G, out, K, A, n, D, ldx, ldg, ldo);
        BDE_CHECK_LAUNCH();
        return BDE_OK;
    }
    switch (n) {
#define X_(N_) \
    case N_:   \
        return launch_apply<N_>(X, G, out, K, A, D, ldx, ldg, ldo, st);
            BDE_FOR_EACH_N(X_)
#undef X_
        default:
            return BDE_ERR_UNSUPPORTED_N;
    }
}

int apply_opt_impl(float* X, const float* G, const float* K, const float* A, int n, int64_t D, int64_t ldx,
                   int64_t ldg, const BaseOptParams& o, cudaStream_t st, const NextDistParams* next, size_t ws_bytes) {
    pdl_for_this_apply() = take_chain_hint(st);
    if (!X || !G || !K || !A || n < 1 || n > BDE_MAX_PARTICLES || D < 0 || ldx < D || ldg < D) return BDE_ERR_INVALID_ARG;
    if (n > kOptMaxParticles) return BDE_ERR_UNSUPPORTED_N;   // no fused base-optimizer form above 32 particles
    if (o.kind != kOptSgd && o.kind != kOptAdam) return BDE_ERR_INVALID_ARG;
    const bool needs_s0 = o.kind == kOptAdam || o.momentum != 0.0f;
    if ((needs_s0 && !o.state0) || (o.kind == kOptAdam && !o.state1)) return BDE_ERR_INVALID_ARG;
    if (next) {
        if (!next->dist || (next->fuse_bandwidth && (!next->bp.K || !next->bp.A || !(next->bp.dataset_size > 0.0))))
            return BDE_ERR_INVALID_ARG;
        size_t need = 0;
        bde_svgd_workspace_bytes(n, &need);
        if (!next->ws || ws_bytes < need) return BDE_ERR_WORKSPACE;
    }
    const bool vec_all = aligned16(X) && aligned16(G) && (ldx % 4 == 0) && (ldg % 4 == 0) &&
                         (!needs_s0 || aligned16(o.state0)) && (o.kind != kOptAdam || aligned16(o.state1)) &&
                         (!o.out_last || aligned16(o.out_last));
    if (next && (D == 0 || n < 2 || n > kNextDistMaxParticles || !vec_all || !has_fast_path(n))) {
        // no single-pass form for this shape: fused update, then K1 (+K1b) on the updated particles
        const int rc = apply_opt_impl(X, G, K, A, n, D, ldx, ldg, o, st, nullptr, 0);
        if (rc != BDE_OK) return rc;
        return pairdist_impl(X, n, D, ldx, next->dist, 0, next->ws, ws_bytes, next->fuse_bandwidth, next->bp, st);
    }
    if (D == 0) return BDE_OK;
    const size_t span_x = sizeof(float) * (static_cast<size_t>(n - 1) * ldx + D);
    const size_t span_g = sizeof(float) * (static_cast<size_t>(n - 1) * ldg + D);
    if (overlaps(X, span_x, G, span_g)) return BDE_ERR_INVALID_ARG;
    const bool vec_ok = aligned16(X) && aligned16(G) && (ldx % 4 == 0) && (ldg % 4 == 0) &&
                        (!needs_s0 || aligned16(o.state0)) && (o.kind != kOptAdam || aligned16(o.state1)) &&
                        (!o.out_last || aligned16(o.out_last));
    if (!vec_ok || !has_fast_path(n)) {
        int64_t want = (D + 255) / 256;
        const int64_t cap = static_cast<int64_t>(sm_count_cached()) * 4;
        if (want > cap) want = cap;
        if (o.kind == kOptSgd)
            svgd_apply_opt_scalar_kernel<kOptSgd><<<static_cast<unsigned>(want), 256, 0, st>>>(X, G, K, A, n, D, ldx, ldg, o);
        else
            svgd_apply_opt_scalar_kernel<kOptAdam><<<static_cast<unsigned>(want), 256, 0, st>>>(X, G, K, A, n, D, ldx, ldg, o);
        BDE_CHECK_LAUNCH();
        return BDE_OK;
    }
    switch (n) {
#define X_(N_) \
    case N_:   \
        return launch_apply_fused<N_>(X, G, K, A, D, ldx, ldg, o, st, next);
        BDE_FOR_EACH_N(X_)
#undef X_
        default:
            return BDE_ERR_UNSUPPORTED_N;
    }
}

// --- chain hint (programmatic dependent launch of K2 behind K1) ---
namespace {
thread_local cudaStream_t g_chain_stream = nullptr;
thread_local bool g_chain_armed = false;
}  // namespace
bool take_chain_hint(cudaStream_t st) {
    const bool ok = g_chain_armed && g_chain_stream == st;
    g_chain_armed = false;
    return ok;
}
bool& pdl_for_this_apply() {
    thread_local bool v = false;
    return v;
}

}  // namespace bde

using namespace bde;

extern "C" int bde_svgd_chain_next(bde_stream_t stream) {
    g_chain_stream = static_cast<cudaStream_t>(stream);
    g_chain_armed = true;
    return BDE_OK;
}

extern "C" int bde_svgd_workspace_bytes(int n, size_t* bytes) {
    if (!bytes || n < 1 || n > BDE_MAX_PARTICLES) return BDE_ERR_INVALID_ARG;
    const int P = pair_count(n) > 0 ? pair_count(n) : 1;
    *bytes = grid_reduce_ws_bytes(n > kGenericMaxParticles ? kManyMaxCtas : kMaxCtasPairdist, P);
    return BDE_OK;
}

extern "C" int bde_svgd_pairdist(const float* X, int n, int64_t D, int64_t ld, double* dist, int accumulate,
                                 void* workspace, size_t workspace_bytes, bde_stream_t stream) {
    BandwidthParams bp{};
    return pairdist_impl(X, n, D, ld, dist, accumulate, workspace, workspace_bytes, 0, bp,
                         static_cast<cudaStream_t>(stream));
}

extern "C" int bde_svgd_pairdist_bandwidth(const float* X, int n, int64_t D, int64_t ld, double l2_reg,
                                           double kernel_grad_scale, double dataset_size, double h_override,
                                           double* dist, float* K, float* A, double* info, int32_t* sel,
                                           void* workspace, size_t workspace_bytes, bde_stream_t stream) {
    if (!K || !A || !(dataset_size > 0.0)) return BDE_ERR_INVALID_ARG;
    BandwidthParams bp{l2_reg, kernel_grad_scale, dataset_size, h_override, K, A, info, sel};
    return pairdist_impl(X, n, D, ld, dist, 0, workspace, workspace_bytes, 1, bp, static_cast<cudaStream_t>(stream));
}

extern "C" int bde_svgd_bandwidth(const double* dist, int n, double l2_reg, double kernel_grad_scale,
                                  double dataset_size, double h_override, float* K, float* A, double* info,
                                  int32_t* sel, bde_stream_t stream) {
    if (!dist || !K || !A || n < 1 || n > BDE_MAX_PARTICLES || !(dataset_size > 0.0)) return BDE_ERR_INVALID_ARG;
    BandwidthParams bp{l2_reg, kernel_grad_scale, dataset_size, h_override, K, A, info, sel};
    if (n > kGenericMaxParticles) return bandwidth_many(dist, n, bp, static_cast<cudaStream_t>(stream));
    svgd_bandwidth_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(dist, n, bp, nullptr);
    BDE_CHECK_LAUNCH();
    return BDE_OK;
}

extern "C" int bde_svgd_apply(const float* X, const float* G, float* out, const float* K, const float* A, int n,
                              int64_t D, int64_t ld, bde_stream_t stream) {
    return apply_impl(X, G, out, K, A, n, D, ld, ld, ld, static_cast<cudaStream_t>(stream));
}

extern "C" int bde_svgd_step(const float* X, const float* G, float* out, int n, int64_t D, int64_t ld, double l2_reg,
                             double kernel_grad_scale, double dataset_size, double h_override, double* dist, float* K,
                             float* A, double* info, int32_t* sel, void* workspace, size_t workspace_bytes,
                             bde_stream_t stream) {
    if (!K || !A || !(dataset_size > 0.0)) return BDE_ERR_INVALID_ARG;
    BandwidthParams bp{l2_reg, kernel_grad_scale, dataset_size, h_override, K, A, info, sel};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = pairdist_impl(X, n, D, ld, dist, 0, workspace, workspace_bytes, 1, bp, st);
    if (rc != BDE_OK) return rc;
    bde_svgd_chain_next(stream);   // K2 directly behind K1: programmatic dependent launch
    return apply_impl(X, G, out, K, A, n, D, ld, ld, ld, st);
}

static BaseOptParams sgd_params(float* momentum_buf, int buf_initialized, double lr, double momentum, double dampening,
                                double weight_decay, int nesterov, float* out_last) {
    BaseOptParams o;
    o.kind = kOptSgd;
    o.lr = static_cast<float>(lr);
    o.momentum = static_cast<float>(momentum);
    o.one_minus_dampening = static_cast<float>(1.0 - dampening);
    o.weight_decay = static_cast<float>(weight_decay);
    o.nesterov = nesterov ? 1 : 0;
    o.buf_initialized = buf_initialized ? 1 : 0;
    o.state0 = momentum_buf;
    o.out_last = out_last;
    return o;
}

extern "C" int bde_svgd_apply_sgd(float* X, const float* G, const float* K, const float* A, int n, int64_t D, int64_t ld,
                                  float* momentum_buf, int buf_initialized, double lr, double momentum, double dampening,
                                  double weight_decay, int nesterov, float* out_last, bde_stream_t stream) {
    const BaseOptParams o = sgd_params(momentum_buf, buf_initialized, lr, momentum, dampening, weight_decay, nesterov, out_last);
    return apply_opt_impl(X, G, K, A, n, D, ld, ld, o, static_cast<cudaStream_t>(stream));
}

static BaseOptParams adam_params(int n, float* exp_avg, float* exp_avg_sq, int64_t step0, double lr, double beta1,
                                 double beta2, double eps, double weight_decay, int decoupled_weight_decay,
                                 float* out_last) {
    BaseOptParams o;
    o.kind = kOptAdam;
    o.lr = static_cast<float>(lr);
    o.beta1 = static_cast<float>(beta1);
    o.one_minus_beta1 = static_cast<float>(1.0 - beta1);
    o.beta2 = static_cast<float>(beta2);
    o.one_minus_beta2 = static_cast<float>(1.0 - beta2);
    o.eps = static_cast<float>(eps);
    o.weight_decay = static_cast<float>(weight_decay);
    o.decoupled_wd = decoupled_weight_decay ? 1 : 0;
    o.decay_factor = static_cast<float>(1.0 - lr * weight_decay);
    for (int i = 0; i < n; ++i) {
        // python-side scalars of _single_tensor_adam, folded in double like eager PyTorch does
        const double t = static_cast<double>(step0 + i + 1);
        const double bc1 = 1.0 - pow(beta1, t), bc2 = 1.0 - pow(beta2, t);
        o.step_size[i] = static_cast<float>(lr / bc1);
        o.inv_bc2_sqrt[i] = static_cast<float>(1.0 / sqrt(bc2));
    }
    o.state0 = exp_avg;
    o.state1 = exp_avg_sq;
    o.out_last = out_last;
    return o;
}

extern "C" int bde_svgd_apply_adam(float* X, const float* G, const float* K, const float* A, int n, int64_t D, int64_t ld,
                                   float* exp_avg, float* exp_avg_sq, int64_t step0, double lr, double beta1,
                                   double beta2, double eps, double weight_decay, int decoupled_weight_decay,
                                   float* out_last, bde_stream_t stream) {
    if (n < 1 || n > BDE_MAX_PARTICLES || step0 < 0) return BDE_ERR_INVALID_ARG;
    if (n > kOptMaxParticles) return BDE_ERR_UNSUPPORTED_N;
    const BaseOptParams o = adam_params(n, exp_avg, exp_avg_sq, step0, lr, beta1, beta2, eps, weight_decay,
                                        decoupled_weight_decay, out_last);
    return apply_opt_impl(X, G, K, A, n, D, ld, ld, o, static_cast<cudaStream_t>(stream));
}

static NextDistParams next_params(double* dist_next, int fuse_bandwidth, double l2_reg, double kernel_grad_scale,
                                  double dataset_size, double h_override, float* K_next, float* A_next, double* info,
                                  int32_t* sel, void* workspace) {
    NextDistParams nd;
    nd.dist = dist_next;
    nd.ws = workspace;
    nd.fuse_bandwidth = fuse_bandwidth ? 1 : 0;
    nd.bp = BandwidthParams{l2_reg, kernel_grad_scale, dataset_size, h_override, K_next, A_next, info, sel};
    return nd;
}

extern "C" int bde_svgd_train_step_sgd(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                                       int64_t ld, float* momentum_buf, int buf_initialized, double lr, double momentum,
                                       double dampening, double weight_decay, int nesterov, float* out_last,
                                       double* dist_next, int fuse_bandwidth, double l2_reg, double kernel_grad_scale,
                                       double dataset_size, double h_override, float* K_next, float* A_next,
                                       double* info, int32_t* sel, void* workspace, size_t workspace_bytes,
                                       bde_stream_t stream) {
    const BaseOptParams o = sgd_params(momentum_buf, buf_initialized, lr, momentum, dampening, weight_decay, nesterov, out_last);
    const NextDistParams nd = next_params(dist_next, fuse_bandwidth, l2_reg, kernel_grad_scale, dataset_size, h_override,
                                          K_next, A_next, info, sel, workspace);
    return apply_opt_impl(X, G, K, A, n, D, ld, ld, o, static_cast<cudaStream_t>(stream), &nd, workspace_bytes);
}

extern "C" int bde_svgd_train_step_adam(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                                        int64_t ld, float* exp_avg, float* exp_avg_sq, int64_t step0, double lr,
                                        double beta1, double beta2, double eps, double weight_decay,
                                        int decoupled_weight_decay, float* out_last, double* dist_next,
                                        int fuse_bandwidth, double l2_reg, double kernel_grad_scale, double dataset_size,
                                        double h_override, float* K_next, float* A_next, double* info, int32_t* sel,
                                        void* workspace, size_t workspace_bytes, bde_stream_t stream) {
    if (n < 1 || n > BDE_MAX_PARTICLES || step0 < 0) return BDE_ERR_INVALID_ARG;
    if (n > kOptMaxParticles) return BDE_ERR_UNSUPPORTED_N;
    const BaseOptParams o = adam_params(n, exp_avg, exp_avg_sq, step0, lr, beta1, beta2, eps, weight_decay,
                                        decoupled_weight_decay, out_last);
    const NextDistParams nd = next_params(dist_next, fuse_bandwidth, l2_reg, kernel_grad_scale, dataset_size, h_override,
                                          K_next, A_next, info, sel, workspace);
    return apply_opt_impl(X, G, K, A, n, D, ld, ld, o, static_cast<cudaStream_t>(stream), &nd, workspace_bytes);
}
