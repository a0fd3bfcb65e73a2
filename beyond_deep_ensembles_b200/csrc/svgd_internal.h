// svgd_internal.h — internal (non-ABI) entry points shared between svgd.cu and host_api.cu.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

namespace bde {

struct BandwidthParams {
    double l2_reg, kernel_grad_scale, dataset_size, h_override;
    float* K;
    float* A;
    double* info;
    int32_t* sel;
};

// f1: the base optimizer's update fused into K2 (svgd.py:92-103: ONE optimizer whose state is shared by all
// particles and stepped once per particle, in particle order).  kind 0 = plain K2.
constexpr int kOptNone = 0, kOptSgd = 1, kOptAdam = 2;
constexpr int kOptMaxParticles = 32;
struct BaseOptParams {
    int kind = kOptNone;
    // torch.optim.SGD
    float lr = 0.f, momentum = 0.f, one_minus_dampening = 1.f, weight_decay = 0.f;
    int nesterov = 0;
    int buf_initialized = 0;     // 0: the very first optimizer step ever (momentum_buffer = clone(grad))
    // torch.optim.Adam / AdamW
    float beta1 = 0.f, one_minus_beta1 = 0.f, beta2 = 0.f, one_minus_beta2 = 0.f, eps = 0.f;
    int decoupled_wd = 0;
    float decay_factor = 1.f;                    // AdamW: 1 - lr*weight_decay
    float step_size[kOptMaxParticles] = {};      // lr / (1 - beta1^t) for t = step0 + i + 1
    float inv_bc2_sqrt[kOptMaxParticles] = {};   // 1 / sqrt(1 - beta2^t)
    float* state0 = nullptr;     // momentum_buffer | exp_avg      [D]
    float* state1 = nullptr;     // exp_avg_sq                      [D]
    float* out_last = nullptr;   // optional: new gradient of the LAST particle (what svgd.py:94 leaves in param.grad)
};

// Training-step form of the fused kernel: the same pass also accumulates the pair distances of the UPDATED
// particles (the K1 of the next SVGD step), reduces them over the grid like K1 does and, with fuse_bandwidth,
// lets the last CTA run K1b for the next step (bp.K / bp.A may alias the K / A this launch reads).
struct NextDistParams {
    double* dist = nullptr;   // [n*n], written (not accumulated)
    void* ws = nullptr;       // grid-reduction workspace (bde_svgd_workspace_bytes)
    int fuse_bandwidth = 0;
    BandwidthParams bp{};
};
constexpr int kNextDistMaxParticles = 10;  // all pairs of a column quad in one thread's registers

// Particle counts of the generic runtime-n kernels, the fused base-optimizer forms, the host-staged entries and
// the in-kernel peer exchange.  n in (kGenericMaxParticles, BDE_MAX_PARTICLES] runs the particle-tiled kernels of
// svgd_many.cu (K1, K1b, K2 only; 16-byte aligned rows).
constexpr int kGenericMaxParticles = 32;
constexpr int kManyMaxCtas = 256;   // grid bound of the particle-tiled K1 (one CTA per SM): sizes its workspace

// peer.cu: is `ws` attached (bde_peer_attach) to a peer set of more than one rank?
bool peer_attached(const void* ws);

// svgd_many.cu: n in 33..64, X (and G, out) 16-byte aligned with ld % 4 == 0 (checked by the callers)
int pairdist_many(const float* X, int n, int64_t D, int64_t ld, double* dist, int accumulate, void* ws, int fuse,
                  const BandwidthParams& bp, cudaStream_t st);
int bandwidth_many(const double* dist, int n, const BandwidthParams& bp, cudaStream_t st);
int apply_many(const float* X, const float* G, float* out, const float* K, const float* A, int n, int64_t D,
               int64_t ldx, int64_t ldg, int64_t ldo, cudaStream_t st);

int pairdist_impl(const float* X, int n, int64_t D, int64_t ld, double* dist, int accumulate, void* ws,
                  size_t ws_bytes, int fuse, const BandwidthParams& bp, cudaStream_t st);
int apply_impl(const float* X, const float* G, float* out, const float* K, const float* A, int n, int64_t D,
               int64_t ldx, int64_t ldg, int64_t ldo, cudaStream_t st);
// fused form: X is updated in place, `out` is not written (o.out_last receives row n-1 if non-null)
int apply_opt_impl(float* X, const float* G, const float* K, const float* A, int n, int64_t D, int64_t ldx,
                   int64_t ldg, const BaseOptParams& o, cudaStream_t st, const NextDistParams* next = nullptr,
                   size_t ws_bytes = 0);

}  // namespace bde
