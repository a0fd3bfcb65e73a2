/*
 * bde_b200.h — C-ABI of the B200-native posterior-update kernels.
 *
 * This is the drop-in boundary of the hot path inside the reference's
 * BayesianOptimizer.step (Feuermagier/Beyond_Deep_Ensembles, src/algos).  The
 * reference has no FFI for this path (it is inline eager PyTorch), so each entry
 * point below cites the reference lines whose arithmetic it replaces.  The Python
 * host classes in beyond_deep_ensembles_b200/ (same names and constructor
 * signatures as the reference's optimizers) call these through ctypes.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - functions never allocate, never synchronise and never throw; the caller
 *     passes workspaces (sizes from the *_workspace_bytes queries, zero-filled
 *     once when allocated — kernels leave them zeroed again);
 *   - return value: 0 = ok, >0 = a cudaError_t, <0 = one of BDE_ERR_*;
 *   - matrices are row-major fp32, `ld` = row stride in elements;
 *   - Philox4x32-10 noise is keyed by (seed, stream_id) and counted by the GLOBAL
 *     element index (`elem0` + local index) so results do not depend on how the
 *     parameter dimension is sharded over GPUs.  `elem0` must be a multiple of 4.
 *     When an `eps` pointer is non-NULL the injected noise is used instead.
 */
#ifndef BDE_B200_H
#define BDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BDE_OK 0
#define BDE_ERR_INVALID_ARG (-1)
#define BDE_ERR_ALIGNMENT (-2)
#define BDE_ERR_WORKSPACE (-3)
#define BDE_ERR_UNSUPPORTED_N (-4)

/*
 * Particle counts: every SVGD entry accepts 1 <= n <= BDE_MAX_PARTICLES (BDE_ERR_INVALID_ARG otherwise).
 *   n <= 32: every SVGD entry, any alignment.
 *   33 <= n <= 64: bde_svgd_workspace_bytes, bde_svgd_pairdist, bde_svgd_bandwidth, bde_svgd_pairdist_bandwidth,
 *     bde_svgd_apply and bde_svgd_step only, on 16-byte aligned base pointers with ld % 4 == 0 (BDE_ERR_ALIGNMENT
 *     otherwise); the fused base-optimizer entries (bde_svgd_apply_sgd / _adam, bde_svgd_train_step_*) and the
 *     host-buffer entries (bde_svgd_host_*, bde_svgd_step_host) return BDE_ERR_UNSUPPORTED_N, and so does K1 on a
 *     workspace attached to a peer set (bde_peer_attach; the exchange carries at most 32*31/2 sums): D-sharded jobs
 *     all-reduce `dist` between bde_svgd_pairdist and bde_svgd_bandwidth instead.
 */
#define BDE_MAX_PARTICLES 64

typedef void* bde_stream_t;

/* ---- library ------------------------------------------------------------- */
int bde_version(void);
const char* bde_error_string(int code);
/*
 * Launch-geometry override for tuning sweeps: key is "pairdist_ctas_per_sm",
 * "apply_ctas_per_sm", "ew_ctas_per_sm", or "pairdist_variant" / "apply_variant" /
 * "ew_variant" (1 = direct-LDG kernels, 2 = TMA-staged kernels), "apply_tile_sets" (the
 * alternative consumer geometry of the staged K2: 3 or 4 tile sets at n > 12, 1 set x 512 or
 * 3 sets x 256 columns at n <= 12), "swag_batch" (draws per pass of bde_swag_sample_batch:
 * 2, 4, 8 or 16; 1 = the general kernels of both batched samplers instead of the fast ones),
 * "batch_prefetch" (fast batched samplers: L2 prefetch distance in grid-stride iterations,
 * 9 = off) or "batch_splits" (partner CTAs per pass of the fast batched SWAG sampler: 2, 4);
 * value 0 restores the automatic choice.
 */
int bde_tune(const char* key, int value);
/* number of SMs of the current device (grid sizing is done inside the library) */
int bde_device_sm_count(int* sm_count);

/* ---- SVGD (reference: src/algos/svgd.py) ---------------------------------- */

/* Workspace for bde_svgd_pairdist / bde_kl_* reductions (bytes). */
int bde_svgd_workspace_bytes(int n, size_t* bytes);
/* Workspace of the scalar value reductions (bde_kl_*, bde_l2_*, bde_prior_terms_*). */
int bde_value_workspace_bytes(size_t* bytes);

/*
 * K1: partial squared pairwise distances of the n particle rows over the local D
 * columns: dist[i*n+j] (+)= sum_c (X[i,c]-X[j,c])^2, symmetric, zero diagonal, fp64.
 * Replaces torch.cdist(particles, particles, p=2)**2, svgd.py:15 (direct
 * differences, fp32 per-thread partials combined in fp64, deterministic order).
 * accumulate != 0 adds into dist (used when the columns arrive in chunks).
 * Under D-sharding the caller sum-all-reduces `dist` (n*n doubles) across ranks.
 */
int bde_svgd_pairdist(const float* X, int n, int64_t D, int64_t ld, double* dist,
                      int accumulate, void* workspace, size_t workspace_bytes,
                      bde_stream_t stream);

/*
 * K1b: median-heuristic bandwidth, RBF kernel matrix and the fused coefficient
 * matrix.  Replaces svgd.py:17-21 (quantile over all n*n entries with linear
 * interpolation, h = sqrt(0.5*median/ln(n+1)) + 1e-8, K = exp(-d/(2h^2))) and folds
 * svgd.py:23,31,86,89 into A = (l2_reg/2 + c) K - c diag(rowsum K),
 * c = kernel_grad_scale / (dataset_size h^2), so that the new gradient of
 * particle i is  sum_j K_ij g_j + sum_j A_ij x_j.
 * h_override > 0 replaces the median heuristic (svgd.py:19-20).
 * Outputs: K, A fp32 [n*n]; info fp64 [4] = {h, median, d_lo, d_hi};
 * sel int32 [2] = flat indices i*n+j (i<=j) of the two order statistics used.
 */
int bde_svgd_bandwidth(const double* dist, int n, double l2_reg, double kernel_grad_scale,
                       double dataset_size, double h_override, float* K, float* A,
                       double* info, int32_t* sel, bde_stream_t stream);

/*
 * K2: out[i,:] = sum_j K[i,j] G[j,:] + sum_j A[i,j] X[j,:]  (one pass, FP32 FFMA2).
 * Replaces svgd.py:86-97 (prior term, K@(-G), grad_kernel, scatter of -phi).
 * `out` must not overlap X or G.
 */
int bde_svgd_apply(const float* X, const float* G, float* out, const float* K, const float* A,
                   int n, int64_t D, int64_t ld, bde_stream_t stream);

/*
 * K1 with K1b fused into its tail (the last CTA to finish runs the n*n epilogue): the
 * single-GPU form, one launch instead of two.  Arguments as in the two calls above.
 */
int bde_svgd_pairdist_bandwidth(const float* X, int n, int64_t D, int64_t ld, double l2_reg,
                                double kernel_grad_scale, double dataset_size, double h_override,
                                double* dist, float* K, float* A, double* info, int32_t* sel,
                                void* workspace, size_t workspace_bytes, bde_stream_t stream);

/*
 * Single-GPU convenience: K1(+K1b) + K2 on one stream (no collective in between).
 */
/* Declares that the NEXT bde_svgd_apply / bde_svgd_apply_sgd / _adam / bde_svgd_train_step_* launch on `stream` directly
 * follows a bde_svgd_pairdist_bandwidth / bde_svgd_bandwidth launch of this library on the same stream, with NOTHING
 * else enqueued in between.  The staged apply kernel is then launched as a programmatic dependent of K1: it becomes
 * resident and fills its shared-memory ring with X / G tiles while K1 is still in its tail (grid reduction, cross-rank
 * exchange, K1b), and waits for K1's completion before it reads K / A or writes anything.  The hint is consumed by the
 * next apply launch of the calling thread whatever kernel that launch selects.  bde_svgd_step does this itself. */
int bde_svgd_chain_next(bde_stream_t stream);
int bde_svgd_step(const float* X, const float* G, float* out, int n, int64_t D, int64_t ld,
                  double l2_reg, double kernel_grad_scale, double dataset_size,
                  double h_override, double* dist, float* K, float* A, double* info,
                  int32_t* sel, void* workspace, size_t workspace_bytes, bde_stream_t stream);

/*
 * K2 fused with the base optimizer's update (SURVEY.md §8 f1).  Replaces svgd.py:92-103: the new
 * gradient of particle i (row i of K G + A X) is handed to ONE torch.optim optimizer whose state is
 * shared by all particles and which steps once per particle, in particle order 0..n-1.  Here the
 * n sequential steps run in registers per column: X is updated IN PLACE, the n*D gradient matrix
 * never reaches HBM.  out_last (nullable, [D]) receives the new gradient of particle n-1 — what the
 * reference leaves in param.grad.  X and G must not overlap.
 *
 * bde_svgd_apply_sgd  = torch.optim.SGD (weight_decay, momentum, dampening, nesterov; maximize=False):
 *   momentum_buf [D] is the shared momentum_buffer (NULL iff momentum == 0); buf_initialized == 0 on the
 *   optimizer's very first step (buffer := clone of particle 0's gradient, torch/optim/sgd.py).
 * bde_svgd_apply_adam = torch.optim.Adam / AdamW (amsgrad=False, maximize=False): exp_avg, exp_avg_sq [D]
 *   shared; step0 = the optimizer's step count BEFORE this call (particle i takes step step0+i+1);
 *   decoupled_weight_decay != 0 selects AdamW's param *= 1 - lr*wd.
 */
int bde_svgd_apply_sgd(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                       int64_t ld, float* momentum_buf, int buf_initialized, double lr,
                       double momentum, double dampening, double weight_decay, int nesterov,
                       float* out_last, bde_stream_t stream);
int bde_svgd_apply_adam(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                        int64_t ld, float* exp_avg, float* exp_avg_sq, int64_t step0, double lr,
                        double beta1, double beta2, double eps, double weight_decay,
                        int decoupled_weight_decay, float* out_last, bde_stream_t stream);

/*
 * Training-step form of the two entries above: the SAME pass also accumulates the squared pair
 * distances of the UPDATED particles — the K1 of the next SVGD step (svgd.py:15 on the next call of
 * step()), so that a training loop reads X once per step instead of twice.  dist_next [n*n] fp64 is
 * written (symmetric, zero diagonal; under D-sharding it is this rank's partial sum, to be all-reduced).
 * fuse_bandwidth != 0 additionally runs K1b on dist_next in the tail of the same launch and writes the
 * NEXT step's K_next / A_next / info / sel (K_next / A_next may alias K / A: every CTA has consumed the
 * current coefficients before the last CTA writes the new ones).  workspace as for bde_svgd_pairdist.
 * One launch for n <= 10 on 16-byte-aligned rows; any other shape runs the fused update followed by K1.
 */
int bde_svgd_train_step_sgd(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                            int64_t ld, float* momentum_buf, int buf_initialized, double lr,
                            double momentum, double dampening, double weight_decay, int nesterov,
                            float* out_last, double* dist_next, int fuse_bandwidth, double l2_reg,
                            double kernel_grad_scale, double dataset_size, double h_override,
                            float* K_next, float* A_next, double* info, int32_t* sel, void* workspace,
                            size_t workspace_bytes, bde_stream_t stream);
int bde_svgd_train_step_adam(float* X, const float* G, const float* K, const float* A, int n, int64_t D,
                             int64_t ld, float* exp_avg, float* exp_avg_sq, int64_t step0, double lr,
                             double beta1, double beta2, double eps, double weight_decay,
                             int decoupled_weight_decay, float* out_last, double* dist_next,
                             int fuse_bandwidth, double l2_reg, double kernel_grad_scale,
                             double dataset_size, double h_override, float* K_next, float* A_next,
                             double* info, int32_t* sel, void* workspace, size_t workspace_bytes,
                             bde_stream_t stream);

/*
 * Host-buffer entries (the end-to-end path): X_host/G_host/out_host are HOST arrays
 * [n, D] with row stride ld_host (pinned memory gives full PCIe bandwidth).  The
 * columns are streamed through the device in `chunk_cols`-wide pieces (a multiple of 4)
 * on the library's own copy/compute streams so that PCIe traffic in both directions
 * overlaps the kernels.  Caller-provided device staging: dX [n, ld_dev] with
 * ld_dev = D rounded up to 4 (X stays resident between the two phases), dG and dOut
 * [2][n, chunk_cols].  Both calls block until their results are complete.
 *   bde_svgd_host_pairdist: per chunk H2D X -> K1(accumulate); dist = local partial sums.
 *   (D-sharded jobs all-reduce `dist` here.)
 *   bde_svgd_host_apply:    K1b, then per chunk H2D G -> K2 -> D2H out.
 *   bde_svgd_step_host:     both, for a single rank.  info_host[4], sel_host[2] may be NULL.
 */
int bde_svgd_host_pairdist(const float* X_host, int n, int64_t D, int64_t ld_host, int64_t chunk_cols,
                           float* dX, double* dist, void* workspace, size_t workspace_bytes);
int bde_svgd_host_apply(const float* G_host, float* out_host, int n, int64_t D, int64_t ld_host,
                        double l2_reg, double kernel_grad_scale, double dataset_size,
                        double h_override, int64_t chunk_cols, const float* dX, float* dG, float* dOut,
                        const double* dist, float* K, float* A, double* info, int32_t* sel,
                        double* info_host, int32_t* sel_host);
int bde_svgd_step_host(const float* X_host, const float* G_host, float* out_host, int n,
                       int64_t D, int64_t ld_host, double l2_reg, double kernel_grad_scale,
                       double dataset_size, double h_override, int64_t chunk_cols,
                       float* dX, float* dG, float* dOut, double* dist, float* K, float* A,
                       double* info, int32_t* sel, void* workspace, size_t workspace_bytes,
                       double* info_host, int32_t* sel_host);

/* ---- SWAG (reference: src/algos/swag.py) ---------------------------------- */

/*
 * K3: running moments + one deviation column, swag.py:98-104 with `updates` the
 * value AFTER the increment at swag.py:98:
 *   mean <- (updates*mean + theta)/(updates+1);  sq <- (updates*sq + theta^2)/(updates+1);
 *   dev_row <- theta - mean_new.
 * dev_row is the ring-buffer row that replaces the reference's roll(-1)+last-column
 * write (the buffer is [K, D] row-major on device instead of [D, K] on the host).
 */
int bde_swag_update(const float* theta, float* mean, float* sq, float* dev_row, int64_t D,
                    int64_t updates, bde_stream_t stream);

/*
 * K4: theta = mean + sum_k dev[(head+k)%K,:] * z[k]/sqrt(2(K-1))
 *             + sqrt(0.5*(relu(sq-mean^2)+1e-6)) * eps,
 * swag.py:112-114 + LowRankMultivariateNormal.rsample (draw order z then eps),
 * swag.py:57.  `head` = physical row of the OLDEST column (= updates % K).
 * eps_k: K device floats (the low-rank noise, identical on every rank) or NULL
 * (Philox counter = k on stream_id^0x5741); eps_d: D device floats or NULL (Philox).
 */
int bde_swag_sample(const float* mean, const float* sq, const float* dev, int K, int head,
                    int64_t D, int64_t ld, const float* eps_k, const float* eps_d,
                    uint64_t seed, uint64_t stream_id, int64_t elem0, float* theta,
                    bde_stream_t stream);

/*
 * K4 batched: S draws from the same posterior in one pass (SURVEY §8 f3; what
 * DeepEnsemble.predict, ensemble.py:37-43, asks for with `samples // members` consecutive
 * sample_parameters() calls).  theta: [S, ld_out]; draw s equals bde_swag_sample with
 * stream_id + s bit for bit.  eps_k: [S, K] or NULL; eps_d: [S, ld_eps] or NULL.
 * Reads mean, sq and the K deviation rows once per 16 draws.
 */
int bde_swag_sample_batch(const float* mean, const float* sq, const float* dev, int K, int head,
                          int64_t D, int64_t ld, int S, const float* eps_k, const float* eps_d,
                          int64_t ld_eps, uint64_t seed, uint64_t stream_id, int64_t elem0,
                          float* theta, int64_t ld_out, bde_stream_t stream);

/* ---- iVON (reference: src/algos/ivorn.py) --------------------------------- */

/*
 * K5: delta = eps / sqrt(N_eff*max(prec,1e-4)) (0 if deterministic); theta = mean+delta;
 * delta_sum = first ? delta : delta_sum + delta.   ivorn.py:102-115.
 */
int bde_ivon_sample(const float* mean, const float* prec, float* delta_sum, float* theta,
                    int64_t D, double n_eff, int first, int deterministic, const float* eps,
                    uint64_t seed, uint64_t stream_id, int64_t elem0, bde_stream_t stream);

/*
 * K5 batched: S consecutive draws in one pass (SURVEY §8 f3, DeepEnsemble.predict).  theta: [S, ld_out];
 * draw s equals bde_ivon_sample with stream_id + s*stream_stride bit for bit (stream_stride = number of
 * parameter groups, which take their stream ids round-robin); delta_sum ends as after S single calls.
 * eps: [S, ld_eps] or NULL.
 */
int bde_ivon_sample_batch(const float* mean, const float* prec, float* delta_sum, float* theta,
                          int64_t ld_out, int64_t D, int S, double n_eff, int first, int deterministic,
                          const float* eps, int64_t ld_eps, uint64_t seed, uint64_t stream_id,
                          uint64_t stream_stride, int64_t elem0, bde_stream_t stream);

/* K6: acc = first ? grad : acc + grad.   ivorn.py:120-127. */
int bde_ivon_accumulate(float* acc, const float* grad, int64_t D, int first, bde_stream_t stream);

/*
 * K7: the update block ivorn.py:79-89 for one parameter group.  `step` is the value
 * after the increment at ivorn.py:68.  mean uses the OLD precision.
 */
int bde_ivon_update(const float* acc_grad, const float* delta_sum, float* mean, float* momentum,
                    float* prec, int64_t D, int mc_samples, int64_t step, double lr, double beta1,
                    double beta2, double prior_prec, double n_eff, double tempering,
                    double damping, bde_stream_t stream);

/* ---- BBB / Rank-1 (reference: src/algos/bbb.py, util.py:151-186) ----------- */

/* K8 fwd: w = mu + eps * softplus(rho).   util.py:170-171,181-183. */
int bde_gauss_sample_fwd(const float* mu, const float* rho, float* w, int64_t P, const float* eps,
                         uint64_t seed, uint64_t stream_id, int64_t elem0, bde_stream_t stream);

/* K8 bwd: grad_rho = grad_w * eps * exp(rho)/(exp(rho)+1) (grad_mu aliases grad_w). */
int bde_gauss_sample_bwd(const float* grad_w, const float* rho, float* grad_rho, int64_t P,
                         const float* eps, uint64_t seed, uint64_t stream_id, int64_t elem0,
                         bde_stream_t stream);

/*
 * K9: Gaussian-prior KL of N(mu, softplus(rho)^2) against N(prior_mu, prior_sigma^2),
 * bbb.py:18-21 via util.py:173-174, summed in fp64 into *value (device double, may be
 * NULL), and its analytic gradient times grad_scale (host) times *grad_scale_dev
 * (device float, may be NULL) written (accumulate=0) or added (accumulate=1) to
 * grad_mu / grad_rho (both may be NULL for value only).
 */
int bde_kl_gauss_value_and_grad(const float* mu, const float* rho, int64_t P, double prior_mu,
                                double prior_sigma, double* value, float* grad_mu,
                                float* grad_rho, double grad_scale, const float* grad_scale_dev,
                                int accumulate, void* workspace, size_t workspace_bytes,
                                bde_stream_t stream);

/*
 * K9b: scale-mixture prior, bbb.py:23-37: value = -sum logaddexp(ln pi + clamp(lnN(mu;0,s1),-23,0),
 * ln(1-pi) + clamp(lnN(mu;0,s2),-23,0)); gradient w.r.t. mu only (rho does not enter).
 */
int bde_kl_mixture_value_and_grad(const float* mu, int64_t P, double pi, double sigma1,
                                  double sigma2, double* value, float* grad_mu,
                                  double grad_scale, const float* grad_scale_dev, int accumulate,
                                  void* workspace, size_t workspace_bytes, bde_stream_t stream);

/*
 * K10: L2 term of the deterministic parameters, bbb.py:75-76:
 * value = l2_scale/2 * sum theta^2 (fp64), grad (+)= l2_scale * theta * scale.
 */
int bde_l2_value_and_grad(const float* theta, int64_t D, double l2_scale, double* value,
                          float* grad, double grad_scale, const float* grad_scale_dev,
                          int accumulate, void* workspace, size_t workspace_bytes,
                          bde_stream_t stream);

/*
 * K9 + K10 over a LIST of tensors in one launch: the whole prior term of BBBOptimizer.step,
 * bbb.py:69-76 — sum over the Gaussian parameters of their KL plus sum over the deterministic
 * parameters of l2_scale/2 * ||theta||^2 — and its gradient.  All *_host arguments are HOST arrays of
 * `count` entries (the table travels in the kernel parameters, like bde_multi_tensor_copy):
 *   kinds_host[i]   0 = Gaussian parameter under the Gaussian prior N(prior_p0, prior_p1^2):
 *                       a = mu, b = rho, gradients to grad_a / grad_b;
 *                   1 = Gaussian parameter under the scale-mixture prior (pi = prior_p0,
 *                       sigma1 = prior_p1, sigma2 = prior_p2): a = mu, gradient to grad_a only;
 *                   2 = deterministic tensor: a = theta, l2_scales_host[i], gradient to grad_a.
 *   a_host/b_host/grad_a_host/grad_b_host   device pointers as integers (grad_a_host == NULL: value only;
 *                   a zero entry: no gradient for that tensor); sizes_host: element counts.
 * Kinds 0 and 1 cannot be mixed in one call (one prior per call).  *value (device double, may be NULL) is
 * overwritten with the fp64 sum; gradients are multiplied by grad_scale * *grad_scale_dev and written
 * (accumulate_grad == 0) or added.  Per-element arithmetic is that of the single-tensor entries above.
 */
int bde_prior_terms_value_and_grad(int count, const int32_t* kinds_host, const uint64_t* a_host,
                                   const uint64_t* b_host, const uint64_t* grad_a_host,
                                   const uint64_t* grad_b_host, const int64_t* sizes_host,
                                   const double* l2_scales_host, double prior_p0, double prior_p1,
                                   double prior_p2, double* value, double grad_scale,
                                   const float* grad_scale_dev, int accumulate_grad, void* workspace,
                                   size_t workspace_bytes, bde_stream_t stream);

/* ---- D-sharded jobs: in-kernel exchange over NVLink (SURVEY.md 8e) --------- */

/*
 * Every GPU holds a column slice [n, D/R] of the particles; the only cross-rank quantity of an
 * SVGD step is the sum of the n*n partial pair distances (svgd.py:15 over all D columns).  With a
 * peer set attached to the reduction workspace, the last CTA of bde_svgd_pairdist /
 * bde_svgd_pairdist_bandwidth / bde_svgd_step / bde_svgd_train_step_* finishes that sum ACROSS
 * RANKS inside the same launch: P2P stores of its partial sums into every peer's exchange buffer,
 * a release/acquire epoch flag per rank, and a rank-ordered fp64 sum — the result is bit-identical
 * on every rank, and a D-sharded step needs no separate all-reduce launch (the NCCL all-reduce of
 * `dist` remains the portable form).  Every rank must issue the same sequence of launches on the
 * attached workspaces of one peer set, from one stream.  A peer that never arrives poisons the
 * sums with NaN after the attach-time timeout instead of hanging the GPU (bde_peer_status and the host status word
 * report it).
 *
 * Protocol (the caller owns everything; the library only remembers which workspaces are attached):
 *   1. each rank: bde_peer_alloc -> device buffer + a BDE_PEER_HANDLE_BYTES CUDA-IPC handle;
 *   2. exchange the handles between the ranks (any host transport, e.g. torch.distributed);
 *   3. each rank: bde_peer_open on every OTHER rank's handle -> mapped device pointers;
 *   4. bde_peer_attach(workspace, ..., world, rank, bufs_host) with bufs_host[r] = rank r's buffer
 *      as seen from this process (own buffer for r == rank);
 *   5. teardown after a barrier: bde_peer_detach, bde_peer_close (mapped), bde_peer_free (own).
 * bde_peer_alloc / open / close / free / status are setup calls: they allocate and synchronise.
 */
#define BDE_PEER_HANDLE_BYTES 64
#define BDE_PEER_MAX_RANKS 16
int bde_peer_buffer_bytes(size_t* bytes);
int bde_peer_alloc(void** buf, unsigned char* ipc_handle_host);
int bde_peer_open(const unsigned char* ipc_handle_host, void** mapped);
int bde_peer_close(void* mapped);
int bde_peer_free(void* buf);
/* timeout_seconds: how long the last CTA waits for its peers (<= 0: 120 s).  host_status (nullable): one pinned,
 * device-addressable host word that receives the count of abandoned exchanges, so the caller can notice a failure
 * without synchronising.  After a timeout the workspace is marked failed: sums are poisoned with NaN, K1b is not run
 * (K / A keep their previous values) and every later exchange returns at once, until bde_peer_attach is called again. */
int bde_peer_attach(void* workspace, size_t workspace_bytes, int world, int rank, const uint64_t* bufs_host,
                    double timeout_seconds, uint64_t* host_status, bde_stream_t stream);
int bde_peer_detach(void* workspace, size_t workspace_bytes, bde_stream_t stream);
/* exchanges completed / abandoned on this rank's buffer (synchronous device read) */
int bde_peer_status(const void* buf, uint64_t* epoch_host, uint64_t* timeouts_host);
/* How long this rank's exchanges waited for their slowest peer (rank skew): number of exchanges, summed and longest
 * wait in ns since the last reset.  Synchronises; reset != 0 clears the counters. */
int bde_peer_wait_stats(void* buf, uint64_t* exchanges_host, uint64_t* wait_ns_sum_host, uint64_t* wait_ns_max_host,
                        int reset);

/* ---- utilities ------------------------------------------------------------ */

/* out = standard normals from the library's Philox stream (for tests/diagnostics). */
int bde_philox_normal(float* out, int64_t count, uint64_t seed, uint64_t stream_id, int64_t elem0,
                      bde_stream_t stream);

/*
 * Multi-tensor gather/scatter between a list of scattered tensors and a flat arena
 * row (replaces parameters_to_vector / the cat+stack at svgd.py:83-84 and the
 * slice+clone scatter at svgd.py:92-97).  ptrs_host / offsets_host / sizes_host are HOST
 * arrays of `count` entries: device pointers of the tensors, their element offsets into
 * `flat` (ascending, non-overlapping) and their element counts; the table is passed to
 * the kernel by value.  mode 0: flat <- tensors, 1: flat <- flat + tensors,
 * 2: tensors <- flat.
 */
int bde_multi_tensor_copy(float* flat, const uint64_t* ptrs_host, const int64_t* offsets_host,
                          const int64_t* sizes_host, int count, int mode, bde_stream_t stream);

/*
 * The gather modes (0, 1) of bde_multi_tensor_copy fused with GradScaler.unscale_ (algo.py:65-73, i.e. torch's
 * _amp_foreach_non_finite_check_and_unscale_): flat (+)= tensor * *inv_scale, and *found_inf is raised to 1.0f if
 * any source value is not finite.  inv_scale / found_inf are DEVICE scalars (no host sync); the source tensors
 * are left untouched (still scaled).  SURVEY §8 f2.
 */
int bde_multi_tensor_unscale_copy(float* flat, const uint64_t* ptrs_host, const int64_t* offsets_host,
                                  const int64_t* sizes_host, int count, int mode, const float* inv_scale,
                                  float* found_inf, bde_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------
 * f4 (SURVEY.md §8f): BBBLinear's local-reparameterisation forward, src/algos/bbb_layers.py:61-88 (CUDA branch)
 *   mean = b_mu + x W_mu^T;  var = clamp(softplus(b_rho)^2, 1e-4) + clamp(x^2, 1e-4) clamp(softplus(W_rho)^2, 1e-4)^T
 *   out  = (mean + sqrt(var) * eps) / mc_sample
 * as one tcgen05 kernel (3xTF32 tensor-core products with fp32-level accuracy, TMEM accumulators, tensor-map TMA
 * loads, deterministic split-K over in_features / 32).  x: [batch, in] row-major with row stride ldx; W_mu, W_rho:
 * [out, in] contiguous; b_mu / b_rho: [out] or both null; eps: [batch, out] injected noise or null (Philox keyed by
 * (seed, stream_id), counter = element index / 4); act_std / eps_out (nullable) receive sqrt(var) and the noise used,
 * for the backward pass.  in_features % 4 == 0 and 16-byte aligned x / W (BDE_ERR_ALIGNMENT otherwise — callers then
 * keep the reference's own forward).  workspace: bde_bbb_linear_workspace_bytes, zero-filled once by the caller. */
int bde_bbb_linear_workspace_bytes(int batch, int in_features, int out_features, size_t* bytes);
int bde_bbb_linear_fwd(const float* x, int64_t ldx, int batch, int in_features, int out_features, const float* w_mu,
                       const float* w_rho, const float* b_mu, const float* b_rho, const float* eps, uint64_t seed,
                       uint64_t stream_id, double mc_sample, float* out, float* act_std, float* eps_out, void* workspace,
                       size_t workspace_bytes, bde_stream_t stream);

/* f4, second half: the Rank-1 VI linear layer src/algos/rank1.py:50-64 —
 *   s = s_mu + eps_s * softplus(s_rho) [in],  r = r_mu + eps_r * softplus(r_rho) [out],  out = linear(x * s, W) * r + bias
 * — with the prologue / epilogue scaling fused around the same tcgen05 product as bde_bbb_linear_fwd (exact 3-way tf32
 * split, TMEM accumulator, deterministic split-K).  W: [out, in] contiguous; bias: [out] (the component's row) or null;
 * eps_s / eps_r: injected noise or null (Philox streams sid_s / sid_r, counter = element index / 4, i.e. the values
 * bde_gauss_sample_fwd draws for the same stream ids).  lin receives linear(x * s, W); s_out / r_out / eps_s_out /
 * eps_r_out the sampled vectors and their noise (backward pass).  Workspace: bde_bbb_linear_workspace_bytes. */
int bde_rank1_linear_fwd(const float* x, int64_t ldx, int batch, int in_features, int out_features, const float* W,
                         const float* s_mu, const float* s_rho, const float* r_mu, const float* r_rho, const float* bias,
                         const float* eps_s, const float* eps_r, uint64_t seed, uint64_t sid_s, uint64_t sid_r, float* out,
                         float* lin, float* s_out, float* r_out, float* eps_s_out, float* eps_r_out, void* workspace,
                         size_t workspace_bytes, bde_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* BDE_B200_H */
