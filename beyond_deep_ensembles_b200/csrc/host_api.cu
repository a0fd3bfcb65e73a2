// host_api.cu — host-buffer entry of the SVGD step (the end-to-end path).
// Streams the columns of host-resident X / G through the device in chunks on separate
// copy and compute streams so that PCIe transfers in both directions overlap the kernels:
//   phase 1: H2D X chunk -> K1 (accumulating partial distances)            ... -> K1b
//   phase 2: H2D G chunk -> K2 on (resident X chunk, G chunk) -> D2H out chunk
#include "common.cuh"
#include "svgd_internal.h"

namespace bde {

struct HostPipe {
    bool ready = false;
    cudaStream_t h2d = nullptr, comp = nullptr, d2h = nullptr;
    cudaEvent_t ev_x = nullptr, ev_g[2] = {nullptr, nullptr}, ev_k2[2] = {nullptr, nullptr},
                ev_out[2] = {nullptr, nullptr};
};

static int get_pipe(HostPipe** out) {
    static HostPipe pipes[64];
    int dev = 0;
    BDE_RETURN_IF_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return BDE_ERR_INVALID_ARG;
    HostPipe& p = pipes[dev];
    if (!p.ready) {
        BDE_RETURN_IF_CUDA(cudaStreamCreateWithFlags(&p.h2d, cudaStreamNonBlocking));
        BDE_RETURN_IF_CUDA(cudaStreamCreateWithFlags(&p.comp, cudaStreamNonBlocking));
        BDE_RETURN_IF_CUDA(cudaStreamCreateWithFlags(&p.d2h, cudaStreamNonBlocking));
        BDE_RETURN_IF_CUDA(cudaEventCreateWithFlags(&p.ev_x, cudaEventDisableTiming));
        for (int b = 0; b < 2; ++b) {
            BDE_RETURN_IF_CUDA(cudaEventCreateWithFlags(&p.ev_g[b], cudaEventDisableTiming));
            BDE_RETURN_IF_CUDA(cudaEventCreateWithFlags(&p.ev_k2[b], cudaEventDisableTiming));
            BDE_RETURN_IF_CUDA(cudaEventCreateWithFlags(&p.ev_out[b], cudaEventDisableTiming));
        }
        p.ready = true;
    }
    *out = &p;
    return BDE_OK;
}

}  // namespace bde

using namespace bde;

extern "C" int bde_svgd_host_pairdist(const float* X_host, int n, int64_t D, int64_t ld_host, int64_t chunk_cols,
                                      float* dX, double* dist, void* workspace, size_t workspace_bytes) {
    if (!X_host || !dX || !dist || n < 1 || n > BDE_MAX_PARTICLES || D < 1 || ld_host < D || chunk_cols < 4 ||
        (chunk_cols & 3))
        return BDE_ERR_INVALID_ARG;
    if (n > kGenericMaxParticles) return BDE_ERR_UNSUPPORTED_N;   // the host-staged path stops at 32 particles
    HostPipe* p = nullptr;
    int rc = get_pipe(&p);
    if (rc != BDE_OK) return rc;
    const int64_t ld_dev = (D + 3) & ~static_cast<int64_t>(3);
    const int64_t nchunks = (D + chunk_cols - 1) / chunk_cols;
    const size_t fsz = sizeof(float);
    for (int64_t c = 0; c < nchunks; ++c) {
        const int64_t col0 = c * chunk_cols;
        const int64_t w = (D - col0 < chunk_cols) ? D - col0 : chunk_cols;
        BDE_RETURN_IF_CUDA(cudaMemcpy2DAsync(dX + col0, ld_dev * fsz, X_host + col0, ld_host * fsz, w * fsz, n,
                                             cudaMemcpyHostToDevice, p->h2d));
        BDE_RETURN_IF_CUDA(cudaEventRecord(p->ev_x, p->h2d));
        BDE_RETURN_IF_CUDA(cudaStreamWaitEvent(p->comp, p->ev_x, 0));
        BandwidthParams none{};
        rc = pairdist_impl(dX + col0, n, w, ld_dev, dist, c > 0 ? 1 : 0, workspace, workspace_bytes, 0, none, p->comp);
        if (rc != BDE_OK) return rc;
    }
    BDE_RETURN_IF_CUDA(cudaStreamSynchronize(p->comp));
    return BDE_OK;
}

extern "C" int bde_svgd_host_apply(const float* G_host, float* out_host, int n, int64_t D, int64_t ld_host,
                                   double l2_reg, double kernel_grad_scale, double dataset_size, double h_override,
                                   int64_t chunk_cols, const float* dX, float* dG, float* dOut, const double* dist,
                                   float* K, float* A, double* info, int32_t* sel, double* info_host,
                                   int32_t* sel_host) {
    if (!G_host || !out_host || !dX || !dG || !dOut || !dist || !K || !A || n < 1 || n > BDE_MAX_PARTICLES || D < 1 ||
        ld_host < D || chunk_cols < 4 || (chunk_cols & 3) || !(dataset_size > 0.0))
        return BDE_ERR_INVALID_ARG;
    if (n > kGenericMaxParticles) return BDE_ERR_UNSUPPORTED_N;
    HostPipe* p = nullptr;
    int rc = get_pipe(&p);
    if (rc != BDE_OK) return rc;
    const int64_t ld_dev = (D + 3) & ~static_cast<int64_t>(3);
    const int64_t nchunks = (D + chunk_cols - 1) / chunk_cols;
    const size_t fsz = sizeof(float);
    rc = bde_svgd_bandwidth(dist, n, l2_reg, kernel_grad_scale, dataset_size, h_override, K, A, info, sel, p->comp);
    if (rc != BDE_OK) return rc;
    if (info_host && info)
        BDE_RETURN_IF_CUDA(cudaMemcpyAsync(info_host, info, 4 * sizeof(double), cudaMemcpyDeviceToHost, p->comp));
    if (sel_host && sel)
        BDE_RETURN_IF_CUDA(cudaMemcpyAsync(sel_host, sel, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, p->comp));
    for (int64_t c = 0; c < nchunks; ++c) {
        const int b = static_cast<int>(c & 1);
        const int64_t col0 = c * chunk_cols;
        const int64_t w = (D - col0 < chunk_cols) ? D - col0 : chunk_cols;
        float* g_buf = dG + static_cast<size_t>(b) * n * chunk_cols;
        float* o_buf = dOut + static_cast<size_t>(b) * n * chunk_cols;
        if (c >= 2) BDE_RETURN_IF_CUDA(cudaStreamWaitEvent(p->h2d, p->ev_k2[b], 0));  // g_buf consumed
        BDE_RETURN_IF_CUDA(cudaMemcpy2DAsync(g_buf, chunk_cols * fsz, G_host + col0, ld_host * fsz, w * fsz, n,
                                             cudaMemcpyHostToDevice, p->h2d));
        BDE_RETURN_IF_CUDA(cudaEventRecord(p->ev_g[b], p->h2d));
        BDE_RETURN_IF_CUDA(cudaStreamWaitEvent(p->comp, p->ev_g[b], 0));
        if (c >= 2) BDE_RETURN_IF_CUDA(cudaStreamWaitEvent(p->comp, p->ev_out[b], 0));  // o_buf drained
        rc = apply_impl(dX + col0, g_buf, o_buf, K, A, n, w, ld_dev, chunk_cols, chunk_cols, p->comp);
        if (rc != BDE_OK) return rc;
        BDE_RETURN_IF_CUDA(cudaEventRecord(p->ev_k2[b], p->comp));
        BDE_RETURN_IF_CUDA(cudaStreamWaitEvent(p->d2h, p->ev_k2[b], 0));
        BDE_RETURN_IF_CUDA(cudaMemcpy2DAsync(out_host + col0, ld_host * fsz, o_buf, chunk_cols * fsz, w * fsz, n,
                                             cudaMemcpyDeviceToHost, p->d2h));
        BDE_RETURN_IF_CUDA(cudaEventRecord(p->ev_out[b], p->d2h));
    }
    BDE_RETURN_IF_CUDA(cudaStreamSynchronize(p->comp));
    BDE_RETURN_IF_CUDA(cudaStreamSynchronize(p->d2h));
    return BDE_OK;
}

extern "C" int bde_svgd_step_host(const float* X_host, const float* G_host, float* out_host, int n, int64_t D,
                                  int64_t ld_host, double l2_reg, double kernel_grad_scale, double dataset_size,
                                  double h_override, int64_t chunk_cols, float* dX, float* dG, float* dOut,
                                  double* dist, float* K, float* A, double* info, int32_t* sel, void* workspace,
                                  size_t workspace_bytes, double* info_host, int32_t* sel_host) {
    int rc = bde_svgd_host_pairdist(X_host, n, D, ld_host, chunk_cols, dX, dist, workspace, workspace_bytes);
    if (rc != BDE_OK) return rc;
    return bde_svgd_host_apply(G_host, out_host, n, D, ld_host, l2_reg, kernel_grad_scale, dataset_size, h_override,
                               chunk_cols, dX, dG, dOut, dist, K, A, info, sel, info_host, sel_host);
}
