// peer.cu — host side of the in-kernel NVLink exchange (common.cuh: peer_allreduce_fp64).
//
// D-sharded SVGD (SURVEY.md §8e) needs ONE cross-rank step: the sum of the n*n partial pair distances.
// Instead of a separate all-reduce launch, each rank owns a small exchange buffer (PeerBuf, ~130 KB,
// cudaMalloc'ed so that it can be exported with CUDA IPC); every rank maps the buffers of all peers and
// writes the table of mapped pointers into the header of its reduction workspace.  From then on the last
// CTA of every grid reduction that uses this workspace completes the sum across ranks inside the launch.
// The caller owns the buffer, the mappings and the workspace; the library only remembers which workspaces are
// attached, so that K1 above 32 particles (more sums than an exchange slot holds) can refuse them.
#include <cstring>
#include <mutex>
#include <set>

#include "common.cuh"
#include "svgd_internal.h"

namespace bde {
namespace {
std::mutex g_attached_mu;
std::set<const void*> g_attached;   // workspaces attached to a peer set of more than one rank
void set_attached(const void* ws, bool on) {
    std::lock_guard<std::mutex> lock(g_attached_mu);
    if (on)
        g_attached.insert(ws);
    else
        g_attached.erase(ws);
}
}  // namespace
bool peer_attached(const void* ws) {
    std::lock_guard<std::mutex> lock(g_attached_mu);
    return g_attached.count(ws) != 0;
}
}  // namespace bde

using namespace bde;

extern "C" int bde_peer_buffer_bytes(size_t* bytes) {
    if (!bytes) return BDE_ERR_INVALID_ARG;
    *bytes = sizeof(PeerBuf);
    return BDE_OK;
}

extern "C" int bde_peer_alloc(void** buf, unsigned char* ipc_handle_host) {
    if (!buf || !ipc_handle_host) return BDE_ERR_INVALID_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == BDE_PEER_HANDLE_BYTES, "IPC handle size");
    void* p = nullptr;
    BDE_RETURN_IF_CUDA(cudaMalloc(&p, sizeof(PeerBuf)));
    cudaError_t e = cudaMemset(p, 0, sizeof(PeerBuf));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return static_cast<int>(e);
    }
    memcpy(ipc_handle_host, &h, sizeof(h));
    *buf = p;
    return BDE_OK;
}

extern "C" int bde_peer_open(const unsigned char* ipc_handle_host, void** mapped) {
    if (!ipc_handle_host || !mapped) return BDE_ERR_INVALID_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle_host, sizeof(h));
    void* p = nullptr;
    BDE_RETURN_IF_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *mapped = p;
    return BDE_OK;
}

extern "C" int bde_peer_close(void* mapped) {
    if (!mapped) return BDE_ERR_INVALID_ARG;
    BDE_RETURN_IF_CUDA(cudaIpcCloseMemHandle(mapped));
    return BDE_OK;
}

extern "C" int bde_peer_free(void* buf) {
    if (!buf) return BDE_ERR_INVALID_ARG;
    BDE_RETURN_IF_CUDA(cudaFree(buf));
    return BDE_OK;
}

extern "C" int bde_peer_attach(void* workspace, size_t workspace_bytes, int world, int rank, const uint64_t* bufs_host,
                               double timeout_seconds, uint64_t* host_status, bde_stream_t stream) {
    if (!workspace || workspace_bytes < kWsHeaderBytes || world < 1 || world > kPeerMaxRanks || rank < 0 || rank >= world ||
        (world > 1 && !bufs_host))
        return BDE_ERR_INVALID_ARG;
    WsHeader h{};
    h.peer_world = world;
    h.peer_rank = rank;
    h.timeout_ns = timeout_seconds > 0.0 ? static_cast<unsigned long long>(timeout_seconds * 1e9) : 0ull;
    h.host_status = reinterpret_cast<unsigned long long*>(host_status);   // pinned host memory is device-addressable (UVA)
    for (int r = 0; r < world && world > 1; ++r) {
        if (!bufs_host[r]) return BDE_ERR_INVALID_ARG;
        h.peer[r] = reinterpret_cast<PeerBuf*>(static_cast<uintptr_t>(bufs_host[r]));
    }
    // the ticket (first word) is zero between launches, so the whole header can be rewritten in stream order
    BDE_RETURN_IF_CUDA(cudaMemcpyAsync(workspace, &h, sizeof(h), cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
    BDE_RETURN_IF_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));  // h lives on this stack frame
    set_attached(workspace, world > 1);
    return BDE_OK;
}

extern "C" int bde_peer_detach(void* workspace, size_t workspace_bytes, bde_stream_t stream) {
    if (!workspace || workspace_bytes < kWsHeaderBytes) return BDE_ERR_INVALID_ARG;
    BDE_RETURN_IF_CUDA(cudaMemsetAsync(workspace, 0, sizeof(WsHeader), static_cast<cudaStream_t>(stream)));
    set_attached(workspace, false);
    return BDE_OK;
}

extern "C" int bde_peer_status(const void* buf, uint64_t* epoch_host, uint64_t* timeouts_host) {
    if (!buf) return BDE_ERR_INVALID_ARG;
    unsigned long long v[2] = {0, 0};
    BDE_RETURN_IF_CUDA(cudaMemcpy(v, buf, sizeof(v), cudaMemcpyDeviceToHost));
    if (epoch_host) *epoch_host = v[0];
    if (timeouts_host) *timeouts_host = v[1];
    return BDE_OK;
}

extern "C" int bde_peer_wait_stats(void* buf, uint64_t* exchanges_host, uint64_t* wait_ns_sum_host, uint64_t* wait_ns_max_host,
                                   int reset) {
    if (!buf) return BDE_ERR_INVALID_ARG;
    PeerBuf* pb = static_cast<PeerBuf*>(buf);
    unsigned long long v[3] = {0, 0, 0};   // wait_ns_sum, wait_ns_max, waits are consecutive fields
    BDE_RETURN_IF_CUDA(cudaMemcpy(v, &pb->wait_ns_sum, sizeof(v), cudaMemcpyDeviceToHost));
    if (wait_ns_sum_host) *wait_ns_sum_host = v[0];
    if (wait_ns_max_host) *wait_ns_max_host = v[1];
    if (exchanges_host) *exchanges_host = v[2];
    if (reset) BDE_RETURN_IF_CUDA(cudaMemset(&pb->wait_ns_sum, 0, sizeof(v)));
    return BDE_OK;
}
