"""Tensor-level wrappers over the C-ABI (include/bde_b200.h).

Every function validates dtype / device / strides, extracts raw device pointers and the
current CUDA stream, and calls the library through ctypes.  No arithmetic happens here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _lib



def require_cuda(*tensors: torch.Tensor) -> None:
    """The product path is CUDA-only; anything else is an error, never a fallback.  All tensors of one call must
    live on ONE device (the kernels take raw pointers and run on that device's current stream)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.BdeError("beyond_deep_ensembles_b200 runs on CUDA tensors only (no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise _lib.BdeError(f"tensors of one kernel call span devices ({dev} and {t.device})")


def _rows(t: torch.Tensor):
    """(n, D, ld) of a row-major 2-D fp32 matrix whose rows are contiguous."""
    if t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise ValueError("expected a 2-D tensor with contiguous rows")
    n, D = t.shape
    ld = t.stride(0) if n > 1 else max(D, 1)
    return n, D, ld


def _vec(t: torch.Tensor | None):
    if t is not None and (t.dim() != 1 or (t.numel() > 1 and t.stride(0) != 1)):
        raise ValueError("expected a contiguous 1-D tensor")
    return t


def _s(t: torch.Tensor) -> int:
    return _lib.stream_ptr(t.device)


def zeros_bytes(nbytes: int, device) -> torch.Tensor:
    return torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device=device)


# --------------------------------------------------------------------------------------
# SVGD
# --------------------------------------------------------------------------------------
@dataclass
class SvgdScratch:
    """Per-(device, n) scratch of the SVGD kernels: all small and allocated once."""
    n: int
    dist: torch.Tensor   # [n, n] fp64
    K: torch.Tensor      # [n, n] fp32
    A: torch.Tensor      # [n, n] fp32
    info: torch.Tensor   # [4] fp64: h, median, d_lo, d_hi
    sel: torch.Tensor    # [2] int32
    ws: torch.Tensor     # reduction workspace (zero-filled once)
    peers: object = None  # dist.PeerSet once attached: launches on this scratch then sum over all ranks in-kernel

    @staticmethod
    def allocate(n: int, device) -> "SvgdScratch":
        nbytes = C.c_size_t(0)
        _lib.check(_lib.get().bde_svgd_workspace_bytes(n, C.byref(nbytes)), "bde_svgd_workspace_bytes")
        return SvgdScratch(
            n=n,
            dist=torch.zeros((n, n), dtype=torch.float64, device=device),
            K=torch.zeros((n, n), dtype=torch.float32, device=device),
            A=torch.zeros((n, n), dtype=torch.float32, device=device),
            info=torch.zeros(4, dtype=torch.float64, device=device),
            sel=torch.zeros(2, dtype=torch.int32, device=device),
            ws=zeros_bytes(nbytes.value, device),
        )

    @property
    def ws_bytes(self) -> int:
        return self.ws.numel() * 8

    def exact_redo(self) -> bool:
        """Did the last centred-Gram K1 launch on this scratch (n = 16 / 20, csrc/svgd_gram.cuh) fail its
        cancellation guard, i.e. were the distances recomputed by the direct kernel?  (WsHeader.redo; syncs.)"""
        return ((int(self.ws[1].item()) >> 32) & 0xFFFFFFFF) != 0


def svgd_pairdist(X: torch.Tensor, sc: SvgdScratch, accumulate: bool = False) -> torch.Tensor:
    """K1: sc.dist (+)= squared pair distances over X's columns (svgd.py:15)."""
    require_cuda(X)
    _lib.require_f32(X)
    n, D, ld = _rows(X)
    assert n == sc.n
    _lib.call("bde_svgd_pairdist", X.data_ptr(), n, D, ld, sc.dist.data_ptr(), int(accumulate), sc.ws.data_ptr(),
              sc.ws_bytes, _s(X))
    return sc.dist


def svgd_bandwidth(sc: SvgdScratch, l2_reg: float, kernel_grad_scale: float, dataset_size: float,
                   h_override: float = 0.0) -> None:
    """K1b: median heuristic, K and A from sc.dist (svgd.py:17-31,86,89)."""
    require_cuda(sc.dist)
    _lib.call("bde_svgd_bandwidth", sc.dist.data_ptr(), sc.n, float(l2_reg), float(kernel_grad_scale),
              float(dataset_size), float(h_override or 0.0), sc.K.data_ptr(), sc.A.data_ptr(), sc.info.data_ptr(),
              sc.sel.data_ptr(), _s(sc.dist))


def svgd_apply(X: torch.Tensor, G: torch.Tensor, out: torch.Tensor, sc: SvgdScratch) -> torch.Tensor:
    """K2: out = K G + A X (svgd.py:86-97)."""
    require_cuda(X, G, out)
    _lib.require_f32(X, G, out)
    n, D, ld = _rows(X)
    if _rows(G) != (n, D, ld) or _rows(out) != (n, D, ld):
        raise ValueError("X, G and out must share shape and row stride")
    _lib.call("bde_svgd_apply", X.data_ptr(), G.data_ptr(), out.data_ptr(), sc.K.data_ptr(), sc.A.data_ptr(), n, D, ld,
              _s(X))
    return out


NEXT_KERNEL_MAX_PARTICLES = 10  # single-pass training-step form (kNextDistMaxParticles in csrc/svgd_internal.h)
MAX_PARTICLES = 64              # BDE_MAX_PARTICLES: K1, K1b and K2 (include/bde_b200.h)
FUSED_MAX_PARTICLES = 32        # kGenericMaxParticles: fused base-optimizer forms, host-staged entries, peer exchange


@dataclass
class NextKernel:
    """Ask the fused apply kernels for the training-step form: the same pass leaves the pair distances
    of the UPDATED particles in sc.dist (this rank's partial sums) and, with fuse_bandwidth, the next
    step's K / A / info / sel in `sc` (K1b in the tail of the launch; single-rank jobs)."""
    fuse_bandwidth: bool
    l2_reg: float
    kernel_grad_scale: float
    dataset_size: float
    h_override: float = 0.0

    def args(self, sc: "SvgdScratch"):
        return (sc.dist.data_ptr(), int(self.fuse_bandwidth), float(self.l2_reg), float(self.kernel_grad_scale),
                float(self.dataset_size), float(self.h_override or 0.0), sc.K.data_ptr(), sc.A.data_ptr(),
                sc.info.data_ptr(), sc.sel.data_ptr(), sc.ws.data_ptr(), sc.ws_bytes)


def svgd_apply_sgd(X: torch.Tensor, G: torch.Tensor, sc: SvgdScratch, momentum_buf, *, buf_initialized: bool, lr: float,
                   momentum: float = 0.0, dampening: float = 0.0, weight_decay: float = 0.0, nesterov: bool = False,
                   out_last=None, next_kernel: NextKernel | None = None) -> None:
    """K2 fused with n shared-state torch.optim.SGD steps (svgd.py:92-103); X is updated in place.
    With `next_kernel` the launch also produces the next step's pair distances (see NextKernel)."""
    require_cuda(X, G, momentum_buf, out_last)
    _lib.require_f32(X, G, momentum_buf, out_last)
    n, D, ld = _rows(X)
    if _rows(G) != (n, D, ld):
        raise ValueError("X and G must share shape and row stride")
    for t in (momentum_buf, out_last):
        if t is not None and _vec(t).numel() != D:
            raise ValueError("optimizer state / out_last must be [D]")
    if momentum != 0.0 and momentum_buf is None:
        raise ValueError("momentum needs a momentum buffer")
    args = (X.data_ptr(), G.data_ptr(), sc.K.data_ptr(), sc.A.data_ptr(), n, D, ld,
            _lib.ptr(momentum_buf), int(buf_initialized), float(lr), float(momentum), float(dampening),
            float(weight_decay), int(bool(nesterov)), _lib.ptr(out_last))
    if next_kernel is None:
        _lib.call("bde_svgd_apply_sgd", *args, _s(X))
    else:
        _lib.call("bde_svgd_train_step_sgd", *args, *next_kernel.args(sc), _s(X))


def svgd_apply_adam(X: torch.Tensor, G: torch.Tensor, sc: SvgdScratch, exp_avg, exp_avg_sq, *, step0: int, lr: float,
                    beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8, weight_decay: float = 0.0,
                    decoupled_weight_decay: bool = False, out_last=None, next_kernel: NextKernel | None = None) -> None:
    """K2 fused with n shared-state torch.optim.Adam / AdamW steps; particle i takes step step0+i+1.
    With `next_kernel` the launch also produces the next step's pair distances (see NextKernel)."""
    require_cuda(X, G, exp_avg, exp_avg_sq, out_last)
    _lib.require_f32(X, G, exp_avg, exp_avg_sq, out_last)
    n, D, ld = _rows(X)
    if _rows(G) != (n, D, ld):
        raise ValueError("X and G must share shape and row stride")
    for t in (exp_avg, exp_avg_sq, out_last):
        if t is not None and _vec(t).numel() != D:
            raise ValueError("optimizer state / out_last must be [D]")
    args = (X.data_ptr(), G.data_ptr(), sc.K.data_ptr(), sc.A.data_ptr(), n, D, ld,
            exp_avg.data_ptr(), exp_avg_sq.data_ptr(), int(step0), float(lr), float(beta1), float(beta2), float(eps),
            float(weight_decay), int(bool(decoupled_weight_decay)), _lib.ptr(out_last))
    if next_kernel is None:
        _lib.call("bde_svgd_apply_adam", *args, _s(X))
    else:
        _lib.call("bde_svgd_train_step_adam", *args, *next_kernel.args(sc), _s(X))


def svgd_pairdist_bandwidth(X: torch.Tensor, sc: SvgdScratch, l2_reg: float, kernel_grad_scale: float,
                            dataset_size: float, h_override: float = 0.0) -> None:
    """K1 with K1b fused into its tail (single-GPU form, one launch)."""
    require_cuda(X)
    _lib.require_f32(X)
    n, D, ld = _rows(X)
    assert n == sc.n
    _lib.call("bde_svgd_pairdist_bandwidth", X.data_ptr(), n, D, ld, float(l2_reg), float(kernel_grad_scale),
              float(dataset_size), float(h_override or 0.0), sc.dist.data_ptr(), sc.K.data_ptr(), sc.A.data_ptr(),
              sc.info.data_ptr(), sc.sel.data_ptr(), sc.ws.data_ptr(), sc.ws_bytes, _s(X))


def svgd_step(X: torch.Tensor, G: torch.Tensor, out: torch.Tensor, sc: SvgdScratch, l2_reg: float,
              kernel_grad_scale: float, dataset_size: float, h_override: float = 0.0) -> torch.Tensor:
    """Single-GPU posterior update: K1(+K1b) then K2 — two launches, K2 as a programmatic dependent of K1 (it fills
    its ring during K1's tail)."""
    svgd_pairdist_bandwidth(X, sc, l2_reg, kernel_grad_scale, dataset_size, h_override)
    svgd_chain_next(X)
    return svgd_apply(X, G, out, sc)


def svgd_chain_next(t: torch.Tensor) -> None:
    """The next svgd_apply* launch on t's stream directly follows the K1 / K1b launch just made, nothing in between
    (bde_svgd_chain_next): call it only back to back with both."""
    _lib.get().bde_svgd_chain_next(_s(t))


# --------------------------------------------------------------------------------------
# SWAG
# --------------------------------------------------------------------------------------
def swag_update(theta, mean, sq, dev_row, updates: int) -> None:
    """K3 (swag.py:98-104); `updates` is the count after the increment."""
    require_cuda(theta, mean, sq, dev_row)
    _lib.require_f32(theta, mean, sq, dev_row)
    D = _vec(theta).numel()
    assert _vec(mean).numel() == D and _vec(sq).numel() == D and _vec(dev_row).numel() == D
    _lib.call("bde_swag_update", theta.data_ptr(), mean.data_ptr(), sq.data_ptr(), dev_row.data_ptr(), D, int(updates),
              _s(theta))


def swag_sample(mean, sq, dev, head: int, theta, *, eps_k=None, eps_d=None, seed: int = 0, stream_id: int = 0,
                elem0: int = 0) -> None:
    """K4 (swag.py:53-58,107-114).  dev: [K, ld] ring buffer, head = physical row of the oldest column."""
    require_cuda(mean, sq, dev, theta, eps_k, eps_d)
    _lib.require_f32(mean, sq, dev, theta, eps_k, eps_d)
    D = _vec(mean).numel()
    K, Dd, ld = _rows(dev)
    assert Dd == D and _vec(sq).numel() == D and _vec(theta).numel() == D
    if eps_k is not None:
        assert _vec(eps_k).numel() == K
    if eps_d is not None:
        assert _vec(eps_d).numel() == D
    _lib.call("bde_swag_sample", mean.data_ptr(), sq.data_ptr(), dev.data_ptr(), K, int(head), D, ld, _lib.ptr(eps_k),
              _lib.ptr(eps_d), int(seed), int(stream_id), int(elem0), theta.data_ptr(), _s(mean))


def swag_sample_batch(mean, sq, dev, head: int, theta, *, eps_k=None, eps_d=None, seed: int = 0, stream_id: int = 0,
                      elem0: int = 0) -> None:
    """K4 batched: theta [S, ld_out] receives S draws in one pass over the moments; draw s is what swag_sample
    returns for stream_id + s.  eps_k: [S, K], eps_d: [S, D] (row stride free) or None for Philox."""
    require_cuda(mean, sq, dev, theta, eps_k, eps_d)
    _lib.require_f32(mean, sq, dev, theta, eps_k, eps_d)
    D = _vec(mean).numel()
    K, Dd, ld = _rows(dev)
    S, Do, ld_out = _rows(theta)
    assert Dd == D and Do == D and _vec(sq).numel() == D
    ld_eps = 0
    if eps_k is not None:
        assert eps_k.is_contiguous() and tuple(eps_k.shape) == (S, K)
    if eps_d is not None:
        Se, De, ld_eps = _rows(eps_d)
        assert (Se, De) == (S, D)
    _lib.call("bde_swag_sample_batch", mean.data_ptr(), sq.data_ptr(), dev.data_ptr(), K, int(head), D, ld, S,
              _lib.ptr(eps_k), _lib.ptr(eps_d), ld_eps, int(seed), int(stream_id), int(elem0), theta.data_ptr(), ld_out,
              _s(mean))


# --------------------------------------------------------------------------------------
# iVON
# --------------------------------------------------------------------------------------
def ivon_sample(mean, prec, delta_sum, theta, *, n_eff: float, first: bool, deterministic: bool = False, eps=None,
                seed: int = 0, stream_id: int = 0, elem0: int = 0) -> None:
    """K5 (ivorn.py:102-115)."""
    require_cuda(mean, prec, delta_sum, theta, eps)
    _lib.require_f32(mean, prec, delta_sum, theta, eps)
    D = _vec(mean).numel()
    assert _vec(prec).numel() == D and _vec(delta_sum).numel() == D and _vec(theta).numel() == D
    _lib.call("bde_ivon_sample", mean.data_ptr(), prec.data_ptr(), delta_sum.data_ptr(), theta.data_ptr(), D,
              float(n_eff), int(first), int(deterministic), _lib.ptr(_vec(eps)), int(seed), int(stream_id), int(elem0),
              _s(mean))


def ivon_sample_batch(mean, prec, delta_sum, theta, *, n_eff: float, first: bool, deterministic: bool = False, eps=None,
                      seed: int = 0, stream_id: int = 0, stream_stride: int = 1, elem0: int = 0) -> None:
    """K5 batched: theta [S, ld_out] receives S consecutive draws; draw s is what ivon_sample returns for
    stream_id + s * stream_stride, delta_sum ends as after S single calls.  eps: [S, D] (row stride free) or None."""
    require_cuda(mean, prec, delta_sum, theta, eps)
    _lib.require_f32(mean, prec, delta_sum, theta, eps)
    D = _vec(mean).numel()
    S, Do, ld_out = _rows(theta)
    assert Do == D and _vec(prec).numel() == D and _vec(delta_sum).numel() == D
    ld_eps = 0
    if eps is not None:
        Se, De, ld_eps = _rows(eps)
        assert (Se, De) == (S, D)
    _lib.call("bde_ivon_sample_batch", mean.data_ptr(), prec.data_ptr(), delta_sum.data_ptr(), theta.data_ptr(), ld_out, D,
              S, float(n_eff), int(first), int(deterministic), _lib.ptr(eps), ld_eps, int(seed), int(stream_id),
              int(stream_stride), int(elem0), _s(mean))


def ivon_accumulate(acc, grad, first: bool) -> None:
    """K6 (ivorn.py:120-127)."""
    require_cuda(acc, grad)
    _lib.require_f32(acc, grad)
    D = _vec(acc).numel()
    assert _vec(grad).numel() == D
    _lib.call("bde_ivon_accumulate", acc.data_ptr(), grad.data_ptr(), D, int(first), _s(acc))


def ivon_update(acc_grad, delta_sum, mean, momentum, prec, *, mc_samples: int, step: int, lr: float, beta1: float,
                beta2: float, prior_prec: float, n_eff: float, tempering: float, damping: float) -> None:
    """K7 (ivorn.py:66-89)."""
    require_cuda(acc_grad, delta_sum, mean, momentum, prec)
    _lib.require_f32(acc_grad, delta_sum, mean, momentum, prec)
    D = _vec(mean).numel()
    for t in (acc_grad, delta_sum, momentum, prec):
        assert _vec(t).numel() == D
    _lib.call("bde_ivon_update", acc_grad.data_ptr(), delta_sum.data_ptr(), mean.data_ptr(), momentum.data_ptr(),
              prec.data_ptr(), D, int(mc_samples), int(step), float(lr), float(beta1), float(beta2), float(prior_prec),
              float(n_eff), float(tempering), float(damping), _s(mean))


# --------------------------------------------------------------------------------------
# BBB / Rank-1
# --------------------------------------------------------------------------------------
def gauss_sample_fwd(mu, rho, w, *, eps=None, seed: int = 0, stream_id: int = 0, elem0: int = 0) -> None:
    """K8 forward (util.py:170-171)."""
    require_cuda(mu, rho, w, eps)
    _lib.require_f32(mu, rho, w, eps)
    P = mu.numel()
    assert rho.numel() == P and w.numel() == P and mu.is_contiguous() and rho.is_contiguous() and w.is_contiguous()
    _lib.call("bde_gauss_sample_fwd", mu.data_ptr(), rho.data_ptr(), w.data_ptr(), P, _lib.ptr(eps), int(seed),
              int(stream_id), int(elem0), _s(mu))


def gauss_sample_bwd(grad_w, rho, grad_rho, *, eps=None, seed: int = 0, stream_id: int = 0, elem0: int = 0) -> None:
    """K8 backward: grad_rho (grad_mu aliases grad_w)."""
    require_cuda(grad_w, rho, grad_rho, eps)
    _lib.require_f32(grad_w, rho, grad_rho, eps)
    P = rho.numel()
    assert grad_w.numel() == P and grad_rho.numel() == P and grad_w.is_contiguous() and rho.is_contiguous()
    _lib.call("bde_gauss_sample_bwd", grad_w.data_ptr(), rho.data_ptr(), grad_rho.data_ptr(), P, _lib.ptr(eps),
              int(seed), int(stream_id), int(elem0), _s(rho))


def bbb_linear_fwd(x, w_mu, w_rho, b_mu, b_rho, *, eps=None, seed: int = 0, stream_id: int = 0, mc_sample: float = 1.0,
                   workspace=None):
    """f4: BBBLinear's local-reparameterisation forward (bbb_layers.py:61-88) as one tcgen05 kernel.
    x [batch, in] (rows contiguous), w_mu / w_rho [out, in], b_mu / b_rho [out] (or both None), eps [batch, out] or
    None (Philox).  Returns (out, act_std, eps_used), each [batch, out].  workspace: callable (device, nbytes) ->
    zero-filled int64 tensor, or None to allocate one."""
    require_cuda(x, w_mu, w_rho, b_mu, b_rho, eps)
    _lib.require_f32(x, w_mu, w_rho, b_mu, b_rho, eps)
    batch, fin, ldx = _rows(x)
    fout = w_mu.shape[0]
    if tuple(w_mu.shape) != (fout, fin) or tuple(w_rho.shape) != (fout, fin) or not (w_mu.is_contiguous() and w_rho.is_contiguous()):
        raise ValueError("w_mu / w_rho must be contiguous [out_features, in_features]")
    for t in (b_mu, b_rho):
        if t is not None and _vec(t).numel() != fout:
            raise ValueError("bias parameters must be [out_features]")
    if eps is not None and (tuple(eps.shape) != (batch, fout) or not eps.is_contiguous()):
        raise ValueError("eps must be contiguous [batch, out_features]")
    nbytes = C.c_size_t(0)
    _lib.check(_lib.get().bde_bbb_linear_workspace_bytes(batch, fin, fout, C.byref(nbytes)), "bde_bbb_linear_workspace_bytes")
    ws = workspace(x.device, nbytes.value) if workspace is not None else zeros_bytes(nbytes.value, x.device)
    out = torch.empty((batch, fout), dtype=torch.float32, device=x.device)
    act_std = torch.empty_like(out)
    eps_used = torch.empty_like(out)
    _lib.call("bde_bbb_linear_fwd", x.data_ptr(), ldx, batch, fin, fout, w_mu.data_ptr(), w_rho.data_ptr(), _lib.ptr(b_mu),
              _lib.ptr(b_rho), _lib.ptr(eps), int(seed), int(stream_id), float(mc_sample), out.data_ptr(), act_std.data_ptr(),
              eps_used.data_ptr(), ws.data_ptr(), ws.numel() * 8, _s(x))
    return out, act_std, eps_used


def rank1_linear_fwd(x, weight, s_mu, s_rho, r_mu, r_rho, bias=None, *, eps_s=None, eps_r=None, seed: int = 0,
                     stream_id_s: int = 0, stream_id_r: int = 0, workspace=None):
    """f4 (second half): Rank1Linear.forward (rank1.py:50-64) as one tcgen05 kernel — s and r sampled inside, the x * s
    prologue and the * r + bias epilogue fused around the product.  x [batch, in] (rows contiguous), weight [out, in],
    s_* [in], r_* [out], bias [out] or None, eps_s [in] / eps_r [out] or None (Philox).
    Returns (out, lin, s, r, eps_s_used, eps_r_used) with lin = linear(x * s, weight)."""
    require_cuda(x, weight, s_mu, s_rho, r_mu, r_rho, bias, eps_s, eps_r)
    _lib.require_f32(x, weight, s_mu, s_rho, r_mu, r_rho, bias, eps_s, eps_r)
    batch, fin, ldx = _rows(x)
    fout = weight.shape[0]
    if tuple(weight.shape) != (fout, fin) or not weight.is_contiguous():
        raise ValueError("weight must be contiguous [out_features, in_features]")
    for t, size, name in ((s_mu, fin, "s_mu"), (s_rho, fin, "s_rho"), (r_mu, fout, "r_mu"), (r_rho, fout, "r_rho"),
                          (bias, fout, "bias"), (eps_s, fin, "eps_s"), (eps_r, fout, "eps_r")):
        if t is not None and (_vec(t).numel() != size or not t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous vector of {size} elements")
    nbytes = C.c_size_t(0)
    _lib.check(_lib.get().bde_bbb_linear_workspace_bytes(batch, fin, fout, C.byref(nbytes)), "bde_bbb_linear_workspace_bytes")
    ws = workspace(x.device, nbytes.value) if workspace is not None else zeros_bytes(nbytes.value, x.device)
    out = torch.empty((batch, fout), dtype=torch.float32, device=x.device)
    lin = torch.empty_like(out)
    s, es = torch.empty(fin, dtype=torch.float32, device=x.device), torch.empty(fin, dtype=torch.float32, device=x.device)
    r, er = torch.empty(fout, dtype=torch.float32, device=x.device), torch.empty(fout, dtype=torch.float32, device=x.device)
    _lib.call("bde_rank1_linear_fwd", x.data_ptr(), ldx, batch, fin, fout, weight.data_ptr(), s_mu.data_ptr(), s_rho.data_ptr(),
              r_mu.data_ptr(), r_rho.data_ptr(), _lib.ptr(bias), _lib.ptr(eps_s), _lib.ptr(eps_r), int(seed), int(stream_id_s),
              int(stream_id_r), out.data_ptr(), lin.data_ptr(), s.data_ptr(), r.data_ptr(), es.data_ptr(), er.data_ptr(),
              ws.data_ptr(), ws.numel() * 8, _s(x))
    return out, lin, s, r, es, er


def value_workspace(device) -> torch.Tensor:
    nbytes = C.c_size_t(0)
    _lib.check(_lib.get().bde_value_workspace_bytes(C.byref(nbytes)), "bde_value_workspace_bytes")
    return zeros_bytes(nbytes.value, device)


def kl_gauss(mu, rho, prior_mu: float, prior_sigma: float, *, value=None, grad_mu=None, grad_rho=None,
             grad_scale: float = 1.0, grad_scale_dev=None, accumulate: bool = False, ws=None) -> None:
    """K9 (bbb.py:18-21): value (fp64 device scalar) and/or analytic gradient."""
    require_cuda(mu, rho, value, grad_mu, grad_rho, grad_scale_dev)
    _lib.require_f32(mu, rho, grad_mu, grad_rho, grad_scale_dev)
    P = mu.numel()
    assert rho.numel() == P and mu.is_contiguous() and rho.is_contiguous()
    if value is not None:
        assert value.dtype == torch.float64 and ws is not None
    _lib.call("bde_kl_gauss_value_and_grad", mu.data_ptr(), rho.data_ptr(), P, float(prior_mu), float(prior_sigma),
              _lib.ptr(value), _lib.ptr(grad_mu), _lib.ptr(grad_rho), float(grad_scale), _lib.ptr(grad_scale_dev),
              int(accumulate), _lib.ptr(ws), 0 if ws is None else ws.numel() * 8, _s(mu))


def kl_mixture(mu, pi: float, sigma1: float, sigma2: float, *, value=None, grad_mu=None, grad_scale: float = 1.0,
               grad_scale_dev=None, accumulate: bool = False, ws=None) -> None:
    """K9b (bbb.py:23-37)."""
    require_cuda(mu, value, grad_mu, grad_scale_dev)
    _lib.require_f32(mu, grad_mu, grad_scale_dev)
    P = mu.numel()
    assert mu.is_contiguous()
    if value is not None:
        assert value.dtype == torch.float64 and ws is not None
    _lib.call("bde_kl_mixture_value_and_grad", mu.data_ptr(), P, float(pi), float(sigma1), float(sigma2),
              _lib.ptr(value), _lib.ptr(grad_mu), float(grad_scale), _lib.ptr(grad_scale_dev), int(accumulate),
              _lib.ptr(ws), 0 if ws is None else ws.numel() * 8, _s(mu))


PRIOR_GAUSS, PRIOR_MIXTURE, PRIOR_L2 = 0, 1, 2


def prior_terms(kinds, a, b, sizes=None, *, l2_scales=None, prior=(0.0, 1.0, 0.0), value=None, grad_a=None, grad_b=None,
                grad_scale: float = 1.0, grad_scale_dev=None, accumulate: bool = False, ws=None) -> None:
    """K9 + K10 over a list of tensors in one launch (bbb.py:69-76).

    kinds[i]: PRIOR_GAUSS (a[i] = mu, b[i] = rho), PRIOR_MIXTURE (a[i] = mu) or PRIOR_L2 (a[i] = theta,
    l2_scales[i]); prior = (mu_p, sigma_p, -) or (pi, sigma1, sigma2); grad_a / grad_b: lists of output
    tensors (None entries: no gradient for that tensor) or None for the value only."""
    count = len(kinds)
    if count == 0:
        if value is not None:
            value.zero_()
        return
    tensors = [t for t in list(a) + list(b or []) + list(grad_a or []) + list(grad_b or []) if t is not None]
    require_cuda(*tensors, value, grad_scale_dev)
    _lib.require_f32(*tensors, grad_scale_dev)
    for t in tensors:
        if not t.is_contiguous():
            raise ValueError("prior_terms needs contiguous tensors")
    if value is not None:
        assert value.dtype == torch.float64 and ws is not None
    u64, i64 = C.c_uint64 * count, C.c_int64 * count

    def table(ts):
        return u64(*[0 if t is None else t.data_ptr() for t in ts])

    b_list = list(b) if b is not None else [None] * count
    sizes_arr = i64(*[t.numel() for t in a])
    for i, k in enumerate(kinds):
        if k == PRIOR_GAUSS and (b_list[i] is None or b_list[i].numel() != a[i].numel()):
            raise ValueError("a Gaussian parameter needs a rho tensor of the same size")
        for g in (grad_a, grad_b):
            if g is not None and g[i] is not None and g[i].numel() != a[i].numel():
                raise ValueError("gradient tensor size mismatch")
    l2 = (C.c_double * count)(*[float(x) for x in (l2_scales if l2_scales is not None else [0.0] * count)])
    p0, p1, p2 = (float(x) for x in prior)
    _lib.call("bde_prior_terms_value_and_grad", count, C.cast((C.c_int32 * count)(*[int(k) for k in kinds]), C.c_void_p),
              C.cast(table(a), C.c_void_p), C.cast(table(b_list), C.c_void_p),
              None if grad_a is None else C.cast(table(grad_a), C.c_void_p),
              None if grad_b is None else C.cast(table(grad_b), C.c_void_p),
              C.cast(sizes_arr, C.c_void_p), C.cast(l2, C.c_void_p), p0, p1, p2, _lib.ptr(value), float(grad_scale),
              _lib.ptr(grad_scale_dev), int(accumulate), _lib.ptr(ws), 0 if ws is None else ws.numel() * 8, _s(a[0]))


def l2_term(theta, l2_scale: float, *, value=None, grad=None, grad_scale: float = 1.0, grad_scale_dev=None,
            accumulate: bool = False, ws=None) -> None:
    """K10 (bbb.py:75-76)."""
    require_cuda(theta, value, grad, grad_scale_dev)
    _lib.require_f32(theta, grad, grad_scale_dev)
    D = theta.numel()
    assert theta.is_contiguous()
    if value is not None:
        assert value.dtype == torch.float64 and ws is not None
    _lib.call("bde_l2_value_and_grad", theta.data_ptr(), D, float(l2_scale), _lib.ptr(value), _lib.ptr(grad),
              float(grad_scale), _lib.ptr(grad_scale_dev), int(accumulate), _lib.ptr(ws),
              0 if ws is None else ws.numel() * 8, _s(theta))


# --------------------------------------------------------------------------------------
# utilities
# --------------------------------------------------------------------------------------
def philox_normal(out: torch.Tensor, seed: int, stream_id: int, elem0: int = 0) -> torch.Tensor:
    require_cuda(out)
    _lib.require_f32(out)
    _lib.call("bde_philox_normal", out.data_ptr(), out.numel(), int(seed), int(stream_id), int(elem0), _s(out))
    return out


class CopyTable:
    """Host-side half of a multi_tensor_copy call that does not change between calls: the flat offsets and the
    element counts of the tensors (ctypes arrays built once) and a reusable pointer array.  Built once per
    parameter layout; per call only the data pointers are refreshed (autograd may hand out new .grad storage)."""

    def __init__(self, offsets, numels):
        self.count = len(offsets)
        self.numels = [int(n) for n in numels]
        self.offs = (C.c_int64 * self.count)(*[int(o) for o in offsets])
        self.sizes = (C.c_int64 * self.count)(*self.numels)
        self.offs_p = C.cast(self.offs, C.c_void_p)
        self.sizes_p = C.cast(self.sizes, C.c_void_p)


def multi_tensor_copy(flat_row: torch.Tensor, tensors, offsets, mode: int, table: CopyTable | None = None,
                      inv_scale: torch.Tensor | None = None, found_inf: torch.Tensor | None = None) -> None:
    """Gather (mode 0), gather-add (1) or scatter (2) between `tensors` and a flat arena row.

    offsets: element offsets of each tensor inside flat_row (ascending); `table` (a CopyTable for the same
    offsets and tensor sizes) skips rebuilding the constant part of the argument tables.  With `inv_scale` /
    `found_inf` (fp32 device scalars) the gather is fused with GradScaler.unscale_: values are multiplied by
    inv_scale on the way and found_inf is raised on any non-finite source value."""
    count = len(tensors)
    if count == 0:
        return
    require_cuda(flat_row)
    _lib.require_f32(flat_row)
    if table is None:
        table = CopyTable(offsets, [t.numel() for t in tensors])
    elif table.count != count:
        raise ValueError("multi_tensor_copy: tensor list does not match the copy table")
    # one pass over the tensors (this runs once per particle / MC sample over up to a few hundred gradients): the common
    # case costs four attribute reads per tensor, the error branch says which check failed
    f32, dev, ptrs = torch.float32, flat_row.device, []
    for t, numel in zip(tensors, table.numels):
        if t.dtype is f32 and t.device == dev and t.numel() == numel and t.is_contiguous():
            ptrs.append(t.data_ptr())
            continue
        if t.dtype is not f32:
            raise TypeError(f"expected float32 tensor, got {t.dtype}")
        if t.device != dev:
            require_cuda(flat_row, t)   # raises: not a CUDA tensor / tensors span devices
            raise _lib.BdeError(f"tensors of one kernel call span devices ({dev} and {t.device})")
        if not t.is_contiguous():
            raise ValueError("multi_tensor_copy needs contiguous tensors")
        raise ValueError("multi_tensor_copy: tensor size does not match the copy table")
    cptrs = (C.c_uint64 * count)(*ptrs)
    if inv_scale is None:
        _lib.call("bde_multi_tensor_copy", flat_row.data_ptr(), C.cast(cptrs, C.c_void_p), table.offs_p, table.sizes_p,
                  count, int(mode), _s(flat_row))
        return
    require_cuda(inv_scale, found_inf)
    _lib.require_f32(inv_scale, found_inf)
    if inv_scale.numel() != 1 or found_inf.numel() != 1 or mode not in (0, 1):
        raise ValueError("unscaling gather: inv_scale / found_inf must be scalars and the mode a gather")
    _lib.call("bde_multi_tensor_unscale_copy", flat_row.data_ptr(), C.cast(cptrs, C.c_void_p), table.offs_p,
              table.sizes_p, count, int(mode), inv_scale.data_ptr(), found_inf.data_ptr(), _s(flat_row))


# --------------------------------------------------------------------------------------
# host-buffer (end-to-end) SVGD step
# --------------------------------------------------------------------------------------
@dataclass
class HostStaging:
    """Device staging of the host-buffer path: X resident, G / out double-buffered chunks."""
    n: int
    D: int
    chunk_cols: int
    dX: torch.Tensor    # [n, ld_dev]
    dG: torch.Tensor    # [2, n, chunk_cols]
    dOut: torch.Tensor  # [2, n, chunk_cols]

    @staticmethod
    def allocate(n: int, D: int, chunk_cols: int, device, dX: torch.Tensor | None = None) -> "HostStaging":
        chunk_cols = max(4, (min(chunk_cols, D) + 3) // 4 * 4)
        ld_dev = (D + 3) // 4 * 4
        if dX is None:
            dX = torch.empty((n, ld_dev), dtype=torch.float32, device=device)
        assert dX.shape == (n, ld_dev) and dX.is_contiguous()
        return HostStaging(n, D, chunk_cols, dX,
                           torch.empty((2, n, chunk_cols), dtype=torch.float32, device=device),
                           torch.empty((2, n, chunk_cols), dtype=torch.float32, device=device))


def _host_rows(t: torch.Tensor):
    if t.is_cuda or t.dtype != torch.float32 or t.dim() != 2 or t.stride(1) != 1:
        raise ValueError("expected a 2-D fp32 HOST tensor with contiguous rows")
    return t.shape[0], t.shape[1], t.stride(0)


def svgd_host_pairdist(X_host: torch.Tensor, st: HostStaging, sc: SvgdScratch) -> None:
    """Phase 1 of the end-to-end step: stream X up, accumulate the local partial distances (blocks)."""
    n, D, ld = _host_rows(X_host)
    assert (n, D) == (st.n, st.D)
    _lib.call("bde_svgd_host_pairdist", X_host.data_ptr(), n, D, ld, st.chunk_cols, st.dX.data_ptr(),
              sc.dist.data_ptr(), sc.ws.data_ptr(), sc.ws_bytes)


def svgd_host_apply(G_host: torch.Tensor, out_host: torch.Tensor, st: HostStaging, sc: SvgdScratch, l2_reg: float,
                    kernel_grad_scale: float, dataset_size: float, h_override: float = 0.0) -> None:
    """Phase 2: K1b, then stream G up / out down through K2 (blocks until out_host is complete)."""
    n, D, ld = _host_rows(G_host)
    assert (n, D) == (st.n, st.D) and _host_rows(out_host) == (n, D, ld)
    _lib.call("bde_svgd_host_apply", G_host.data_ptr(), out_host.data_ptr(), n, D, ld, float(l2_reg),
              float(kernel_grad_scale), float(dataset_size), float(h_override or 0.0), st.chunk_cols, st.dX.data_ptr(),
              st.dG.data_ptr(), st.dOut.data_ptr(), sc.dist.data_ptr(), sc.K.data_ptr(), sc.A.data_ptr(),
              sc.info.data_ptr(), sc.sel.data_ptr(), None, None)


def svgd_step_host(X_host, G_host, out_host, st: HostStaging, sc: SvgdScratch, l2_reg: float, kernel_grad_scale: float,
                   dataset_size: float, h_override: float = 0.0, group=None) -> None:
    """End-to-end SVGD posterior update on HOST buffers (this rank's column slice when D-sharded)."""
    from . import dist as bdist
    if sc.peers is not None:
        # the chunked host path launches K1 once per chunk on the library's own streams; ranks whose slices differ
        # by a column could disagree on the chunk count, so it keeps the all-reduce form
        raise ValueError("svgd_step_host needs a scratch that is not attached to a peer set")
    svgd_host_pairdist(X_host, st, sc)
    bdist.allreduce_dist(sc, group)
    if bdist.world(group) > 1:
        torch.cuda.current_stream(sc.dist.device).synchronize()  # phase 2 runs on the library's streams
    svgd_host_apply(G_host, out_host, st, sc, l2_reg, kernel_grad_scale, dataset_size, h_override)
