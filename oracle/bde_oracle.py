"""bde_oracle — CPU restatement of the reference's posterior-update arithmetic.

TEST INFRASTRUCTURE ONLY.  This module is the parity checker for the CUDA path in
beyond_deep_ensembles_b200/: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import it.  The product never does.

Parity pinning: the reference (Feuermagier/Beyond_Deep_Ensembles @ b805d6f) ships no tests or
golden vectors for this path, so the oracle is pinned against outputs of the reference itself:
oracle/gen_golden.py imports the unmodified reference from /root/reference, runs it on seeded
inputs with injected noise and commits the results under tests/golden/; tests/test_oracle_golden.py
checks every function below against those fixtures.

Two evaluation modes for every function:
  dtype=float32 — the reference's own op sequence in fp32 (what eager PyTorch computes);
  dtype=float64 — the same sequence on double inputs; this is the accuracy oracle for large D,
                  where the reference's fp32 distance reduction itself drifts (SURVEY.md §8c).

Everything is numpy / torch-CPU tensor arithmetic; there are no Python loops over elements.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------
# SVGD — reference: src/algos/svgd.py
# --------------------------------------------------------------------------------------


def svgd_pairdist(X: torch.Tensor, dtype=torch.float64, chunk: int = 1 << 20) -> torch.Tensor:
    """Squared pairwise distances by direct differences, svgd.py:15 (`torch.cdist(p=2)**2`).

    Accumulated in `dtype` over column chunks (partial sums are exactly what D-sharded ranks
    all-reduce).  Returns the [n, n] matrix of SUMS (no sqrt round trip; see svgd_bandwidth).
    """
    n, D = X.shape
    out = torch.zeros((n, n), dtype=dtype)
    for c0 in range(0, D, chunk):
        x = X[:, c0:c0 + chunk].to(dtype)
        diff = x.unsqueeze(1) - x.unsqueeze(0)  # [n, n, c]
        out += (diff * diff).sum(dim=2)
    return out


def svgd_bandwidth(dist_sums: torch.Tensor, l2_reg: float, kernel_grad_scale: float, dataset_size: float,
                   h_override: float | None = None):
    """Median heuristic + RBF kernel + fused coefficient matrix, svgd.py:15-31,86,89 (fp64).

    dist_sums: [n, n] sums of squared differences.  Mirrors cdist's sqrt followed by **2,
    torch.quantile(q=0.5) over all n*n entries (stable sort, linear interpolation with torch's
    lerp formula), h = sqrt(0.5*med/ln(n+1)) + 1e-8, K = exp(-d/(2h^2)).
    A = (l2/2 + c) K - c diag(rowsum K) with c = kernel_grad_scale/(dataset_size h^2) so that
    new_grad_i = sum_j K_ij g_j + A_ij x_j  ==  -(K @ -(G + l2/2 X) + s*grad_K/N)_i.
    Returns dict(K, A, h, median, d_lo, d_hi, sel=(flat_lo, flat_hi) canonical i<=j indices).
    """
    d = dist_sums.to(torch.float64)
    n = d.shape[0]
    # correctly rounded sqrt, then one correctly rounded multiplication, as the kernel does: torch.sqrt on CPU
    # float64 tensors can be one ulp off (vectorised: torch.sqrt(11000313.0) != math.sqrt(11000313.0)), which
    # moves the median by an ulp, and by how much depends on the host's SIMD path
    r = torch.from_numpy(np.sqrt(d.cpu().numpy()))
    d = r * r
    flat = d.reshape(-1)
    nn_ = flat.numel()
    order = torch.sort(flat, stable=True).indices
    pos = 0.5 * (nn_ - 1)
    lo, hi = int(math.floor(pos)), int(math.ceil(pos))
    w = pos - lo
    a, b = flat[order[lo]].item(), flat[order[hi]].item()
    med = a + w * (b - a) if w < 0.5 else b - (b - a) * (1.0 - w)

    def canon(e: int) -> int:
        i, j = divmod(e, n)
        return e if i <= j else j * n + i

    sel = (canon(int(order[lo])), canon(int(order[hi])))
    h = math.sqrt(0.5 * med / math.log(n + 1)) + 1e-8
    if h_override is not None and h_override > 0:
        h = float(h_override)
    K = torch.exp(-d / (2.0 * h * h))
    c = kernel_grad_scale / (dataset_size * h * h)
    off = K.sum(dim=1) - torch.diagonal(K)
    A = (0.5 * l2_reg + c) * K
    A[range(n), range(n)] = 0.5 * l2_reg * torch.diagonal(K) - c * off
    return dict(K=K, A=A, h=h, median=med, d_lo=a, d_hi=b, sel=sel)


def svgd_apply(X: torch.Tensor, G: torch.Tensor, K: torch.Tensor, A: torch.Tensor, dtype=torch.float64) -> torch.Tensor:
    """out = K G + A X (the new .grad of every particle), svgd.py:86-97 fused."""
    return K.to(dtype) @ G.to(dtype) + A.to(dtype) @ X.to(dtype)


def svgd_step_fused(X, G, l2_reg, kernel_grad_scale, dataset_size, h_override=None, dtype=torch.float64):
    """K1 + K1b + K2 in one call; returns (out, info dict)."""
    info = svgd_bandwidth(svgd_pairdist(X, dtype=torch.float64), l2_reg, kernel_grad_scale, dataset_size, h_override)
    return svgd_apply(X, G, info["K"], info["A"], dtype=dtype), info


def svgd_step_reference_order(X: torch.Tensor, G: torch.Tensor, l2_reg: float, kernel_grad_scale: float,
                              dataset_size: float, dtype=torch.float32) -> torch.Tensor:
    """The reference's own op sequence (svgd.py:86-89 + rbf :15-31) on [n, D] inputs.

    Same ATen ops in the same order as the reference (cdist, quantile, exp, matmul and the
    elementwise temporaries), so timing this on the host cores is the CPU baseline ("port"),
    and in fp64 it is the accuracy oracle.  Returns -phi, i.e. the gradients the reference
    scatters into the particles at svgd.py:95.
    """
    P = X.to(dtype)
    Gv = G.to(dtype).clone()
    Gv += l2_reg / 2 * P                                            # :86
    d = torch.cdist(P, P, p=2) ** 2                                 # :15
    h = torch.sqrt(0.5 * torch.quantile(d, 0.5) / np.log(P.shape[0] + 1)) + 1e-8  # :18
    Kmat = torch.exp(-d / (2 * h ** 2))                             # :21
    gK = Kmat.sum(dim=1).unsqueeze(-1) * P - torch.matmul(Kmat, P)  # :23
    gK /= h ** 2                                                    # :31
    phi = torch.matmul(Kmat, -Gv) + kernel_grad_scale * gK / dataset_size  # :89
    return -phi                                                     # :95


def svgd_base_optimizer_steps(X: torch.Tensor, new_grads: torch.Tensor, kind: str, hyper: dict, state: dict | None = None):
    """svgd.py:92-103: ONE torch.optim optimizer (its state shared by all particles) takes one step
    per particle, in particle order, on `param.data = particle_i`, `param.grad = new_grads[i]`.

    This literally drives torch.optim.SGD / Adam / AdamW on a single CPU parameter, exactly like the
    reference does with the caller's base optimizer.  `state` carries the optimizer state between
    SVGD steps ({} on the very first call): momentum_buffer | (step, exp_avg, exp_avg_sq).
    Returns (X_new [n, D], state).  X and new_grads are not modified.
    """
    X = X.detach().clone().float()
    G = new_grads.detach().float()
    p = torch.nn.Parameter(X[0].clone())
    cls = {"sgd": torch.optim.SGD, "adam": torch.optim.Adam, "adamw": torch.optim.AdamW}[kind]
    opt = cls([p], foreach=False, **hyper)
    if state:
        opt.state[p] = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in state.items()}
    for i in range(X.shape[0]):
        p.data = X[i]            # the particle IS the parameter's storage (svgd.py:96)
        p.grad = G[i].clone()    # svgd.py:94
        opt.step()
    return X, dict(opt.state[p])


# --------------------------------------------------------------------------------------
# SWAG — reference: src/algos/swag.py
# --------------------------------------------------------------------------------------


def swag_update(theta, mean, sq, updates: int, dtype=torch.float32):
    """swag.py:98-104 with `updates` the value after the increment at :98.

    Returns (mean_new, sq_new, deviation_column)."""
    t, m, s = theta.to(dtype), mean.to(dtype), sq.to(dtype)
    m_new = (updates * m + t) / (updates + 1)
    s_new = (updates * s + t ** 2) / (updates + 1)
    return m_new, s_new, t - m_new


def swag_roll_deviations(dev_DK: torch.Tensor, column: torch.Tensor) -> torch.Tensor:
    """swag.py:103-104 on the reference's [D, K] layout."""
    out = torch.roll(dev_DK, -1, 1)
    out[:, -1] = column
    return out


def swag_ring_to_reference(dev_ring_KD: torch.Tensor, updates: int) -> torch.Tensor:
    """Ring buffer [K, D] (row updates%K is the oldest column) -> reference [D, K] roll order."""
    K = dev_ring_KD.shape[0]
    head = updates % K
    idx = [(head + k) % K for k in range(K)]
    return dev_ring_KD[idx].t().contiguous()


def swag_sample(mean, sq, dev_DK, eps_k, eps_d, dtype=torch.float32):
    """swag.py:112-114 + LowRankMultivariateNormal.rsample (loc + W@eps_W + sqrt(diag)*eps_D)."""
    m, s, dev = mean.to(dtype), sq.to(dtype), dev_DK.to(dtype)
    K = dev.shape[1]
    diag = 0.5 * (torch.relu(s - m ** 2) + 1e-6)
    # K == 1 divides by zero exactly as the reference's math.sqrt(2*(K-1)) does (inf/nan)
    den = math.sqrt(2 * (K - 1))
    cov_factor = dev / den if den > 0 else dev / torch.zeros((), dtype=dtype)
    return m + cov_factor @ eps_k.to(dtype) + diag.sqrt() * eps_d.to(dtype)


# --------------------------------------------------------------------------------------
# iVON — reference: src/algos/ivorn.py
# --------------------------------------------------------------------------------------


def ivon_sample(mean, prec, delta_sum, eps, n_eff: float, deterministic=False, dtype=torch.float32):
    """ivorn.py:102-115.  delta_sum=None on the first MC sample.  Returns (theta, delta_sum_new)."""
    m, p = mean.to(dtype), prec.to(dtype)
    if deterministic:
        delta = torch.zeros_like(p)
    else:
        delta = 1 / (n_eff * p.clamp(min=1e-4)).sqrt() * eps.to(dtype)
    theta = m + delta
    return theta, (delta if delta_sum is None else delta_sum.to(dtype) + delta)


def ivon_update(acc_grad, delta_sum, mean, momentum, prec, *, mc_samples: int, step: int, lr: float,
                betas=(0.9, 0.999), prior_prec: float, n_eff: float, tempering: float = 1.0, damping: float = 0.0,
                dtype=torch.float32):
    """ivorn.py:66-89 for one group; `step` is the value after the increment at :68.

    Returns (mean_new, momentum_new, prec_new)."""
    acc, ds = acc_grad.to(dtype), delta_sum.to(dtype)
    mean, momentum, prec = mean.to(dtype).clone(), momentum.to(dtype).clone(), prec.to(dtype).clone()
    beta1, beta2 = betas
    t = step
    N = n_eff
    delta = tempering * prior_prec / N
    gradient = acc / mc_samples
    g_mu = delta * mean + gradient
    momentum = beta1 * momentum + (1 - beta1) * g_mu
    g_s = delta - prec + (N * prec * ds / mc_samples) * gradient + damping
    corrected_momentum = momentum / (1 - beta1 ** t)
    corrected_precision = prec / (1 - beta2 ** t)
    mean = mean - lr * corrected_momentum / corrected_precision
    prec = prec + ((1 - beta2) + 0.5 * (1 - beta2) ** 2 * g_s / prec) * g_s
    return mean, momentum, prec


# --------------------------------------------------------------------------------------
# BBB / Rank-1 — reference: src/algos/util.py:151-186, src/algos/bbb.py
# --------------------------------------------------------------------------------------


def softplus(rho):
    return torch.nn.functional.softplus(rho)


def gauss_sample_fwd(mu, rho, eps, dtype=torch.float32):
    """util.py:170-171: mean + normal_like(std) * std."""
    return mu.to(dtype) + eps.to(dtype) * softplus(rho.to(dtype))


def gauss_sample_bwd(grad_w, rho, eps, dtype=torch.float32):
    """Autograd of gauss_sample_fwd: returns (grad_mu, grad_rho)."""
    r = rho.to(dtype)
    return grad_w.to(dtype), grad_w.to(dtype) * eps.to(dtype) * torch.sigmoid(r)


def kl_gauss(mu, rho, prior_mu: float, prior_sigma: float, dtype=torch.float32):
    """bbb.py:18-21 through util.py:173-174.  Returns (value, grad_mu, grad_rho) (analytic)."""
    m, r = mu.to(dtype), rho.to(dtype)
    sigma = softplus(r)
    kl = 0.5 * (2 * torch.log(prior_sigma / sigma) - 1 + (sigma / prior_sigma).pow(2) + ((prior_mu - m) / prior_sigma).pow(2))
    g_mu = (m - prior_mu) / prior_sigma ** 2
    g_rho = (-1.0 / sigma + sigma / prior_sigma ** 2) * torch.sigmoid(r)
    return kl.to(torch.float64).sum(), g_mu, g_rho


def kl_mixture(mu, pi: float, sigma1: float, sigma2: float, dtype=torch.float32):
    """bbb.py:23-37.  Returns (value, grad_mu) with the gradient taken by autograd."""
    pit = torch.tensor(pi, dtype=dtype)

    def logp(v, s):
        return -(v ** 2) / (2 * s ** 2) - math.log(s) - math.log(math.sqrt(2 * math.pi))

    with torch.enable_grad():  # may be called from inside an autograd.Function (grad mode off)
        m = mu.detach().to(dtype).clone().requires_grad_(True)
        p1 = torch.log(pit) + torch.clamp(logp(m, sigma1), -23, 0)
        p2 = torch.log(1 - pit) + torch.clamp(logp(m, sigma2), -23, 0)
        val = -torch.logaddexp(p1, p2).to(torch.float64).sum()
        (g,) = torch.autograd.grad(val, m)
    return val.detach(), g


def l2_term(theta, l2_scale: float, dtype=torch.float32):
    """bbb.py:75-76.  Returns (value, grad)."""
    t = theta.to(dtype)
    return l2_scale / 2 * t.to(torch.float64).pow(2).sum(), l2_scale * t


# --------------------------------------------------------------------------------------
# Philox4x32-10 + Box-Muller (the library's noise stream), Salmon et al. 2011
# --------------------------------------------------------------------------------------

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)


def philox4x32_10(quads: np.ndarray, seed: int, stream_id: int) -> np.ndarray:
    """quads: uint64 [m] counter values -> uint32 [m, 4] (bit-exact with the CUDA library)."""
    q = quads.astype(np.uint64)
    c0 = (q & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    c1 = (q >> np.uint64(32)).astype(np.uint32)
    c2 = np.full_like(c0, np.uint32(stream_id & 0xFFFFFFFF))
    c3 = np.full_like(c0, np.uint32((stream_id >> 32) & 0xFFFFFFFF))
    k0, k1 = np.uint32(seed & 0xFFFFFFFF), np.uint32((seed >> 32) & 0xFFFFFFFF)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _M0 * c0.astype(np.uint64)
            p1 = _M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), p0.astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), p1.astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = np.uint32(k0 + _W0)
            k1 = np.uint32(k1 + _W1)
    return np.stack([c0, c1, c2, c3], axis=1)


def philox_normal(count: int, seed: int, stream_id: int, elem0: int = 0) -> np.ndarray:
    """Standard normals for global elements elem0 .. elem0+count-1 (elem0 % 4 == 0), fp32."""
    assert elem0 % 4 == 0
    nq = (count + 3) // 4
    r = philox4x32_10(np.arange(nq, dtype=np.uint64) + np.uint64(elem0 // 4), seed, stream_id)

    def bm(r0, r1):
        # the kernel's uniforms (common.cuh:box_muller): the low 23 bits x of a Philox word as the float 2^23 + x, one fp32 FMA each
        x0 = (r0 & np.uint32(0x7FFFFF)).astype(np.float64)
        x1 = (r1 & np.uint32(0x7FFFFF)).astype(np.float64)
        u = (2.0 * x0 + 1.0) * 2.0 ** -24                                   # exact in fp32, in (0, 1)
        k = float(np.float32(2.0 * np.pi * 2.0 ** -23))
        ang = ((2.0 ** 23 + x1) * k + float(np.float32(-3.0 * np.pi))).astype(np.float32).astype(np.float64)   # [-pi, pi)
        rad = np.sqrt(-2.0 * np.log(u))
        return rad * np.cos(ang), rad * np.sin(ang)

    z0, z1 = bm(r[:, 0], r[:, 1])
    z2, z3 = bm(r[:, 2], r[:, 3])
    return np.stack([z0, z1, z2, z3], axis=1).reshape(-1)[:count].astype(np.float32)


def bbb_linear_fwd(x, w_mu, w_rho, b_mu, b_rho, eps, mc_sample: float = 1.0, dtype=torch.float32):
    """BBBLinear.forward, sampling == "activations" (bbb_layers.py:61-88; the CPU branch :72-74 states the same
    arithmetic as the stacked baddbmm of the CUDA branch :66-71).  Returns (out, act_std)."""
    x, w_mu, w_rho, eps = x.to(dtype), w_mu.to(dtype), w_rho.to(dtype), eps.to(dtype)
    b_mean = b_mu.to(dtype) if b_mu is not None else None
    b_var = (F.softplus(b_rho.to(dtype)) ** 2).clamp(min=1e-4) if b_rho is not None else None
    mean = F.linear(x, w_mu, b_mean)
    var = F.linear((x ** 2).clamp(min=1e-4), (F.softplus(w_rho) ** 2).clamp(min=1e-4), b_var)
    std = torch.sqrt(var)
    return (mean + std * eps) / mc_sample, std


def rank1_linear_fwd(x, weight, s_mu, s_rho, r_mu, r_rho, bias, eps_s, eps_r, dtype=torch.float32):
    """Rank1Linear.forward (rank1.py:50-64) with GaussianParameter.sample (util.py:170-171) written out:
    s = s_mu + eps_s * softplus(s_rho), r likewise; out = linear(x * s, weight) * r (+ bias).  Returns (out, lin, s, r)."""
    c = lambda t: t.to(dtype)
    s = c(s_mu) + c(eps_s) * F.softplus(c(s_rho))
    r = c(r_mu) + c(eps_r) * F.softplus(c(r_rho))
    lin = F.linear(c(x) * s, c(weight))
    out = lin * r
    if bias is not None:
        out = out + c(bias).unsqueeze(0)
    return out, lin, s, r
