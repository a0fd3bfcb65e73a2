"""SVGD with 33 to 64 particles: the particle-tiled K1 (+K1b) and K2 of csrc/svgd_many.cu, the C-ABI routing and
refusals, and SVGDOptimizer above 32 particles.

Exact-arithmetic inputs come from tests/test_svgd_matrix.py.  Its value range keeps every fp32 partial sum exact for
the widest flush window of the older K1 forms; the tiled K1 sums 256 * kManyFlushTiles columns of one pair in fp32
before it flushes to fp64, which `test_many_flush_window_fits_the_exact_inputs` checks against that window, so the
generator carries over unchanged.
"""
from __future__ import annotations

import copy
import ctypes as C
import re
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

import golden_models as gm
from conftest import ATOL, RTOL
from oracle import bde_oracle as O
from test_svgd_matrix import (BW, CSRC, FP32_EXACT, G_RANGE, COEF_EIGHTHS, assert_apply_exact,
                              assert_bandwidth_matches_oracle, assert_same_bandwidth, dyadic_coefficients,
                              exact_apply_chunks, exact_gradients, exact_pairdist, exact_particles, flush_windows,
                              nan_like, need_free_memory, on_device, standalone_bandwidth, tie_particles, value_range)

MANY_N = list(range(33, 65))
EXACT_D = [1, 255, 256, 257, 65_539, 4_194_311]
BDE_ERR_INVALID_ARG, BDE_ERR_ALIGNMENT, BDE_ERR_UNSUPPORTED_N = -1, -2, -4


def _many_constant(name: str) -> int:
    m = re.search(rf"constexpr\s+int\s+{name}\s*=\s*(\d+)\s*;", (CSRC / "svgd_many.cu").read_text())
    return int(m.group(1))


# ---------------------------------------------------------------------------------------------------- CPU checks
def test_many_flush_window_fits_the_exact_inputs():
    """The tiled K1's fp32 window (all columns of a tile, kManyFlushTiles tiles) is no wider than the widest window
    value_range() already provides for, and the K2 sums at n = 64 stay exact in eighths."""
    window = 256 * _many_constant("kManyFlushTiles")   # kManyPdTC = kTmaBoxCols = 256 columns per tile
    assert window <= max(w for w in flush_windows().values() if w is not None)
    for D in EXACT_D + [34_000_001]:
        assert min(D, window) * (2 * value_range(D)) ** 2 < FP32_EXACT
    assert 2 * 64 * COEF_EIGHTHS * max(value_range(1), G_RANGE) < FP32_EXACT


def test_many_kernels_sass():
    """The new kernels are built for sm_100a with tensor-map TMA loads (UTMALDG.2D) and packed FP32 (FFMA2)."""
    from beyond_deep_ensembles_b200 import build_ext
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not Path(cuobjdump).exists():
        pytest.skip("cuobjdump not found")
    lib = build_ext.build(verbose=False)
    sass = subprocess.run([cuobjdump, "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    funcs = {}
    for chunk in re.split(r"\n\s*Function : ", sass)[1:]:
        funcs[chunk.split("\n", 1)[0].strip()] = chunk
    for kernel in ("svgd_pairdist_many_kernel", "svgd_apply_many_kernel"):
        body = [b for name, b in funcs.items() if kernel in name]
        assert len(body) == 1, kernel
        assert "UTMALDG.2D" in body[0], kernel
        assert "FFMA2" in body[0], kernel
        assert "STL" not in body[0] and "LDL" not in body[0], f"{kernel}: local-memory spills"


# ---------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def ops(cuda_lib):
    from beyond_deep_ensembles_b200 import ops as _ops
    return _ops


def many_particles(n: int, D: int, seed: int) -> torch.Tensor:
    """Exact integer particles; at D = 1 no n > 32 particles in [-64, 64] can have distinct distances, so there the
    draws are plain (ties cannot hide a swapped slot when every slot is checked against the exact sum anyway)."""
    if D == 1:
        g = torch.Generator(device="cuda").manual_seed(seed)
        return torch.randint(-value_range(1), value_range(1) + 1, (n, 1), generator=g, device="cuda").float()
    return exact_particles(n, D, seed=seed, device="cuda")


def k1_exact(ops, X, dX, n, what):
    """K1 plain / again / accumulate, K1 + K1b fused, against the exact sums; fused K1b against standalone K1b."""
    ref = exact_pairdist(X)
    ref_bw = standalone_bandwidth(ops, ref)
    assert_bandwidth_matches_oracle(ref_bw, ref, what)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist(dX, sc)
    assert torch.equal(sc.dist, ref), f"{what}: distances differ from the exact sums"
    ops.svgd_pairdist(dX, sc)
    assert torch.equal(sc.dist, ref), f"{what}: a second launch changed the bits"
    ops.svgd_pairdist(dX, sc, accumulate=True)
    assert torch.equal(sc.dist, 2 * ref), f"{what}: accumulate"
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist_bandwidth(dX, sc, *BW)
    assert torch.equal(sc.dist, ref), f"{what}: fused distances"
    assert_same_bandwidth(sc, ref_bw, what)
    return ref, ref_bw


def k2_exact(ops, X, G, n, seed, what):
    """K2 on dyadic K / A, alone and armed behind a K1 launch (programmatic dependent launch), bit for bit."""
    K, A = dyadic_coefficients(n, seed)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    out = nan_like(X)
    sc.K.copy_(K)
    sc.A.copy_(A)
    ops.svgd_apply(X, G, out, sc)
    assert_apply_exact(out, X, G, K, A, f"{what}, K2 alone")
    # chained: K1 (distances only, so K / A keep the dyadic values) directly followed by the armed K2
    out.fill_(float("nan"))
    ops.svgd_pairdist(X, sc)
    ops.svgd_chain_next(X)
    ops.svgd_apply(X, G, out, sc)
    assert_apply_exact(out, X, G, K, A, f"{what}, K2 chained behind K1")


# ---------------------------------------------------------------------------------------------------- exact matrix
@pytest.mark.gpu
@pytest.mark.parametrize("D", EXACT_D)
@pytest.mark.parametrize("n", MANY_N)
def test_many_exact(ops, n, D):
    """Every n in 33..64 at D from one column to ~4 M (ragged tiles, one tile, several rings): K1, K1 accumulate,
    K1 + K1b fused and standalone K1b, and K2 (armed and not), bit for bit against the exact results."""
    X = many_particles(n, D, seed=n * 7919 + D)
    dX = on_device(X)
    k1_exact(ops, X, dX, n, f"n={n} D={D}")
    G = on_device(exact_gradients(n, D, seed=n + D, device="cuda"))
    k2_exact(ops, dX, G, n, n + D, f"n={n} D={D}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [33, 64])
def test_many_sliced_columns_emulate_d_sharding(ops, n):
    """D-sharding emulated on one GPU: K1 with accumulate over 2, 3 and 5 column slices (16-byte aligned starts),
    then K1b, equals the whole-matrix result bit for bit."""
    D = 70_001
    X = exact_particles(n, D, seed=n + 5, device="cuda")
    dX = on_device(X)
    ref = exact_pairdist(X)
    ref_bw = standalone_bandwidth(ops, ref)
    for parts in (2, 3, 5):
        bounds = [min(D, (D * k // parts + 3) // 4 * 4) for k in range(parts)] + [D]
        sc = ops.SvgdScratch.allocate(n, "cuda")
        for k, (a, b) in enumerate(zip(bounds, bounds[1:])):
            ops.svgd_pairdist(dX[:, a:b], sc, accumulate=k > 0)
        assert torch.equal(sc.dist, ref), f"n={n}: {parts} slices"
        ops.svgd_bandwidth(sc, *BW)
        assert_same_bandwidth(sc, ref_bw, f"n={n}: {parts} slices")


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["duplicate", "equidistant"])
def test_many_ties_n64(ops, case):
    """Duplicate and equidistant particles at n = 64: median selection indices and median equal the oracle's,
    from the standalone K1b and from K1's tail."""
    n = 64
    X = tie_particles(n, case).cuda()
    ref = exact_pairdist(X)
    ref_bw = standalone_bandwidth(ops, ref)
    assert_bandwidth_matches_oracle(ref_bw, ref, f"n=64 {case}")
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist_bandwidth(on_device(X), sc, *BW)
    assert torch.equal(sc.dist, ref)
    assert_same_bandwidth(sc, ref_bw, f"n=64 {case} fused")


# ---------------------------------------------------------------------------------------------------- against the oracle
@pytest.mark.gpu
@pytest.mark.parametrize("D", [65_539, 20_000_000])
@pytest.mark.parametrize("n", [33, 48, 64])
def test_many_against_oracle(ops, n, D):
    """Seeded C5-style inputs (distinct per-particle scales): distances within 2e-6 relative of fp64, median selection
    identical, h / K / A within the fp32 tolerance, K2 within rtol 1e-5 / atol 1e-6 of the fp64 product."""
    g = torch.Generator(device="cuda").manual_seed(n * 31 + D)
    scale = 0.05 * (1 + 0.1 * torch.arange(n, dtype=torch.float32, device="cuda")).unsqueeze(1)
    X = on_device(scale * torch.randn(n, D, generator=g, device="cuda"))
    G = on_device(1e-3 * torch.randn(n, D, generator=g, device="cuda"))
    d_ref = exact_pairdist(X)   # fp64 sums of fp64 squares of exact differences
    sc = ops.SvgdScratch.allocate(n, "cuda")
    out = nan_like(X)
    ops.svgd_step(X, G, out, sc, *BW)
    np.testing.assert_allclose(sc.dist.cpu().numpy(), d_ref.cpu().numpy(), rtol=2e-6, atol=1e-12)
    bw = O.svgd_bandwidth(d_ref.cpu(), *BW)
    assert tuple(sc.sel.tolist()) == bw["sel"]
    np.testing.assert_allclose(sc.info[0].item(), bw["h"], rtol=1e-6)
    np.testing.assert_allclose(sc.K.cpu().numpy(), bw["K"].numpy(), rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(sc.A.cpu().numpy(), bw["A"].numpy(), rtol=RTOL, atol=ATOL)
    for sl, ref in exact_apply_chunks(X, G, bw["K"].double(), bw["A"].double()):
        torch.testing.assert_close(out[:, sl].double(), ref, rtol=RTOL, atol=ATOL)


# ---------------------------------------------------------------------------------------------------- past 2^31 elements
@pytest.mark.gpu
def test_large_offset_svgd_n64(ops):
    """n = 64 x D = 34,000,001 (2.2e9 elements per matrix): K1 + K1b and K2, each checked over the whole matrix."""
    n, D = 64, 34_000_001
    elems = n * ((D + 3) // 4 * 4)
    need_free_memory(3 * elems * 4 + 8 * (1 << 22) * n * 6 + (4 << 30))
    X = on_device(exact_particles(n, D, seed=3, device="cuda"))
    G = on_device(exact_gradients(n, D, seed=3, device="cuda"))
    torch.cuda.empty_cache()
    ref = exact_pairdist(X)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist_bandwidth(X, sc, *BW)
    assert torch.equal(sc.dist, ref)
    assert_same_bandwidth(sc, standalone_bandwidth(ops, ref), "n=64 large")
    K, A = dyadic_coefficients(n, seed=3)
    sc.K.copy_(K)
    sc.A.copy_(A)
    out = nan_like(X)
    ops.svgd_apply(X, G, out, sc)
    assert_apply_exact(out, X, G, K, A, "n=64 large")


# ---------------------------------------------------------------------------------------------------- SVGDOptimizer
SGD_H = dict(lr=1e-2, momentum=0.9, nesterov=True, weight_decay=1e-3)
ADAM_H = dict(lr=1e-3)


def build_many(n: int, base_cls, hyper: dict, seed: int = 0):
    from beyond_deep_ensembles_b200 import SVGDOptimizer
    torch.manual_seed(seed)
    model = gm.make_mlp().cuda()
    inits = [torch.cat([p.detach().reshape(-1) for p in gm.make_mlp().parameters()]).numpy() for _ in range(n - 1)]
    k = {"k": 0}

    def reset():
        gm.load_flat(model.parameters(), inits[k["k"]])
        k["k"] += 1

    base = base_cls(model.parameters(), **hyper)
    opt = SVGDOptimizer(model.parameters(), reset, base, particle_count=n, dataset_size=768, l2_reg=0.01,
                        kernel_grad_scale=1.0)
    return model, opt


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sgd", "adam"])
@pytest.mark.parametrize("n", [40, 64])
def test_many_optimizer_steps_match_reference(ops, monkeypatch, n, kind):
    """Three SVGDOptimizer steps at n = 40 / 64 with a shared SGD (momentum, Nesterov, weight decay) or Adam base
    optimizer: each step equals the reference op sequence (fp64) on the same particles and gradients followed by the
    reference's n base-optimizer steps.  Only K1 + K1b and K2 are called: no fused, training-step or host entry."""
    from beyond_deep_ensembles_b200 import _lib
    base_cls, hyper = (torch.optim.SGD, SGD_H) if kind == "sgd" else (torch.optim.Adam, ADAM_H)
    model, opt = build_many(n, base_cls, hyper, seed=n)
    assert opt._plan_for(opt.get_base_optimizer(), None, list(opt._params())) is None
    calls = []
    real_call = _lib.call
    monkeypatch.setattr(_lib, "call", lambda name, *a: (calls.append(name), real_call(name, *a))[1])
    g = torch.Generator().manual_seed(n)
    state = {}
    for s in range(3):
        x = torch.randn(64, 8, generator=g).cuda()
        y = torch.randn(64, generator=g).cuda()
        X0 = opt._X.detach().clone()
        fwd, bwd = gm.mse_closures(model, x, y)
        opt.step(fwd, bwd)
        new_grads = O.svgd_step_reference_order(X0.cpu(), opt._G.detach().cpu(), 0.01, 1.0, 768, dtype=torch.float64)
        X_ref, state = O.svgd_base_optimizer_steps(X0.cpu(), new_grads.float(), kind, hyper, state)
        np.testing.assert_allclose(opt._X.detach().cpu().numpy(), X_ref.numpy(), rtol=3e-5, atol=3e-6,
                                   err_msg=f"step {s}")
    used = set(calls)
    assert {"bde_svgd_pairdist_bandwidth", "bde_svgd_apply"} <= used, used
    refused = {c for c in used if re.match(r"bde_svgd_(apply_sgd|apply_adam|train_step|host|step_host)", c)}
    assert not refused, refused


@pytest.mark.gpu
def test_many_state_dict_roundtrip_n64(ops):
    n = 64
    model, opt = build_many(n, torch.optim.Adam, ADAM_H, seed=1)
    x, y = torch.randn(32, 8).cuda(), torch.randn(32).cuda()
    opt.step(*gm.mse_closures(model, x, y))
    sd = copy.deepcopy(opt.state_dict())
    assert set(sd["state"][0].keys()) == {f"particle_{i}" for i in range(n)}
    model2, opt2 = build_many(n, torch.optim.Adam, ADAM_H, seed=2)
    opt2.load_state_dict(sd)
    assert torch.equal(opt._X, opt2._X)
    assert opt2.state[next(iter(opt2._params()))]["particle_0"].data_ptr() == opt2._xviews[0][0].data_ptr()


# ---------------------------------------------------------------------------------------------------- refusals
@pytest.mark.gpu
def test_many_particle_count_65_raises(ops):
    with pytest.raises(ValueError):
        build_many(65, torch.optim.SGD, dict(lr=1e-2))


@pytest.mark.gpu
def test_many_abi_refusals(cuda_lib):
    lib = cuda_lib
    D = 1024
    X = torch.zeros(65, D + 8, device="cuda")
    G, out = torch.zeros_like(X), torch.zeros_like(X)
    dist = torch.zeros(65 * 65, dtype=torch.float64, device="cuda")
    K, A = torch.zeros(65 * 65, device="cuda"), torch.zeros(65 * 65, device="cuda")
    info, sel = torch.zeros(4, dtype=torch.float64, device="cuda"), torch.zeros(2, dtype=torch.int32, device="cuda")
    nbytes = C.c_size_t(0)
    assert lib.bde_svgd_workspace_bytes(65, C.byref(nbytes)) == BDE_ERR_INVALID_ARG
    assert lib.bde_svgd_workspace_bytes(64, C.byref(nbytes)) == 0
    ws = torch.zeros(nbytes.value // 8 + 1, dtype=torch.float64, device="cuda")
    p = lambda t: t.data_ptr()
    ld = D + 8
    # n = 65: out of range everywhere
    assert lib.bde_svgd_pairdist(p(X), 65, D, ld, p(dist), 0, p(ws), nbytes.value, None) == BDE_ERR_INVALID_ARG
    assert lib.bde_svgd_bandwidth(p(dist), 65, *BW, 0.0, p(K), p(A), p(info), p(sel), None) == BDE_ERR_INVALID_ARG
    assert lib.bde_svgd_apply(p(X), p(G), p(out), p(K), p(A), 65, D, ld, None) == BDE_ERR_INVALID_ARG
    assert lib.bde_svgd_step(p(X), p(G), p(out), 65, D, ld, *BW, 0.0, p(dist), p(K), p(A), p(info), p(sel), p(ws),
                             nbytes.value, None) == BDE_ERR_INVALID_ARG
    # n = 33: fused base-optimizer, training-step and host entries
    n = 33
    buf = torch.zeros(D, device="cuda")
    assert lib.bde_svgd_apply_sgd(p(X), p(G), p(K), p(A), n, D, ld, p(buf), 0, 1e-2, 0.9, 0.0, 0.0, 0, None,
                                  None) == BDE_ERR_UNSUPPORTED_N
    assert lib.bde_svgd_apply_adam(p(X), p(G), p(K), p(A), n, D, ld, p(buf), p(buf), 0, 1e-3, 0.9, 0.999, 1e-8,
                                   0.0, 0, None, None) == BDE_ERR_UNSUPPORTED_N
    assert lib.bde_svgd_train_step_sgd(p(X), p(G), p(K), p(A), n, D, ld, p(buf), 0, 1e-2, 0.9, 0.0, 0.0, 0, None,
                                       p(dist), 1, *BW, 0.0, p(K), p(A), p(info), p(sel), p(ws), nbytes.value,
                                       None) == BDE_ERR_UNSUPPORTED_N
    assert lib.bde_svgd_train_step_adam(p(X), p(G), p(K), p(A), n, D, ld, p(buf), p(buf), 0, 1e-3, 0.9, 0.999, 1e-8,
                                        0.0, 0, None, p(dist), 1, *BW, 0.0, p(K), p(A), p(info), p(sel), p(ws),
                                        nbytes.value, None) == BDE_ERR_UNSUPPORTED_N
    Xh = torch.zeros(n, D)
    dX = torch.zeros(n, D, device="cuda")
    stage = torch.zeros(2 * n * 256, device="cuda")
    assert lib.bde_svgd_host_pairdist(p(Xh), n, D, D, 256, p(dX), p(dist), p(ws), nbytes.value) == BDE_ERR_UNSUPPORTED_N
    assert lib.bde_svgd_host_apply(p(Xh), p(Xh), n, D, D, *BW, 0.0, 256, p(dX), p(stage), p(stage), p(dist), p(K),
                                   p(A), p(info), p(sel), None, None) == BDE_ERR_UNSUPPORTED_N
    assert lib.bde_svgd_step_host(p(Xh), p(Xh), p(Xh), n, D, D, *BW, 0.0, 256, p(dX), p(stage), p(stage), p(dist),
                                  p(K), p(A), p(info), p(sel), p(ws), nbytes.value, None, None) == BDE_ERR_UNSUPPORTED_N
    # n = 40: a base pointer 4 bytes off, or a row stride that is not a multiple of 4
    n = 40
    off = X.data_ptr() + 4
    assert lib.bde_svgd_pairdist(off, n, D, ld, p(dist), 0, p(ws), nbytes.value, None) == BDE_ERR_ALIGNMENT
    assert lib.bde_svgd_pairdist(p(X), n, D, ld - 1, p(dist), 0, p(ws), nbytes.value, None) == BDE_ERR_ALIGNMENT
    assert lib.bde_svgd_apply(p(X), p(G), out.data_ptr() + 4, p(K), p(A), n, D, ld, None) == BDE_ERR_ALIGNMENT
    assert lib.bde_svgd_apply(off, p(G), p(out), p(K), p(A), n, D, ld, None) == BDE_ERR_ALIGNMENT
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_many_attached_workspace_refused(cuda_lib):
    """K1 above 32 particles refuses a workspace attached to a peer set of two ranks (the in-kernel exchange
    carries at most 496 sums) instead of returning rank-local sums; detached, the same workspace works again.  The
    refusal comes before any launch, so one exchange buffer standing in for both ranks is enough."""
    lib, n, D = cuda_lib, 40, 1024
    nbytes = C.c_size_t(0)
    assert lib.bde_svgd_workspace_bytes(n, C.byref(nbytes)) == 0
    assert nbytes.value <= 256 + 8 * 256 * (n * (n - 1) // 2)   # sized for the tiled K1's grid, not the direct K1's
    ws = torch.zeros(nbytes.value // 8 + 1, dtype=torch.float64, device="cuda")
    X = torch.ones(n, D, device="cuda")
    dist = torch.zeros(n * n, dtype=torch.float64, device="cuda")
    buf, handle = C.c_void_p(), C.create_string_buffer(64)
    assert lib.bde_peer_alloc(C.byref(buf), handle) == 0
    try:
        bufs = (C.c_uint64 * 2)(buf.value, buf.value)
        assert lib.bde_peer_attach(ws.data_ptr(), nbytes.value, 2, 0, bufs, 1.0, None, None) == 0
        rc = lib.bde_svgd_pairdist(X.data_ptr(), n, D, D, dist.data_ptr(), 0, ws.data_ptr(), nbytes.value, None)
        assert rc == BDE_ERR_UNSUPPORTED_N
        assert lib.bde_peer_detach(ws.data_ptr(), nbytes.value, None) == 0
        assert lib.bde_svgd_pairdist(X.data_ptr(), n, D, D, dist.data_ptr(), 0, ws.data_ptr(), nbytes.value, None) == 0
        torch.cuda.synchronize()
        assert torch.equal(dist, torch.zeros_like(dist))
    finally:
        torch.cuda.synchronize()
        lib.bde_peer_free(buf)


@pytest.mark.gpu
@pytest.mark.parametrize("n,D", [(40, 501), (64, 1000)])
def test_many_rbf(ops, n, D):
    """bde.rbf above 32 particles, also on a row length that is not a multiple of 4: kernel matrix and its gradient
    against the fp64 oracle."""
    from beyond_deep_ensembles_b200 import rbf
    g = torch.Generator().manual_seed(n + D)
    scale = 0.05 * (1 + 0.1 * torch.arange(n, dtype=torch.float32)).unsqueeze(1)
    X = scale * torch.randn(n, D, generator=g)
    K, grad = rbf(X.cuda())
    bw = O.svgd_bandwidth(O.svgd_pairdist(X), 0.0, 1.0, 1.0)
    np.testing.assert_allclose(K.cpu().numpy(), bw["K"].numpy(), rtol=RTOL, atol=ATOL)
    ref = -(bw["A"].double() @ X.double())
    np.testing.assert_allclose(grad.cpu().numpy(), ref.numpy(), rtol=RTOL, atol=ATOL * max(1.0, ref.abs().max().item()))
