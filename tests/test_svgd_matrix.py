"""Exact-arithmetic matrix of every SVGD kernel instantiation and launch form.

Each particle count with a register-resident fast path (BDE_FOR_EACH_N in csrc/svgd.cu: n = 2..12, 16, 20) is its own
template instantiation with its own geometry (pair groups and slots, threads per CTA, ring depth, tile columns and
tile sets, transposed coefficient tables); every other n and every unaligned input runs the generic runtime-n
kernels.  Tolerance checks on Gaussian data cannot show that every pair landed in its own slot, so these tests feed
inputs whose correct output is known exactly:

* particles are integers in [-R, R]: differences, squares and every fp32 partial sum of K1 are exact integers as long
  as no fp32 value a warp accumulates between two fp64 flushes can reach 2^24 (`flush_windows`, `value_range`,
  checked without a GPU by `test_exact_inputs_are_exact_and_distinct`), and all n(n-1)/2 distances are distinct, so
  two swapped slots cannot cancel out.  The reference distances are exact fp64 sums of integers, computed on the
  device in column chunks by elementwise torch ops;
* K / A are multiples of 1/8 that are NOT symmetric: K G + A X is then exact in any summation order, so every K2 form
  must match the reference bit for bit, and an i/j mix-up in the transposed coefficient tables shows.

The large-offset tests (matrices of more than 2^31 elements) can be selected on their own with `-k large_offset`; they
skip, with the reason, when the GPU has too little free memory.
"""
from __future__ import annotations

import math
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import ATOL, RTOL
from oracle import bde_oracle as O

CSRC = Path(__file__).resolve().parent.parent / "beyond_deep_ensembles_b200" / "csrc"
FAST_N = [2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 16, 20]
GENERIC_N = [1, 13, 14, 15, 17, 18, 19, *range(21, 33)]
NEXT_MAX_N = 10                        # kNextDistMaxParticles: single-pass training-step form
SMALL_D = [3, 37, 4099, 70_001]        # below one quad, one tile, one ring; ragged everywhere
FP32_EXACT = 1 << 24                   # integers up to here are exact in fp32
MAX_RANGE = 64                         # particle values never exceed [-64, 64]
G_RANGE = 64                           # gradients: integers in [-64, 64] (no flush bound applies to K2)
COEF_EIGHTHS = 17                      # K / A entries: multiples of 1/8 with |value| <= 17/8
BW = (0.01, 1.0, 768.0)                # l2_reg, kernel_grad_scale, dataset_size of every K1b call
B200_SMS = 148


# ---------------------------------------------------------------------------------------------------- exact inputs
def _constant(name: str) -> int:
    """A `constexpr int` of the SVGD kernel sources."""
    for f in ("svgd_kernels.cuh", "svgd_gram.cuh"):
        m = re.search(rf"constexpr\s+int\s+{name}\s*=\s*(\d+)\s*;", (CSRC / f).read_text())
        if m:
            return int(m.group(1))
    raise LookupError(name)


def flush_windows() -> dict:
    """Columns whose squared differences (Gram form: products of centred rows) one warp sums in fp32 before they
    are flushed to fp64: 32 lanes x one column quad per lane and iteration / tile x the flush period, plus the
    ragged tail (< 4 columns) that joins the last period.  None: the form has no periodic flush (the direct
    training-step kernel keeps its partials until the end, so its window is every column a warp sees, <= D)."""
    quad_warp = 32 * 4
    return {
        "direct K1": quad_warp * _constant("kFlushIters") + 4,
        "staged K1": quad_warp * _constant("kFlushTiles") + 4,
        "Gram K1": quad_warp * _constant("kGramFlushTiles"),
        "staged training step": quad_warp * _constant("kFlushTiles") + 4,
        "direct training step": None,
    }


def value_range(D: int) -> int:
    """Largest R (<= MAX_RANGE) for which min(D, window) * (2R)^2 < 2^24 for every flushing K1 form."""
    w = min(D, max(v for v in flush_windows().values() if v is not None))
    return min(MAX_RANGE, math.isqrt((FP32_EXACT - 1) // w) // 2)


def direct_next_is_exact(D: int) -> bool:
    """The direct training-step kernel never flushes: exact only while all D columns fit the fp32 bound."""
    return D * (2 * value_range(D)) ** 2 < FP32_EXACT


def exact_pairdist(X: torch.Tensor, chunk: int = 1 << 22) -> torch.Tensor:
    """[n, n] fp64 sums of squared differences on X's device.  For integer X every partial sum is an integer below
    2^53, so the result is exact whatever the order (elementwise ops only, no library call)."""
    n, D = X.shape
    d = torch.zeros(n, n, dtype=torch.float64, device=X.device)
    for c0 in range(0, D, chunk):
        x = X[:, c0:c0 + chunk].double()
        for i in range(n - 1):
            d[i, i + 1:] += ((x[i + 1:] - x[i]) ** 2).sum(1)
    return d + d.T


def _first_duplicate(d: torch.Tensor):
    n = d.shape[0]
    iu = torch.triu_indices(n, n, 1)
    vals = d[iu[0], iu[1]]
    order = torch.sort(vals, stable=True).indices
    same = (vals[order[1:]] == vals[order[:-1]]).nonzero()
    if same.numel() == 0:
        return None
    p = int(order[int(same[0]) + 1])
    return int(iu[0, p]), int(iu[1, p])


def exact_particles(n: int, D: int, seed: int, device="cpu") -> torch.Tensor:
    """Integer-valued fp32 particles [n, D] in [-R, R] (R = value_range(D)) whose n(n-1)/2 squared pair distances
    are pairwise distinct.  Random draws first; then, while two distances coincide, one entry of one of the two
    particles is redrawn and the distances are updated exactly."""
    R = value_range(D)
    g = torch.Generator(device=device).manual_seed(seed)
    X = torch.randint(-R, R + 1, (n, D), generator=g, device=device, dtype=torch.int32).float()
    d = exact_pairdist(X).cpu()
    rng = np.random.default_rng(seed)
    for _ in range(200 * n * n + 10):
        dup = _first_duplicate(d)
        if dup is None:
            return X
        r = dup[int(rng.integers(2))]
        c, v = int(rng.integers(D)), float(rng.integers(-R, R + 1))
        col = X[:, c].double().cpu()
        delta = (v - col) ** 2 - (col[r] - col) ** 2
        delta[r] = 0.0
        d[r, :] += delta
        d[:, r] += delta
        X[r, c] = v
    raise AssertionError(f"no distinct distances for n={n}, D={D}")


def exact_gradients(n: int, D: int, seed: int, device="cpu") -> torch.Tensor:
    g = torch.Generator(device=device).manual_seed(seed + 1)
    return torch.randint(-G_RANGE, G_RANGE + 1, (n, D), generator=g, device=device, dtype=torch.int32).float()


def dyadic_coefficients(n: int, seed: int):
    """K, A: multiples of 1/8 in [-17/8, 17/8] with K_ij != K_ji and A_ij != A_ji for every i != j."""
    g = torch.Generator().manual_seed(seed + 2)
    mats = []
    for _ in range(2):
        m = torch.randint(-16, 17, (n, n), generator=g).float()
        upper = torch.triu(torch.ones(n, n, dtype=torch.bool), 1)
        m[upper & (m == m.T)] += 1.0
        mats.append(m / 8.0)
    return mats


def exact_apply_chunks(X, G, K, A, chunk: int = 1 << 22):
    """(column slice, exact K G + A X in fp64) over X's device, chunk by chunk (elementwise ops only)."""
    n, D = X.shape
    Kd, Ad = K.double().to(X.device), A.double().to(X.device)
    for c0 in range(0, D, chunk):
        sl = slice(c0, min(D, c0 + chunk))
        x, g = X[:, sl].double(), G[:, sl].double()
        ref = torch.zeros_like(x)
        for j in range(n):
            ref += Kd[:, j:j + 1] * g[j] + Ad[:, j:j + 1] * x[j]
        yield sl, ref


def assert_apply_exact(out, X, G, K, A, what):
    for sl, ref in exact_apply_chunks(X, G, K, A):
        got = out[:, sl].double()
        if not torch.equal(got, ref):
            bad = (got != ref).nonzero()[0].tolist()
            raise AssertionError(f"{what}: K2 differs from the exact result at row {bad[0]}, column {sl.start + bad[1]}: "
                                 f"{got[bad[0], bad[1]].item()} != {ref[bad[0], bad[1]].item()}")


def wrap_columns(sm_count: int) -> int:
    """D at which every persistent CTA wraps its ring at least twice: (2 x deepest ring + 1) tiles per CTA of the
    widest tile.  Rings: pd_stages / apply_stages cap at 8 stages, the Gram ring holds up to 12 stages of 256
    columns; the widest tile is K1's 1024 columns at one pair group (pd_tile_cols).  Plus an odd remainder."""
    return sm_count * max((2 * 8 + 1) * 1024, (2 * 12 + 1) * 256) + 4 * 257 + 3


def alt_tile_sets(n: int, opt: bool, nxt: bool) -> int:
    """The `apply_tile_sets` value that selects the staged K2's alternative geometry (launch_apply_opt: TS_ALT)."""
    small = n > 12 or (nxt and n >= 9) or (not opt and n >= 8)
    rolled = n > 16 or (n == 16 and opt)
    ts0 = 1 if not small else (4 if rolled else 3)
    return 3 if not small else (7 - ts0 if n > 12 else 1)


def test_exact_inputs_are_exact_and_distinct():
    """No GPU: the value range keeps every fp32 partial sum of K1 exact for every D of this file, the K2 sums fit
    fp32 in units of 1/8, and the generator gives pairwise distinct distances for every n it is used with."""
    windows = flush_windows()
    assert windows["direct K1"] >= windows["staged K1"] > 4 and windows["Gram K1"] > 0
    all_d = SMALL_D + [wrap_columns(B200_SMS), 230_000_003, 115_000_001, 1000, 2051]
    for D in all_d:
        R = value_range(D)
        assert R >= 1, D
        for name, w in windows.items():
            if w is not None:
                assert min(D, w) * (2 * R) ** 2 < FP32_EXACT, (name, D, R)
        # K2: |sum| <= 2 n * 17/8 * max(R, G_RANGE), counted in eighths, for the largest n
        assert 2 * 32 * COEF_EIGHTHS * max(R, G_RANGE) < FP32_EXACT
    assert direct_next_is_exact(3) and direct_next_is_exact(4099) and not direct_next_is_exact(70_001)
    for n in sorted(set(FAST_N + GENERIC_N)):
        for D in (3, 37, 4099):
            X = exact_particles(n, D, seed=n * 1000 + D)
            R = value_range(D)
            assert torch.equal(X, X.round()) and X.abs().max() <= R
            d = exact_pairdist(X)
            iu = torch.triu_indices(n, n, 1)
            vals = d[iu[0], iu[1]]
            assert vals.unique().numel() == vals.numel(), (n, D)
            assert torch.equal(d, O.svgd_pairdist(X)), (n, D)
    X = exact_particles(20, 70_001, seed=5)
    vals = exact_pairdist(X)[torch.triu_indices(20, 20, 1).unbind()]
    assert vals.unique().numel() == vals.numel()
    # the oracle's cdist round trip squares the correctly rounded sqrt by one multiplication, as the kernel does
    # (torch.sqrt on a CPU float64 tensor can be one ulp off for this value)
    d = torch.tensor([[0.0, 11000313.0], [11000313.0, 0.0]], dtype=torch.float64)
    r = math.sqrt(11000313.0)
    assert O.svgd_bandwidth(d, *BW)["d_hi"] == r * r
    K, A = dyadic_coefficients(9, 3)
    off = ~torch.eye(9, dtype=torch.bool)
    assert (K != K.T)[off].all() and (A != A.T)[off].all()
    assert torch.equal(K * 8, (K * 8).round()) and K.abs().max() <= COEF_EIGHTHS / 8


# ---------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def ops(cuda_lib):
    from beyond_deep_ensembles_b200 import ops as _ops
    return _ops


@pytest.fixture
def tune(cuda_lib):
    """bde_tune(key, value) for this test; every key it set goes back to 0 (automatic) on teardown."""
    keys = set()

    def set_(key: str, value: int):
        keys.add(key)
        assert cuda_lib.bde_tune(key.encode(), int(value)) == 0, key
    yield set_
    for k in keys:
        cuda_lib.bde_tune(k.encode(), 0)


def sm_count() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


def resolve_D(D):
    return wrap_columns(sm_count()) if D == "wrap" else D


def nan_like(x: torch.Tensor, layout: str = "aligned") -> torch.Tensor:
    """A NaN-filled [n, D] GPU matrix: `aligned` rows padded to a multiple of 4 (fast paths), `odd-ld` a row stride
    that is not a multiple of 4, `misaligned` a 16-byte aligned stride on a base 4 bytes off (both: generic kernels)."""
    n, D = x.shape
    ld = (D + 3) // 4 * 4
    mis = 0
    if layout == "odd-ld":
        ld = D + 1 if (D + 1) % 4 else D + 2
    elif layout == "misaligned":
        mis = 1
    buf = torch.full((n * ld + mis + 4,), float("nan"), device="cuda")
    return torch.as_strided(buf, (n, D), (ld, 1), storage_offset=mis)


def on_device(x: torch.Tensor, layout: str = "aligned") -> torch.Tensor:
    """Copy [n, D] to the GPU in one of the layouts of nan_like."""
    view = nan_like(x, layout)
    view.copy_(x)
    return view


def state_vec(D: int, layout: str) -> torch.Tensor:
    mis = 1 if layout == "misaligned" else 0
    return torch.zeros(D + 8, device="cuda")[mis:mis + D]


def standalone_bandwidth(ops, dist: torch.Tensor):
    """K1b alone (bde_svgd_bandwidth) on the given distances: (K, A, info, sel)."""
    sc = ops.SvgdScratch.allocate(dist.shape[0], "cuda")
    sc.dist.copy_(dist)
    ops.svgd_bandwidth(sc, *BW)
    return sc.K.clone(), sc.A.clone(), sc.info.clone(), sc.sel.clone()


def assert_same_bandwidth(sc, ref, what):
    for name, got, want in zip(("K", "A", "info", "sel"), (sc.K, sc.A, sc.info, sc.sel), ref):
        assert torch.equal(got, want), f"{what}: K1b {name} differs from the standalone K1b on the same distances"


def assert_bandwidth_matches_oracle(ref, dist, what):
    K, A, info, sel = (t.cpu() for t in ref)
    bw = O.svgd_bandwidth(dist.cpu(), *BW)
    assert tuple(sel.tolist()) == bw["sel"], what
    assert info[1].item() == bw["median"], f"{what}: median {info[1].item()!r} != {bw['median']!r}"
    assert info[2].item() == bw["d_lo"] and info[3].item() == bw["d_hi"], what
    np.testing.assert_allclose(info[0].item(), bw["h"], rtol=1e-6, err_msg=what)
    np.testing.assert_allclose(K.numpy(), bw["K"].numpy(), rtol=1e-5, atol=1e-7, err_msg=what)
    np.testing.assert_allclose(A.numpy(), bw["A"].numpy(), rtol=1e-5, atol=1e-9, err_msg=what)


SGD = ("sgd", dict(lr=1e-3, momentum=0.9, dampening=0.0, weight_decay=1e-2, nesterov=True))
ADAM = ("adam", dict(lr=1e-2, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2))
ADAMW = ("adamw", dict(lr=1e-2, betas=(0.9, 0.999), eps=1e-8, weight_decay=5e-2))
SGD_FROZEN = ("sgd", dict(lr=0.0, momentum=0.0, dampening=0.0, weight_decay=0.0, nesterov=False))


def fused_step(ops, opt, dX, dG, sc, D, layout, next_kernel=None):
    """One K2f launch (one optimizer step per particle, fresh state); returns (state0, state1, out_last)."""
    kind, h = opt
    s0, s1, last = state_vec(D, layout), state_vec(D, layout), state_vec(D, layout)
    if kind == "sgd":
        ops.svgd_apply_sgd(dX, dG, sc, s0 if h["momentum"] else None, buf_initialized=False, out_last=last,
                           next_kernel=next_kernel, **h)
    else:
        ops.svgd_apply_adam(dX, dG, sc, s0, s1, step0=0, lr=h["lr"], beta1=h["betas"][0], beta2=h["betas"][1],
                            eps=h["eps"], weight_decay=h["weight_decay"], decoupled_weight_decay=(kind == "adamw"),
                            out_last=last, next_kernel=next_kernel)
    return s0, s1, last


def check_fused(X0, G, K, A, dX, last, opt, what):
    """out_last is the exact K2 row n-1 bit for bit; X matches the optimizer oracle fed with the exact K2 output."""
    n = X0.shape[0]
    out = torch.empty_like(X0)
    for sl, ref in exact_apply_chunks(X0, G, K, A):
        out[:, sl] = ref.float()
    assert torch.equal(last, out[n - 1]), f"{what}: out_last differs from the exact K2 row n-1"
    x_ref, _ = O.svgd_base_optimizer_steps(X0, out, opt[0], opt[1], None)
    got = dX.detach().clone()
    torch.testing.assert_close(got, x_ref, rtol=RTOL, atol=5 * ATOL, msg=lambda m: f"{what}: {m}")


# ---------------------------------------------------------------------------------------------------- K1 (+ K1b)
CASES = [(n, D) for n in FAST_N for D in SMALL_D + ["wrap"]]


def _k1_forms(ops, tune, X, dX, n, variants, what):
    ref = exact_pairdist(X)
    ref_bw = standalone_bandwidth(ops, ref)
    assert_bandwidth_matches_oracle(ref_bw, ref, what)
    for v in variants:
        tune("pairdist_variant", v)
        sc = ops.SvgdScratch.allocate(n, "cuda")
        tag = f"{what}, pairdist_variant {v}"
        if v != 3:   # the Gram form exists only with K1b fused
            ops.svgd_pairdist(dX, sc)
            assert torch.equal(sc.dist, ref), f"{tag}: distances differ from the exact sums"
            first = sc.dist.clone()
            ops.svgd_pairdist(dX, sc)
            assert torch.equal(sc.dist, first), f"{tag}: a second launch changed the bits"
            ops.svgd_pairdist(dX, sc, accumulate=True)
            assert torch.equal(sc.dist, 2 * ref), f"{tag}: accumulate"
        sc = ops.SvgdScratch.allocate(n, "cuda")
        ops.svgd_pairdist_bandwidth(dX, sc, *BW)
        assert torch.equal(sc.dist, ref), f"{tag}: fused distances differ from the exact sums"
        assert_same_bandwidth(sc, ref_bw, tag)
        if v == 3 and X.shape[1] >= 4099:
            assert not sc.exact_redo(), f"{tag}: the Gram guard sent the case to the direct kernel"
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("n,D", CASES)
def test_pairdist_exact(ops, tune, n, D):
    """K1 direct and staged (and the centred Gram form at n = 16 / 20): plain, accumulate (2 x exact) and with K1b
    fused, bit for bit against the exact sums; the fused K1b bit for bit against K1b alone on the same distances."""
    D = resolve_D(D)
    X = exact_particles(n, D, seed=n * 7919 + D, device="cuda")
    _k1_forms(ops, tune, X, on_device(X), n, [1, 2] + ([3] if n in (16, 20) else []), f"n={n} D={D}")


# ---------------------------------------------------------------------------------------------------- K2 / K2f
def _apply_forms(n, opt: bool, nxt: bool = False):
    """(apply_variant, apply_tile_sets) of every K2 geometry: direct, staged default, staged alternative."""
    return [(1, 0), (2, 0), (2, alt_tile_sets(n, opt, nxt))]


@pytest.mark.gpu
@pytest.mark.parametrize("n,D", CASES)
def test_apply_exact(ops, tune, n, D):
    """Plain K2 with non-symmetric dyadic K / A: every form (direct, staged in both tile geometries, automatic) is
    bit for bit the exact K G + A X."""
    D = resolve_D(D)
    X = exact_particles(n, D, seed=n * 31 + D, device="cuda")
    G = exact_gradients(n, D, seed=n * 31 + D, device="cuda")
    K, A = dyadic_coefficients(n, seed=n + D)
    dX, dG = on_device(X), on_device(G)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    sc.K.copy_(K)
    sc.A.copy_(A)
    for v, ts in _apply_forms(n, False) + [(0, 0)]:
        tune("apply_variant", v)
        tune("apply_tile_sets", ts)
        out = nan_like(X)
        ops.svgd_apply(dX, dG, out, sc)
        assert_apply_exact(out, X, G, K, A, f"n={n} D={D} apply_variant {v} tile_sets {ts}")


@pytest.mark.gpu
@pytest.mark.parametrize("opt", [SGD, ADAM, ADAMW], ids=["sgd-nesterov-wd", "adam", "adamw"])
@pytest.mark.parametrize("n,D", CASES)
def test_fused_apply_exact(ops, tune, n, D, opt):
    """K2f (K2 + n shared-state optimizer steps) in every form: out_last is the exact K2 row n-1 bit for bit, the
    particles match the optimizer oracle fed with the exact K2 output."""
    D = resolve_D(D)
    X = exact_particles(n, D, seed=n * 37 + D, device="cuda")
    G = exact_gradients(n, D, seed=n * 37 + D, device="cuda")
    K, A = dyadic_coefficients(n, seed=2 * n + D)
    dG = on_device(G)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    sc.K.copy_(K)
    sc.A.copy_(A)
    for v, ts in _apply_forms(n, True):
        tune("apply_variant", v)
        tune("apply_tile_sets", ts)
        dX = on_device(X)
        _, _, last = fused_step(ops, opt, dX, dG, sc, D, "aligned")
        check_fused(X, G, K, A, dX, last, opt, f"n={n} D={D} {opt[0]} apply_variant {v} tile_sets {ts}")


# ---------------------------------------------------------------------------------------------------- training step
TRAIN_CASES = [(n, D) for n in FAST_N if n <= NEXT_MAX_N for D in SMALL_D + ["wrap"]]


def _train_step(ops, n, D, X, G, K, A, opt, fuse, layout="aligned"):
    dX, dG = on_device(X, layout), on_device(G, layout)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    sc.K.copy_(K)
    sc.A.copy_(A)
    _, _, last = fused_step(ops, opt, dX, dG, sc, D, layout, next_kernel=ops.NextKernel(fuse, *BW))
    return dX, sc, last


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", [True, False], ids=["k1b", "no-k1b"])
@pytest.mark.parametrize("n,D", TRAIN_CASES)
def test_train_step_exact(ops, tune, n, D, fuse):
    """Training-step form (K2f + the next step's K1, optionally K1b, in one launch), direct and staged in both
    geometries.  lr = 0 leaves the integer particles in place, so the next-step distances must be the exact sums
    (the direct form only while D fits its single fp32 window); with real SGD / Adam steps they match fp64
    distances of the returned particles to 2e-6.  The fused K1b is bit for bit K1b alone on the distances the launch
    left; without it K / A stay untouched."""
    D = resolve_D(D)
    X = exact_particles(n, D, seed=n * 41 + D, device="cuda")
    G = exact_gradients(n, D, seed=n * 41 + D, device="cuda")
    K, A = dyadic_coefficients(n, seed=3 * n + D)
    ref = exact_pairdist(X)
    for v, ts in _apply_forms(n, True, True):
        tune("apply_variant", v)
        tune("apply_tile_sets", ts)
        for opt in (SGD_FROZEN, SGD, ADAM):
            what = f"n={n} D={D} {opt[0]} lr={opt[1]['lr']} apply_variant {v} tile_sets {ts}"
            dX, sc, last = _train_step(ops, n, D, X, G, K, A, opt, fuse)
            check_fused(X, G, K, A, dX, last, opt, what)
            if opt is SGD_FROZEN:
                assert torch.equal(dX, X), what
                if v == 2 or direct_next_is_exact(D):
                    assert torch.equal(sc.dist, ref), f"{what}: next-step distances differ from the exact sums"
                else:
                    torch.testing.assert_close(sc.dist, ref, rtol=2e-6, atol=1e-12)
            else:
                torch.testing.assert_close(sc.dist, exact_pairdist(dX), rtol=2e-6, atol=1e-12,
                                           msg=lambda m: f"{what}: {m}")
            if fuse:
                assert_same_bandwidth(sc, standalone_bandwidth(ops, sc.dist), what)
            else:
                assert torch.equal(sc.K.cpu(), K) and torch.equal(sc.A.cpu(), A), what


# ---------------------------------------------------------------------------------------------------- generic paths
GENERIC_CASES = ([(n, D, "aligned") for n in GENERIC_N for D in (3, 4099)]
                 + [(n, D, lay) for n in FAST_N for D in (37, 4099) for lay in ("odd-ld", "misaligned")])


@pytest.mark.gpu
@pytest.mark.parametrize("n,D,layout", GENERIC_CASES)
def test_generic_paths_exact(ops, tune, n, D, layout):
    """Runtime-n kernels (n without a fast path, or any n on an unaligned layout): K1 plain / accumulate / fused,
    K2, K2f and the two-launch training-step fallback on the same exact inputs."""
    what = f"n={n} D={D} {layout}"
    X = exact_particles(n, D, seed=n * 53 + D, device="cuda")
    G = exact_gradients(n, D, seed=n * 53 + D, device="cuda")
    K, A = dyadic_coefficients(n, seed=5 * n + D)
    dX = on_device(X, layout)
    ref = _k1_forms(ops, tune, X, dX, n, [0], what)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    sc.K.copy_(K)
    sc.A.copy_(A)
    out = nan_like(X, layout)
    ops.svgd_apply(dX, on_device(G, layout), out, sc)
    assert_apply_exact(out, X, G, K, A, what)
    for opt in (SGD, ADAM):
        dXf = on_device(X, layout)
        _, _, last = fused_step(ops, opt, dXf, on_device(G, layout), sc, D, layout)
        check_fused(X, G, K, A, dXf, last, opt, f"{what} {opt[0]}")
    for fuse in (True, False):
        dXn, scn, last = _train_step(ops, n, D, X, G, K, A, SGD_FROZEN, fuse, layout)
        assert torch.equal(dXn, X) and torch.equal(scn.dist, ref), f"{what}: training-step fallback distances"
        if fuse:
            assert_same_bandwidth(scn, standalone_bandwidth(ops, ref), f"{what}: training-step fallback")


# ---------------------------------------------------------------------------------------------------- K1b in every host
def tie_particles(n: int, case: str, D: int = 37) -> torch.Tensor:
    """duplicate: exact particles with copies (exact zero off-diagonal distances); equidistant: X_i = 3 e_i, every
    off-diagonal distance is 18."""
    if case == "equidistant":
        X = torch.zeros(n, max(D, n))
        X[range(n), range(n)] = 3.0
        return X
    X = exact_particles(n, D, seed=n)
    if n >= 2:
        X[1] = X[0]
    if n >= 4:
        X[n - 1] = X[n // 2]
    return X


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["distinct", "duplicate", "equidistant"])
@pytest.mark.parametrize("n", list(range(1, 33)))
def test_bandwidth_in_every_host(ops, tune, n, case):
    """K1b runs standalone and as the tail of the direct K1, the staged K1, the Gram K1 (n = 16 / 20), the generic K1
    (+ standalone K1b) and the training-step kernel: all must leave the same K, A, info and sel bit for bit.  On tie-
    heavy distances the median selection and the median itself must equal the oracle's exactly."""
    X = tie_particles(n, case) if case != "distinct" else exact_particles(n, 37, seed=n + 99)
    Xd = X.cuda()
    ref = exact_pairdist(Xd)
    ref_bw = standalone_bandwidth(ops, ref)
    assert_bandwidth_matches_oracle(ref_bw, ref, f"n={n} {case}")
    fast = n in FAST_N
    hosts = [(0, "odd-ld")] + ([(1, "aligned"), (2, "aligned")] if fast else [(0, "aligned")])
    if n in (16, 20):
        hosts.append((3, "aligned"))
    for v, layout in hosts:
        tune("pairdist_variant", v)
        sc = ops.SvgdScratch.allocate(n, "cuda")
        ops.svgd_pairdist_bandwidth(on_device(Xd, layout), sc, *BW)
        assert torch.equal(sc.dist, ref), f"n={n} {case} pairdist_variant {v} {layout}: distances"
        assert_same_bandwidth(sc, ref_bw, f"n={n} {case} pairdist_variant {v} {layout}")
    if 2 <= n <= NEXT_MAX_N:
        D = Xd.shape[1]
        G = exact_gradients(n, D, seed=n, device="cuda")
        K, A = dyadic_coefficients(n, seed=n)
        for v in (1, 2):
            tune("apply_variant", v)
            dXn, scn, _ = _train_step(ops, n, D, Xd, G, K, A, SGD_FROZEN, True)
            assert torch.equal(scn.dist, ref), f"n={n} {case} training step apply_variant {v}: distances"
            assert_same_bandwidth(scn, ref_bw, f"n={n} {case} training step apply_variant {v}")


# ---------------------------------------------------------------------------------------------------- past 2^31 elements
def need_free_memory(nbytes: int):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 2**30:.0f} GiB of free GPU memory, {free / 2**30:.0f} GiB free")


@pytest.mark.gpu
def test_large_offset_svgd_n10(ops, tune):
    """n = 10 x D = 230,000,003 (2.3e9 elements per matrix): K1 + K1b, automatic K2 (n * ld is past the limit where
    plain K2 switches its tile geometry), K2 forced to the direct kernel, K2f SGD and the training step, each
    checked over the whole vector."""
    n, D = 10, 230_000_003
    elems = n * ((D + 3) // 4 * 4)
    need_free_memory(4 * elems * 4 + 8 * (1 << 22) * n * 6 + (4 << 30))
    X = on_device(exact_particles(n, D, seed=1, device="cuda"))
    G = on_device(exact_gradients(n, D, seed=1, device="cuda"))
    torch.cuda.empty_cache()
    K, A = dyadic_coefficients(n, seed=1)
    ref = exact_pairdist(X)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist_bandwidth(X, sc, *BW)
    assert torch.equal(sc.dist, ref)
    assert_same_bandwidth(sc, standalone_bandwidth(ops, ref), "n=10 large")
    sc.K.copy_(K)
    sc.A.copy_(A)
    out = nan_like(X)
    # automatic (n * ld > kApplySmallTileMaxElems: the 1 x 512 geometry), staged forced to its 3 x 256 default, direct
    for v, ts in ((0, 0), (2, 3), (1, 0)):
        tune("apply_variant", v)
        tune("apply_tile_sets", ts)
        out.fill_(float("nan"))
        ops.svgd_apply(X, G, out, sc)
        assert_apply_exact(out, X, G, K, A, f"n=10 large apply_variant {v} tile_sets {ts}")
    tune("apply_variant", 0)
    tune("apply_tile_sets", 0)
    del out
    # K2f SGD on a copy of X (same padded layout), against the exact K2 of the original chunk by chunk
    X_new = on_device(X)
    kind, h = SGD
    buf, last = torch.zeros(D, device="cuda"), torch.zeros(D, device="cuda")
    ops.svgd_apply_sgd(X_new, G, sc, buf, buf_initialized=False, out_last=last, **h)
    for sl, ref_out in exact_apply_chunks(X, G, K, A):
        assert torch.equal(last[sl], ref_out[n - 1].float())
        x_ref, _ = O.svgd_base_optimizer_steps(X[:, sl], ref_out.float(), kind, h, None)
        torch.testing.assert_close(X_new[:, sl], x_ref, rtol=RTOL, atol=5 * ATOL)
    # training step (automatic form) on the updated particles: next-step distances of what it returns
    del X
    buf.zero_()
    ops.svgd_apply_sgd(X_new, G, sc, buf, buf_initialized=False, out_last=last,
                       next_kernel=ops.NextKernel(True, *BW), **h)
    torch.testing.assert_close(sc.dist, exact_pairdist(X_new), rtol=2e-6, atol=1e-12)
    assert_same_bandwidth(sc, standalone_bandwidth(ops, sc.dist), "n=10 large training step")


@pytest.mark.gpu
def test_large_offset_svgd_n20_gram(ops, tune):
    """n = 20 x D = 115,000,001 (2.3e9 elements): the centred-Gram K1 with K1b, and K2, over the whole vector."""
    n, D = 20, 115_000_001
    elems = n * ((D + 3) // 4 * 4)
    need_free_memory(3 * elems * 4 + 8 * (1 << 22) * n * 6 + (4 << 30))
    X = on_device(exact_particles(n, D, seed=2, device="cuda"))
    G = on_device(exact_gradients(n, D, seed=2, device="cuda"))
    torch.cuda.empty_cache()
    K, A = dyadic_coefficients(n, seed=2)
    ref = exact_pairdist(X)
    tune("pairdist_variant", 3)
    sc = ops.SvgdScratch.allocate(n, "cuda")
    ops.svgd_pairdist_bandwidth(X, sc, *BW)
    assert not sc.exact_redo()
    assert torch.equal(sc.dist, ref)
    assert_same_bandwidth(sc, standalone_bandwidth(ops, ref), "n=20 large Gram")
    sc.K.copy_(K)
    sc.A.copy_(A)
    out = nan_like(X)
    ops.svgd_apply(X, G, out, sc)
    assert_apply_exact(out, X, G, K, A, "n=20 large")


@pytest.mark.gpu
def test_large_offset_swag(ops):
    """SWAG with K = 10 and D = 240,000,007: ring row 9 starts past element 2^31.  K + 2 updates (the ring wraps)
    bit-exact against the fp32 oracle on a column sample that includes the first and last columns of every row, and
    one draw on the same columns."""
    K, D = 10, 240_000_007
    assert (K - 1) * D > 2**31
    need_free_memory((K + 6) * D * 4 + (2 << 30))
    g = torch.Generator(device="cuda").manual_seed(7)
    mean = torch.randn(D, device="cuda", generator=g) * 0.3
    sq = mean * mean + 0.01 * torch.rand(D, device="cuda", generator=g)
    ring = torch.zeros(K, D, device="cuda")
    cols = torch.randint(0, D, (4096,), generator=torch.Generator().manual_seed(1))
    cols = torch.unique(torch.cat([cols, torch.arange(64), torch.arange(D - 64, D)]))
    cd = cols.cuda()
    m_ref, s_ref = mean[cd].cpu(), sq[cd].cpu()
    ring_ref = torch.zeros(K, cols.numel())
    for updates in range(1, K + 3):
        theta = mean + 0.05 * torch.randn(D, device="cuda", generator=g)
        ops.swag_update(theta, mean, sq, ring[(updates - 1) % K], updates)
        m_ref, s_ref, col = O.swag_update(theta[cd].cpu(), m_ref, s_ref, updates)
        ring_ref[(updates - 1) % K] = col
        del theta
    assert torch.equal(mean[cd].cpu(), m_ref) and torch.equal(sq[cd].cpu(), s_ref)
    assert torch.equal(ring[:, cd].cpu(), ring_ref)
    eps_k = torch.randn(K, generator=torch.Generator().manual_seed(5))
    eps_d = torch.randn(D, device="cuda", generator=g)
    out = torch.empty(D, device="cuda")
    ops.swag_sample(mean, sq, ring, updates % K, out, eps_k=eps_k.cuda(), eps_d=eps_d)
    ref = O.swag_sample(m_ref, s_ref, O.swag_ring_to_reference(ring_ref, updates), eps_k, eps_d[cd].cpu(),
                        dtype=torch.float64)
    np.testing.assert_allclose(out[cd].cpu().numpy(), ref.numpy(), rtol=RTOL, atol=ATOL)
