"""Mixed precision for D-sharded jobs: torch's ShardedGradScaler over the optimizer's ranks.

Each rank checks only its own columns for non-finite gradients.  The bar: a sharded run with a ShardedGradScaler
equals the unsharded run with a plain GradScaler, in every scenario of tests/sharded_scaler_script.py, although the
planted inf gradient reaches one rank only: the same skipped base-optimizer steps, the same `get_scale()` trajectory,
bit-identical concatenated slices for the elementwise family (SWAG, iVON, BBB) where the gradients are exact, SVGD
to fp32 rounding.  gloo + the oracle-backed ABI double in spawned ranks; on one GPU the ranks are emulated one after
the other over the real kernels; NCCL with two GPUs."""
from __future__ import annotations

import math
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import fake_abi
import sharded_scaler_script as script


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _same(a, b):
    """Bit-identical, NaN where NaN (iVON loses the planted column: it never skips its update)."""
    return a.shape == b.shape and torch.equal(torch.nan_to_num(a, nan=7.0, posinf=8.0, neginf=9.0),
                                              torch.nan_to_num(b, nan=7.0, posinf=8.0, neginf=9.0)) \
        and torch.equal(a.isnan(), b.isnan())


def compare(parts, full, concat: bool, exact):
    """parts: one result dict per rank; concat: the vectors are the ranks' slices (else every rank holds them
    whole); exact(algo) -> bit-identical or fp32 rounding."""
    assert parts[0].keys() == full.keys()
    for algo, want in full.items():
        for r, p in enumerate(parts):
            assert p[algo]["scales"] == want["scales"], f"{algo}: rank {r} scale trajectory"
            assert p[algo]["base_steps"] == want["base_steps"], f"{algo}: rank {r} skipped other base steps"
        # the planted overflow was caught: one step backed the scale off
        assert any(b < a for a, b in zip([script.INIT_SCALE] + want["scales"], want["scales"])), algo
        for key, vec in want.items():
            if key in ("scales", "base_steps"):
                continue
            got = [torch.cat([p[algo][key] for p in parts], dim=1)] if concat else [p[algo][key] for p in parts]
            for g in got:
                if exact(algo):
                    assert _same(g, vec), f"{algo}.{key} differs from the unsharded run"
                else:   # NaN where NaN here too
                    np.testing.assert_allclose(g.numpy(), vec.numpy(), rtol=2e-5, atol=2e-6, err_msg=f"{algo}.{key}")


def spawn(tmp_path, world, backend, mode):
    out_path = str(tmp_path / f"{mode}{world}")
    mp.spawn(script.worker, args=(world, free_port(), out_path, backend, mode), nprocs=world, join=True)
    return [torch.load(f"{out_path}.{r}") for r in range(world)]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_grad_scaler_gloo(tmp_path, monkeypatch, world):
    torch.set_num_threads(1)
    fake_abi.install(monkeypatch)
    cpu = torch.device("cpu")
    slices, wrapped = script.run_slices(cpu, 1, 0, None, False), script.run_wrapped(cpu, 1, 0, None, False)
    parts = spawn(tmp_path, world, "gloo", "agree")
    compare([p["slices"] for p in parts], slices, True, lambda algo: not algo.startswith("svgd"))
    # ColumnShardedModel averages R equal gradients: exact at R = 2 only
    compare([p["wrapped"] for p in parts], wrapped, False, lambda algo: world == 2 and not algo.startswith("svgd"))


def test_sharded_optimizers_accept_only_a_sharded_scaler_over_their_ranks_gloo(tmp_path):
    """Optimizer over ranks {0, 1} of a 3-rank job: a plain GradScaler, a ShardedGradScaler over the whole job and one
    over ranks {1, 2} are refused before anything changes; a ShardedGradScaler over another group object with the
    same ranks steps."""
    parts = spawn(tmp_path, 3, "gloo", "refuse")
    assert parts[2] == {}
    for res in parts[:2]:
        assert res["sharded_same_ranks"] == "ok"
        for name in ("plain", "sharded_world", "sharded_other_ranks"):
            assert "ShardedGradScaler over the same ranks" in res[name], name


def test_single_rank_jobs_keep_any_scaler(monkeypatch):
    """A one-rank job (no process group) keeps its plain GradScaler path: no check, no collective."""
    torch.set_num_threads(1)
    fake_abi.install(monkeypatch)
    monkeypatch.setattr(dist, "all_reduce", lambda *a, **k: pytest.fail("collective in a one-rank job"))
    out = script.run_slices(torch.device("cpu"), 1, 0, None, False)
    assert out["swag"]["base_steps"] == [1, 0, 1, 1] and out["svgd_fused"]["base_steps"] == [4, 0, 4]


# ---------------------------------------------------------------------------------------------------- one GPU
class _FakeGroup:
    def __init__(self, world, rank):
        self.world, self.rank = world, rank


class _Collectives:
    """torch.distributed.all_reduce for ranks emulated one after the other in one process, as a fixed point: each
    round runs every rank and records the local input of each of its all-reduces; the next round answers call k with
    the reduction (SUM / MAX) over the ranks' inputs to call k in the previous round.  Once the inputs stop changing,
    every rank ran with the true reductions — the closed form of the group's collectives."""

    def __init__(self, world):
        self.world, self.prev, self.rank = world, None, 0
        self.rec = [[] for _ in range(world)]

    def all_reduce(self, tensor, op=dist.ReduceOp.SUM, group=None, async_op=False):
        k = len(self.rec[self.rank])
        self.rec[self.rank].append(tensor.detach().clone())
        if self.prev is not None and all(k < len(p) for p in self.prev):
            stack = torch.stack([p[k].to(tensor.device) for p in self.prev])
            tensor.copy_(stack.amax(0) if op == dist.ReduceOp.MAX else stack.sum(0))

        class _Done:
            def wait(self):
                return True
        return _Done() if async_op else None

    def next_round(self) -> bool:
        """True when this round's inputs equal the previous round's (converged)."""
        same = self.prev is not None and all(len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
                                             for a, b in zip(self.rec, self.prev))
        self.prev, self.rec = self.rec, [[] for _ in range(self.world)]
        return same


def _emulated_parts(dev, world, monkeypatch):
    from beyond_deep_ensembles_b200 import bbb as bbb_mod
    from beyond_deep_ensembles_b200 import dist as bdist
    from beyond_deep_ensembles_b200.layout import shard_bounds

    def fake_column_shard(local_size, group=None):
        lo, hi = shard_bounds(script.D_GLOBAL, group.world, group.rank)
        assert hi - lo == local_size
        return bdist.ColumnShard(group, group.world, group.rank, lo, local_size, script.D_GLOBAL, script.SEED)

    def fake_place(self):
        lo, _ = shard_bounds(script.D_GLOBAL, self._group.world, self._group.rank)
        for param in self._params():
            owner = getattr(getattr(param, "get_parameter_kl", None), "__self__", None)
            if owner is not None and getattr(owner, "mean", None) is param:
                owner.column_offset, owner.noise_seed = lo, script.SEED

    coll = _Collectives(world)
    monkeypatch.setenv("BDE_PEER_EXCHANGE", "0")
    monkeypatch.setattr(bdist, "column_shard", fake_column_shard)
    monkeypatch.setattr(bdist, "world", lambda group=None: group.world if isinstance(group, _FakeGroup) else 1)
    monkeypatch.setattr(bbb_mod.BBBOptimizer, "_place_gaussian_slices", fake_place)
    monkeypatch.setattr(dist, "all_reduce", coll.all_reduce)
    for _ in range(16):
        parts = []
        for r in range(world):
            coll.rank = r
            parts.append(script.run_slices(dev, world, r, _FakeGroup(world, r), True))
        if coll.next_round():
            return parts
    pytest.fail("the emulated collectives did not reach a fixed point")


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_grad_scaler_emulated_on_one_gpu(cuda_lib, monkeypatch, world):
    """R ranks' slices one after the other on cuda:0 through the real kernels; only torch.distributed.all_reduce
    (pair distances, BBB's prior value, the scaler's and the fused gather's found_inf) is replaced by its closed form."""
    dev = torch.device("cuda", 0)
    full = script.run_slices(dev, 1, 0, None, False)
    parts = _emulated_parts(dev, world, monkeypatch)
    compare(parts, full, True, lambda algo: not algo.startswith("svgd"))


@pytest.mark.gpu
def test_one_rank_sharded_grad_scaler_equals_the_plain_scaler(cuda_lib, tmp_path):
    """A one-rank process group on cuda:0 (NCCL): ShardedGradScaler's collectives run for real and change nothing."""
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    plain = {"slices": script.run_slices(dev, 1, 0, None, False), "wrapped": script.run_wrapped(dev, 1, 0, None, False)}
    dist.init_process_group("nccl", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1, device_id=dev)
    try:
        g = dist.group.WORLD
        sharded = {"slices": script.run_slices(dev, 1, 0, g, True), "wrapped": script.run_wrapped(dev, 1, 0, g, True)}
        torch.cuda.synchronize()
    finally:
        dist.destroy_process_group()
    for family in ("slices", "wrapped"):
        for algo, want in plain[family].items():
            for key, vec in want.items():
                got = sharded[family][algo][key]
                assert got == vec if isinstance(vec, list) else _same(got, vec), f"{family}.{algo}.{key}"


@pytest.mark.gpu
def test_sharded_grad_scaler_autocast_nccl(tmp_path):
    """NCCL x 2, ColumnShardedModel, fp16 autocast in the forward closure: sharded SWAG and SVGD against the unsharded
    run with a plain GradScaler, one planted one-rank overflow each."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    full = script.run_wrapped(torch.device("cuda", 0), 1, 0, None, False, algos=("swag", "svgd"), autocast=True)
    parts = spawn(tmp_path, 2, "nccl", "autocast")
    for algo, want in full.items():
        for p in parts:
            got = p["wrapped"][algo]
            assert got["scales"] == want["scales"] and got["base_steps"] == want["base_steps"], algo
            for key, vec in want.items():
                if key not in ("scales", "base_steps"):
                    np.testing.assert_allclose(got[key].numpy(), vec.numpy(), rtol=1e-4, atol=1e-5, err_msg=algo)
    assert math.isclose(full["swag"]["scales"][1], full["swag"]["scales"][0] / 2)   # step 2 backed off
