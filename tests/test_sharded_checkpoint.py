"""Checkpoints of D-sharded training (`ColumnShardedModel.full_state_dict` / `load_full_state_dict`).

The bar: a sharded job's full state dict is the dict the plain class returns when it runs the same steps on the whole
model (keys, indices, shapes, dtypes, devices, values), on every rank the same; a job saved at R ranks and resumed at
another R continues as the uninterrupted job does — particles, moments, base-optimizer state and SWAG's next Philox draw.
Values are bit-exact where the sharded-closure suite already promises it (SWAG / iVON when the ranks see the same batch
and R is 1 or 2: averaging two equal gradients is exact), otherwise equal to fp32 rounding (SVGD's n x n distance sums,
the mean of three gradients).  gloo + the oracle-backed ABI double here, the CUDA library on a B200, NCCL on two."""
from __future__ import annotations

import copy
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import fake_abi
import sharded_checkpoint_script as script

RTOL, ATOL = 2e-5, 2e-6      # the sharded-closure suite's tolerance


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def assert_same(got, want, exact, devices=True, path="sd"):
    """`got` has `want`'s structure, keys, shapes, dtypes (and devices) and values — `__base_optimizer` excepted: a
    full dict carries None there, a plain one the optimizer object."""
    if isinstance(want, dict):
        assert isinstance(got, dict) and set(got) == set(want), f"{path}: keys {sorted(map(str, got))} vs {sorted(map(str, want))}"
        for k in want:
            if k == "__base_optimizer":
                assert got[k] is None or isinstance(got[k], torch.optim.Optimizer), path
                continue
            assert_same(got[k], want[k], exact, devices, f"{path}[{k!r}]")
    elif torch.is_tensor(want):
        assert torch.is_tensor(got), path
        assert got.shape == want.shape and got.dtype == want.dtype, f"{path}: {got.shape} {got.dtype} vs {want.shape} {want.dtype}"
        if devices:
            assert got.device == want.device, f"{path}: {got.device} vs {want.device}"
        if exact:
            assert torch.equal(got.cpu(), want.cpu()), f"{path} differs"
        else:
            np.testing.assert_allclose(got.cpu().numpy(), want.cpu().numpy(), rtol=RTOL, atol=ATOL, err_msg=path)
    elif isinstance(want, (list, tuple)):
        assert type(got) is type(want) and len(got) == len(want), path
        for i, (g, w) in enumerate(zip(got, want)):
            assert_same(g, w, exact, devices, f"{path}[{i}]")
    else:
        assert got == want, f"{path}: {got!r} vs {want!r}"


def exact_for(case, *worlds):
    return not case.startswith("svgd") and all(w <= 2 for w in worlds)


# ---------------------------------------------------------------------- spawned jobs (gloo, CPU double)
_RUNS = {}


def spawn(tmp_path, world, backend, mode, ckpt=None):
    """Every rank's exported dicts of a `world`-rank job (mode "save", or "resume" from the host dict `ckpt`)."""
    out_path = str(tmp_path / f"{mode}{world}")
    ckpt_path = None
    if ckpt is not None:
        ckpt_path = str(tmp_path / f"ckpt_for_{mode}{world}")
        torch.save(script.to_cpu(ckpt), ckpt_path)
    mp.spawn(script.worker, args=(world, free_port(), out_path, backend, mode, ckpt_path), nprocs=world, join=True)
    return [torch.load(f"{out_path}.{r}") for r in range(world)]


@pytest.fixture
def cpu_double(monkeypatch):
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    fake_abi.install(monkeypatch)
    yield torch.device("cpu")
    torch.set_num_threads(threads)


@pytest.fixture
def plain(cpu_double):
    """The uninterrupted plain run (in process, on the CPU double)."""
    if "plain" not in _RUNS:
        _RUNS["plain"] = script.uninterrupted(cpu_double)
    return _RUNS["plain"]


def saved(tmp_path_factory, world):
    """The checkpoint of a `world`-rank gloo job after STEPS steps: one dict per rank."""
    if ("save", world) not in _RUNS:
        _RUNS[("save", world)] = spawn(tmp_path_factory.mktemp(f"save{world}"), world, "gloo", "save")
    return _RUNS[("save", world)]


@pytest.mark.parametrize("world", [2, 3])
def test_full_state_dict_equals_the_unsharded_twin_gloo(tmp_path_factory, plain, world):
    parts = saved(tmp_path_factory, world)
    for case in script.CASES:
        want = plain["ckpt"][case]
        for r, part in enumerate(parts):
            got = part[case]
            assert_same(got["sd"], want["sd"], exact_for(case, world), path=f"{case} rank {r}")
            if want["bsd"] is not None:
                assert_same(got["bsd"], want["bsd"], exact_for(case, world), path=f"{case} base rank {r}")
            # every rank exported the same dict
            assert_same(got, parts[0][case], True, path=f"{case} rank {r} vs rank 0")
        assert parts[0][case]["sd"]["state"].get("__base_optimizer", None) is None


@pytest.mark.parametrize("src,dst", [(1, 2), (2, 3), (3, 1), (2, 1), (1, 3), (3, 2)])
def test_resume_at_another_rank_count_gloo(tmp_path_factory, tmp_path, cpu_double, plain, src, dst):
    """Save after STEPS steps at R = src, resume at R = dst, STEPS more: the uninterrupted run's state and next SWAG
    draw.  R = 1 is the plain class on the whole model: its own state_dict() is the checkpoint, and its own
    load_state_dict() takes a full dict unchanged."""
    ckpt = plain["ckpt"] if src == 1 else saved(tmp_path_factory, src)[0]
    if dst == 1:
        res = [script.resume(cpu_double, copy.deepcopy(script.to_cpu(ckpt)))]
    else:
        res = spawn(tmp_path, dst, "gloo", "resume", ckpt)
    for case in script.CASES:
        want = plain["final"][case]
        exact = exact_for(case, src, dst)
        for r, part in enumerate(res):
            assert_same(part[case]["sd"], want["sd"], exact, path=f"{case} {src}->{dst} rank {r}")
            if want["bsd"] is not None:
                assert_same(part[case]["bsd"], want["bsd"], exact, path=f"{case} base {src}->{dst} rank {r}")
            if case == "swag":      # Philox continuity: the resumed job draws what the uninterrupted one draws
                assert_same(part[case]["sample"], want["sample"], exact, path=f"swag sample {src}->{dst} rank {r}")


# ---------------------------------------------------------------------- one rank, in process
def test_one_rank_job_loads_the_plain_checkpoint_and_rehomes_the_fused_base_state(cpu_double, plain):
    """A checkpoint written by the plain class loads into a one-rank sharded job.  SVGD's fused base-optimizer plan
    keeps momentum_buffer / exp_avg / exp_avg_sq as views of its arenas: a load replaces them with fresh tensors, and
    the next step's bind_state() copies them back into the arenas (the run still equals the uninterrupted one)."""
    for case in script.CASES:
        ckpt = plain["ckpt"][case]              # as the plain class wrote it, its base optimizer object included
        job = script.Job(case, cpu_double, wrap=True, weights=ckpt["weights"])
        job.load(ckpt["sd"], ckpt["bsd"])
        keys = {"svgd_sgd": ("momentum_buffer",), "svgd_adam": ("exp_avg", "exp_avg_sq")}.get(case, ())
        for key in keys:
            assert job.base.state[job.sm.param][key].numel() == job.sm.shard
        job.steps()
        if keys:
            plan = job.opt._fused_plan
            assert plan is not None and plan.base is job.base
            arenas = (plan.state0, plan.state1)
            for key, arena in zip(keys, arenas):
                assert job.base.state[job.sm.param][key].data_ptr() == arena.data_ptr(), key
        sd, bsd = job.export()
        want = plain["final"][case]
        assert_same(sd, want["sd"], not case.startswith("svgd"), path=case)
        if bsd is not None:
            assert_same(bsd, want["bsd"], not case.startswith("svgd"), path=f"{case} base")
        if case == "swag":
            assert_same(job.sample(), want["sample"], True, path="swag sample")


def _state(opt):
    return copy.deepcopy(script.to_cpu(opt.state_dict()))


def test_refusals_leave_the_optimizer_unchanged(cpu_double):
    import beyond_deep_ensembles_b200 as bde
    import golden_models as gm
    dev = cpu_double
    swag = script.Job("swag", dev, wrap=True)
    svgd = script.Job("svgd_sgd", dev, wrap=True)
    for job in (swag, svgd):
        job.steps(1)
    swag_sd, swag_bsd = swag.export()
    svgd_sd, svgd_bsd = svgd.export()

    def refused(job, sd, match, target=None):
        target = job.opt if target is None else target
        before, before_base = _state(job.opt), _state(job.base)
        with pytest.raises(ValueError, match=match):
            job.sm.load_full_state_dict(target, sd)
        assert_same(_state(job.opt), before, True)
        assert_same(_state(job.base), before_base, True)

    # another logical size: the checkpoint of a narrower model
    torch.manual_seed(0)
    small = gm.make_mlp(hidden=40)
    sm_small = bde.ColumnShardedModel(small)
    base_small = torch.optim.SGD([sm_small.param], lr=0.05, momentum=0.9)
    swag_small = bde.SwagOptimizer([sm_small.param], base_small, update_interval=1, deviation_samples=3)
    refused(swag, sm_small.full_state_dict(swag_small), "shape")
    # a parameter of another shape (same element count)
    bad = copy.deepcopy(svgd_sd)
    bad["state"][0] = {k: v.reshape(8, 50) for k, v in bad["state"][0].items()}
    refused(svgd, bad, "shape")
    # another particle_count / deviation_samples
    bad = copy.deepcopy(svgd_sd)
    bad["state"]["__particle_count"] = 3
    for k in range(4):
        del bad["state"][k]["particle_3"]
    refused(svgd, bad, "particle_count")
    bad = copy.deepcopy(swag_sd)
    bad["state"]["__deviations"] = bad["state"]["__deviations"][:, :2].contiguous()
    refused(swag, bad, "deviation_samples")
    # a base-optimizer dict of another shape into the base optimizer
    bad = copy.deepcopy(svgd_bsd)
    bad["state"][1]["momentum_buffer"] = bad["state"][1]["momentum_buffer"][:10]
    refused(svgd, bad, "shape", target=svgd.base)

    # optimizers that are not over [sm.param], and BBB
    twin = torch.optim.SGD(swag.model.parameters(), lr=0.1)
    with pytest.raises(ValueError, match=r"\[sm.param\]"):
        swag.sm.full_state_dict(twin)
    with pytest.raises(ValueError, match=r"\[sm.param\]"):
        swag.sm.load_full_state_dict(twin, swag_bsd)
    other = bde.ColumnShardedModel(gm.make_mlp())
    with pytest.raises(ValueError, match=r"\[sm.param\]"):
        other.full_state_dict(swag.opt)
    bbb = bde.BBBOptimizer.__new__(bde.BBBOptimizer)        # refused by its class, before anything is read
    with pytest.raises(ValueError, match="BBBOptimizer"):
        swag.sm.full_state_dict(bbb)
    with pytest.raises(ValueError, match="BBBOptimizer"):
        swag.sm.load_full_state_dict(bbb, swag_sd)

    # and the good dicts still load afterwards
    swag.load(swag_sd, swag_bsd)
    svgd.load(svgd_sd, svgd_bsd)


def test_plain_classes_keep_their_base_optimizer_on_a_full_dict(cpu_double):
    """A full dict carries `__base_optimizer = None`; the plain class that loads it keeps its own base optimizer."""
    plain = script.Job("svgd_adam", cpu_double)
    job = script.Job("svgd_adam", cpu_double, wrap=True)
    job.steps(1)
    sd, _ = job.export()
    plain.opt.load_state_dict(sd)
    assert plain.opt.get_base_optimizer() is plain.base


# ---------------------------------------------------------------------- the CUDA library
@pytest.mark.gpu
@pytest.mark.parametrize("case", script.CASES)
def test_one_rank_checkpoint_is_bit_exact_on_the_gpu(case):
    """One B200, one-rank ColumnShardedModel, the CUDA library (SVGD through the fused SGD / Adam plans), a loss whose
    gradient is elementwise: the full dict equals the plain twin's state_dict() bit for bit; a reload of it, and a
    load of the plain twin's own checkpoint, followed by STEPS more steps equal the uninterrupted run bit for bit."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from beyond_deep_ensembles_b200 import _lib
    _lib.get()
    dev = torch.device("cuda", 0)
    twin = script.Job(case, dev, elementwise=True)
    twin.steps()
    sd3, bsd3 = twin.export()
    weights = twin.weights()
    twin.steps()
    sd6, bsd6 = twin.export()
    sample6 = twin.sample() if case == "swag" else None

    job = script.Job(case, dev, wrap=True, elementwise=True)
    job.steps()
    f3, fb3 = job.export()
    assert_same(f3, sd3, True, path=f"{case} full")
    if bsd3 is not None:
        assert_same(fb3, bsd3, True, path=f"{case} base full")
    for label, (sd, bsd) in (("reload", (f3, fb3)), ("plain checkpoint", (sd3, bsd3))):
        job = script.Job(case, dev, wrap=True, weights=weights, elementwise=True)
        job.load(sd, bsd)
        job.steps()
        if case.startswith("svgd"):
            plan = job.opt._fused_plan
            assert plan is not None and job.base.state[job.sm.param]["exp_avg" if case == "svgd_adam"
                                                                     else "momentum_buffer"].data_ptr() == plan.state0.data_ptr()
        f6, fb6 = job.export()
        assert_same(f6, sd6, True, path=f"{case} {label}")
        if bsd6 is not None:
            assert_same(fb6, bsd6, True, path=f"{case} base {label}")
        if case == "swag":
            assert_same(job.sample(), sample6, True, path=f"swag sample {label}")


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", [(2, 1), (1, 2)])
def test_resume_at_another_rank_count_nccl(tmp_path, src, dst):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    dev = torch.device("cuda", 0)
    plain = script.uninterrupted(dev)
    ckpt = plain["ckpt"] if src == 1 else spawn(tmp_path, src, "nccl", "save")[0]
    if dst == 1:
        res = [script.resume(dev, {c: {k: script.to_cpu(v) for k, v in d.items()} for c, d in ckpt.items()})]
    else:
        res = spawn(tmp_path, dst, "nccl", "resume", ckpt)
    for case in script.CASES:
        want = plain["final"][case]
        for r, part in enumerate(res):     # library GEMMs in the closures: fp32 rounding on the GPU
            assert_same(part[case]["sd"], want["sd"], False, devices=False, path=f"{case} {src}->{dst} rank {r}")
            if want["bsd"] is not None:
                assert_same(part[case]["bsd"], want["bsd"], False, devices=False, path=f"{case} base rank {r}")
            if case == "swag":
                assert_same(part[case]["sample"], want["sample"], False, devices=False, path=f"swag sample rank {r}")
