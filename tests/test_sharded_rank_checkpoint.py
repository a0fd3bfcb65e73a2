"""Per-rank checkpoints of D-sharded training (`ColumnShardedModel.shard_state_dict` / `load_shard_state_dicts`,
`checkpoint.consolidate`).

The bar: every rank saves its own columns with no collective, a job at any rank count loads the saved files (mmap)
into the rank-local state the full-dict route gives, bit for bit, and continues like the uninterrupted job —
particles, moments, base-optimizer state and SWAG's next Philox draw, to the tolerance of tests/test_sharded_checkpoint.py;
`consolidate` turns the files into the full dict in one process.  gloo + the oracle-backed ABI double here, the CUDA
library on a B200, NCCL on two."""
from __future__ import annotations

import copy

import pytest
import torch
import torch.multiprocessing as mp

import fake_abi
import rank_checkpoint_script as rscript
import sharded_checkpoint_script as script
from test_sharded_checkpoint import assert_same, exact_for, free_port

WORLDS = (1, 2, 3)
_RUNS = {}


def spawn(tmp_path, world, backend, mode, ckpt_dir, full=None):
    out_path = str(tmp_path / f"{mode}{world}")
    full_path = None
    if full is not None:
        full_path = str(tmp_path / f"full_for_{mode}{world}")
        torch.save(script.to_cpu(full), full_path)
    mp.spawn(rscript.worker, args=(world, free_port(), out_path, backend, mode, str(ckpt_dir), full_path),
             nprocs=world, join=True)
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
    if "plain" not in _RUNS:
        _RUNS["plain"] = script.uninterrupted(cpu_double)
    return _RUNS["plain"]


def saved(tmp_path_factory, cpu_double, world):
    """(checkpoint directory of per-rank files, rank 0's full-dict export) of a `world`-rank job after STEPS steps."""
    if ("save", world) not in _RUNS:
        d = tmp_path_factory.mktemp(f"rank_ckpt{world}")
        if world == 1:
            full = rscript.save(cpu_double, d)
        else:
            full = spawn(d, world, "gloo", "save", d)[0]
        _RUNS[("save", world)] = (d, full)
    return _RUNS[("save", world)]


def loaded(tmp_path_factory, cpu_double, src, dst):
    """Every rank's result of resuming the `src`-rank checkpoint at `dst` ranks."""
    if ("load", src, dst) not in _RUNS:
        d, full = saved(tmp_path_factory, cpu_double, src)
        if dst == 1:
            res = [rscript.load(cpu_double, d, copy.deepcopy(full))]
        else:
            res = spawn(tmp_path_factory.mktemp(f"load{src}to{dst}"), dst, "gloo", "load", d, full)
        _RUNS[("load", src, dst)] = res
    return _RUNS[("load", src, dst)]


def test_each_rank_writes_only_its_columns(tmp_path_factory, cpu_double):
    d, _ = saved(tmp_path_factory, cpu_double, 3)
    for case in script.CASES:
        for which in ("opt", "base") if case != "ivon" else ("opt",):
            shards = rscript.files(d, case, which)
            assert sorted(s["rank"] for s in shards) == [0, 1, 2]
            for s in shards:
                assert s["format"] == "bde-column-shard" and s["version"] == 1 and s["world"] == 3
                assert (s["lo"], s["hi"]) == (s["rank"] * s["shard"], (s["rank"] + 1) * s["shard"])
                assert s["state_dict"]["state"].get("__base_optimizer") is None

                def walk(o):
                    if torch.is_tensor(o):
                        assert o.device.type == "cpu" and (o.dim() == 0 or o.shape[0] == s["shard"]), o.shape
                    elif isinstance(o, dict):
                        for v in o.values():
                            walk(v)
                    elif isinstance(o, (list, tuple)):
                        for v in o:
                            walk(v)
                walk(s["state_dict"])


@pytest.mark.parametrize("src", WORLDS)
@pytest.mark.parametrize("dst", WORLDS)
def test_rank_route_equals_full_route_gloo(tmp_path_factory, cpu_double, src, dst):
    """The rank-local state after `load_shard_state_dicts` of the per-rank files equals the state after
    `load_full_state_dict(full_state_dict(...))` of the same job, bit for bit, on every rank."""
    for r, part in enumerate(loaded(tmp_path_factory, cpu_double, src, dst)):
        for case in script.CASES:
            full_opt, full_base = part[case]["full_route"]
            rank_opt, rank_base = part[case]["rank_route"]
            assert_same(rank_opt, full_opt, True, path=f"{case} {src}->{dst} rank {r}")
            if full_base is not None:
                assert_same(rank_base, full_base, True, path=f"{case} base {src}->{dst} rank {r}")


@pytest.mark.parametrize("src,dst", [(1, 2), (2, 3), (3, 1), (2, 1), (1, 3), (3, 2)])
def test_resume_from_rank_files_at_another_rank_count_gloo(tmp_path_factory, cpu_double, plain, src, dst):
    """Saved per rank at R = src, loaded from the files with mmap at R = dst, STEPS more steps: the uninterrupted
    run's state and next SWAG draw."""
    for r, part in enumerate(loaded(tmp_path_factory, cpu_double, src, dst)):
        for case in script.CASES:
            want = plain["final"][case]
            exact = exact_for(case, src, dst)
            assert_same(part[case]["sd"], want["sd"], exact, path=f"{case} {src}->{dst} rank {r}")
            if want["bsd"] is not None:
                assert_same(part[case]["bsd"], want["bsd"], exact, path=f"{case} base {src}->{dst} rank {r}")
            if case == "swag":
                assert_same(part[case]["sample"], want["sample"], exact, path=f"swag sample {src}->{dst} rank {r}")


@pytest.mark.parametrize("world", WORLDS)
def test_consolidate_equals_the_full_state_dict(tmp_path_factory, cpu_double, world):
    """One process, no torch.distributed: the per-rank files become the job's full dict, and the plain classes load
    it into the state the full dict gives them."""
    from beyond_deep_ensembles_b200 import checkpoint
    d, full = saved(tmp_path_factory, cpu_double, world)
    for case in script.CASES:
        sd = checkpoint.consolidate(rscript.files(d, case, "opt"))
        assert_same(sd, full[case]["sd"], True, path=f"{case} R={world}")
        bsd = None
        if full[case]["bsd"] is not None:
            bsd = checkpoint.consolidate(rscript.files(d, case, "base"))
            assert_same(bsd, full[case]["bsd"], True, path=f"{case} base R={world}")
        a, b = script.Job(case, cpu_double), script.Job(case, cpu_double)
        a.load(copy.deepcopy(full[case]["sd"]), copy.deepcopy(full[case]["bsd"]))
        b.load(sd, bsd)
        assert_same(rscript.state(b.opt), rscript.state(a.opt), True, path=f"{case} plain R={world}")
        if a.base is not None:
            assert_same(rscript.state(b.base), rscript.state(a.base), True, path=f"{case} plain base R={world}")


def test_refusals_leave_the_optimizer_unchanged(tmp_path_factory, cpu_double):
    import beyond_deep_ensembles_b200 as bde
    import golden_models as gm
    dev = cpu_double
    d2, full2 = saved(tmp_path_factory, cpu_double, 2)
    d3, _ = saved(tmp_path_factory, cpu_double, 3)
    swag = rscript.job("swag", dev, None)
    svgd = rscript.job("svgd_adam", dev, None)
    for j in (swag, svgd):
        j.steps(1)

    def refused(j, shards, match, target=None):
        target = j.opt if target is None else target
        before, before_base = rscript.state(j.opt), rscript.state(j.base)
        with pytest.raises(ValueError, match=match):
            j.sm.load_shard_state_dicts(target, shards)
        assert_same(rscript.state(j.opt), before, True)
        assert_same(rscript.state(j.base), before_base, True)

    swag2, svgd2 = rscript.files(d2, "swag", "opt"), rscript.files(d2, "svgd_adam", "opt")
    # not this format: a full dict, an empty list
    refused(swag, [full2["swag"]["sd"]], "format")
    refused(swag, [], "format")
    # shards that do not tile: a missing rank, a duplicate rank, dicts of two jobs
    refused(swag, swag2[:1], "tile")
    refused(swag, [swag2[0], swag2[0]], "tile")
    refused(swag, [swag2[0], rscript.files(d3, "swag", "opt")[1]], "different jobs")
    bad = [copy.deepcopy(s) for s in swag2]
    bad[1]["lo"] += 64
    refused(swag, bad, "tile")
    # another logical size: the per-rank checkpoint of a narrower model
    torch.manual_seed(0)
    sm_small = bde.ColumnShardedModel(gm.make_mlp(hidden=40))
    base_small = torch.optim.SGD([sm_small.param], lr=0.05, momentum=0.9)
    swag_small = bde.SwagOptimizer([sm_small.param], base_small, update_interval=1, deviation_samples=3)
    refused(swag, [sm_small.shard_state_dict(swag_small)], "shapes")
    # another optimizer class: SWAG's files into SVGD, SGD's into Adam
    refused(svgd, swag2, "SwagOptimizer")
    refused(svgd, rscript.files(d2, "svgd_sgd", "base"), "SGD", target=svgd.base)
    # another particle_count / deviation_samples
    bad = [copy.deepcopy(s) for s in svgd2]
    for s in bad:
        s["state_dict"]["state"]["__particle_count"] = 3
        del s["state_dict"]["state"][0]["particle_3"]
    refused(svgd, bad, "particle_count")
    bad = [copy.deepcopy(s) for s in swag2]
    for s in bad:
        s["state_dict"]["state"]["__deviations"] = s["state_dict"]["state"]["__deviations"][:, :2].contiguous()
    refused(swag, bad, "deviation_samples")
    # shards that disagree about a scalar: SWAG's update count, Adam's step, a hyper-parameter
    bad = [copy.deepcopy(s) for s in swag2]
    bad[1]["state_dict"]["state"]["__updates"] += 1
    refused(swag, bad, "disagree")
    bad = rscript.files(d2, "svgd_adam", "base")
    bad[0]["state_dict"]["state"][0]["step"] = bad[0]["state_dict"]["state"][0]["step"] + 1
    refused(svgd, bad, "disagree", target=svgd.base)
    bad = rscript.files(d2, "svgd_adam", "base")
    bad[1]["state_dict"]["param_groups"][0]["lr"] = 0.5
    refused(svgd, bad, "disagree", target=svgd.base)
    # BBB, both ways
    bbb = bde.BBBOptimizer.__new__(bde.BBBOptimizer)
    with pytest.raises(ValueError, match="BBBOptimizer"):
        swag.sm.shard_state_dict(bbb)
    with pytest.raises(ValueError, match="BBBOptimizer"):
        swag.sm.load_shard_state_dicts(bbb, swag2)

    # and the good files still load afterwards
    swag.sm.load_shard_state_dicts(swag.opt, swag2)
    svgd.sm.load_shard_state_dicts(svgd.opt, svgd2)


# ---------------------------------------------------------------------- the CUDA library
@pytest.mark.gpu
@pytest.mark.parametrize("case", script.CASES)
def test_one_rank_rank_files_are_bit_exact_on_the_gpu(tmp_path, case):
    """One B200, one-rank ColumnShardedModel on the CUDA library, a loss whose gradient is elementwise: save the
    per-rank file after STEPS steps, load it with mmap into a fresh job and run STEPS more — the uninterrupted job's
    state and next SWAG draw, bit for bit."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from beyond_deep_ensembles_b200 import _lib
    _lib.get()
    dev = torch.device("cuda", 0)
    j = rscript.job(case, dev, None, elementwise=True)
    j.steps()
    rscript.save_shards(j, tmp_path, case)
    weights = j.weights()
    j.steps()
    want_sd, want_bsd = j.export()
    want_sample = j.sample() if case == "swag" else None

    r = rscript.job(case, dev, None, weights=weights, elementwise=True)
    rscript.load_shards(r, tmp_path, case)
    r.steps()
    sd, bsd = r.export()
    assert_same(sd, want_sd, True, path=case)
    if want_bsd is not None:
        assert_same(bsd, want_bsd, True, path=f"{case} base")
    if case == "swag":
        assert_same(r.sample(), want_sample, True, path="swag sample")


@pytest.mark.gpu
def test_nccl_save_at_two_resume_on_one_and_two(tmp_path):
    """Save per rank at two GPUs (NCCL), resume on one GPU and on two; the device-memory increase of a per-rank save
    or load stays below twice the rank-local optimizer state plus 64 MB."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    dev = torch.device("cuda", 0)
    ckpt = tmp_path / "ckpt"
    ckpt.mkdir()
    mp.spawn(rscript.memory_worker, args=(2, free_port(), str(ckpt), str(tmp_path / "save")), nprocs=2, join=True)
    saved = [torch.load(tmp_path / f"save.{r}") for r in range(2)]
    for r, part in enumerate(saved):
        for case in script.CASES:
            s = part[case]
            print(f"rank {r} {case}: rank-local state {s['state_bytes']} B, peak increase save {s['peaks']['save']} B, "
                  f"load {s['peaks']['load']} B")
            for what in ("save", "load"):
                assert s["peaks"][what] < 2 * s["state_bytes"] + (64 << 20), (r, case, what)
    full = saved[0]
    plain = script.uninterrupted(dev)
    res = [rscript.load(dev, ckpt, full)]
    res += spawn(tmp_path, 2, "nccl", "load", ckpt, full)
    for i, part in enumerate(res):
        for case in script.CASES:
            assert_same(part[case]["rank_route"], part[case]["full_route"], True, devices=False,
                        path=f"{case} routes {i}")
            want = plain["final"][case]    # library GEMMs in the closures: fp32 rounding on the GPU
            assert_same(part[case]["sd"], want["sd"], False, devices=False, path=f"{case} resume {i}")
            if want["bsd"] is not None:
                assert_same(part[case]["bsd"], want["bsd"], False, devices=False, path=f"{case} base resume {i}")
            if case == "swag":
                assert_same(part[case]["sample"], want["sample"], False, devices=False, path=f"swag sample {i}")
