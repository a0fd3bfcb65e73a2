"""Per-rank checkpoint jobs of tests/test_sharded_rank_checkpoint.py (`ColumnShardedModel.shard_state_dict` /
`load_shard_state_dicts`), over the four jobs of sharded_checkpoint_script.

`save` runs STEPS steps, writes every rank's per-rank dicts to `<ckpt_dir>/<case>.{opt,base}.<rank>` and returns the
full-dict route's export (collective) and the model weights.  `load` resumes from a checkpoint directory at this job's
rank count twice — once through the full dicts, once through the per-rank files loaded with mmap=True — returns both
rank-local states, then runs STEPS more steps on the per-rank resume.  While the per-rank functions run,
torch.distributed's collectives raise."""
from __future__ import annotations

import contextlib
import os
import sys
from pathlib import Path

import torch

import sharded_checkpoint_script as script

COLLECTIVES = ("all_gather", "all_gather_into_tensor", "all_gather_object", "all_reduce", "all_to_all",
               "all_to_all_single", "barrier", "broadcast", "broadcast_object_list", "gather", "gather_object",
               "reduce", "reduce_scatter", "reduce_scatter_tensor", "scatter", "scatter_object_list", "send", "recv",
               "isend", "irecv")


@contextlib.contextmanager
def no_collectives(sm):
    """torch.distributed's collectives raise inside; `sm.collectives` must not move."""
    import torch.distributed as dist
    saved = {name: getattr(dist, name) for name in COLLECTIVES if hasattr(dist, name)}

    def refuse(*args, **kwargs):
        raise AssertionError("a collective was issued")
    count = sm.collectives
    for name in saved:
        setattr(dist, name, refuse)
    try:
        yield
    finally:
        for name, fn in saved.items():
            setattr(dist, name, fn)
    assert sm.collectives == count


def files(ckpt_dir, case, which):
    """Every rank's file of `case` ("opt" or "base") in a checkpoint directory, loaded with mmap."""
    paths = sorted(Path(ckpt_dir).glob(f"{case}.{which}.*"))
    return [torch.load(p, map_location="cpu", mmap=True) for p in paths]


def state(opt):
    return script.to_cpu(script.snapshot(opt.state_dict()))


def job(case, dev, group, weights=None, elementwise=False):
    return script.Job(case, dev, group, wrap=True, weights=weights, elementwise=elementwise)


def save_shards(j, ckpt_dir, case):
    rank = j.sm.rank
    with no_collectives(j.sm):
        torch.save(j.sm.shard_state_dict(j.opt), Path(ckpt_dir) / f"{case}.opt.{rank}")
        if j.base is not None:
            torch.save(j.sm.shard_state_dict(j.base), Path(ckpt_dir) / f"{case}.base.{rank}")


def load_shards(j, ckpt_dir, case):
    with no_collectives(j.sm):
        j.sm.load_shard_state_dicts(j.opt, files(ckpt_dir, case, "opt"))
        if j.base is not None:
            j.sm.load_shard_state_dicts(j.base, files(ckpt_dir, case, "base"))


def save(dev, ckpt_dir, group=None):
    out = {}
    for case in script.CASES:
        j = job(case, dev, group)
        j.steps()
        save_shards(j, ckpt_dir, case)
        sd, bsd = j.export()
        out[case] = {"sd": sd, "bsd": bsd, "weights": j.weights()}
    return out


def load(dev, ckpt_dir, full, group=None):
    """`full`: what `save` returned (rank 0's) for the checkpoint in ckpt_dir."""
    out = {}
    for case in script.CASES:
        weights = {k: v.to(dev) for k, v in full[case]["weights"].items()}
        via_full = job(case, dev, group, weights)
        via_full.load(full[case]["sd"], full[case]["bsd"])
        j = job(case, dev, group, weights)
        load_shards(j, ckpt_dir, case)
        res = {"full_route": (state(via_full.opt), None if j.base is None else state(via_full.base)),
               "rank_route": (state(j.opt), None if j.base is None else state(j.base))}
        j.steps()
        res["sd"], res["bsd"] = j.export()
        if case == "swag":
            res["sample"] = j.sample()
        out[case] = res
    return out


def worker(rank: int, world: int, port: int, out_path: str, backend: str, mode: str, ckpt_dir: str,
           full_path: str | None = None):
    """One rank of a D-sharded job, mode "save" (into ckpt_dir) or "load" (from ckpt_dir and the full dicts at
    full_path); writes its result, on the host, to out_path.<rank>."""
    root = Path(__file__).resolve().parent.parent
    sys.path.insert(0, str(root))
    sys.path.insert(0, str(root / "tests"))
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dev = torch.device("cpu")
        dist.init_process_group("gloo", rank=rank, world_size=world)
        torch.set_num_threads(1)
        import fake_abi
        fake_abi.install(script._Patch())
    from beyond_deep_ensembles_b200 import dist as bdist
    if mode == "save":
        res = save(dev, ckpt_dir, dist.group.WORLD)
    else:
        res = load(dev, ckpt_dir, torch.load(full_path), dist.group.WORLD)
    if dev.type == "cuda":
        torch.cuda.synchronize()
    torch.save(script.to_cpu(res), f"{out_path}.{rank}")
    dist.barrier()
    bdist.shutdown_peer_exchange()
    dist.destroy_process_group()


def state_bytes(*opts):
    """Device bytes of the optimizers' rank-local state."""
    def walk(o):
        if torch.is_tensor(o):
            return o.numel() * o.element_size() if o.is_cuda else 0
        if isinstance(o, dict):
            return sum(walk(v) for k, v in o.items() if k != "__base_optimizer")
        if isinstance(o, (list, tuple)):
            return sum(walk(v) for v in o)
        return 0
    return sum(walk(o.state_dict()) for o in opts if o is not None)


def memory_worker(rank: int, world: int, port: int, ckpt_dir: str, out_path: str):
    """One rank of an NCCL job: STEPS steps, a per-rank save into ckpt_dir, then a reload of every rank's files into
    the same job.  Records the peak increase of allocated device memory around each against the rank-local optimizer
    state, then exports the full dicts and weights (rank 0's is the checkpoint's full-dict twin)."""
    root = Path(__file__).resolve().parent.parent
    sys.path.insert(0, str(root))
    sys.path.insert(0, str(root / "tests"))
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from beyond_deep_ensembles_b200 import dist as bdist
    out = {}
    for case in script.CASES:
        j = job(case, dev, dist.group.WORLD)
        j.steps()
        res = {"state_bytes": state_bytes(j.opt, j.base), "peaks": {}}
        for what, fn in (("save", save_shards), ("load", load_shards)):
            if what == "load":
                dist.barrier()          # every rank's files are written
            torch.cuda.synchronize(dev)
            torch.cuda.reset_peak_memory_stats(dev)
            before = torch.cuda.memory_allocated(dev)
            fn(j, ckpt_dir, case)
            torch.cuda.synchronize(dev)
            res["peaks"][what] = torch.cuda.max_memory_allocated(dev) - before
        res["sd"], res["bsd"] = j.export()
        res["weights"] = j.weights()
        out[case] = res
    torch.save(script.to_cpu(out), f"{out_path}.{rank}")
    dist.barrier()
    bdist.shutdown_peer_exchange()
    dist.destroy_process_group()
