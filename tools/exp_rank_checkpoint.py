"""Checkpoint cost of D-sharded training: the full-dict route against the per-rank route, save and load.

Two shapes, each one flat fp32 weight vector (the model left out, as in bench.py's sharded_closure section):
  swag   SwagOptimizer over SGD (momentum), D = 23,880,950 (ResNet-50 size), K = 10
  svgd   SVGDOptimizer over SGD (momentum), n = 20 particles, D = 5e7
at R = 1 and, with two or more GPUs, R = 2 (NCCL).  The job runs two steps on the loss sum(w^2) first, so that every
state vector is allocated and written.

Routes, each timed on every rank with a host clock around work that ends in a device synchronise:
  full save  sm.full_state_dict(opt) and (base) -> rank 0 torch.save's one file
  full load  every rank torch.load's that file (map_location="cpu") -> sm.load_full_state_dict(opt / base)
  rank save  torch.save(sm.shard_state_dict(opt / base), f"{path}.{rank}") on every rank
  rank load  every rank torch.load's the R files with mmap=True -> sm.load_shard_state_dicts(opt / base)
Peak device memory is torch.cuda.max_memory_allocated() above what was allocated before the phase; peak host memory is
the largest resident set (/proc/self/statm, sampled every millisecond by a thread) above the resident set before it.
Files go to a temporary directory; loads read them back right after they were written (the page cache, not a cold
disk).  A row reports the largest value over the ranks.

    python tools/exp_rank_checkpoint.py --out profiles/r03_rank_checkpoint.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import socket
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

SHAPES = {"swag": dict(D=23_880_950, K=10), "svgd": dict(D=50_000_000, n=20)}
PAGE = os.sysconf("SC_PAGE_SIZE")


def rss() -> int:
    with open("/proc/self/statm") as f:
        return int(f.read().split()[1]) * PAGE


class Peak:
    """Peak device and host memory above the values at entry, and the wall time, of a phase."""

    def __init__(self, dev):
        self.dev = dev

    def __enter__(self):
        torch.cuda.synchronize(self.dev)
        torch.cuda.reset_peak_memory_stats(self.dev)
        self.dev0, self.host0 = torch.cuda.memory_allocated(self.dev), rss()
        self.host_peak, self.stop = self.host0, False

        def poll():
            while not self.stop:
                self.host_peak = max(self.host_peak, rss())
                time.sleep(0.001)
        self.thread = threading.Thread(target=poll, daemon=True)
        self.thread.start()
        self.t0 = time.perf_counter()
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize(self.dev)
        self.seconds = time.perf_counter() - self.t0
        self.stop = True
        self.thread.join()
        self.host_peak = max(self.host_peak, rss())
        self.device_bytes = torch.cuda.max_memory_allocated(self.dev) - self.dev0
        self.host_bytes = self.host_peak - self.host0


def build(shape, dev, group):
    import beyond_deep_ensembles_b200 as bde
    from beyond_deep_ensembles_b200 import noise
    noise.set_seed(5)
    torch.manual_seed(5)
    D = SHAPES[shape]["D"]
    w = torch.nn.Parameter(0.01 * torch.randn(D, device=dev))
    sm = bde.ColumnShardedModel([w], group)
    base = torch.optim.SGD([sm.param], lr=1e-3, momentum=0.9)
    if shape == "swag":
        opt = bde.SwagOptimizer([sm.param], base, update_interval=1, deviation_samples=SHAPES[shape]["K"],
                                process_group=group)
    else:
        def reset():
            with torch.no_grad():
                w.normal_(0.0, 0.01)
        opt = bde.SVGDOptimizer([sm.param], sm.reset_closure(reset), base, particle_count=SHAPES[shape]["n"],
                                dataset_size=1000, l2_reg=0.01, process_group=group)
    fwd, bwd = sm.closures(lambda: (w * w).sum(), lambda loss: loss.backward())
    for _ in range(2):
        opt.step(fwd, bwd)
    return sm, opt, base


def state_bytes(*opts):
    def walk(o):
        if torch.is_tensor(o):
            return o.numel() * o.element_size()
        if isinstance(o, dict):
            return sum(walk(v) for k, v in o.items() if k != "__base_optimizer")
        if isinstance(o, (list, tuple)):
            return sum(walk(v) for v in o)
        return 0
    return sum(walk(o.state_dict()) for o in opts)


def run(rank, world, port, shape, tmp, out_path):
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        group = dist.group.WORLD

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    sm, opt, base = build(shape, dev, group)
    rows = {"state_bytes": state_bytes(opt, base)}
    full_path, rank_path = Path(tmp) / "full.pt", Path(tmp) / "rank"

    def full_save():
        ckpt = {"opt": sm.full_state_dict(opt), "base": sm.full_state_dict(base)}
        if rank == 0:
            torch.save(ckpt, full_path)

    def full_load():
        ckpt = torch.load(full_path, map_location="cpu")
        sm.load_full_state_dict(opt, ckpt["opt"])
        sm.load_full_state_dict(base, ckpt["base"])

    def rank_save():
        torch.save({"opt": sm.shard_state_dict(opt), "base": sm.shard_state_dict(base)}, f"{rank_path}.{rank}")

    def rank_load():
        shards = [torch.load(f"{rank_path}.{r}", map_location="cpu", mmap=True) for r in range(world)]
        sm.load_shard_state_dicts(opt, [s["opt"] for s in shards])
        sm.load_shard_state_dicts(base, [s["base"] for s in shards])

    for name, fn in (("full_save", full_save), ("full_load", full_load), ("rank_save", rank_save),
                     ("rank_load", rank_load)):
        barrier()
        with Peak(dev) as p:
            fn()
        barrier()
        rows[name] = dict(seconds=p.seconds, device_peak_bytes=p.device_bytes, host_peak_bytes=p.host_bytes)
    rows["full_file_bytes"] = full_path.stat().st_size
    rows["rank_file_bytes"] = [Path(f"{rank_path}.{r}").stat().st_size for r in range(world)]
    torch.save(rows, f"{out_path}.{rank}")
    if world > 1:
        dist.barrier()
        from beyond_deep_ensembles_b200 import dist as bdist
        bdist.shutdown_peer_exchange()
        dist.destroy_process_group()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def gpu_identity() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count(),
            "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="swag,svgd")
    ap.add_argument("--worlds", default="1,2")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import torch.multiprocessing as mp
    rows = [dict(kind="identity", **gpu_identity())]
    print(json.dumps(rows[0]), flush=True)
    for shape in a.shapes.split(","):
        for world in map(int, a.worlds.split(",")):
            if world > torch.cuda.device_count():
                row = dict(kind="rank_checkpoint", shape=shape, world=world, skipped="fewer GPUs than ranks")
                rows.append(row)
                print(json.dumps(row), flush=True)
                continue
            tmp = tempfile.mkdtemp(prefix="bde_rank_ckpt_")
            try:
                out_path = str(Path(tmp) / "result")
                mp.spawn(run, args=(world, free_port(), shape, tmp, out_path), nprocs=world, join=True)
                ranks = [torch.load(f"{out_path}.{r}") for r in range(world)]
            finally:
                shutil.rmtree(tmp, ignore_errors=True)
            row = dict(kind="rank_checkpoint", shape=shape, world=world, **SHAPES[shape],
                       rank_local_state_bytes=max(r["state_bytes"] for r in ranks),
                       full_file_bytes=ranks[0]["full_file_bytes"], rank_file_bytes=ranks[0]["rank_file_bytes"])
            for phase in ("full_save", "full_load", "rank_save", "rank_load"):
                row[phase] = {k: max(r[phase][k] for r in ranks) for k in ranks[0][phase]}
            rows.append(row)
            print(json.dumps(row), flush=True)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()
