"""Checkpoint / resume jobs of tests/test_sharded_checkpoint.py, run in the test process (the plain classes, or a
one-rank ColumnShardedModel) and by every rank of a spawned D-sharded job (`worker`).

Four jobs, each seeded on its own so that a section does not depend on what ran before it: SWAG over SGD with momentum,
iVON with 2 MC samples, SVGD with 4 particles over SGD (momentum, Nesterov, weight decay) and over Adam — the last two
take the fused base-optimizer plan.  `save` runs STEPS steps and exports (opt dict, base dict, model weights);
`resume` builds a fresh job from the weights, loads the dicts and runs STEPS more; `uninterrupted` runs 2 * STEPS with
the plain classes and exports after STEPS and at the end.  Plain jobs export with `state_dict()` and load with
`load_state_dict()`; sharded ones with `sm.full_state_dict` / `sm.load_full_state_dict`."""
from __future__ import annotations

import os
import sys
from pathlib import Path

import torch

import golden_models as gm

SEED = 991
BATCH = 48
STEPS = 3
CASES = ("swag", "ivon", "svgd_sgd", "svgd_adam")


class Job:
    def __init__(self, case, dev, group=None, wrap=False, weights=None, elementwise=False):
        """group None and wrap False: the plain class over model.parameters(); otherwise the optimizer runs over a
        ColumnShardedModel's one parameter (group None + wrap: a one-rank "group", no collective).
        elementwise: a loss whose gradient is elementwise in the weights (no GEMM between runs to compare)."""
        import beyond_deep_ensembles_b200 as bde
        from beyond_deep_ensembles_b200 import noise
        self.case = case
        noise.set_seed(SEED)
        torch.manual_seed(3)
        self.model = model = gm.make_mlp().to(dev)
        if weights is not None:
            model.load_state_dict(weights)
        sharded = group is not None or wrap
        self.sm = sm = bde.ColumnShardedModel(model, group) if sharded else None
        params = [sm.param] if sharded else list(model.parameters())
        if elementwise:
            g = torch.Generator().manual_seed(8)
            targets = [torch.randn(p.shape, generator=g).to(dev) for p in model.parameters()]

            def fwd():
                return sum(((p - t) ** 2).sum() for p, t in zip(model.parameters(), targets))
        else:
            g = torch.Generator().manual_seed(5)
            x, y = torch.randn(BATCH, 8, generator=g).to(dev), torch.randn(BATCH, generator=g).to(dev)
            fwd, _ = gm.mse_closures(model, x, y)

        def bwd(loss):
            loss.backward()
        self.fwd, self.bwd = sm.closures(fwd, bwd) if sharded else (fwd, bwd)
        self.base = None
        if case == "swag":
            self.base = torch.optim.SGD(params, lr=0.05, momentum=0.9)
            self.opt = bde.SwagOptimizer(params, self.base, update_interval=1, deviation_samples=3, process_group=group)
        elif case == "ivon":
            self.opt = bde.iVONOptimizer(params, lr=0.01, prior_prec=10.0, dataset_size=1000, mc_samples=2,
                                         damping=1e-3, process_group=group)
        else:
            if case == "svgd_sgd":
                self.base = torch.optim.SGD(params, lr=0.02, momentum=0.9, nesterov=True, weight_decay=1e-4)
            else:
                self.base = torch.optim.Adam(params, lr=1e-3, weight_decay=1e-4)

            def reset_fn():
                for m in model:
                    if hasattr(m, "reset_parameters"):
                        m.reset_parameters()
            reset = sm.reset_closure(reset_fn) if sharded else reset_fn
            torch.manual_seed(11)
            self.opt = bde.SVGDOptimizer(params, reset, self.base, particle_count=4, dataset_size=BATCH, l2_reg=0.01,
                                         process_group=group)

    def steps(self, count=STEPS):
        for _ in range(count):
            self.opt.step(self.fwd, self.bwd)

    def export(self):
        """(optimizer dict, base-optimizer dict or None) in the reference layout, detached from the live arenas."""
        if self.sm is None:
            return (snapshot(self.opt.state_dict()),
                    None if self.base is None else snapshot(self.base.state_dict()))
        return (self.sm.full_state_dict(self.opt),
                None if self.base is None else self.sm.full_state_dict(self.base))

    def load(self, sd, bsd):
        if self.sm is None:
            self.opt.load_state_dict(sd)
            if self.base is not None:
                self.base.load_state_dict(bsd)
        else:
            self.sm.load_full_state_dict(self.opt, sd)
            if self.base is not None:
                self.sm.load_full_state_dict(self.base, bsd)

    def weights(self):
        """The model's weights as the plain job's model holds them (a sharded job gathers its current slices)."""
        if self.sm is not None:
            self.sm.gather()
        return {k: v.detach().clone() for k, v in self.model.state_dict().items()}

    def sample(self):
        self.opt.sample_parameters()
        if self.sm is not None:
            self.sm.gather()
        return torch.cat([p.detach().reshape(-1) for p in self.model.parameters()]).cpu().clone()


def snapshot(obj):
    """Tensors cloned (the plain classes' dicts hold views of live arenas); optimizer objects kept as they are."""
    if torch.is_tensor(obj):
        return obj.detach().clone()
    if isinstance(obj, dict):
        return {k: snapshot(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [snapshot(v) for v in obj]
    return obj


def to_cpu(obj):
    if torch.is_tensor(obj):
        return obj.detach().cpu()
    if isinstance(obj, dict):
        return {k: (None if k == "__base_optimizer" else to_cpu(v)) for k, v in obj.items()}
    if isinstance(obj, list):
        return [to_cpu(v) for v in obj]
    return obj


def save(dev, group=None):
    out = {}
    for case in CASES:
        job = Job(case, dev, group)
        job.steps()
        sd, bsd = job.export()
        out[case] = {"sd": sd, "bsd": bsd, "weights": job.weights()}
    return out


def resume(dev, ckpt, group=None):
    out = {}
    for case in CASES:
        job = Job(case, dev, group, weights={k: v.to(dev) for k, v in ckpt[case]["weights"].items()})
        job.load(ckpt[case]["sd"], ckpt[case]["bsd"])
        job.steps()
        sd, bsd = job.export()
        out[case] = {"sd": sd, "bsd": bsd}
        if case == "swag":
            out[case]["sample"] = job.sample()
    return out


def uninterrupted(dev):
    """The plain classes over 2 * STEPS steps: the checkpoint after STEPS ("ckpt", as `save` returns it) and the
    state at the end ("final", as `resume` returns it)."""
    ckpt, final = {}, {}
    for case in CASES:
        job = Job(case, dev)
        job.steps()
        sd, bsd = job.export()
        ckpt[case] = {"sd": sd, "bsd": bsd, "weights": job.weights()}
        job.steps()
        sd, bsd = job.export()
        final[case] = {"sd": sd, "bsd": bsd}
        if case == "swag":
            final[case]["sample"] = job.sample()
    return {"ckpt": ckpt, "final": final}


class _Patch:
    def setattr(self, obj, name, value):
        setattr(obj, name, value)


def worker(rank: int, world: int, port: int, out_path: str, backend: str, mode: str, ckpt_path: str | None = None):
    """One rank of a D-sharded job: mode "save" or "resume" (from the checkpoint file at ckpt_path); writes what it
    exported, on the host, to out_path.<rank>."""
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
        fake_abi.install(_Patch())
    from beyond_deep_ensembles_b200 import dist as bdist
    if mode == "save":
        res = save(dev, dist.group.WORLD)
    else:
        res = resume(dev, torch.load(ckpt_path), dist.group.WORLD)
    if dev.type == "cuda":
        torch.cuda.synchronize()
    torch.save(to_cpu(res), f"{out_path}.{rank}")
    dist.barrier()
    bdist.shutdown_peer_exchange()
    dist.destroy_process_group()
