"""One script, run by every rank of a D-sharded job with torch's ShardedGradScaler and by the test process with a
plain GradScaler on the whole problem (world = 1, group None).  In every scenario one backward pass gets an inf
gradient in ONE global column, so only the rank that owns that column sees it; the job must still skip the same
steps and follow the same loss-scale trajectory as the unsharded run.

Two families:
  * slices: the optimizers over this rank's column slice of separable problems (as tests/sharded_script.py);
  * wrapped: the optimizers over `ColumnShardedModel(model).param` with its closures (as
    tests/sharded_closure_script.py); all ranks see the same batch.
SVGD runs with the fused unscale-and-gather and with the reference's unscale_-then-gather (`fuse_unscale_into_gather`);
the scaler turns the fused base-optimizer launch and gradient prebinding off in both."""
from __future__ import annotations

import os

import torch
import torch.distributed as dist

import golden_models as gm

D_GLOBAL = 64 * 37      # slices of shard_bounds() are whole 64-element blocks
SEED = 4242
PLANT = 64 * 5 + 3      # slices: a column of rank 0 at R = 2 and 3
PLANT_WRAPPED = 480     # wrapped: a weight of the MLP's second layer, in the last rank's columns at R = 2 and 3
INIT_SCALE = 1024.0


def make_scaler(dev, group, sharded: bool):
    kw = dict(init_scale=INIT_SCALE, growth_interval=1)   # the scale moves every step: its trajectory shows skips
    if sharded:
        from torch.distributed.fsdp.sharded_grad_scaler import ShardedGradScaler
        return ShardedGradScaler(dev.type, process_group=group, **kw)
    return torch.amp.GradScaler(dev.type, **kw)


class Job:
    """The scaler, the pass counter of the backward closures and the per-step record of one optimizer's run."""

    def __init__(self, dev, group, sharded, plant_at):
        self.scaler = make_scaler(dev, group, sharded)
        self.plant_at, self.passes = plant_at, 0
        self.scales, self.base_steps, self._count = [], [], [0]

    def count_steps(self, base):
        base.register_step_post_hook(lambda *a: self._count.__setitem__(0, self._count[0] + 1))

    def backward(self, bwd, plant):
        """bwd(loss) runs the scaled backward pass (and hands the gradient to the sharded parameter); then the inf."""
        def run(loss):
            bwd(loss)
            self.passes += 1
            if self.passes == self.plant_at:
                plant()
        return run

    def step(self, opt, fwd, bwd):
        self._count[0] = 0
        opt.step(fwd, bwd, grad_scaler=self.scaler)
        self.scaler.update()
        self.scales.append(float(self.scaler.get_scale()))
        self.base_steps.append(self._count[0])


def _scaled_backward(scaler):
    def bwd(loss):
        scaler.scale(loss).backward()
    return bwd


# ---------------------------------------------------------------------------------------------------- slices
def run_slices(dev, world: int, rank: int, group, sharded: bool):
    import beyond_deep_ensembles_b200 as bde
    from beyond_deep_ensembles_b200 import noise
    from beyond_deep_ensembles_b200.layout import shard_bounds

    noise.set_seed(SEED + (0 if group is None else 1000 * rank))
    lo, hi = shard_bounds(D_GLOBAL, world, rank)
    g = torch.Generator().manual_seed(7)
    W0, W1 = torch.randn(D_GLOBAL, generator=g), torch.randn(D_GLOBAL, generator=g)
    Cv = torch.randn(D_GLOBAL, generator=g)
    c = Cv[lo:hi].to(dev)
    mine = PLANT - lo if lo <= PLANT < hi else None
    out = {}

    def planter(param):
        def plant():
            if mine is not None:
                param.grad.view(-1)[mine] = float("inf")
        return plant

    def loss_of(*params):
        return lambda: sum((0.5 * (p * c) ** 2).sum() for p in params)

    # SWAG: one pass per step, the base optimizer's step is skipped at step 2
    w = torch.nn.Parameter(W0[lo:hi].clone().to(dev))
    base = torch.optim.SGD([w], lr=0.1, momentum=0.9)
    opt = bde.SwagOptimizer([w], base, update_interval=1, deviation_samples=3, process_group=group)
    job = Job(dev, group, sharded, plant_at=2)
    job.count_steps(base)
    opt.init_grad_scaler(job.scaler)
    bwd = job.backward(_scaled_backward(job.scaler), planter(w))
    for _ in range(4):
        job.step(opt, loss_of(w), bwd)
    out["swag"] = _record(job, theta=opt._theta, mean=opt._mean, sq=opt._sq)

    # iVON, 2 MC samples, two parameter groups: the inf sits in the SECOND group of the last sample of the last step
    # (iVON never skips its update, the reference's check being always true: the scale backs off, one column is lost)
    v0, v1 = (torch.nn.Parameter(W[lo:hi].clone().to(dev)) for W in (W0, W1))
    opt = bde.iVONOptimizer([{"params": [v0]}, {"params": [v1]}], lr=0.01, prior_prec=10.0, dataset_size=1000,
                            mc_samples=2, damping=1e-3, process_group=group)
    job = Job(dev, group, sharded, plant_at=4)
    opt.init_grad_scaler(job.scaler)
    bwd = job.backward(_scaled_backward(job.scaler), planter(v1))
    for _ in range(2):
        job.step(opt, loss_of(v0, v1), bwd)
    rows = {f"{k}{gi}": ar["rows"][k] for gi, ar in enumerate(opt._arenas) for k in ("mean", "momentum", "precision")}
    out["ivon"] = _record(job, **rows)

    # SVGD, 4 particles: the inf is in the last particle of step 2, whose flag decides for all four base steps
    for fused in (True, False):
        x = torch.nn.Parameter(W0[lo:hi].clone().to(dev))
        gen = torch.Generator().manual_seed(11)          # the same resets on every rank: one global problem

        def reset():
            with torch.no_grad():
                x.copy_(torch.randn(D_GLOBAL, generator=gen)[lo:hi].to(dev))
        base = torch.optim.SGD([x], lr=0.02, momentum=0.9)
        opt = bde.SVGDOptimizer([x], reset, base, particle_count=4, dataset_size=100, l2_reg=0.01, process_group=group)
        opt.fuse_unscale_into_gather = fused
        job = Job(dev, group, sharded, plant_at=8)
        job.count_steps(base)
        opt.init_grad_scaler(job.scaler)
        bwd = job.backward(_scaled_backward(job.scaler), planter(x))
        for _ in range(3):
            job.step(opt, loss_of(x), bwd)
        out[f"svgd_{'fused' if fused else 'unscale'}"] = _record(job, particles=opt._X)

    # BBB: the inf lands in the deterministic parameter's gradient at step 2
    gp = bde.GaussianParameter((hi - lo,), device=dev)
    det = torch.nn.Parameter(Cv[lo:hi].clone().to(dev))
    with torch.no_grad():
        gp.mean.copy_(0.1 * W0[lo:hi].to(dev))
        gp.rho.copy_(-3.0 + 0.2 * Cv[lo:hi].to(dev))
    params = [gp.mean, gp.rho, det]
    base = torch.optim.SGD(params, lr=0.05)
    opt = bde.BBBOptimizer(params, base, prior=bde.GaussianPrior(0.0, 1.0), dataset_size=100, l2_scale=0.01,
                           process_group=group)
    job = Job(dev, group, sharded, plant_at=2)
    job.count_steps(base)
    opt.init_grad_scaler(job.scaler)
    bwd = job.backward(_scaled_backward(job.scaler), planter(det))
    for _ in range(3):
        job.step(opt, lambda: ((gp.sample() + det) * c).pow(2).sum(), bwd)
    out["bbb"] = _record(job, mean=gp.mean, rho=gp.rho, det=det)
    return out


def _record(job, **vectors):
    return {"scales": job.scales, "base_steps": job.base_steps,
            **{k: v.detach().reshape(-1, v.shape[-1]).cpu().clone() for k, v in vectors.items()}}


# ---------------------------------------------------------------------------------------------------- wrapped
def run_wrapped(dev, world: int, rank: int, group, sharded: bool, algos=("swag", "ivon", "svgd", "bbb"),
                autocast: bool = False):
    """Every vector is returned full length in parameters_to_vector order (the sharded run gathers its slices)."""
    import beyond_deep_ensembles_b200 as bde
    from beyond_deep_ensembles_b200 import noise

    noise.set_seed(SEED + (0 if group is None else 1000 * rank))
    gx = torch.Generator().manual_seed(5)
    x, y = torch.randn(48, 8, generator=gx).to(dev), torch.randn(48, generator=gx).to(dev)
    out = {}

    def build():
        torch.manual_seed(3 + (0 if group is None else 17 * rank))   # rank 0's init is broadcast
        model = gm.make_mlp().to(dev)
        if group is None:
            return model, None, list(model.parameters())
        sm = bde.ColumnShardedModel(model, group)
        return model, sm, [sm.param]

    def closures(model, sm, job):
        fwd, _ = gm.mse_closures(model, x, y)
        if autocast:
            plain_fwd = fwd

            def fwd():
                with torch.autocast(dev.type, dtype=torch.float16):
                    return plain_fwd()
        bwd = _scaled_backward(job.scaler)
        if sm is not None:
            fwd, bwd = sm.closures(fwd, bwd)
        return fwd, job.backward(bwd, _wrapped_planter(model, sm))

    def export(sm, layout, rows):
        rows = rows.reshape(-1, rows.shape[-1])
        return (layout.to_logical(rows) if sm is None else sm.logical(sm.gather_rows(rows))).cpu()

    if "swag" in algos:
        model, sm, params = build()
        base = torch.optim.SGD(params, lr=0.05, momentum=0.9)
        opt = bde.SwagOptimizer(params, base, update_interval=1, deviation_samples=3, process_group=group)
        job = Job(dev, group, sharded, plant_at=2)
        job.count_steps(base)
        opt.init_grad_scaler(job.scaler)
        fwd, bwd = closures(model, sm, job)
        for _ in range(4):
            job.step(opt, fwd, bwd)
        out["swag"] = {"scales": job.scales, "base_steps": job.base_steps,
                       "theta": export(sm, opt._layout, opt._theta), "mean": export(sm, opt._layout, opt._mean)}

    if "ivon" in algos:
        model, sm, params = build()
        opt = bde.iVONOptimizer(params, lr=0.01, prior_prec=10.0, dataset_size=1000, mc_samples=2, damping=1e-3,
                                process_group=group)
        job = Job(dev, group, sharded, plant_at=4)
        opt.init_grad_scaler(job.scaler)
        fwd, bwd = closures(model, sm, job)
        for _ in range(2):
            job.step(opt, fwd, bwd)
        ar = opt._arenas[0]
        out["ivon"] = {"scales": job.scales, "base_steps": job.base_steps,
                       **{k: export(sm, ar["layout"], ar["rows"][k]) for k in ("mean", "momentum", "precision")}}

    if "svgd" in algos:
        for fused in (True, False):
            model, sm, params = build()
            base = torch.optim.SGD(params, lr=0.02, momentum=0.9)

            def reset_fn(model=model):
                for m in model:
                    if hasattr(m, "reset_parameters"):
                        m.reset_parameters()
            reset = reset_fn if sm is None else sm.reset_closure(reset_fn)
            torch.manual_seed(11 + (0 if group is None else 5 * rank))
            opt = bde.SVGDOptimizer(params, reset, base, particle_count=4, dataset_size=48, l2_reg=0.01,
                                    process_group=group)
            opt.fuse_unscale_into_gather = fused
            job = Job(dev, group, sharded, plant_at=8)
            job.count_steps(base)
            opt.init_grad_scaler(job.scaler)
            fwd, bwd = closures(model, sm, job)
            for _ in range(3):
                job.step(opt, fwd, bwd)
            out[f"svgd_{'fused' if fused else 'unscale'}"] = {"scales": job.scales, "base_steps": job.base_steps,
                                                               "particles": export(sm, opt._layout, opt._X)}

    if "bbb" in algos:
        # no Gaussian layers: the prior term is the L2 penalty of the (sharded) deterministic weights
        model, sm, params = build()
        base = torch.optim.SGD(params, lr=0.05)
        opt = bde.BBBOptimizer(params, base, prior=bde.GaussianPrior(0.0, 1.0), dataset_size=100, l2_scale=0.01,
                               process_group=group)
        job = Job(dev, group, sharded, plant_at=2)
        job.count_steps(base)
        opt.init_grad_scaler(job.scaler)
        fwd, bwd = closures(model, sm, job)
        for _ in range(3):
            job.step(opt, fwd, bwd)
        flat = params[0] if sm is not None else None
        out["bbb"] = {"scales": job.scales, "base_steps": job.base_steps,
                      "weights": (sm.logical(sm.gather_rows(flat.detach())).cpu() if sm is not None else
                                  torch.cat([p.detach().reshape(-1) for p in params]).cpu().reshape(1, -1))}
    return out


def _wrapped_planter(model, sm):
    """inf into the gradient of logical column PLANT_WRAPPED: the model's own tensor (unsharded) or the owner rank's
    column of `sm.param.grad` (after the reduce-scatter)."""
    sizes = [p.numel() for p in model.parameters()]
    t = next(i for i in range(len(sizes)) if sum(sizes[:i + 1]) > PLANT_WRAPPED)
    j = PLANT_WRAPPED - sum(sizes[:t])

    def plant():
        if sm is None:
            list(model.parameters())[t].grad.view(-1)[j] = float("inf")
            return
        pos = sm.layout.offsets[t] + j
        if sm.lo <= pos < sm.hi:
            sm.param.grad.view(-1)[pos - sm.lo] = float("inf")
    return plant


# ---------------------------------------------------------------------------------------------------- refusals
def refusals(dev, world: int, rank: int):
    """Collective over the whole job (new_group).  Returns what each scaler did with a sharded SWAG step: "ok" or
    the ValueError's message."""
    import beyond_deep_ensembles_b200 as bde
    from beyond_deep_ensembles_b200 import dist as bdist
    from torch.distributed.fsdp.sharded_grad_scaler import ShardedGradScaler

    first = dist.new_group(list(range(world - 1)))       # the optimizer's group: ranks 0 .. R-2
    first_again = dist.new_group(list(range(world - 1)))  # another group object over the same ranks
    last = dist.new_group(list(range(1, world)))          # ranks 1 .. R-1: overlaps, but other ranks
    res = {}
    if rank == world - 1:
        return res
    kw = dict(init_scale=INIT_SCALE)
    scalers = {"plain": torch.amp.GradScaler(dev.type, **kw),
               "sharded_world": ShardedGradScaler(dev.type, process_group=dist.group.WORLD, **kw),
               "sharded_other_ranks": ShardedGradScaler(dev.type, process_group=last, **kw),
               "sharded_same_ranks": ShardedGradScaler(dev.type, process_group=first_again, **kw)}
    assert bdist.world(first) == world - 1 >= 2
    for name, scaler in scalers.items():
        w = torch.nn.Parameter(torch.randn(64, device=dev))
        opt = bde.SwagOptimizer([w], torch.optim.SGD([w], lr=0.1), update_interval=1, deviation_samples=2,
                                process_group=first)
        before = w.detach().clone()
        try:
            opt.init_grad_scaler(scaler)
            opt.step(lambda: (w ** 2).sum(), _scaled_backward(scaler), grad_scaler=scaler)
            res[name] = "ok"
        except ValueError as e:
            res[name] = str(e)
            assert torch.equal(w.detach(), before)
    return res


# ---------------------------------------------------------------------------------------------------- worker
def worker(rank: int, world: int, port: int, out_path: str, backend: str, mode: str):
    """One rank of a spawned job.  mode: "agree" (both families over the default group), "refuse", "autocast"."""
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

        class _Patch:
            def setattr(self, obj, name, value):
                setattr(obj, name, value)
        fake_abi.install(_Patch())
    from beyond_deep_ensembles_b200 import dist as bdist
    group = dist.group.WORLD
    if mode == "agree":
        res = {"slices": run_slices(dev, world, rank, group, True), "wrapped": run_wrapped(dev, world, rank, group, True)}
    elif mode == "refuse":
        res = refusals(dev, world, rank)
    else:
        res = {"wrapped": run_wrapped(dev, world, rank, group, True, algos=("swag", "svgd"), autocast=True)}
    if dev.type == "cuda":
        torch.cuda.synchronize()
    torch.save(res, f"{out_path}.{rank}")
    dist.barrier()
    bdist.shutdown_peer_exchange()
    dist.destroy_process_group()
