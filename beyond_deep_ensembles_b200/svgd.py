"""Stein Variational Gradient Descent — drop-in for the reference's SVGDOptimizer.

Reference: src/algos/svgd.py:37-136.  Same constructor, same step()/sample_parameters()
semantics (particle/parameter aliasing, one shared base optimizer stepped once per particle,
persistent particle cursor), same state-dict keys.  The arithmetic of svgd.py:83-97 runs as
two CUDA launches on flat [n, D] arenas: K1 (+K1b) and K2.
"""
from __future__ import annotations

import torch
from torch.amp.grad_scaler import OptState

from . import dist as bdist
from . import ops
from .algo import BayesianOptimizer
from .fused_base import FusedBasePlan
from .layout import ParamLayout


def rbf(particles: torch.Tensor, h_override=None):
    """RBF kernel with the median heuristic and its gradient (reference: svgd.py:14-32).

    Returns (kernel [n, n], grad_kernel [n, D]) like the reference; computed by K1/K1b/K2
    (grad_kernel = A X with l2_reg = 0, dataset_size = kernel_grad_scale = 1 and G = 0).
    """
    X = particles.detach().contiguous().float()
    n, D = X.shape
    if n > ops.FUSED_MAX_PARTICLES and D % 4:
        # the kernels for more than 32 particles need rows 16-byte apart: copy into a padded row stride
        X = torch.zeros(n, (D + 3) // 4 * 4, dtype=X.dtype, device=X.device)[:, :D].copy_(X)
    sc = ops.SvgdScratch.allocate(n, X.device)
    ops.svgd_pairdist(X, sc)
    # out = K*0 + A X with A = c K - c diag(rowsum K), c = 1/h^2  ->  -(grad_kernel)
    ops.svgd_bandwidth(sc, 0.0, 1.0, 1.0, 0.0 if h_override is None else float(h_override))
    ld = X.stride(0)
    out = torch.empty(n, ld, dtype=X.dtype, device=X.device)[:, :D]
    ops.svgd_apply(X, torch.zeros(n, ld, dtype=X.dtype, device=X.device)[:, :D], out, sc)
    return sc.K.clone(), -out.contiguous()


class SVGDOptimizer(BayesianOptimizer):
    """Stein Variational Gradient Descent over `particle_count` particles.

    One param_group per tensor (svgd.py:50); `reset_params_closure` is called
    particle_count - 1 times to initialise the particles (svgd.py:58-63);
    `base_optimizer` must optimise the same parameters.  `process_group` (extension, default None = this rank
    works alone like the reference): the torch.distributed group whose ranks each hold a COLUMN SLICE of every
    particle (SURVEY.md §8e); only then are the n x n partial distances summed across ranks.

    `particle_count` is at most ops.MAX_PARTICLES (64); a larger count raises ValueError.

    `fuse_base_optimizer` (class attribute, default True): when the base optimizer is a stock
    torch.optim.SGD / Adam / AdamW and no GradScaler is active, its n per-particle steps
    (svgd.py:92-103) run inside the apply kernel (fused_base.py); set it to False to always call
    `base_optimizer.step()` per particle.  Above 32 particles (ops.FUSED_MAX_PARTICLES) the fused form does not
    exist: K2 writes the new gradients and the base optimizer steps per particle whatever this attribute says.

    `reuse_pair_distances` (class attribute, default True): the fused launch also computes the pair
    distances of the particles it has just updated (n <= 10), which are exactly what `rbf` needs at the
    next step() — so a training loop reads the particles once per step.  The cached kernel is only valid
    while nothing but this optimizer writes the particles: load_state_dict() and every unfused step drop it, and
    every step() compares autograd's version counters of the particle arena (shared by all `particle_i` views) and
    of the model parameters (which alias the last particle between steps) with the values recorded after the
    launch that produced the cache — any tracked in-place write in between (model.load_state_dict(), weight
    clipping, EMA copies, re-initialisation) drops the cache and K1 runs again.  Writes that bypass the counters
    (`param.data.mul_()`, raw-pointer kernels) must call `invalidate_kernel_cache()` (or set the attribute to False).
    """

    fuse_base_optimizer = True
    reuse_pair_distances = True

    def __init__(self, params, reset_params_closure, base_optimizer, particle_count, dataset_size, l2_reg=0.0,
                 kernel_grad_scale=1.0, process_group=None):
        if particle_count > ops.MAX_PARTICLES:
            raise ValueError(f"SVGDOptimizer supports at most {ops.MAX_PARTICLES} particles, got {particle_count}")
        params = list(params)
        super().__init__(map(lambda p: {"params": p}, params), {})
        self.state["__base_optimizer"] = base_optimizer
        self.state["__l2_reg"] = l2_reg
        self.state["__dataset_size"] = dataset_size
        self.state["__current_particle"] = 0
        self.state["__particle_count"] = particle_count
        self.state["__kernel_grad_scale"] = kernel_grad_scale

        plist = list(self._params())
        ops.require_cuda(*plist)
        device = plist[0].device
        self._layout = ParamLayout(plist)
        n = particle_count
        # HBM layout: particles X, their gradients G and the new gradients OUT as [n, size] arenas
        self._X = self._layout.new_arena(n, device)
        self._G = self._layout.new_arena(n, device)
        self._out_full = None                                # [n, size], only the unfused path needs it
        self._out_last = self._layout.new_arena(1, device)   # new gradient of the last particle (svgd.py:94)
        self._fused_plan = None
        self._scratch = ops.SvgdScratch.allocate(n, device)
        # process_group=None means NOT sharded — the reference is rank-local, and under plain data parallelism (DDP)
        # every rank holds ALL columns of its own particles: summing the pair distances over such replicas would
        # scale d, the median and h^2 by the world size.  D-sharding is opt-in: pass the group whose ranks hold the
        # column slices (torch.distributed.group.WORLD for the default group).
        self._group = bdist.SINGLE if process_group is None else process_group
        # D-sharded on one node: exchange the n*n partial distances inside the kernels (collective over the group)
        bdist.enable_peer_exchange(self._scratch, self._group)
        # what self._scratch holds for the CURRENT particles: None, "partial" (this rank's pair-distance sums,
        # not yet all-reduced) or "kernel" (K, A, info, sel ready)
        self._cached = None
        self._cached_hyper = None
        self._cached_versions = None
        self._xviews = [self._layout.views(self._X[i]) for i in range(n)]
        self._gviews = [self._layout.views(self._G[i]) for i in range(n)]
        self._oviews = None
        self._oviews_last = self._layout.views(self._out_last[0])

        for particle_idx in range(n):
            with torch.no_grad():
                for param, view, gview in zip(plist, self._xviews[particle_idx], self._gviews[particle_idx]):
                    view.copy_(param.detach())
                    self.state[param][f"particle_{particle_idx}"] = view
                    view.grad = gview  # the reference keeps particle gradients in particle.grad (svgd.py:133)
            if particle_idx < n - 1:
                reset_params_closure()

    # ------------------------------------------------------------------ step
    def step(self, forward_closure, backward_closure, grad_scaler=None):
        n = self.state["__particle_count"]
        base = self.state["__base_optimizer"]
        plist = list(self._params())
        losses = []
        prebind = self._prebind_active(grad_scaler, self._layout.size, len(plist))
        scaler_on = grad_scaler is not None and grad_scaler.is_enabled()
        if scaler_on:
            self._refuse_scaler_if_sharded(grad_scaler, bdist.world(self._group))
        if prebind:
            self._G.zero_()   # ONE memset for all particles; autograd then accumulates straight into the arena rows
        for particle_idx in range(n):
            if scaler_on:
                self._set_grad_scaler_state(grad_scaler, OptState.READY, base)
            xviews = self._xviews[particle_idx]
            if prebind:
                gviews = self._gviews[particle_idx]
                for param, xview, gview in zip(plist, xviews, gviews):
                    param.data = xview           # _use_particle (svgd.py:120-127): alias, no copy
                    param.grad = gview           # what base.zero_grad() + the gather of svgd.py:74,129-133 amount to
            elif self._base_owns_exactly(base, plist):
                # base.zero_grad() (svgd.py:74) over exactly these parameters is "grad = None" for each of them; folded into
                # the rebinding loop it saves torch's per-call bookkeeping (~0.1 ms per particle at 96 tensors)
                for param, xview in zip(plist, xviews):
                    param.data = xview
                    param.grad = None
            else:
                for param, xview in zip(plist, xviews):
                    param.data = xview
                base.zero_grad()

            loss = forward_closure()
            losses.append(loss.detach())
            backward_closure(loss)
            if prebind and all(p.grad is g for p, g in zip(plist, gviews)):
                continue                         # the gradients already sit in row particle_idx of G
            # gather: the closure replaced a .grad (zero_grad(set_to_none=True) inside it), AMP, or prebinding off
            if not self._store_grads(particle_idx, plist, grad_scaler, base):   # unscale (if AMP) + gather, one launch
                return None
        # mean over the particles (svgd.py:105) in ONE reduction instead of n accumulate launches
        mean_loss = torch.stack(losses).mean() if n > 1 else losses[0].clone()

        if self._scratch.peers is not None:
            self._scratch.peers.check()   # an abandoned in-kernel exchange (straggler rank) is an error, never silent
        with torch.no_grad():
            hyper = (self.state["__l2_reg"], self.state["__kernel_grad_scale"], self.state["__dataset_size"])
            cached = self._cached if (self.reuse_pair_distances and self._cached_hyper == hyper) else None
            if cached is not None and self._cached_versions != self._write_versions(plist):
                cached = None   # something else wrote a particle since the cache was computed
            self._cached = None
            # (the base optimizer's state is bound BEFORE K1 is enqueued: binding may launch torch fills, and the apply
            # kernel below may only be chained to K1 if nothing else sits between the two on the stream)
            plan = self._plan_for(base, grad_scaler, plist)
            bound = plan.bind_state() if plan is not None else None
            if bound is None:
                _ = self._out   # allocate the [n, size] output arena (first unfused step) before K1 as well
            if cached != "kernel":
                # svgd.py:83-89 on the arenas: K1 -> (all-reduce of n*n doubles when D-sharded) -> K1b
                bdist.svgd_kernel_sharded(self._X, self._scratch, *hyper, 0.0, self._group,
                                          have_partial=(cached == "partial"))
                ops.svgd_chain_next(self._X)   # K2 / K2f follows directly: programmatic dependent launch
            if bound is not None:
                # f1: K2 + the n shared-state base-optimizer steps of svgd.py:92-103 in one pass; X in place.
                # Training-step form (n <= 10): the pass also leaves the next step's pair distances in the
                # scratch; a single rank (or a peer set over NVLink) finishes K1b in the same launch, otherwise the
                # D-sharded ranks all-reduce at the next step.
                nk = None
                if self.reuse_pair_distances and 2 <= n <= ops.NEXT_KERNEL_MAX_PARTICLES:
                    nk = ops.NextKernel(bdist.exchanges_in_kernel(self._scratch, self._group), *hyper)
                if plan.launch(self._X, self._G, self._scratch, self._out_last[0], *bound, next_kernel=nk):
                    self._cached = "kernel" if nk.fuse_bandwidth else "partial"
                    self._cached_hyper = hyper
                    self._cached_versions = self._write_versions(plist)
                for param, xview, oview in zip(plist, self._xviews[n - 1], self._oviews_last):
                    param.grad = oview
                    param.data = xview
            else:
                # svgd.py:92-103 literally: hand the new gradients to the ORIGINAL parameters, alias them to
                # the particle and let the (shared) base optimizer step once per particle
                ops.svgd_apply(self._X, self._G, self._out, self._scratch)
                for particle_idx in range(n):
                    for param, xview, oview in zip(plist, self._xviews[particle_idx], self._oviews[particle_idx]):
                        param.grad = oview
                        param.data = xview
                    if grad_scaler is not None:
                        self._set_grad_scaler_state(grad_scaler, OptState.UNSCALED, base)
                        grad_scaler.step(base)
                    else:
                        base.step()

        return mean_loss

    @property
    def _out(self):
        """[n, size] arena of the new gradients (allocated on first use: the fused path never needs it)."""
        if self._out_full is None:
            n = self.state["__particle_count"]
            self._out_full = self._layout.new_arena(n, self._X.device)
            self._oviews = [self._layout.views(self._out_full[i]) for i in range(n)]
        return self._out_full

    def _plan_for(self, base, grad_scaler, plist):
        if (not self.fuse_base_optimizer or (grad_scaler is not None and grad_scaler.is_enabled())
                or self.state["__particle_count"] > ops.FUSED_MAX_PARTICLES):
            return None
        plan = self._fused_plan
        if plan is None or plan.base is not base or not plan.still_valid():
            plan = self._fused_plan = FusedBasePlan.build(base, plist, self._layout, self._X.device)
        return plan

    def _base_owns_exactly(self, base, plist) -> bool:
        """True when the base optimizer holds exactly this optimizer's parameters, zero_grad defaults to
        set_to_none and nobody hooked or overrode it (checked once per base optimizer object)."""
        cached = getattr(self, "_base_zero_fast", None)
        if cached is None or cached[0] is not base:
            import inspect
            ids = {id(p) for g in base.param_groups for p in g["params"]}
            plain = type(base).zero_grad is torch.optim.Optimizer.zero_grad and "zero_grad" not in vars(base)
            default = inspect.signature(torch.optim.Optimizer.zero_grad).parameters["set_to_none"].default is True
            cached = (base, plain and default and ids == {id(p) for p in plist})
            self._base_zero_fast = cached
        return cached[1]

    def _write_versions(self, plist):
        """Autograd version counters that every tracked in-place write to a particle bumps: the X arena's (shared
        by all of its views, i.e. by every state[param]["particle_i"]) and the model parameters' (own counters)."""
        return (self._X._version, tuple(p._version for p in plist))

    def invalidate_kernel_cache(self):
        """Forget the pair distances computed by the last fused launch (see `reuse_pair_distances`)."""
        self._cached = None

    def sample_parameters(self):
        """Cycles through the particles (svgd.py:107-112)."""
        self._use_particle(self.state["__current_particle"])
        self.state["__current_particle"] = (self.state["__current_particle"] + 1) % self.state["__particle_count"]

    # ------------------------------------------------------------------ helpers
    def _params_for_particle(self, particle_idx):
        particle = f"particle_{particle_idx}"
        for group in self.param_groups:
            for param in group["params"]:
                yield self.state[param][particle]

    def _use_particle(self, particle_idx):
        """No copy: the model parameters alias the particle's arena row (svgd.py:120-127)."""
        for param, view in zip(self._params(), self._xviews[particle_idx]):
            param.data = view

    def _store_grads(self, particle_idx, plist, grad_scaler=None, base=None):
        """This particle's gradients -> row `particle_idx` of G in one launch; under AMP the launch also does what
        `grad_scaler.unscale_(base)` does (svgd.py:78-84, algo.py:65-73).  False = do not use the gradients."""
        grads = [p.grad for p in plist]
        if any(g is None for g in grads):
            raise AttributeError("SVGD needs a gradient for every parameter after backward_closure")
        return self._unscale_and_gather(grad_scaler, base, self._G[particle_idx], grads, self._layout)

    def get_base_optimizer(self):
        return self.state["__base_optimizer"]

    # ------------------------------------------------------------------ checkpoints
    def load_state_dict(self, state_dict):
        """Accepts reference-written state dicts: per-parameter `particle_i` tensors are copied
        into the arena rows and the state keeps pointing at the arena views."""
        super().load_state_dict(state_dict)
        self._cached = None
        n = self.state["__particle_count"]
        if n != self._X.shape[0]:
            raise ValueError("particle_count of the checkpoint differs from this optimizer")
        with torch.no_grad():
            for k, param in enumerate(self._params()):
                for i in range(n):
                    loaded = self.state[param][f"particle_{i}"]
                    view = self._xviews[i][k]
                    if loaded.data_ptr() != view.data_ptr():
                        view.copy_(loaded)
                    view.grad = self._gviews[i][k]
                    self.state[param][f"particle_{i}"] = view
