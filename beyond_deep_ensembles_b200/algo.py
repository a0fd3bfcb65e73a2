"""BayesianOptimizer base API and the last-layer wrapper.

Mirrors the reference's public surface (src/algos/algo.py:5-133): same class names, method
names, argument meaning and error behaviour, so training loops written against the reference
(`loss = optimizer.step(forward_closure, backward_closure, grad_scaler=scaler)`,
`optimizer.complete_epoch()`, `optimizer.sample_parameters()`, `get_base_optimizer()`,
`init_grad_scaler()`) run unchanged.  The only arithmetic reachable from this file is the gradient gather of
`_unscale_and_gather` (one C-ABI launch).
"""
from __future__ import annotations

from typing import Any, Dict

import torch
from torch.amp.grad_scaler import OptState
from torch.optim import Optimizer


def _scaler_active(grad_scaler) -> bool:
    return grad_scaler is not None and grad_scaler.is_enabled()


class BayesianOptimizer(Optimizer):
    """An optimizer over a distribution of parameters (reference: algo.py:5-81).

    step() owns the forward/backward passes: `forward_closure()` returns the loss without
    calling backward or clearing gradients, `backward_closure(loss)` runs one backward pass
    (calling grad_scaler.scale(loss) itself when AMP is used).
    """

    def __init__(self, params, defaults):
        super().__init__(params, defaults)
        # tells torch's GradScaler that step() deals with the loss scale itself (algo.py:17)
        self._step_supports_amp_scaling = True

    # ---- checkpoints: the reference's layout plus the position of the Philox stream counter ----
    def state_dict(self):
        """torch's layout (and the reference's keys); one extra top-level entry, ignored by torch / the reference
        when they load it: how many Philox noise streams have been used, so a resumed run does not replay them."""
        from . import noise
        sd = super().state_dict()
        sd["bde_noise_stream"] = noise.stream_position()
        return sd

    def load_state_dict(self, state_dict):
        from . import noise
        base = self.state.get("__base_optimizer")
        super().load_state_dict(state_dict)
        if base is not None and self.state.get("__base_optimizer", base) is None:
            # a full state dict of a D-sharded job (ColumnShardedModel.full_state_dict) carries no base optimizer
            # object (its state is a dict of its own): keep this optimizer's
            self.state["__base_optimizer"] = base
        noise.restore_stream_position(state_dict.get("bde_noise_stream"))

    # ---- what subclasses implement (algo.py:19-56) ----
    def step(self, forward_closure, backward_closure):
        raise NotImplementedError()

    def sample_parameters(self):
        raise NotImplementedError()

    def complete_epoch(self):
        """End-of-epoch bookkeeping; nothing by default."""

    def get_base_optimizer(self):
        """The optimizer that makes the actual parameter updates (the one LR schedulers attach to)."""

    # ---- GradScaler plumbing (algo.py:44-49, 65-81) ----
    def init_grad_scaler(self, grad_scaler):
        # GradScalers initialise lazily on the first step/unscale; the optimizers poke at the
        # per-optimizer state before that, so force the initialisation here.
        if _scaler_active(grad_scaler) and grad_scaler._scale is None:
            grad_scaler._lazy_init_scale_growth_tracker(self._params_device())

    def _prepare_and_check_grads(self, grad_scaler, optimizer=None):
        """Unscale the gradients held by `optimizer` (default: self); True when they may be used."""
        if not _scaler_active(grad_scaler):
            return True
        grad_scaler.unscale_(optimizer if optimizer is not None else self)
        # Kept literally from algo.py:73: this reads the OPTIMIZER's state dict (a defaultdict,
        # so the key springs into existence as {}), not the scaler's found-inf record, hence it
        # is always True — the reference's behaviour, which callers have been trained against.
        found = self.state["found_inf_per_device"]
        return sum(flag.item() for flag in found.values()) == 0

    def _set_grad_scaler_state(self, grad_scaler, stage, optimizer=None):
        if _scaler_active(grad_scaler):
            key = id(optimizer if optimizer is not None else self)
            grad_scaler._per_optimizer_states[key]["stage"] = stage

    def _refuse_scaler_if_sharded(self, grad_scaler, world: int, group=None) -> None:
        """D-sharded optimizers (process_group=`group`) see one rank's columns only, so the non-finite check of an
        active GradScaler must be agreed over the group, or the ranks could disagree about skipping a step and back
        the loss scale off differently.  torch's ShardedGradScaler over the same ranks agrees: its unscale_
        all-reduces found_inf over its process group, and the fused gather route agrees on its flag in
        `_agree_on_found_inf`.  Any other active scaler (a plain GradScaler, a look-alike, a ShardedGradScaler over
        other ranks) is refused loudly."""
        if world <= 1 or not _scaler_active(grad_scaler):
            return
        from torch.distributed.fsdp.sharded_grad_scaler import ShardedGradScaler
        from . import dist as bdist
        if not (isinstance(grad_scaler, ShardedGradScaler) and bdist.same_ranks(grad_scaler.process_group, group)):
            raise ValueError("a D-sharded optimizer (process_group=...) supports an active GradScaler only as a "
                             "torch.distributed.fsdp.sharded_grad_scaler.ShardedGradScaler over the same ranks: the "
                             "non-finite check has to be agreed over the group")

    def _agree_on_found_inf(self, grad_scaler, world: int, optimizer=None) -> None:
        """D-sharded, fused route: MAX over the group of the non-finite flag the gathers of this step left in the
        scaler's record for `optimizer` (default: self), so every rank's grad_scaler.step() / update() decide as the
        unsharded job does.  The reference route needs nothing here (ShardedGradScaler.unscale_ agrees itself).

        Called ONCE per step, after the last gather, not once per gather.  Every gather writes a fresh flag into the
        record, as unscale_ does, and nothing reads it before the next gather replaces it: `_unscale_and_gather`
        returns the literal algo.py:73 check, which reads the optimizer's own state, never the scaler's.  What the
        scaler decides on (SVGD's grad_scaler.step(base) per particle, then update()) is the record after the
        last gather of the step, and the MAX of that flag over the ranks is exactly the unsharded flag.  iVON needs
        the agreement after its last parameter group, too: `_gather_more` raises the same flag."""
        if world <= 1 or not (_scaler_active(grad_scaler) and self.fuse_unscale_into_gather):
            return
        from . import dist as bdist
        record = grad_scaler._per_optimizer_states[id(self if optimizer is None else optimizer)]
        for flag in record["found_inf_per_device"].values():
            bdist.allreduce_max_(flag, grad_scaler.process_group)

    #: with an active GradScaler, fold unscale_ + the non-finite check into the gradient gather (SURVEY §8 f2)
    fuse_unscale_into_gather = True

    #: zero-copy gradient capture (SURVEY §8 f2): before each backward pass every `param.grad` is bound to its slice of
    #: the flat gradient arena (zeroed once per step), so autograd accumulates straight into the arena and the
    #: per-particle / per-sample gather launch disappears.  "auto" = only for FEW, SMALL tensors: with a bound .grad
    #: autograd's AccumulateGrad launches one in-place add per parameter (96 per backward pass for ResNet-20, where the
    #: gather is ONE multi-tensor launch) and moves 12 D bytes per pass against 8 D for the gather.  Measured A/B with
    #: real closures (profiles/r02_prebind_ab.json): UCI MLP (4 tensors) overhead 1.20 -> 0.34 ms per step, ResNet-20
    #: x 20 particles 3.8 -> 4.4-6.4 ms, DistilBERT iVON +0.74 ms.  True / False force it.  Never used with an active
    #: GradScaler (the gather then also unscales).
    prebind_grads = "auto"
    prebind_auto_max_elements = 8_000_000
    prebind_auto_max_tensors = 16

    def _prebind_active(self, grad_scaler, row_elements: int, tensors: int = 0) -> bool:
        if _scaler_active(grad_scaler) or self.prebind_grads is False:
            return False
        return self.prebind_grads is True or (row_elements <= self.prebind_auto_max_elements
                                              and tensors <= self.prebind_auto_max_tensors)

    def _unscale_and_gather(self, grad_scaler, optimizer, row, grads, layout, accumulate=False):
        """Gradients of the pass that just ran -> the flat arena `row` (gather, or gather-add).  Returns what
        `_prepare_and_check_grads` returns.

        Without a scaler this is one multi-tensor launch.  With an active GradScaler the reference first runs
        `grad_scaler.unscale_(optimizer)` — a read-modify-write pass over every gradient plus the non-finite check
        (algo.py:65-73) — and gathers afterwards; here both happen in the gather launch: the values are multiplied
        by 1/scale on their way into the arena and `found_inf` is raised on the device, and the scaler's
        per-optimizer record is left exactly as `unscale_` leaves it (stage UNSCALED, found_inf_per_device), so
        `grad_scaler.step()` / `update()` behave as before.  The `.grad` tensors themselves stay scaled; the
        optimizers replace them before anything reads them again."""
        from . import ops
        opt = self if optimizer is None else optimizer
        mode = 1 if accumulate else 0

        def gather(**kw):
            try:
                ops.multi_tensor_copy(row, grads, layout.offsets, mode=mode, table=layout.copy_table, **kw)
            except ValueError:   # e.g. channels_last gradients: gather from contiguous copies
                ops.multi_tensor_copy(row, [g.contiguous() for g in grads], layout.offsets, mode=mode,
                                      table=layout.copy_table, **kw)

        if _scaler_active(grad_scaler) and self.fuse_unscale_into_gather:
            record = grad_scaler._per_optimizer_states[id(opt)]
            if record["stage"] is OptState.UNSCALED:
                raise RuntimeError("unscale_() has already been called on this optimizer since the last update().")
            if record["stage"] is OptState.STEPPED:
                raise RuntimeError("unscale_() is being called after step().")
            scale = grad_scaler._scale
            assert scale is not None, "call init_grad_scaler(grad_scaler) before the first step"
            inv_scale = scale.double().reciprocal().float()
            found_inf = torch.full((), 0.0, dtype=torch.float32, device=scale.device)
            gather(inv_scale=inv_scale, found_inf=found_inf)
            record["found_inf_per_device"] = {found_inf.device: found_inf}
            record["stage"] = OptState.UNSCALED
            return sum(flag.item() for flag in self.state["found_inf_per_device"].values()) == 0   # algo.py:73, literally
        usable = self._prepare_and_check_grads(grad_scaler, optimizer)
        if usable:
            gather()
        return usable

    # ---- parameter access (algo.py:57-63) ----
    def _params(self):
        for group in self.param_groups:
            yield from group["params"]

    def _params_device(self):
        return next(self._params()).device


class LastLayerBayesianOptimizer(BayesianOptimizer):
    """Bayesian last layer + deterministic body (reference: algo.py:83-133).

    The deterministic gradients are zeroed once and ACCUMULATE over all forward/backward
    passes the Bayesian optimizer makes inside its step before the deterministic optimizer
    steps — exactly the reference's order (algo.py:100-103).  GradScalers are refused, as there.
    """

    _PARTS = ("ll_bayesian_optimizer", "deterministic_optimizer")

    def __init__(self, ll_bayesian_optimizer: BayesianOptimizer, deterministic_optimizer: Optimizer):
        # deliberately no super().__init__(): the reference does not call it either
        self.ll_bayesian_optimizer = ll_bayesian_optimizer
        self.deterministic_optimizer = deterministic_optimizer

    def step(self, forward_closure, backward_closure, grad_scaler=None):
        if _scaler_active(grad_scaler):
            raise ValueError("Doesn't support grad scaler")
        body, head = self.deterministic_optimizer, self.ll_bayesian_optimizer
        body.zero_grad()
        loss = head.step(forward_closure, backward_closure)   # >= 1 backward pass: fills the body's gradients too
        body.step()
        return loss

    def init_grad_scaler(self, grad_scaler):
        if grad_scaler.is_enabled():
            raise RuntimeError("Doesn't support grad scaler")

    def get_base_optimizer(self):
        raise RuntimeError("There is no defined base optimizer on the ll optimizer. Call get_base_optimizer directly "
                           "on the passed ll bayesian optimizer")

    def complete_epoch(self):
        self.ll_bayesian_optimizer.complete_epoch()

    def sample_parameters(self):
        self.ll_bayesian_optimizer.sample_parameters()

    def presample(self, count):
        """Forward DeepEnsemble.predict's batch announcement to the Bayesian part (no-op if it cannot batch)."""
        announce = getattr(self.ll_bayesian_optimizer, "presample", None)
        if announce is not None:
            announce(count)

    def state_dict(self) -> Dict[str, Any]:
        return {part: getattr(self, part).state_dict() for part in self._PARTS}

    def load_state_dict(self, state_dict: Dict[str, Any]) -> None:
        for part in self._PARTS:
            getattr(self, part).load_state_dict(state_dict[part])

    def __repr__(self) -> str:
        bar = "=" * 34
        return (f"LL Bayesian Optimizer: \n\n{self.ll_bayesian_optimizer!r}\n{bar}\n"
                f"Deterministic Optimizer:\n\n{self.deterministic_optimizer!r}")
