"""Improved Variational Online Newton — drop-in for the reference's iVONOptimizer.

Reference: src/algos/ivorn.py:8-127 (the reference spells the module "ivorn").  Per parameter
group the state lives in flat HBM arenas (mean, momentum, precision, delta_sum, acc_grad and the
sampled weights theta that the model parameters alias), so that a step is
  mc_samples x [ K5 sample (1 launch) -> closure fwd/bwd -> K6 gather-accumulate (1 launch) ]
  -> K7 update (1 launch)
instead of ~30 eager ops per tensor.  State-dict keys and shapes match the reference
(state[param]["mean" | "momentum" | "precision" | "delta" | "acc_grad"]).
"""
from __future__ import annotations

import torch
from torch.amp.grad_scaler import OptState

from . import dist as bdist
from . import noise, ops
from .algo import BayesianOptimizer
from .layout import ParamLayout

_ROWS = ("mean", "momentum", "precision", "delta", "acc_grad", "theta")


class iVONOptimizer(BayesianOptimizer):
    """`process_group` (extension, default None = this rank holds every parameter, like the reference): the
    torch.distributed group whose ranks each hold a COLUMN SLICE of every parameter group's state (SURVEY.md §8e).
    Sampling, accumulation and the update stay local; the group only places each rank's slice in the job-wide
    Philox stream (per-element counter = global column index), so the draw does not depend on the rank count."""

    def __init__(self, params, lr, prior_prec, dataset_size, betas=(0.9, 0.999), damping=0.0, tempering=1.0,
                 augmentation=1.0, mc_samples=5, deterministic=False, process_group=None):
        defaults = {
            "lr": lr,
            "betas": betas,
            "prior_prec": prior_prec,
            "damping": damping,
            "tempering": tempering,
            "augmentation": augmentation,
            "N": dataset_size,
            "deterministic": deterministic,
            "step": 0,
        }
        super().__init__(params, defaults)
        ops.require_cuda(*self._params())

        self._arenas = []  # one dict per param_group
        for group in self.param_groups:
            plist = group["params"]
            L = ParamLayout(plist)
            arena = L.new_arena(len(_ROWS), plist[0].device)
            rows = {name: arena[i] for i, name in enumerate(_ROWS)}
            views = {name: L.views(rows[name]) for name in _ROWS}
            with torch.no_grad():
                for k, param in enumerate(plist):
                    views["mean"][k].copy_(param.detach())
                    state = self.state[param]
                    state["mean"] = views["mean"][k]
                    state["momentum"] = views["momentum"][k]
                    state["precision"] = views["precision"][k]
                    state["delta"] = None
                    state["acc_grad"] = None
                # ivorn.py:35: precision starts at prior_prec / N (the padding too, so it stays finite)
                rows["precision"].fill_(group["prior_prec"] / group["N"])
                rows["theta"].copy_(rows["mean"])
                for k, param in enumerate(plist):
                    param.data = views["theta"][k]
            # collective over the group (if any), once per parameter group, in group order on every rank
            shard = bdist.column_shard(L.size, process_group)
            self._arenas.append({"layout": L, "rows": rows, "views": views, "n_samples": 0, "shard": shard})

        assert mc_samples > 0
        self.mc_samples = mc_samples
        # presample(): draws generated ahead of time, handed out by the following sample_parameters() calls
        self._pre_next = self._pre_ready = self._pre_pending = 0

    # ------------------------------------------------------------------ step
    def step(self, forward_closure, backward_closure, grad_scaler=None):
        shard = self._arenas[0]["shard"]
        self._refuse_scaler_if_sharded(grad_scaler, shard.world, shard.group)
        self._reset_state()
        self._drop_presampled(release=True)   # training does not keep the prediction-time sample buffers

        acc_loss = None
        prebind = self._prebind_active(grad_scaler, max(ar["layout"].size for ar in self._arenas),
                                       sum(len(g["params"]) for g in self.param_groups))
        if prebind:
            # zero-copy capture: every MC sample's backward accumulates straight into acc_grad (ivorn.py:120-127 is
            # "acc = grad; acc += grad ..."): one memset per group and step, no gather / accumulate launches
            for ar in self._arenas:
                ar["rows"]["acc_grad"].zero_()
        for _ in range(self.mc_samples):
            # READY so that GradScaler.unscale_ may be called once per MC sample (ivorn.py:47)
            self._set_grad_scaler_state(grad_scaler, OptState.READY)

            self.sample_parameters()
            with torch.enable_grad():
                if prebind:
                    for group, ar in zip(self.param_groups, self._arenas):
                        for param, gview in zip(group["params"], ar["views"]["acc_grad"]):
                            param.grad = gview
                else:
                    self.zero_grad()
                loss = forward_closure()
                backward_closure(loss)

            if acc_loss is None:
                acc_loss = loss
            else:
                acc_loss += loss

            if prebind and self._grads_still_bound():
                for group, ar in zip(self.param_groups, self._arenas):
                    if ar.get("n_grads", 0) == 0:
                        for k, param in enumerate(group["params"]):
                            self.state[param]["acc_grad"] = ar["views"]["acc_grad"][k]
                    ar["n_grads"] = ar.get("n_grads", 0) + 1
                continue
            # gather(-accumulate): prebinding off, AMP, or the closure replaced a .grad (zero_grad inside it) — the
            # arena holds the sum so far (zeros before the first sample), so the ordinary path continues from it
            if not self._store_gradients(grad_scaler):   # unscale (if AMP) + gather-accumulate, one launch per group
                return None
        self._agree_on_found_inf(grad_scaler, shard.world)   # D-sharded: the last sample's flag, all groups raised
        acc_loss /= self.mc_samples

        with torch.no_grad():
            for group, ar in zip(self.param_groups, self._arenas):
                group["step"] += 1
                beta1, beta2 = group["betas"]
                r = ar["rows"]
                ops.ivon_update(r["acc_grad"], r["delta"], r["mean"], r["momentum"], r["precision"],
                                mc_samples=self.mc_samples, step=group["step"], lr=group["lr"], beta1=beta1,
                                beta2=beta2, prior_prec=group["prior_prec"], n_eff=group["N"] * group["augmentation"],
                                tempering=group["tempering"], damping=group["damping"])

        self._set_grad_scaler_state(grad_scaler, OptState.STEPPED)
        return acc_loss

    def _reset_state(self):
        self._drop_presampled()
        for group, ar in zip(self.param_groups, self._arenas):
            ar["n_samples"] = 0
            ar["n_grads"] = 0
            for param in group["params"]:
                state = self.state[param]
                state["delta"] = None
                state["acc_grad"] = None

    def sample_parameters(self):
        """theta = mean + eps / sqrt(N max(prec, 1e-4)); delta_sum (+)= delta (ivorn.py:102-115) — or the next
        row of a presample() batch."""
        if self._pre_ready == 0 and self._pre_pending > 0:
            self._draw_batch()
        if self._pre_ready > 0:
            row = self._pre_next
            self._pre_next += 1
            self._pre_ready -= 1
            for group, ar in zip(self.param_groups, self._arenas):
                for k, param in enumerate(group["params"]):
                    param.data = ar["pre_views"][row][k]
                    self.state[param]["delta"] = ar["views"]["delta"][k]
            return
        for group, ar in zip(self.param_groups, self._arenas):
            L, r, v = ar["layout"], ar["rows"], ar["views"]
            first = ar["n_samples"] == 0
            eps = None
            if not group["deterministic"]:
                eps = noise.draw("ivon", L.logical_size, r["mean"].device)
                if eps is not None:
                    eps = L.from_logical(eps)
            ops.ivon_sample(r["mean"], r["precision"], r["delta"], r["theta"], n_eff=group["N"] * group["augmentation"],
                            first=first, deterministic=bool(group["deterministic"]), eps=eps,
                            seed=self._noise_seed(ar), stream_id=noise.next_stream_id(), elem0=ar["shard"].elem0)
            ar["n_samples"] += 1
            plist = group["params"]
            if first or plist[0].data_ptr() != v["theta"][0].data_ptr():
                for k, param in enumerate(plist):
                    param.data = v["theta"][k]
                    self.state[param]["delta"] = v["delta"][k]

    @staticmethod
    def _noise_seed(ar) -> int:
        """The Philox key: torch's seed, or — D-sharded — the one the group agreed on (rank 0's)."""
        return noise.seed() if ar["shard"].seed is None else ar["shard"].seed

    # ---- batched sampling (SURVEY §8 f3) ----
    #: upper bound of the presample buffers in bytes; larger requests are drawn in several batches
    presample_max_bytes = 1 << 30
    presample_max_rows = 16

    def presample(self, count: int):
        """Announce that the next `count` sample_parameters() calls follow each other without a step() in between
        (what DeepEnsemble.predict does, ensemble.py:37-43): they are generated by ONE K5-batched launch per
        parameter group, reading mean / precision once.  Every draw — and delta_sum afterwards — is bit-identical
        to what `count` single calls produce (same Philox streams, same injected-noise order)."""
        self._drop_presampled()
        self._pre_pending = int(count) if count and count > 1 else 0

    def _drop_presampled(self, release: bool = False):
        """Forget undelivered draws; release=True (every step()) also frees the presample buffers (see swag.py)."""
        self._pre_next = self._pre_ready = self._pre_pending = 0
        if release:
            for ar in self._arenas:
                ar.pop("pre_buf", None)
                ar.pop("pre_views", None)

    def _draw_batch(self):
        groups = len(self.param_groups)
        total = sum(ar["layout"].size for ar in self._arenas)
        rows = int(min(self._pre_pending, self.presample_max_rows, max(1, self.presample_max_bytes // (4 * total))))
        # injected noise is consumed in the order of `rows` sequential calls: one draw per group per call
        eps = [[] for _ in range(groups)]
        for _ in range(rows):
            for g, (group, ar) in enumerate(zip(self.param_groups, self._arenas)):
                if not group["deterministic"]:
                    eps[g].append(noise.draw("ivon", ar["layout"].logical_size, ar["rows"]["mean"].device))
        first_id = noise.reserve_stream_ids(rows * groups)   # call s, group g: first_id + s * groups + g
        for g, (group, ar) in enumerate(zip(self.param_groups, self._arenas)):
            L, r = ar["layout"], ar["rows"]
            if ar.get("pre_buf") is None or ar["pre_buf"].shape[0] < rows:
                ar["pre_buf"] = L.new_arena(rows, r["mean"].device)
                ar["pre_views"] = [L.views(ar["pre_buf"][k]) for k in range(rows)]
            e = None
            if eps[g] and all(z is not None for z in eps[g]):
                e = torch.stack([L.from_logical(z) for z in eps[g]])
            elif any(z is not None for z in eps[g]):
                raise ValueError("a noise injector must supply either every draw of a presampled batch or none")
            ops.ivon_sample_batch(r["mean"], r["precision"], r["delta"], ar["pre_buf"][:rows],
                                  n_eff=group["N"] * group["augmentation"], first=ar["n_samples"] == 0,
                                  deterministic=bool(group["deterministic"]), eps=e, seed=self._noise_seed(ar),
                                  stream_id=first_id + g, stream_stride=groups, elem0=ar["shard"].elem0)
            ar["n_samples"] += rows
        self._pre_next, self._pre_ready = 0, rows
        self._pre_pending -= rows

    def get_base_optimizer(self):
        return self

    def _grads_still_bound(self) -> bool:
        return all(param.grad is gview for group, ar in zip(self.param_groups, self._arenas)
                   for param, gview in zip(group["params"], ar["views"]["acc_grad"]))

    def _store_gradients(self, grad_scaler=None):
        """acc_grad (+)= grad, gathered straight from the scattered .grad tensors (ivorn.py:120-127); under AMP the
        same launch unscales and checks for non-finite values (ivorn.py:60, algo.py:65-73).  False = skip the step."""
        usable = True
        for gi, (group, ar) in enumerate(zip(self.param_groups, self._arenas)):
            L, r, v = ar["layout"], ar["rows"], ar["views"]
            grads = [param.grad for param in group["params"]]
            if any(g is None for g in grads):
                raise TypeError("iVON needs a gradient for every parameter after backward_closure")
            first = ar.get("n_grads", 0) == 0
            if gi == 0:
                usable = self._unscale_and_gather(grad_scaler, None, r["acc_grad"], grads, L, accumulate=not first)
                if not usable:
                    return False
            else:
                # further groups share the scaler record the first group just wrote: gather with the same factor
                self._gather_more(grad_scaler, r["acc_grad"], grads, L, accumulate=not first)
            ar["n_grads"] = ar.get("n_grads", 0) + 1
            if first:
                for k, param in enumerate(group["params"]):
                    self.state[param]["acc_grad"] = v["acc_grad"][k]
        return usable

    def _gather_more(self, grad_scaler, row, grads, layout, accumulate):
        kw = {}
        if grad_scaler is not None and grad_scaler.is_enabled():
            if self.fuse_unscale_into_gather:
                record = grad_scaler._per_optimizer_states[id(self)]
                kw = dict(inv_scale=grad_scaler._scale.double().reciprocal().float(),
                          found_inf=record["found_inf_per_device"][row.device])
            # else: unscale_ of the first group's call already unscaled every .grad of this optimizer in place
        mode = 1 if accumulate else 0
        try:
            ops.multi_tensor_copy(row, grads, layout.offsets, mode=mode, table=layout.copy_table, **kw)
        except ValueError:
            ops.multi_tensor_copy(row, [g.contiguous() for g in grads], layout.offsets, mode=mode,
                                  table=layout.copy_table, **kw)

    # ------------------------------------------------------------------ checkpoints
    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._drop_presampled()
        with torch.no_grad():
            for group, ar in zip(self.param_groups, self._arenas):
                v = ar["views"]
                for k, param in enumerate(group["params"]):
                    state = self.state[param]
                    for name in ("mean", "momentum", "precision", "delta", "acc_grad"):
                        loaded = state.get(name)
                        if loaded is None:
                            continue
                        if loaded.data_ptr() != v[name][k].data_ptr():
                            v[name][k].copy_(loaded)
                        state[name] = v[name][k]
