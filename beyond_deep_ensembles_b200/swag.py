"""Stochastic Weight Averaging-Gaussian — drop-in for the reference's SwagOptimizer.

Reference: src/algos/swag.py:10-114.  The reference keeps mean / second moment / [D, K]
deviations on the HOST and moves the whole parameter vector D2H on every update (swag.py:100)
and (K+2)*D floats H2D before sampling (swag.py:112-114).  Here everything lives in HBM:
  theta  [size]     the training weights (the model's parameters are views of it),
  mean, sq [size]   running moments,
  dev    [K, size]  deviation ring buffer (row updates % K is overwritten next; no roll),
  sample [size]     the last drawn weights (parameters alias it between sample and step).
state_dict()/load_state_dict() convert to/from the reference layout (`__mean`, `__sq_weights`
as [D] CPU tensors, `__deviations` as [D, K] CPU tensor in roll order).
"""
from __future__ import annotations

import math

import torch

from . import dist as bdist
from . import noise, ops
from .algo import BayesianOptimizer
from .layout import ParamLayout


class SwagOptimizer(BayesianOptimizer):
    """`process_group` (extension, default None = this rank holds every parameter, like the reference): the
    torch.distributed group whose ranks each hold a COLUMN SLICE of the weights and of every moment (SURVEY.md
    §8e).  No kernel on this path exchanges data; the group only fixes the noise: the K low-rank coefficients are
    identical on all ranks, the per-weight normals are the ranks' disjoint parts of one Philox stream."""

    def __init__(self, params, base_optimizer, update_interval, start_epoch=0, deviation_samples=30,
                 process_group=None):
        super().__init__(params, {})

        self.start_epoch = start_epoch
        self.update_interval = math.floor(update_interval)
        self.deviation_samples = deviation_samples

        plist = list(self._params())
        ops.require_cuda(*plist)
        device = plist[0].device
        self._layout = ParamLayout(plist)
        L = self._layout
        self._shard = bdist.column_shard(L.size, process_group)   # collective over the group (if any)
        self._theta = L.new_arena(1, device)[0]
        self._sample = L.new_arena(1, device)[0]
        self._mean = L.new_arena(1, device)[0]
        self._sq = L.new_arena(1, device)[0]
        self._dev = L.new_arena(deviation_samples, device)
        self._tviews = L.views(self._theta)
        self._sviews = L.views(self._sample)
        # presample(): rows drawn ahead of time, handed out by the following sample_parameters() calls
        self._pre_buf = None      # [rows, size]
        self._pre_views = []      # per-row parameter views
        self._pre_next = 0        # next row of _pre_buf to hand out
        self._pre_ready = 0       # rows of _pre_buf that hold undelivered draws
        self._pre_pending = 0     # draws promised by presample() but not generated yet

        with torch.no_grad():
            for param, tview in zip(plist, self._tviews):
                tview.copy_(param.detach())
                param.data = tview  # re-home: base-optimizer updates now land in the arena
                self.state[param]["original_param"] = tview
            # swag.py:32-33: the initial weights count as sample 0 of both moments
            self._mean.copy_(self._theta)
            torch.mul(self._theta, self._theta, out=self._sq)

        self.state["__base_optimizer"] = base_optimizer
        self.state["__epoch"] = 0
        self.state["__steps_since_swag_start"] = 0
        self.state["__updates"] = 0
        self.state["__params_dirty"] = False

    # ------------------------------------------------------------------ step
    def step(self, forward_closure, backward_closure, grad_scaler=None):
        # no gather on this path: grad_scaler.step(base) runs the scaler's own unscale_, which a ShardedGradScaler agrees
        self._refuse_scaler_if_sharded(grad_scaler, self._shard.world, self._shard.group)
        self._drop_presampled(release=True)   # the posterior is about to change; training does not keep the buffer
        self._restore_original_params()
        base = self.state["__base_optimizer"]
        base.zero_grad()

        loss = forward_closure()
        backward_closure(loss)

        if grad_scaler is not None:
            grad_scaler.step(base)
        else:
            base.step()

        self._swag_update()
        return loss

    def sample_parameters(self):
        """theta~ = mean + Dev z / sqrt(2(K-1)) + sqrt(diag) eps (swag.py:53-58, 107-114), one launch —
        or the next row of a presample() batch."""
        self._save_original_params()
        self.state["__params_dirty"] = True
        if self._pre_ready == 0 and self._pre_pending > 0:
            self._draw_batch()
        if self._pre_ready > 0:
            views = self._pre_views[self._pre_next]
            self._pre_next += 1
            self._pre_ready -= 1
            for param, view in zip(self._params(), views):
                param.data = view
            return
        K, dev_ = self.deviation_samples, self._theta.device
        eps_k = noise.draw("swag_k", K, dev_)
        eps_d = noise.draw("swag_d", self._layout.logical_size, dev_)
        if eps_d is not None:
            eps_d = self._layout.from_logical(eps_d)
        ops.swag_sample(self._mean, self._sq, self._dev, self.state["__updates"] % K, self._sample, eps_k=eps_k,
                        eps_d=eps_d, seed=self._noise_seed(), stream_id=noise.next_stream_id(),
                        elem0=self._shard.elem0)
        for param, sview in zip(self._params(), self._sviews):
            param.data = sview

    def _noise_seed(self) -> int:
        """The Philox key: torch's seed, or — D-sharded — the one the group agreed on (rank 0's)."""
        return noise.seed() if self._shard.seed is None else self._shard.seed

    # ---- batched sampling (SURVEY §8 f3) ----
    #: upper bound of the presample buffer in bytes; larger requests are drawn in several batches
    presample_max_bytes = 1 << 30
    #: draws generated per _draw_batch call (the kernel reads the moments once per 16 draws: more rows save nothing)
    presample_max_rows = 16

    def presample(self, count: int):
        """Announce that the next `count` sample_parameters() calls draw from the CURRENT posterior (what
        DeepEnsemble.predict does, ensemble.py:37-43): they are generated by one K4-batched launch per 16 draws,
        reading the moments and the deviation matrix once instead of once per draw.  Every draw is bit-identical
        to the one sample_parameters() would have produced on its own (same Philox streams, same injected-noise
        order); each handed-out sample lives in its own row, so earlier samples stay valid until step()."""
        self._drop_presampled()
        self._pre_pending = max(int(count), 0) if count and count > 1 else 0

    def _drop_presampled(self, release: bool = False):
        """Forget undelivered draws; release=True (every step()) also returns the buffer to the allocator, so one
        predict() during validation does not pin up to presample_max_bytes per ensemble member for the rest of
        training (the parameters were re-homed to the sample arena before this is called)."""
        self._pre_ready = self._pre_pending = self._pre_next = 0
        if release:
            self._pre_buf = None
            self._pre_views = []

    def _draw_batch(self):
        L, K, dev_ = self._layout, self.deviation_samples, self._theta.device
        size = self._theta.numel()
        rows = int(min(self._pre_pending, self.presample_max_rows, max(1, self.presample_max_bytes // (4 * size))))
        if self._pre_buf is None or self._pre_buf.shape[0] < rows:
            self._pre_buf = L.new_arena(rows, dev_)
            self._pre_views = [L.views(self._pre_buf[r]) for r in range(rows)]
        # injected noise is consumed in the order of `rows` sequential calls: (swag_k, swag_d) per draw
        eps_k, eps_d = [], []
        for _ in range(rows):
            eps_k.append(noise.draw("swag_k", K, dev_))
            eps_d.append(noise.draw("swag_d", L.logical_size, dev_))
        ek = torch.stack(eps_k) if all(e is not None for e in eps_k) else None
        ed = torch.stack([L.from_logical(e) for e in eps_d]) if all(e is not None for e in eps_d) else None
        if (ek is None and any(e is not None for e in eps_k)) or (ed is None and any(e is not None for e in eps_d)):
            raise ValueError("a noise injector must supply either every draw of a presampled batch or none")
        ops.swag_sample_batch(self._mean, self._sq, self._dev, self.state["__updates"] % K, self._pre_buf[:rows],
                              eps_k=ek, eps_d=ed, seed=self._noise_seed(), stream_id=noise.reserve_stream_ids(rows),
                              elem0=self._shard.elem0)
        self._pre_next, self._pre_ready = 0, rows
        self._pre_pending -= rows

    def complete_epoch(self):
        self.state["__epoch"] += 1

    def get_base_optimizer(self):
        return self.state["__base_optimizer"]

    # ------------------------------------------------------------------ helpers
    def _restore_original_params(self):
        if self.state["__params_dirty"]:
            for param, tview in zip(self._params(), self._tviews):
                param.data = tview
            self.state["__params_dirty"] = False

    def _save_original_params(self):
        if not self.state["__params_dirty"]:
            self._sync_theta()

    def _sync_theta(self):
        """The training weights normally ARE the theta arena.  If a caller re-bound param.data
        to other storage, gather it back (one launch) and re-home the parameters."""
        plist = list(self._params())
        if all(p.data_ptr() == v.data_ptr() for p, v in zip(plist, self._tviews)):
            return
        with torch.no_grad():
            ops.multi_tensor_copy(self._theta, [p.detach().contiguous() for p in plist], self._layout.offsets, mode=0,
                                  table=self._layout.copy_table)
            for param, tview in zip(plist, self._tviews):
                param.data = tview

    def _swag_update(self):
        if self.state["__epoch"] >= self.start_epoch:
            self.state["__steps_since_swag_start"] += 1

            if self.state["__steps_since_swag_start"] % self.update_interval == 0:
                assert not self.state["__params_dirty"]
                with torch.no_grad():
                    self._sync_theta()
                    self.state["__updates"] += 1
                    updates = self.state["__updates"]
                    row = (updates - 1) % self.deviation_samples
                    ops.swag_update(self._theta, self._mean, self._sq, self._dev[row], updates)

    # ------------------------------------------------------------------ checkpoints
    def _export_moments(self):
        L = self._layout
        K, u = self.deviation_samples, self.state["__updates"]
        order = [(u % K + k) % K for k in range(K)]  # oldest ... newest = the reference's roll order
        dev = L.to_logical(self._dev[order])          # [K, D]
        return (L.to_logical(self._mean).cpu(), L.to_logical(self._sq).cpu(), dev.t().contiguous().cpu())

    def state_dict(self):
        mean, sq, dev = self._export_moments()
        self.state["__mean"], self.state["__sq_weights"], self.state["__deviations"] = mean, sq, dev
        try:
            return super().state_dict()
        finally:
            for key in ("__mean", "__sq_weights", "__deviations"):
                del self.state[key]

    def load_state_dict(self, state_dict: dict):
        super().load_state_dict(state_dict)
        self._drop_presampled()
        L, dev_ = self._layout, self._theta.device
        mean = self.state.pop("__mean").to(dev_).float()
        sq = self.state.pop("__sq_weights").to(dev_).float()
        dev = self.state.pop("__deviations").to(dev_).float()  # [D, K], column K-1 newest
        K, u = self.deviation_samples, self.state["__updates"]
        if dev.shape != (L.logical_size, K):
            raise ValueError("checkpoint deviations do not match this optimizer (D, deviation_samples)")
        with torch.no_grad():
            L.from_logical(mean, out=self._mean)
            L.from_logical(sq, out=self._sq)
            ring = L.from_logical(dev.t().contiguous())          # logical column k -> row (u + k) % K
            for k in range(K):
                self._dev[(u % K + k) % K].copy_(ring[k])
            # parameters: keep whatever the model holds, re-homed into the arena
            for param, tview in zip(self._params(), self._tviews):
                loaded = self.state[param].get("original_param")
                if self.state["__params_dirty"] and loaded is not None:
                    tview.copy_(loaded)
                self.state[param]["original_param"] = tview
            if not self.state["__params_dirty"]:
                self._sync_theta()
