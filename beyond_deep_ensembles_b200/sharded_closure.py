"""Model closures for D-sharded posteriors (SURVEY.md §8e last note, §8 f4: "a sharded-closure story").

The D-sharded optimizers (`SVGDOptimizer` / `SwagOptimizer` / `iVONOptimizer(process_group=...)`) keep only a
COLUMN SLICE of every particle / moment / state vector on each rank.  The reference has no notion of that: its
closures (algo.py:19-29) run a whole model on whole parameters.  `ColumnShardedModel` is the piece in between:

    full  [R * shard]   every rank: the flat weight vector the model's parameters are views of (layout.ParamLayout:
                        256-byte aligned tensors, zero padding; the tail beyond the layout is padding too)
    param [shard]       this rank's columns [rank * shard, (rank + 1) * shard) — the ONE nn.Parameter handed to the
                        Bayesian optimizer and to its base optimizer
    grad  [R * shard]   every rank: the model's .grad tensors are pre-bound views of it (zero-copy capture, one memset)

    forward closure  =  all-gather(param.data -> full)  +  the user's forward closure           (ONE collective)
    backward closure =  the user's backward closure  +  reduce-scatter(grad -> param.grad)      (ONE collective)

`param.data` is gathered as it is at that moment — the optimizers re-home it (SVGD: the current particle's arena
row, SWAG / iVON: the drawn sample), which is exactly how the reference's closures see "the current parameters".
The reduce-scatter averages over the ranks (every rank may run its own micro-batch: data parallelism over the same
group, the ZeRO arrangement) and ACCUMULATES into an existing `param.grad` like autograd does, so pre-bound
gradient arenas (svgd.py / ivorn.py `prebind_grads`) and MC-sample accumulation keep working.

Equal shards (`shard` = whole 64-element blocks) so that both collectives are the single-buffer forms
(`all_gather_into_tensor`, `reduce_scatter_tensor`: one NCCL ring / NVLS operation each, no staging copies).
With rank r's Philox counters starting at r * shard (dist.column_shard's prefix sum), a D-sharded run over this
closure equals the unsharded run on the same layout: bit for bit for the elementwise family when the ranks see
the same batch, to rounding for SVGD (the n x n distance sums are added in a different order).

Checkpoints (checkpoint.py), two routes; a job saved at R ranks resumes at any other R by either.
`full_state_dict(optimizer)` / `load_full_state_dict(optimizer, state_dict)` convert between a D-sharded optimizer's (or
its base optimizer's) rank slices and the state dict of the same class constructed unsharded over the model's own
parameters, so the plain classes (or the reference's) load and evaluate its checkpoint on one GPU; it puts the whole
unsharded state on every rank.  `shard_state_dict(optimizer)` returns this rank's columns only, on the host, for each
rank to save on its own; `load_shard_state_dicts(optimizer, shards)` reshards the R saved dicts by range arithmetic,
and `checkpoint.consolidate(shards)` turns them into the full dict in one process.  Neither issues a collective.

Mixed precision: each rank checks only its own columns for non-finite gradients, so the D-sharded optimizers accept an
active scaler only as torch's `ShardedGradScaler` over the optimizer's ranks. The ranks then agree on every skipped step
and on the loss scale. Anything else raises in step(). The scaler's `state_dict()` is the same on every rank: a
checkpoint saves it once beside the optimizer's dicts.

Not covered: BBB / Rank-1 layers (their variational parameters live inside the modules and the layers sample in
`forward`; `BBBOptimizer(process_group=...)` shards them per tensor and has neither checkpoint route), D-sharded optimizers
over slices made without this class (their global shapes are unknown to it), module buffers (rank-local, as under DDP
without buffer broadcast, and not part of the optimizer state dicts), `torch.distributed.checkpoint` formats,
non-fp32 parameters.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import checkpoint
from . import dist as bdist
from .layout import ALIGN, ParamLayout


class ColumnShardedModel:
    """Column shards of a model's flat weight vector over `process_group` + the closures that run the model on them.

    `model`: an nn.Module or an iterable of parameters (those with requires_grad are sharded).  Collective over the
    group at construction (rank 0's initial weights are broadcast unless `broadcast_init=False`).
    `average_grads`: reduce-scatter with AVG (data-parallel mean, default) or SUM.

    Checkpoints: `full_state_dict` / `load_full_state_dict` (the reference-layout dict, gathered on every rank: for
    evaluation on one GPU and for jobs whose whole state fits one rank twice) and `shard_state_dict` /
    `load_shard_state_dicts` (each rank saves its own columns, the loader reshards to any rank count; no collective,
    no length-D buffer).  Not covered by either: BBB / Rank-1 layers, module buffers, `torch.distributed.checkpoint`
    formats.
    """

    def __init__(self, model, process_group=None, average_grads: bool = True, broadcast_init: bool = True):
        params = model.parameters() if isinstance(model, torch.nn.Module) else model
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no trainable parameters to shard")
        if any(p.dtype != torch.float32 for p in self.params):
            raise TypeError("ColumnShardedModel shards fp32 parameters (the posterior arenas are fp32)")
        device = self.params[0].device
        if any(p.device != device for p in self.params):
            raise ValueError("all parameters must live on one device")
        self.group = bdist.SINGLE if process_group is None else process_group
        self.world = bdist.world(self.group)
        self.rank = dist.get_rank(self.group) if self.world > 1 else 0
        self.average_grads = bool(average_grads)
        self.layout = ParamLayout(self.params)
        blocks = -(-self.layout.size // ALIGN)
        self.shard = -(-blocks // self.world) * ALIGN           # columns per rank: whole blocks, equal on all ranks
        self.lo, self.hi = self.rank * self.shard, (self.rank + 1) * self.shard
        total = self.world * self.shard
        self.full = torch.zeros(total, dtype=torch.float32, device=device)
        self.grad = torch.zeros(total, dtype=torch.float32, device=device)
        self._wviews = self.layout.views(self.full[: self.layout.size])
        self._gviews = self.layout.views(self.grad[: self.layout.size])
        self._reduced = None                                    # [shard] landing buffer of the reduce-scatter
        with torch.no_grad():
            for p, w in zip(self.params, self._wviews):
                w.copy_(p.detach())
                p.data = w                                      # re-home: the model now computes on `full`
            if broadcast_init and self.world > 1:
                dist.broadcast(self.full, src=self._src0(), group=self._pg())
        #: this rank's columns — the parameter list of the D-sharded optimizer is `[sharded.param]`
        self.param = torch.nn.Parameter(self.full[self.lo:self.hi].clone())
        self.collectives = 0                                    # all-gathers + reduce-scatters issued (tests, bench)

    # ------------------------------------------------------------------ group plumbing
    def _pg(self):
        """The group argument torch.distributed expects (None = default group)."""
        return None if self.group is bdist.SINGLE else self.group

    def _src0(self) -> int:
        """Global rank of the group's rank 0 (what dist.broadcast's `src` counts in)."""
        return 0 if self._pg() is None else dist.get_global_rank(self.group, 0)

    # ------------------------------------------------------------------ weights
    def gather(self) -> None:
        """all-gather the ranks' CURRENT `param.data` into `full` (collective).  Call it after
        `optimizer.sample_parameters()` before an evaluation forward; the training closures do it themselves."""
        src = self.param.data
        if src.numel() != self.shard or src.dtype != torch.float32:
            raise ValueError("the sharded parameter was re-bound to storage of a different size or dtype")
        src = src.reshape(-1)
        if not src.is_contiguous():
            src = src.contiguous()
        with torch.no_grad():
            self._rehome()
            if self.world > 1:
                dist.all_gather_into_tensor(self.full, src, group=self._pg())
                self.collectives += 1
            elif src.data_ptr() != self.full.data_ptr():
                self.full.copy_(src)

    def _rehome(self) -> None:
        """The model's parameters must still be the views of `full` (somebody may have re-bound .data)."""
        for p, w in zip(self.params, self._wviews):
            if p.data_ptr() != w.data_ptr():
                w.copy_(p.detach())
                p.data = w

    def scatter(self) -> None:
        """`param.data` <- this rank's columns of `full` (in place; no collective): after the model's weights were
        written directly (re-initialisation, loading a model state dict)."""
        with torch.no_grad():
            self._rehome()
            self.param.data.view(-1).copy_(self.full[self.lo:self.hi])

    def reset_closure(self, reset_fn, broadcast: bool = True):
        """A `reset_params_closure` for SVGDOptimizer (svgd.py:58-63): `reset_fn()` re-initialises the MODEL; rank
        0's result is broadcast (the ranks' RNGs need not agree) and this rank's columns land in `param`."""
        def reset():
            reset_fn()
            with torch.no_grad():
                self._rehome()
                if broadcast and self.world > 1:
                    dist.broadcast(self.full, src=self._src0(), group=self._pg())
            self.scatter()
        return reset

    # ------------------------------------------------------------------ closures
    def closures(self, forward_closure, backward_closure):
        """(forward_closure, backward_closure) in the reference's convention (algo.py:19-29) for a D-sharded
        optimizer over `[self.param]`: the forward gathers the weights, the backward hands this rank's columns of
        the (averaged) gradient to `param.grad`."""
        def forward():
            self.gather()
            return forward_closure()

        def backward(loss):
            self.grad.zero_()                                   # ONE memset; autograd accumulates into the views
            for p, g in zip(self.params, self._gviews):
                p.grad = g
            backward_closure(loss)
            self.reduce_grads()
        return forward, backward

    def reduce_grads(self) -> None:
        """reduce-scatter the model's gradients over the group into `param.grad` (collective; accumulates into an
        existing `param.grad`, like autograd)."""
        with torch.no_grad():
            for p, g in zip(self.params, self._gviews):
                if p.grad is not g:                             # the closure replaced a .grad (zero_grad inside it)
                    if p.grad is None:
                        g.zero_()
                    else:
                        g.copy_(p.grad)
                    p.grad = g
            if self.world > 1:
                if self._reduced is None:
                    self._reduced = torch.empty(self.shard, dtype=torch.float32, device=self.grad.device)
                op = dist.ReduceOp.AVG if self.average_grads else dist.ReduceOp.SUM
                dist.reduce_scatter_tensor(self._reduced, self.grad, op=op, group=self._pg())
                self.collectives += 1
                mine = self._reduced
            else:
                mine = self.grad[self.lo:self.hi]
            target = self.param.grad
            if target is None:
                self.param.grad = mine.clone().view_as(self.param)
            else:
                target.add_(mine.view_as(target))

    # ------------------------------------------------------------------ export
    def logical(self, flat: torch.Tensor) -> torch.Tensor:
        """[..., R * shard] (concatenated rank slices) -> [..., D] in the reference's parameters_to_vector order."""
        return self.layout.to_logical(flat[..., : self.layout.size])

    def gather_rows(self, rows: torch.Tensor) -> torch.Tensor:
        """[k, shard] per-rank state rows (particles, moments) -> [k, R * shard] on every rank (collective; export
        and tests only)."""
        rows = rows.reshape(-1, self.shard).contiguous()
        if self.world == 1:
            return rows.clone()
        parts = [torch.empty_like(rows) for _ in range(self.world)]
        dist.all_gather(parts, rows, group=self._pg())
        return torch.cat(parts, dim=1)

    # ------------------------------------------------------------------ checkpoints
    def full_state_dict(self, optimizer) -> dict:
        """The state dict `optimizer`'s class returns when constructed UNSHARDED over the model's own parameters
        (`model.parameters()`, same order) after the same steps: same keys, per-parameter indices, shapes, dtypes and
        devices, and `bde_noise_stream` (the furthest rank's).  `optimizer`: a SVGDOptimizer / SwagOptimizer /
        iVONOptimizer over `[self.param]` with this group, or the torch.optim base optimizer over `[self.param]`.
        `__base_optimizer` is None: save `full_state_dict(base)` beside it.

        Collective over the group (one all_gather_object, one all_gather); every rank gets the same dict.  Memory:
        what the unsharded optimizer holds — every column vector at full length D on `param`'s device on EVERY rank
        (SVGD: n particles x D, iVON: 5 x D), SWAG's mean, second moment and [D, K] deviations on the host — plus one
        [rows, R * shard] gather buffer on the device while it runs."""
        return checkpoint.full_state_dict(self, optimizer)

    def load_full_state_dict(self, optimizer, state_dict: dict) -> None:
        """The inverse of `full_state_dict`: this rank's columns [lo, hi) of every vector, handed to the optimizer's own
        `load_state_dict`.  Accepts a dict written by `full_state_dict` at any rank count, or by the plain class over
        the model's parameters (this package's or the reference's).  The optimizer keeps its own base optimizer; load
        the base optimizer's dict into it the same way.  No collective.

        Raises ValueError — before anything is written — for another logical size or parameter shape, an optimizer
        not over `[self.param]`, another `particle_count` / `deviation_samples`, or BBBOptimizer."""
        checkpoint.load_full_state_dict(self, optimizer, state_dict)

    def shard_state_dict(self, optimizer) -> dict:
        """This rank's part of a per-rank checkpoint: a plain, picklable dict of `optimizer`'s rank-local state dict
        (every tensor copied to the host, `__base_optimizer` None) and the column geometry — `format`, `version`,
        `kind` (the optimizer's class name), `world`, `rank`, `shard`, `lo`, `hi` and the model's parameter `shapes`.
        Nothing in it has length D.  `optimizer`: as for `full_state_dict`.  No collective: each rank
        `torch.save`s its own dict.  Memory: one host copy of the rank-local state."""
        return checkpoint.shard_state_dict(self, optimizer)

    def load_shard_state_dicts(self, optimizer, shards) -> None:
        """Load the R dicts `shard_state_dict` returned on the ranks of a saving job (any order, any R, typically
        `torch.load(..., mmap=True)`): this rank's columns are cut from the saved shards that overlap [lo, hi), padding
        columns keep the optimizer's values, and the rank-local dict goes to the optimizer's own `load_state_dict` —
        the same dict `load_full_state_dict` builds from the full dict of that job.  No collective.

        Raises ValueError — before anything is written — for dicts of another format, shards that do not tile the
        saving job's columns exactly once, another logical size or parameter shape, another optimizer class, another
        `particle_count` / `deviation_samples`, shards that disagree about a scalar, or BBBOptimizer."""
        checkpoint.load_shard_state_dicts(self, optimizer, shards)
