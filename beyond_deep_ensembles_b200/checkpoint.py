"""Reference-layout state dicts of the optimizers that run on `ColumnShardedModel`'s column slices.

A D-sharded optimizer over `[sm.param]` exports this rank's slice: one parameter of `[shard]` columns, SWAG's moments
as `[shard]` / `[shard, K]`.  `full_state_dict` turns the ranks' slices into the dict the same class returns when it is
constructed unsharded over the model's own parameters (same keys, indices, shapes, dtypes and devices), so a
checkpoint can be evaluated on one GPU by the plain classes (or the reference's), and `load_full_state_dict` cuts such
a dict — written at any rank count, or by a plain class — back into this rank's slice.  Philox counters are global
column indices, so the resumed job draws the noise the uninterrupted job would have drawn.

Conversion rules, the same for every class:
  per-parameter state  a tensor shaped like `sm.param` is a column vector: the ranks' [k, shard] rows are gathered,
                       cut to the layout (`ColumnShardedModel.logical`) and split into one tensor per model parameter
                       (its shape, on sm.param's device).  Anything else (Adam's `step`, iVON's `None` entries) must
                       agree over the ranks and is repeated for every model parameter.
  optimizer state      (string keys) a tensor whose first dimension is `shard` holds columns along it (SWAG's
                       `__mean`, `__sq_weights` [shard] and roll-order `__deviations` [shard, K]) -> [D, ...] on its
                       own device (the host, for SWAG).  Scalars (`__current_particle`, `__updates`, ...) must agree.
                       `__base_optimizer` becomes None: its state is a dict of its own (`full_state_dict(base)`), and
                       the optimizers keep their own base optimizer when they load a None entry.
  param_groups         SVGD keeps one group per tensor (svgd.py:50): one group per model parameter; the others one
                       group over all of them.  Hyper-parameters must agree over the ranks.
  bde_noise_stream     the furthest rank's position; loading restores it as `load_state_dict` always does.

Loading takes this rank's columns [lo, hi) of every vector; padding columns (between tensors and in the tail) keep the
values the optimizer holds, as the plain classes' `load_state_dict` leaves their arenas' padding alone.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from .algo import BayesianOptimizer

_BASE = "__base_optimizer"
_STREAM = "bde_noise_stream"


# ---------------------------------------------------------------------- which optimizers
def _kind(optimizer):
    from .ivorn import iVONOptimizer
    from .svgd import SVGDOptimizer
    from .swag import SwagOptimizer
    for cls in (SVGDOptimizer, SwagOptimizer, iVONOptimizer):
        if isinstance(optimizer, cls):
            return cls
    if isinstance(optimizer, torch.optim.Optimizer) and not isinstance(optimizer, BayesianOptimizer):
        return torch.optim.Optimizer
    raise ValueError(f"full state dicts cover SVGDOptimizer, SwagOptimizer, iVONOptimizer and torch.optim base "
                     f"optimizers over [sm.param], not {type(optimizer).__name__} (BBBOptimizer keeps its state in "
                     "the modules and shards it per tensor)")


def _check_over(sm, optimizer, kind) -> None:
    params = [p for g in optimizer.param_groups for p in g["params"]]
    if len(params) != 1 or params[0] is not sm.param:
        raise ValueError("the optimizer must be constructed over [sm.param], the ColumnShardedModel's one parameter")
    from . import dist as bdist
    from .ivorn import iVONOptimizer
    from .svgd import SVGDOptimizer
    from .swag import SwagOptimizer
    if kind is SVGDOptimizer:
        world = bdist.world(optimizer._group)
    elif kind is SwagOptimizer:
        world = optimizer._shard.world
    elif kind is iVONOptimizer:
        world = optimizer._arenas[0]["shard"].world
    else:
        return
    if world != sm.world:
        raise ValueError(f"the optimizer is sharded over {world} rank(s), the model over {sm.world}: pass the "
                         "ColumnShardedModel's process_group to the optimizer")


def _fingerprint(obj):
    """A picklable, comparable stand-in for the non-column part of a state dict."""
    if torch.is_tensor(obj):
        return ("tensor", str(obj.dtype), tuple(obj.shape), obj.detach().cpu().tolist())
    if isinstance(obj, dict):
        return {k: _fingerprint(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return (type(obj).__name__, [_fingerprint(v) for v in obj])
    if isinstance(obj, torch.optim.Optimizer):
        return type(obj).__name__
    return obj


def _logical_offsets(layout):
    offs, o = [], 0
    for n in layout.numels:
        offs.append(o)
        o += n
    return offs


def _my_columns(sm, device):
    """(positions in the logical vector, local columns) of the model's elements in this rank's [lo, hi)."""
    idx = sm.layout.logical_index(device)
    pos = ((idx >= sm.lo) & (idx < sm.hi)).nonzero().squeeze(1)
    return pos, idx[pos] - sm.lo


# ---------------------------------------------------------------------- export
def full_state_dict(sm, optimizer) -> dict:
    kind = _kind(optimizer)
    _check_over(sm, optimizer, kind)
    local = optimizer.state_dict()
    state = local["state"]
    entry = state.get(0, {})
    shard = sm.shard

    # every column vector of this rank as [m, shard] rows: ONE gather for the whole dict
    blocks, rows = [], {}
    for key, v in entry.items():
        if torch.is_tensor(v) and v.shape == sm.param.shape:
            rows[(0, key)] = (sum(b.shape[0] for b in blocks), 1)
            blocks.append(v.detach().reshape(1, shard))
    for key, v in state.items():
        if isinstance(key, str) and torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == shard:
            block = v.detach().reshape(shard, -1).t()
            rows[(None, key)] = (sum(b.shape[0] for b in blocks), block.shape[0])
            blocks.append(block)
    rest = {"state": {k: ({kk: vv for kk, vv in v.items() if (0, kk) not in rows} if k == 0 else v)
                      for k, v in state.items() if (None, k) not in rows},
            "param_groups": local["param_groups"],
            **{k: v for k, v in local.items() if k not in ("state", "param_groups", _STREAM)}}
    stream = local.get(_STREAM)
    if sm.world > 1:
        seen = [None] * sm.world
        dist.all_gather_object(seen, ((_fingerprint(rest), sorted(map(str, rows))), stream), group=sm._pg())
        if any(s[0] != seen[0][0] for s in seen):
            raise ValueError("the ranks disagree about the optimizer's scalar state or hyper-parameters")
        if stream is not None:
            stream = max(s[1] for s in seen)
    if blocks:
        if len({b.dtype for b in blocks}) != 1:
            raise ValueError("column state of one optimizer must share one dtype")
        logical = sm.logical(sm.gather_rows(torch.cat([b.to(sm.full.device) for b in blocks])))    # [rows, D]

    layout = sm.layout
    offs = _logical_offsets(layout)
    P = len(layout.numels)
    out_state = {}
    for key, v in state.items():
        if key == 0:
            for k in range(P):
                e = {}
                for kk, vv in v.items():
                    if (0, kk) in rows:
                        r = rows[(0, kk)][0]
                        e[kk] = logical[r, offs[k]:offs[k] + layout.numels[k]].view(layout.shapes[k]).to(vv.device)
                    else:
                        e[kk] = vv.detach().clone() if torch.is_tensor(vv) else vv
                out_state[k] = e
        elif (None, key) in rows:
            r, m = rows[(None, key)]
            out_state[key] = logical[r:r + m].t().reshape((layout.logical_size,) + tuple(v.shape[1:])) \
                .contiguous().to(v.device)
        elif key == _BASE:
            out_state[key] = None
        else:
            out_state[key] = v
    group = {k: v for k, v in local["param_groups"][0].items() if k != "params"}
    from .svgd import SVGDOptimizer
    if kind is SVGDOptimizer:
        groups = [{**group, "params": [k]} for k in range(P)]
    else:
        groups = [{**group, "params": list(range(P))}]
    out = {}
    for key, v in local.items():
        out[key] = out_state if key == "state" else groups if key == "param_groups" else stream if key == _STREAM else v
    return out


# ---------------------------------------------------------------------- import
def _local_dict(sm, optimizer, kind, state_dict) -> dict:
    """The rank-local dict `optimizer.load_state_dict` accepts.  Raises ValueError before anything is written."""
    from .svgd import SVGDOptimizer
    from .swag import SwagOptimizer
    layout = sm.layout
    P, D = len(layout.numels), layout.logical_size
    groups = state_dict["param_groups"]
    ids = [i for g in groups for i in g["params"]]
    if len(ids) != P:
        raise ValueError(f"the state dict holds {len(ids)} parameters, the model {P}")
    if len(groups) != (P if kind is SVGDOptimizer else 1):
        raise ValueError(f"the state dict has {len(groups)} parameter groups; {kind.__name__} over the whole model "
                         f"has {P if kind is SVGDOptimizer else 1}")
    hyper = [{k: v for k, v in g.items() if k != "params"} for g in groups]
    if any(_fingerprint(h) != _fingerprint(hyper[0]) for h in hyper):
        raise ValueError("parameter groups with different hyper-parameters cannot share one sharded parameter")
    saved = state_dict["state"]
    stray = [k for k in saved if not isinstance(k, str) and k not in ids]
    if stray:
        raise ValueError(f"state for parameter indices {stray} that no parameter group lists")

    cur = optimizer.state_dict()                    # padding columns keep these values
    cur_state = cur["state"]
    cur_entry = cur_state.get(0, {})
    dev = sm.param.device
    pos, cols = _my_columns(sm, dev)

    def columns(flat, current, shape_tail, device):
        base = current if torch.is_tensor(current) and current.shape == (sm.shard,) + shape_tail else None
        base = base.detach().clone() if base is not None else torch.zeros((sm.shard,) + shape_tail,
                                                                            dtype=torch.float32, device=device)
        base[cols.to(base.device)] = flat[pos.to(flat.device)].to(base.device, base.dtype)
        return base

    if kind is SVGDOptimizer and saved.get("__particle_count") != optimizer.state["__particle_count"]:
        raise ValueError(f"particle_count {saved.get('__particle_count')} of the state dict differs from this "
                         f"optimizer's {optimizer.state['__particle_count']}")
    if kind is SwagOptimizer:
        K = optimizer.deviation_samples
        for key, shape in (("__mean", (D,)), ("__sq_weights", (D,)), ("__deviations", (D, K))):
            v = saved.get(key)
            if not torch.is_tensor(v) or tuple(v.shape) != shape:
                raise ValueError(f"{key} of the state dict has shape {None if v is None else tuple(v.shape)}, this "
                                 f"optimizer needs {shape} (logical size D = {D}, deviation_samples = {K})")

    entries = [saved.get(i) for i in ids]
    local_state = {}
    if any(e is not None for e in entries):
        if any(e is None for e in entries) or any(set(e) != set(entries[0]) for e in entries):
            raise ValueError("the parameters' state entries hold different keys")
        if kind is SVGDOptimizer:
            need = {f"particle_{i}" for i in range(optimizer.state["__particle_count"])}
            if not need <= set(entries[0]):
                raise ValueError("the state dict lacks particles of this optimizer's particle_count")
        new = {}
        for key in entries[0]:
            vals = [e[key] for e in entries]
            if any(torch.is_tensor(v) and v.dim() > 0 for v in vals):
                for k, v in enumerate(vals):
                    if not torch.is_tensor(v) or tuple(v.shape) != layout.shapes[k]:
                        raise ValueError(f"state[{ids[k]}][{key!r}] has shape "
                                         f"{tuple(v.shape) if torch.is_tensor(v) else type(v).__name__}, the model's "
                                         f"parameter {k} has shape {layout.shapes[k]}")
                flat = torch.cat([v.detach().reshape(-1).to(dev) for v in vals])
                new[key] = columns(flat, cur_entry.get(key), (), dev)
            else:
                if any(_fingerprint(v) != _fingerprint(vals[0]) for v in vals):
                    raise ValueError(f"state entry {key!r} differs between parameters; one sharded parameter holds one")
                new[key] = vals[0].detach().clone() if torch.is_tensor(vals[0]) else vals[0]
        local_state[0] = new
    for key, v in saved.items():
        if not isinstance(key, str):
            continue
        if key == _BASE and _BASE in optimizer.state:
            local_state[key] = optimizer.state[_BASE]          # this job's own base optimizer, whatever was saved
        elif torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == D:
            cv = cur_state.get(key)
            local_state[key] = columns(v.detach(), cv, tuple(v.shape[1:]),
                                       cv.device if torch.is_tensor(cv) else v.device)
        else:
            local_state[key] = v
    out = {k: v for k, v in state_dict.items() if k not in ("state", "param_groups")}
    out["state"] = local_state
    out["param_groups"] = [{**hyper[0], "params": [0]}]
    return out


def load_full_state_dict(sm, optimizer, state_dict: dict) -> None:
    kind = _kind(optimizer)
    _check_over(sm, optimizer, kind)
    optimizer.load_state_dict(_local_dict(sm, optimizer, kind, state_dict))
