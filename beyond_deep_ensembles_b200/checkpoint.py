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

Per-rank dicts (`shard_state_dict`, format FORMAT): a rank's own state dict on the host plus its column geometry, written
with no collective.  `load_shard_state_dicts` cuts this rank's columns out of the R saved dicts by range arithmetic in
layout space (layout column c of saved shard s is its column c - lo_s; the layout depends only on the parameter shapes)
and reads only the shards that overlap [lo, hi); `consolidate` joins them into the full dict in one process.  Both use
the rules above: the same column classification, scalar agreement and padding rule, so they build the same dicts as the
full-dict route.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from .algo import BayesianOptimizer
from .layout import ParamLayout

_BASE = "__base_optimizer"
_STREAM = "bde_noise_stream"
FORMAT, VERSION = "bde-column-shard", 1


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
    raise ValueError(f"sharded checkpoints cover SVGDOptimizer, SwagOptimizer, iVONOptimizer and torch.optim base "
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


# ---------------------------------------------------------------------- the rules every route shares
def _column_keys(state, n) -> list:
    """The column vectors of a rank-local `state` whose slices are `n` columns wide: `(0, key)` for per-parameter
    tensors shaped [n], `(None, key)` for string-keyed tensors whose first dimension is n (SWAG's moments)."""
    keys = [(0, k) for k, v in state.get(0, {}).items() if torch.is_tensor(v) and tuple(v.shape) == (n,)]
    return keys + [(None, k) for k, v in state.items()
                   if isinstance(k, str) and torch.is_tensor(v) and v.dim() >= 1 and v.shape[0] == n]


def _column(state, key):
    return state[0][key[1]] if key[0] == 0 else state[key[1]]


def _rows(state, columns, n):
    """Every column vector as [m, n] rows (m = 1, or K for SWAG's [n, K] deviations) and where each one starts."""
    blocks, rows = [], {}
    for key in columns:
        block = _column(state, key).detach().reshape(n, -1).t() if key[0] is None else \
            _column(state, key).detach().reshape(1, n)
        rows[key] = (sum(b.shape[0] for b in blocks), block.shape[0])
        blocks.append(block)
    if len({b.dtype for b in blocks}) > 1:
        raise ValueError("column state of one optimizer must share one dtype")
    return blocks, rows


def _agreement(local, columns):
    """What the ranks' dicts must agree on: everything but the column vectors and the noise stream position."""
    state = local["state"]
    rest = {"state": {k: ({kk: vv for kk, vv in v.items() if (0, kk) not in columns} if k == 0 else v)
                      for k, v in state.items() if (None, k) not in columns},
            "param_groups": local["param_groups"],
            **{k: v for k, v in local.items() if k not in ("state", "param_groups", _STREAM)}}
    return _fingerprint(rest), sorted(map(str, columns))


def _agree(seen) -> None:
    if any(s != seen[0] for s in seen):
        raise ValueError("the ranks disagree about the optimizer's scalar state or hyper-parameters")


def _check_counts(optimizer, kind, state, entry_keys, n, width) -> None:
    """particle_count / deviation_samples of a saved dict (`state`: its string-keyed state, `entry_keys`: the keys of
    its per-parameter entries or None) against this optimizer's; its column vectors are `n` long (`width` says what n
    is)."""
    from .svgd import SVGDOptimizer
    from .swag import SwagOptimizer
    if kind is SVGDOptimizer:
        count = optimizer.state["__particle_count"]
        if state.get("__particle_count") != count:
            raise ValueError(f"particle_count {state.get('__particle_count')} of the state dict differs from this "
                             f"optimizer's {count}")
        if entry_keys is not None and not {f"particle_{i}" for i in range(count)} <= set(entry_keys):
            raise ValueError("the state dict lacks particles of this optimizer's particle_count")
    if kind is SwagOptimizer:
        K = optimizer.deviation_samples
        for key, shape in (("__mean", (n,)), ("__sq_weights", (n,)), ("__deviations", (n, K))):
            v = state.get(key)
            if not torch.is_tensor(v) or tuple(v.shape) != shape:
                raise ValueError(f"{key} of the state dict has shape {None if v is None else tuple(v.shape)}, this "
                                 f"optimizer needs {shape} ({width}, deviation_samples = {K})")


def _base(current, shape, device):
    """This rank's vector before a load writes the saved columns into it: a copy of the optimizer's own, so that
    padding columns keep their values, or zeros where the optimizer holds none yet."""
    if torch.is_tensor(current) and tuple(current.shape) == shape:
        return current.detach().clone()
    return torch.zeros(shape, dtype=torch.float32, device=device)


def _reference_dict(layout, local, rows, logical, stream, group_per_parameter) -> dict:
    """The reference-layout dict: `local` (a rank-local dict) with its column vectors replaced by `logical`
    ([rows, D], `rows` says where each one starts) split into the model's parameters."""
    state = local["state"]
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
    if group_per_parameter:
        groups = [{**group, "params": [k]} for k in range(P)]
    else:
        groups = [{**group, "params": list(range(P))}]
    out = {}
    for key, v in local.items():
        out[key] = out_state if key == "state" else groups if key == "param_groups" else stream if key == _STREAM else v
    return out


# ---------------------------------------------------------------------- export
def full_state_dict(sm, optimizer) -> dict:
    kind = _kind(optimizer)
    _check_over(sm, optimizer, kind)
    local = optimizer.state_dict()
    columns = _column_keys(local["state"], sm.shard)
    blocks, rows = _rows(local["state"], columns, sm.shard)     # ONE gather for the whole dict
    stream = local.get(_STREAM)
    if sm.world > 1:
        seen = [None] * sm.world
        dist.all_gather_object(seen, (_agreement(local, columns), stream), group=sm._pg())
        _agree([s[0] for s in seen])
        if stream is not None:
            stream = max(s[1] for s in seen)
    logical = None
    if blocks:
        logical = sm.logical(sm.gather_rows(torch.cat([b.to(sm.full.device) for b in blocks])))    # [rows, D]
    from .svgd import SVGDOptimizer
    return _reference_dict(sm.layout, local, rows, logical, stream, kind is SVGDOptimizer)


# ---------------------------------------------------------------------- import
def _local_dict(sm, optimizer, kind, state_dict) -> dict:
    """The rank-local dict `optimizer.load_state_dict` accepts.  Raises ValueError before anything is written."""
    from .svgd import SVGDOptimizer
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
        base = _base(current, (sm.shard,) + shape_tail, device)
        base[cols.to(base.device)] = flat[pos.to(flat.device)].to(base.device, base.dtype)
        return base

    entries = [saved.get(i) for i in ids]
    stated = any(e is not None for e in entries)
    if stated and (any(e is None for e in entries) or any(set(e) != set(entries[0]) for e in entries)):
        raise ValueError("the parameters' state entries hold different keys")
    _check_counts(optimizer, kind, saved, entries[0] if stated else None, D, f"logical size D = {D}")
    local_state = {}
    if stated:
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


# ---------------------------------------------------------------------- per-rank dicts
def _host(obj):
    """A copy of a state dict with every tensor on the host (copied: the optimizers' dicts hold views of live arenas)
    and `__base_optimizer` None."""
    if torch.is_tensor(obj):
        return obj.detach().to("cpu", copy=True)
    if isinstance(obj, dict):
        return {k: (None if k == _BASE else _host(v)) for k, v in obj.items()}
    if isinstance(obj, list):
        return [_host(v) for v in obj]
    return obj


def shard_state_dict(sm, optimizer) -> dict:
    kind = _kind(optimizer)
    _check_over(sm, optimizer, kind)
    return {"format": FORMAT, "version": VERSION, "kind": type(optimizer).__name__,
            "world": sm.world, "rank": sm.rank, "shard": sm.shard, "lo": sm.lo, "hi": sm.hi,
            "shapes": [tuple(s) for s in sm.layout.shapes], "state_dict": _host(optimizer.state_dict())}


def _tiling(shards):
    """`shards` sorted by rank, after checking that they are the per-rank dicts of one job and tile [0, R * shard)
    exactly once.  Returns (shards, layout of their parameter shapes)."""
    shards = list(shards)
    if not shards or any(not isinstance(s, dict) or s.get("format") != FORMAT for s in shards):
        raise ValueError(f"not a per-rank checkpoint: expected the dicts of format {FORMAT!r} that "
                         "ColumnShardedModel.shard_state_dict returns")
    if any(s.get("version") != VERSION for s in shards):
        raise ValueError(f"per-rank checkpoint versions {sorted({s.get('version') for s in shards})}; this package "
                         f"reads version {VERSION}")

    def job(s):
        return s["world"], s["shard"], s["kind"], [tuple(x) for x in s["shapes"]]
    if any(job(s) != job(shards[0]) for s in shards):
        raise ValueError("the per-rank dicts come from different jobs: their rank count, shard width, optimizer or "
                         "parameter shapes differ")
    R, n = shards[0]["world"], shards[0]["shard"]
    shards.sort(key=lambda s: s["rank"])
    layout = ParamLayout.from_shapes(job(shards[0])[3])
    if [s["rank"] for s in shards] != list(range(R)) or \
            any((s["lo"], s["hi"]) != (s["rank"] * n, (s["rank"] + 1) * n) for s in shards) or R * n < layout.size:
        raise ValueError(f"the per-rank dicts do not tile [0, {R} * {n}) exactly once: ranks "
                         f"{[s['rank'] for s in shards]} of a {R}-rank job")
    return shards, layout


def _shard_columns(shards, optimizer=None, kind=None):
    """The column keys the per-rank dicts share, after the scalar and hyper-parameter checks (and, given the
    optimizer, the particle_count / deviation_samples checks)."""
    n = shards[0]["shard"]
    sds = [s["state_dict"] for s in shards]
    columns = _column_keys(sds[0]["state"], n)
    _agree([_agreement(sd, _column_keys(sd["state"], n)) for sd in sds])
    saved = sds[0]["state"]
    if optimizer is not None:
        _check_counts(optimizer, kind, saved, saved[0].keys() if 0 in saved else None, n, f"shard width {n}")
    odd = [kk for kk, vv in saved.get(0, {}).items() if torch.is_tensor(vv) and vv.dim() > 0 and (0, kk) not in columns]
    if odd:
        raise ValueError(f"per-parameter state {odd} of the per-rank dicts is not shaped [{n}] like their columns")
    return columns


def _stream(shards):
    streams = [s["state_dict"].get(_STREAM) for s in shards]
    return None if streams[0] is None else max(streams)


def _runs(layout, a, b):
    """The layout-space column ranges inside [a, b) that hold parameter elements (padding excluded)."""
    return [(max(o, a), min(o + n, b)) for o, n in zip(layout.offsets, layout.numels) if max(o, a) < min(o + n, b)]


def _local_from_shards(sm, optimizer, kind, shards) -> dict:
    """The rank-local dict `optimizer.load_state_dict` accepts, from the per-rank dicts of a job at any rank count:
    layout column c of saved shard s is its column c - lo_s.  Reads only the shards that overlap [lo, hi).  Raises
    ValueError before anything is written."""
    shards, layout = _tiling(shards)
    if layout.shapes != sm.layout.shapes:
        raise ValueError(f"the checkpoint's parameter shapes {layout.shapes} (logical size {layout.logical_size}) "
                         f"differ from this model's {sm.layout.shapes} (logical size {sm.layout.logical_size})")
    if shards[0]["kind"] != type(optimizer).__name__:
        raise ValueError(f"the checkpoint holds the state of a {shards[0]['kind']}, not of a "
                         f"{type(optimizer).__name__}")
    columns = _shard_columns(shards, optimizer, kind)
    overlaps = [(s, _runs(layout, max(sm.lo, s["lo"]), min(sm.hi, s["hi"]))) for s in shards]
    overlaps = [(s, runs) for s, runs in overlaps if runs]

    def fill(key, current, device):
        tail = tuple(_column(shards[0]["state_dict"]["state"], key).shape[1:])
        base = _base(current, (sm.shard,) + tail, device)
        for s, runs in overlaps:
            src = _column(s["state_dict"]["state"], key)
            a, b = runs[0][0], runs[-1][1]
            piece = src[a - s["lo"]:b - s["lo"]].to(base.device)
            for x, y in runs:
                base[x - sm.lo:y - sm.lo].copy_(piece[x - a:y - a])
        return base

    cur = optimizer.state_dict()["state"]           # padding columns keep these values
    saved = shards[0]["state_dict"]["state"]
    local_state = {}
    for key, v in saved.items():
        if key == 0:
            local_state[0] = {kk: fill((0, kk), cur.get(0, {}).get(kk), sm.param.device) if (0, kk) in columns
                              else vv.detach().clone() if torch.is_tensor(vv) else vv for kk, vv in v.items()}
        elif (None, key) in columns:
            cv = cur.get(key)
            local_state[key] = fill((None, key), cv, cv.device if torch.is_tensor(cv) else v.device)
        elif key == _BASE and _BASE in optimizer.state:
            local_state[key] = optimizer.state[_BASE]          # this job's own base optimizer
        else:
            local_state[key] = v
    out = {k: v for k, v in shards[0]["state_dict"].items() if k != "state"}
    out["state"] = local_state
    if _STREAM in out:
        out[_STREAM] = _stream(shards)
    return out


def load_shard_state_dicts(sm, optimizer, shards) -> None:
    kind = _kind(optimizer)
    _check_over(sm, optimizer, kind)
    optimizer.load_state_dict(_local_from_shards(sm, optimizer, kind, shards))


def consolidate(shards) -> dict:
    """The reference-layout dict of a job saved per rank (the R dicts of `ColumnShardedModel.shard_state_dict`, in
    any order): what `ColumnShardedModel.full_state_dict` returns for the same job, with every tensor on the host.  One
    process, no torch.distributed, no GPU.  Raises ValueError for dicts that do not tile one job's columns or
    disagree about a scalar."""
    shards, layout = _tiling(shards)
    columns = _shard_columns(shards)
    n = shards[0]["shard"]
    parts = [_rows(s["state_dict"]["state"], columns, n) for s in shards]
    rows = parts[0][1]
    logical = None
    if columns:
        logical = layout.to_logical(torch.cat([torch.cat(blocks) for blocks, _ in parts], dim=1)[:, :layout.size])
    return _reference_dict(layout, shards[0]["state_dict"], rows, logical, _stream(shards),
                           shards[0]["kind"] == "SVGDOptimizer")
