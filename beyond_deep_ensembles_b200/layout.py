"""Flat-arena layout of a parameter list in HBM.

The reference gathers parameters with parameters_to_vector / cat+stack on every step
(svgd.py:83-84, swag.py:100).  Here every parameter list gets ONE flat fp32 row layout, decided
once: tensor k occupies [offset_k, offset_k + numel_k) with offset_k aligned to ALIGN elements
(256 B, so that the model's own GEMM/conv kernels keep seeing well-aligned weights when
param.data is re-homed into the arena).  Rows of an arena ([rows, size]) are particles, MC
state vectors, SWAG deviation columns, ...; the padding elements are zero and contribute
nothing to any kernel on the path.

`logical` order = the reference's parameters_to_vector order without padding; it is only
used when exporting / importing state dicts in the reference's layout.
"""
from __future__ import annotations

import torch

ALIGN = 64  # elements (256 bytes)


class ParamLayout:
    def __init__(self, params, align: int = ALIGN):
        self.params = list(params)
        if not self.params:
            raise ValueError("empty parameter list")
        self.shapes = [tuple(p.shape) for p in self.params]
        self.numels = [p.numel() for p in self.params]
        self.offsets = []
        off = 0
        for n in self.numels:
            self.offsets.append(off)
            off += -(-n // align) * align
        self.size = max(off, align)            # padded row length (multiple of `align`)
        self.logical_size = sum(self.numels)
        self._index = {}
        self._copy_table = None

    @classmethod
    def from_shapes(cls, shapes, align: int = ALIGN) -> "ParamLayout":
        """The layout of parameters of these shapes (it depends on nothing else): meta tensors, no storage."""
        return cls([torch.empty(s, device="meta") for s in shapes], align)

    @property
    def copy_table(self):
        """The constant argument tables of ops.multi_tensor_copy for this layout (built on first use)."""
        if self._copy_table is None:
            from . import ops
            self._copy_table = ops.CopyTable(self.offsets, self.numels)
        return self._copy_table

    def new_arena(self, rows: int, device, dtype=torch.float32) -> torch.Tensor:
        return torch.zeros((rows, self.size), dtype=dtype, device=device)

    def views(self, row: torch.Tensor):
        """Per-parameter views (zero-copy) of one arena row."""
        assert row.dim() == 1 and row.numel() == self.size
        return [row[o:o + n].view(s) for o, n, s in zip(self.offsets, self.numels, self.shapes)]

    def logical_index(self, device) -> torch.Tensor:
        key = str(device)
        if key not in self._index:
            idx = torch.cat([torch.arange(o, o + n, dtype=torch.int64) for o, n in zip(self.offsets, self.numels)])
            self._index[key] = idx.to(device)
        return self._index[key]

    def to_logical(self, arena: torch.Tensor) -> torch.Tensor:
        """[..., size] -> [..., logical_size] (export only; not on the hot path)."""
        return arena.index_select(-1, self.logical_index(arena.device))

    def from_logical(self, vec: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """[..., logical_size] -> [..., size] with zero padding (import / noise injection only)."""
        shape = tuple(vec.shape[:-1]) + (self.size,)
        if out is None:
            out = torch.zeros(shape, dtype=vec.dtype, device=vec.device)
        else:
            out.zero_()
        out.index_copy_(-1, self.logical_index(vec.device), vec)
        return out


def shard_bounds(D: int, world: int, rank: int, align: int = ALIGN):
    """Column range [lo, hi) of `rank` when D columns are split over `world` ranks in
    `align`-element blocks (the first D % world blocks go to the lowest ranks)."""
    blocks = -(-D // align)
    base, extra = divmod(blocks, world)
    lo_b = rank * base + min(rank, extra)
    hi_b = lo_b + base + (1 if rank < extra else 0)
    return min(lo_b * align, D), min(hi_b * align, D)
