"""D-sharded execution: every rank holds a column slice of every particle.

Only the n*n partial squared-distance matrix crosses NVLink; every other kernel on the path is
local to its slice (SURVEY.md §8e).  Rank r of R owns the columns layout.shard_bounds(D, R, r).

Two forms of the exchange:
  * portable: one NCCL (or gloo) sum all-reduce of n*n doubles between K1 and K1b (3 launches + the
    collective per step);
  * peer exchange (`PeerSet`, one node, CUDA IPC): the ranks map each other's small exchange
    buffers once; afterwards the last CTA of K1 — or of the fused training-step kernel — writes its
    partial sums straight into the peers' memory over NVLink, waits for theirs and runs K1b in the
    same launch.  A D-sharded step is then launched exactly like a single-GPU step.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import torch
import torch.distributed as dist

from . import _lib, ops


class _Single:
    """Sentinel group: this rank works alone, whatever torch.distributed's state (plain data-parallel jobs)."""

    def __repr__(self):
        return "bde.dist.SINGLE"


SINGLE = _Single()


def world(group=None) -> int:
    """Ranks that hold column slices of ONE problem.  The functional API below takes torch.distributed's
    convention (group=None = the default group); SVGDOptimizer passes SINGLE unless a group was given explicitly."""
    if group is SINGLE:
        return 1
    return dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1


def allreduce_dist(sc: "ops.SvgdScratch", group=None) -> None:
    """Sum the partial pair distances over the ranks holding the other column slices."""
    if world(group) > 1:
        dist.all_reduce(sc.dist, op=dist.ReduceOp.SUM, group=group)


# --------------------------------------------------------------------------------------
# column shards of the elementwise family (SWAG, iVON, Gaussian parameters): no data-path collective
# --------------------------------------------------------------------------------------
class ColumnShard:
    """Where this rank's slice of a flat state vector sits in the job-wide vector (SURVEY.md §8e, second bullet).

    The elementwise kernels need no exchange; what makes a D-sharded posterior ONE posterior is the noise: the
    per-element Philox counter is `elem0` + local index (so the ranks draw disjoint parts of the same stream —
    with elem0 = 0 everywhere every rank would replay the same normals on its slice), and everything drawn per
    VECTOR rather than per element (SWAG's K low-rank coefficients) comes from the same (seed, stream id) on every
    rank.  `seed` is rank 0's; the stream counter is advanced to the furthest rank's at construction."""

    __slots__ = ("group", "world", "rank", "elem0", "local", "total", "seed")

    def __init__(self, group, world_size, rank, elem0, local, total, seed):
        self.group, self.world, self.rank = group, world_size, rank
        self.elem0, self.local, self.total, self.seed = elem0, local, total, seed

    def __repr__(self):
        return f"ColumnShard(rank {self.rank}/{self.world}, columns [{self.elem0}, {self.elem0 + self.local}) of {self.total})"


def column_shard(local_size: int, group=None) -> ColumnShard:
    """Collective over `group` (one all_gather_object): exclusive prefix sum of the ranks' arena lengths.  Arena
    lengths are multiples of layout.ALIGN, so every elem0 is a multiple of 4 as the kernels require.
    group=None / SINGLE: this rank holds everything (elem0 = 0, seed follows torch)."""
    from . import noise
    if group is None:
        group = SINGLE
    w = world(group)
    if w <= 1:
        return ColumnShard(group, 1, 0, 0, int(local_size), int(local_size), None)
    rank = dist.get_rank(group)
    rows = [None] * w
    dist.all_gather_object(rows, (int(local_size), noise.seed(), noise.stream_position()), group=group)
    sizes = [r[0] for r in rows]
    if any(s % 4 for s in sizes):
        raise ValueError("column shards must be multiples of 4 elements long (flat arenas are)")
    # per-vector draws must agree: one key for the whole group, and no rank re-uses a stream id another has spent
    noise.restore_stream_position(max(r[2] for r in rows))
    return ColumnShard(group, w, rank, sum(sizes[:rank]), sizes[rank], sum(sizes), int(rows[0][1]))


def check_noise_in_step(shard: ColumnShard) -> None:
    """Collective debugging aid: raise unless every rank of the shard's group stands at the same Philox stream
    position (they do when all ranks make the same sampling calls — the SPMD contract of a D-sharded job)."""
    from . import noise
    if shard.world <= 1:
        return
    rows = [None] * shard.world
    dist.all_gather_object(rows, noise.stream_position(), group=shard.group)
    if len(set(rows)) != 1:
        raise RuntimeError(f"ranks of a D-sharded posterior have drawn different numbers of noise streams: {rows}")


def allreduce_scalar_value(value: torch.Tensor, group) -> torch.Tensor:
    """Sum of a scalar over the ranks holding the other column slices, as a VALUE: the gradient flows to this
    rank's term only (the other ranks differentiate theirs).  Used for the logged KL / L2 prior term of BBB."""
    if world(group) <= 1:
        return value
    total = value.detach().clone()
    dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
    return value + (total - value.detach())


def same_ranks(a, b) -> bool:
    """True when groups `a` and `b` hold the same global ranks (None = the default group).  False for a group this
    rank is not a member of (torch.distributed.new_group hands non-members a placeholder)."""
    if a is b:
        return True
    try:
        return sorted(dist.get_process_group_ranks(a)) == sorted(dist.get_process_group_ranks(b))
    except (KeyError, RuntimeError, ValueError):
        return False


def allreduce_max_(flag: torch.Tensor, group) -> torch.Tensor:
    """In place: the largest value of a device scalar over the ranks holding the other column slices (the non-finite
    flag of a gradient gather).  Enqueued on the stream like any collective; no host synchronisation."""
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    return flag


# --------------------------------------------------------------------------------------
# in-kernel exchange over peer memory
# --------------------------------------------------------------------------------------
class PeerSet:
    """The exchange buffers of all ranks of `group`, mapped into this process (include/bde_b200.h,
    "D-sharded jobs").  Collective: every rank of the group must construct it at the same point."""

    def __init__(self, group=None):
        self.group = group
        self.world = world(group)
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self._own = None
        self._mapped = []
        self._attached = []
        lib = _lib.get()
        own, handle = C.c_void_p(), C.create_string_buffer(64)
        _lib.check(lib.bde_peer_alloc(C.byref(own), handle), "bde_peer_alloc")
        self._own = own.value
        handles = [None] * self.world
        dist.all_gather_object(handles, handle.raw, group=group)
        bufs, ok = [0] * self.world, 1
        for r, h in enumerate(handles):
            if r == self.rank:
                bufs[r] = self._own
                continue
            mapped = C.c_void_p()
            if lib.bde_peer_open(h, C.byref(mapped)) != 0 or not mapped.value:
                ok = 0
                break
            self._mapped.append(mapped.value)
            bufs[r] = mapped.value
        # all ranks must agree before anyone starts waiting on a peer inside a kernel
        flag = torch.tensor([ok], dtype=torch.int32, device=torch.device("cuda", torch.cuda.current_device()))
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 0:
            self.close(barrier=False)
            raise _lib.BdeError("CUDA IPC mapping of a peer's exchange buffer failed on at least one rank")
        self._bufs = (C.c_uint64 * self.world)(*bufs)
        # pinned (device-addressable) host word: the kernels store the number of abandoned exchanges here, so
        # check() can see a failure without a synchronising device read
        self._host_status = torch.zeros(1, dtype=torch.int64).pin_memory()
        self.timeout_s = float(os.environ.get("BDE_PEER_TIMEOUT_S", "120"))

    def attach(self, sc: "ops.SvgdScratch") -> None:
        """From now on the grid reductions that use sc.ws produce sums over all ranks of the group."""
        _lib.check(_lib.get().bde_peer_attach(sc.ws.data_ptr(), sc.ws_bytes, self.world, self.rank, self._bufs,
                                              self.timeout_s, self._host_status.data_ptr(),
                                              _lib.stream_ptr(sc.ws.device)), "bde_peer_attach")
        sc.peers = self
        self._attached.append(weakref.ref(sc))

    def check(self) -> None:
        """Raise if an in-kernel exchange of this peer set was abandoned (a peer did not arrive within
        `timeout_s`).  Reads a pinned host word — no synchronisation — so a failure is reported by the first call
        AFTER the failing launch has finished; from that launch on the kernels leave K / A untouched and skip
        further exchanges, so no NaN reaches the particles in between."""
        bad = int(self._host_status[0])
        if bad:
            raise _lib.BdeError(
                f"in-kernel peer exchange abandoned {bad} time(s): a rank of the D-sharded group did not reach its "
                f"SVGD step within {self.timeout_s:g} s (BDE_PEER_TIMEOUT_S); the sums were discarded and the kernel "
                "matrix was left unchanged.  Re-synchronise the ranks and rebuild the optimizer (or set "
                "BDE_PEER_EXCHANGE=0 to use the NCCL all-reduce form).")

    def status(self):
        """(exchanges completed, exchanges abandoned on a timeout) of this rank — synchronises."""
        e, t = C.c_uint64(0), C.c_uint64(0)
        _lib.check(_lib.get().bde_peer_status(self._own, C.byref(e), C.byref(t)), "bde_peer_status")
        return e.value, t.value

    def wait_stats(self, reset: bool = False):
        """(exchanges, summed wait ns, longest wait ns) of this rank's in-kernel exchanges since the last reset: the
        time the last CTA of K1 spent waiting for its slowest peer — rank skew, not link time.  Synchronises."""
        n, s, m = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _lib.check(_lib.get().bde_peer_wait_stats(self._own, C.byref(n), C.byref(s), C.byref(m), int(reset)),
                   "bde_peer_wait_stats")
        return n.value, s.value, m.value

    def close(self, barrier: bool = True) -> None:
        """Detach the workspaces, unmap the peers and free this rank's buffer.  Collective when barrier=True:
        no rank may free its buffer while a peer's kernel can still write into it."""
        if self._own is None:
            return
        lib = _lib.get()
        for ref in self._attached:
            sc = ref()
            if sc is not None and getattr(sc, "peers", None) is self:
                lib.bde_peer_detach(sc.ws.data_ptr(), sc.ws_bytes, _lib.stream_ptr(sc.ws.device))
                sc.peers = None
        self._attached = []
        torch.cuda.synchronize()
        if barrier and self.world > 1:
            dist.barrier(group=self.group)
        for m in self._mapped:
            lib.bde_peer_close(m)
        self._mapped = []
        lib.bde_peer_free(self._own)
        self._own = None


_PEER_SETS: dict = {}


def enable_peer_exchange(sc: "ops.SvgdScratch", group=None) -> bool:
    """Attach `sc` to the group's peer set (created on first use).  Collective over the group.  Returns
    False — leaving the NCCL all-reduce form in place — for a single rank, CPU tensors, when
    BDE_PEER_EXCHANGE=0, when the ranks cannot map each other's memory (not one node / no P2P), or above
    ops.FUSED_MAX_PARTICLES particles (the in-kernel exchange carries at most 32 * 31 / 2 sums)."""
    if (world(group) <= 1 or not sc.ws.is_cuda or os.environ.get("BDE_PEER_EXCHANGE", "1") == "0"
            or sc.n > ops.FUSED_MAX_PARTICLES):
        return False
    if getattr(sc, "peers", None) is not None:
        return True
    key = id(group) if group is not None else None
    ps = _PEER_SETS.get(key)
    if ps is None:
        try:
            ps = PeerSet(group)
        except _lib.BdeError:
            ps = False
        _PEER_SETS[key] = ps
    if ps is False:
        return False
    ps.attach(sc)
    return True


def shutdown_peer_exchange() -> None:
    """Collective teardown of every peer set of this process (call before destroy_process_group)."""
    for key, ps in list(_PEER_SETS.items()):
        if ps:
            ps.close()
        del _PEER_SETS[key]


def exchanges_in_kernel(sc: "ops.SvgdScratch", group=None) -> bool:
    """True when a launch on `sc` already yields cross-rank sums (single rank, or peer set attached)."""
    return world(group) == 1 or getattr(sc, "peers", None) is not None


# --------------------------------------------------------------------------------------
# the sharded step
# --------------------------------------------------------------------------------------
def svgd_kernel_sharded(X: torch.Tensor, sc: "ops.SvgdScratch", l2_reg: float, kernel_grad_scale: float,
                        dataset_size: float, h_override: float = 0.0, group=None, have_partial: bool = False) -> None:
    """K1 (local partial distances) -> sum over ranks -> K1b (identical on every rank): leaves K and A in `sc`.
    With a single rank, or with a peer set attached to `sc`, all of it is ONE launch.  have_partial: sc.dist
    already holds this rank's partial sums for the current X (left by the previous training-step launch)."""
    if exchanges_in_kernel(sc, group):
        if have_partial:
            ops.svgd_bandwidth(sc, l2_reg, kernel_grad_scale, dataset_size, h_override)
        else:
            ops.svgd_pairdist_bandwidth(X, sc, l2_reg, kernel_grad_scale, dataset_size, h_override)
        return
    if not have_partial:
        ops.svgd_pairdist(X, sc)
    allreduce_dist(sc, group)
    ops.svgd_bandwidth(sc, l2_reg, kernel_grad_scale, dataset_size, h_override)


def svgd_step_sharded(X: torch.Tensor, G: torch.Tensor, out: torch.Tensor, sc: "ops.SvgdScratch", l2_reg: float,
                      kernel_grad_scale: float, dataset_size: float, h_override: float = 0.0, group=None) -> torch.Tensor:
    """One SVGD posterior update on this rank's [n, D/R] slices.

    K1 (local partial distances) -> sum over ranks -> K1b (identical on every rank) -> K2 (local).
    Single rank or peer set attached: the fused two-launch path; otherwise K1, all-reduce, K1b, K2.
    """
    svgd_kernel_sharded(X, sc, l2_reg, kernel_grad_scale, dataset_size, h_override, group)
    return ops.svgd_apply(X, G, out, sc)
