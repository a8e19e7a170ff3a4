"""Table-wise sharded embeddings across the GPUs of one box (new functionality: DLRM.jl is
single-process; BASELINE.json's north_star asks for table-wise model parallelism with the dense
MLPs and the interaction data-parallel).

One process per GPU.  Every table lives whole on one rank.  Per step:

  forward   each rank sends the index columns of its local batch to the tables' owners
            (all-to-all, a few hundred KB), owners pool their tables for the GLOBAL batch in one
            lookup launch, and a second all-to-all delivers to every rank the pooled rows of its
            local samples, which land in the interaction input T [B_local][1 + ntab][D];
  backward  the mirror all-to-all returns dT slices to the owners, which run the fused sparse SGD
            locally over the global batch; dense gradients are summed with one all-reduce.

The routing logic here is pure tensor plumbing over ``torch.distributed`` (NCCL on GPUs, gloo in
the CPU tests); the compute is injected (`lookup_fn`, `update_fn`) and in the product is always the
CUDA library.
"""
from __future__ import annotations

from dataclasses import dataclass
from fractions import Fraction
from typing import Callable, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.distributed as dist


@dataclass
class TableSharding:
    """Which rank owns which table, balanced by LOOKUP COUNT first (every table receives
    B_global * P lookups per step whatever its size), then by bytes: tables are dealt in
    descending row count, snake order, so the big tables land on different ranks.

    With per-table pooling factors P_k (not all equal) table k receives B_global * P_k lookups, so the
    tables are dealt longest first instead: descending P_k, then rows, then id, each to the rank with the
    smallest sum of P_k so far (ties: fewer rows, then the lower rank).  Equal P_k give the snake plan.

    With ``max_col_shards`` S > 1 a table hotter than the even share may be split by columns into c_k slices
    (``shards``), slice j on rank ``holders[k][j]`` (columns [j D / c_k, (j + 1) D / c_k)); see :meth:`build`.
    Then ``local[r]`` lists every table of which rank r holds a slice and ``owner[k]`` is the holder of slice 0."""
    rows: List[int]
    world: int
    owner: List[int]
    local: List[List[int]]      # local[r] = global table ids owned by rank r, ascending
    _slot_cache: Optional[dict] = None
    P: Optional[Tuple[int, ...]] = None     # per-table pooling factors the plan was built for (None: one P)
    D: Optional[int] = None                 # embedding width of a column-wise plan
    shards: Optional[Tuple[int, ...]] = None        # c_k of a plan that splits a table (None: every table whole)
    holders: Optional[List[List[int]]] = None       # holders[k][j] = rank holding slice j of table k

    @property
    def split(self) -> bool:
        """Whether the plan splits a table by columns."""
        return self.shards is not None

    def groups(self, r: int) -> List[Tuple[int, List[int]]]:
        """Rank r's units grouped by width: [(c, tables ascending)] in ascending c, i.e. whole tables (width D)
        first, then slices of width D / 2, D / 4, ...  One EmbeddingTables handle serves each group."""
        if not self.split:
            return [(1, list(self.local[r]))]
        by_c = {}
        for k in range(len(self.rows)):
            if r in self.holders[k]:
                by_c.setdefault(self.shards[k], []).append(k)
        return sorted(by_c.items())

    def slice_of(self, k: int, r: int) -> int:
        """Index j of the slice of table k that rank r holds."""
        return self.holders[k].index(r) if self.split else 0

    def slot_index(self, r: int, device) -> torch.Tensor:
        """Device tensor of the interaction slots (1 + table id) of rank r's tables (cached: no
        host-to-device copy inside the step, which also keeps the step CUDA-graph capturable)."""
        if self._slot_cache is None:
            self._slot_cache = {}
        key = (r, str(device))
        if key not in self._slot_cache:
            self._slot_cache[key] = torch.tensor([1 + k for k in self.local[r]], dtype=torch.int64, device=device)
        return self._slot_cache[key]

    def owner_order(self, device) -> torch.Tensor:
        """Table ids grouped by owner rank (the send order of the index all-to-all), cached."""
        if self._slot_cache is None:
            self._slot_cache = {}
        key = ("order", str(device))
        if key not in self._slot_cache:
            order = [k for r in range(self.world) for k in self.local[r]]
            self._slot_cache[key] = torch.tensor(order, dtype=torch.int64, device=device)
        return self._slot_cache[key]

    @classmethod
    def build(cls, rows: Sequence[int], world: int, P: Optional[Sequence[int]] = None, *, D: Optional[int] = None,
              max_col_shards: int = 1) -> "TableSharding":
        """The same rule as dlrmb_shard_plan (``P`` None or all equal) / dlrmb_shard_plan_mp, and with
        ``max_col_shards`` S > 1 as dlrmb_shard_plan_cw: while the table with the largest P_k / c_k (ties: more rows,
        then the lower id) is above the even share (P_k * world > c_k * sum(P)) and 2 c_k <= min(S, world), its c_k
        doubles.  Nothing split: the table-wise plan.  Otherwise the slices are dealt longest first (descending
        P_k / c_k, then rows, then k, then j), each to the rank with the smallest sum of P_k / c_k among those
        holding no slice of k (ties: fewer rows * D / c_k, then the lower rank).  ``P`` None counts one lookup per
        table.  S must be a power of two and, when S > 1, D / S a multiple of 4."""
        rows = [int(r) for r in rows]
        S = int(max_col_shards)
        if S < 1 or S & (S - 1):
            raise ValueError(f"max_col_shards must be a power of two, got {max_col_shards}")
        if S > 1 and (D is None or int(D) < 1 or int(D) % S or (int(D) // S) % 4):
            raise ValueError(f"D / max_col_shards must be a multiple of 4 (D = {D}, max_col_shards = {S})")
        Pt = None
        if P is not None:
            if world < 1 or not rows:
                raise ValueError(f"a shard plan needs world >= 1 and a table (world {world}, {len(rows)} tables)")
            Pt = tuple(int(p) for p in P)
            if len(Pt) != len(rows) or min(Pt) < 1:
                raise ValueError(f"P must hold one pooling factor >= 1 per table ({len(rows)} tables), got {list(Pt)}")
        if S > 1:
            plan = cls._build_cw(rows, world, Pt or (1,) * len(rows), int(D), S, Pt)
            if plan is not None:
                return plan
        owner = [0] * len(rows)
        if Pt is None or len(set(Pt)) == 1:
            order = sorted(range(len(rows)), key=lambda k: (-rows[k], k))
            for i, k in enumerate(order):
                rnd, pos = divmod(i, world)
                owner[k] = pos if rnd % 2 == 0 else world - 1 - pos
        else:
            load, size = [0] * world, [0] * world
            for k in sorted(range(len(rows)), key=lambda k: (-Pt[k], -rows[k], k)):
                r = min(range(world), key=lambda r: (load[r], size[r], r))
                owner[k] = r
                load[r] += Pt[k]
                size[r] += rows[k]
        local = [[k for k in range(len(rows)) if owner[k] == r] for r in range(world)]
        return cls(rows, world, owner, local, P=Pt, D=None if D is None else int(D))

    @classmethod
    def _build_cw(cls, rows, world, P, D, S, Pt) -> Optional["TableSharding"]:
        """The column-wise plan, or None when it splits nothing (exact arithmetic: fractions as cross products)."""
        n, total = len(rows), sum(P)
        c = [1] * n
        cmax = min(S, world)
        while True:
            k = 0
            for i in range(1, n):
                lhs, rhs = P[i] * c[k], P[k] * c[i]
                if lhs > rhs or (lhs == rhs and rows[i] > rows[k]):
                    k = i
            if P[k] * world <= c[k] * total or 2 * c[k] > cmax:
                break
            c[k] *= 2
        M = max(c)
        if M == 1:
            return None
        units = sorted(((k, j) for k in range(n) for j in range(c[k])),
                       key=lambda u: (Fraction(-P[u[0]], c[u[0]]), -rows[u[0]], u[0], u[1]))
        load, size = [0] * world, [0] * world            # in units of 1 / M
        holders = [[-1] * c[k] for k in range(n)]
        for k, j in units:
            r = min((r for r in range(world) if r not in holders[k]), key=lambda r: (load[r], size[r], r))
            holders[k][j] = r
            load[r] += P[k] * (M // c[k])
            size[r] += rows[k] * (M // c[k])
        local = [[k for k in range(n) if r in holders[k]] for r in range(world)]
        return cls(rows, world, [h[0] for h in holders], local, P=Pt, D=D, shards=tuple(c), holders=holders)

    def lookups_per_rank(self) -> List[Union[int, Fraction]]:
        """Sum of P_k over each rank's tables (per sample of the global batch); a slice of a split table counts
        P_k / c_k (exact fractions)."""
        P = self.P or (1,) * len(self.rows)
        if self.split:
            return [sum((Fraction(P[k], self.shards[k]) for k in l), Fraction(0)) for l in self.local]
        return [sum(P[k] for k in l) for l in self.local]

    def counts(self) -> List[int]:
        return [len(l) for l in self.local]

    def bytes_per_rank(self, D: int) -> List[int]:
        if self.split:
            return [sum(self.rows[k] * (D // self.shards[k]) for k in l) * 4 for l in self.local]
        return [sum(self.rows[k] for k in l) * D * 4 for l in self.local]

    def _unit_index(self, r: int, c: int, ks: Sequence[int], device) -> Tuple[torch.Tensor, torch.Tensor]:
        """(slots, slice ids) of rank r's group of width D / c as device tensors (cached)."""
        if self._slot_cache is None:
            self._slot_cache = {}
        key = ("units", r, c, str(device))
        if key not in self._slot_cache:
            self._slot_cache[key] = (torch.tensor([1 + k for k in ks], dtype=torch.int64, device=device),
                                     torch.tensor([self.slice_of(k, r) for k in ks], dtype=torch.int64, device=device))
        return self._slot_cache[key]


def _a2a(out: torch.Tensor, inp: torch.Tensor, out_splits, in_splits, group) -> None:
    dist.all_to_all_single(out, inp, output_split_sizes=out_splits, input_split_sizes=in_splits, group=group)


def _require_uniform_pooling(idx) -> None:
    """The table-sharded path takes one pooling factor for all tables."""
    from .embedding import PackedIndices
    mixed = isinstance(idx, PackedIndices) or (
        isinstance(idx, (list, tuple)) and len({int(np.asarray(s).reshape(np.asarray(s).shape[0], -1).shape[1])
                                                for s in idx}) > 1)
    if mixed:
        raise ValueError("per-table pooling factors (mixed multi-hot widths) are not supported by the "
                         "table-sharded path; give every table the same P or use EmbeddingTables")


def exchange_indices(idx_local: torch.Tensor, sh: TableSharding, rank: int, group=None) -> torch.Tensor:
    """idx_local [ntab][B_local][P] (this rank's samples, all tables) ->
    [t_mine][B_global][P] (all samples, this rank's tables; sample order = rank-major)."""
    _require_uniform_pooling(idx_local)
    ntab, Bl, P = idx_local.shape
    W = sh.world
    if W == 1:
        return idx_local
    send = idx_local.index_select(0, sh.owner_order(idx_local.device))                 # grouped by owner
    t_mine = len(sh.local[rank])
    recv = torch.empty((W, t_mine, Bl, P), dtype=idx_local.dtype, device=idx_local.device)
    in_splits = [len(sh.local[r]) * Bl * P for r in range(W)]
    out_splits = [t_mine * Bl * P] * W
    _a2a(recv.view(-1), send.view(-1), out_splits, in_splits, group)
    # [W][t][Bl][P] -> [t][W*Bl][P]
    return recv.permute(1, 0, 2, 3).reshape(t_mine, W * Bl, P).contiguous()


def exchange_indices_mp(packed, sh: TableSharding, rank: int, group=None):
    """Per-table pooling factors: ``packed`` (:class:`~dlrm_jl_b200.embedding.PackedIndices` of this rank's
    B_local samples, every table) -> this rank's tables in the owner layout: a PackedIndices at B_global of
    the owned tables in ascending id (table j's [B_global][P_j] block after the blocks of the owned tables
    before it, rank h's samples in its rows [h * B_local, (h + 1) * B_local)), which the `_mp` lookup, sort
    and update read as is."""
    from .embedding import PackedIndices
    W = sh.world
    if W == 1:
        return packed
    P, Bl, flat = packed.P, packed.B, packed.flat
    mine = sh.local[rank]
    offs = np.concatenate([[0], np.cumsum([Bl * p for p in P])]).tolist()
    order = [k for r in range(W) for k in sh.local[r]]                                  # grouped by owner
    send = torch.cat([flat[offs[k]:offs[k + 1]] for k in order]) if order else flat[:0]
    in_splits = [Bl * sum(P[k] for k in sh.local[r]) for r in range(W)]
    per_rank = Bl * sum(P[k] for k in mine)
    recv = torch.empty((W * per_rank,), dtype=flat.dtype, device=flat.device)
    _a2a(recv, send.contiguous(), [per_rank] * W, in_splits, group)
    # [h][j][B_local][P_j] -> [j][h][B_local][P_j]
    parts, o = [], 0
    for k in mine:
        n = Bl * P[k]
        parts.extend(recv[h * per_rank + o:h * per_rank + o + n] for h in range(W))
        o += n
    owned = torch.cat(parts) if parts else recv[:0]
    return PackedIndices(owned.contiguous(), tuple(P[k] for k in mine), Bl * W)


def gloo_group(group=None):
    """``group`` when it runs on gloo, else a new gloo group over every rank of the job.  The per-step lookup counts of
    jagged batches travel over it, so the host never waits on the device.  ``dist.new_group`` must be entered by every
    rank of the default group, which the ranks of a proper subgroup cannot arrange among themselves: a non-gloo
    ``group`` must span the whole job (pass a gloo group otherwise)."""
    if dist.get_backend(group) == "gloo":
        return group
    if group is not None and dist.get_world_size(group) != dist.get_world_size():
        raise ValueError(f"the lookup counts of jagged batches travel over a gloo group, and group (backend "
                         f"{dist.get_backend(group)}, {dist.get_world_size(group)} of {dist.get_world_size()} ranks) is "
                         "neither gloo nor the whole job: pass count_group, a gloo group over the same ranks")
    return dist.new_group(backend="gloo")


def exchange_jagged_counts(jag_local, group=None) -> np.ndarray:
    """Every rank's lookup counts of this step: [world][ntab] int64, row h = rank h's ``L``.  ``jag_local`` is this
    rank's :class:`~dlrm_jl_b200.embedding.JaggedIndices`; ``group`` a gloo (CPU) group.  The jagged kernels size
    their grids from host counts, so an owner needs the counts of its tables summed over the ranks and a sender the
    counts of the ranks before it.  Every rank raises ValueError when the ranks disagree on B_local, the pooling or
    whether the batch is weighted."""
    W = dist.get_world_size(group)
    mine = torch.tensor(list(jag_local.L) + [jag_local.B, jag_local.pooling_code, int(jag_local.weights is not None)],
                        dtype=torch.int64)
    got = [torch.empty_like(mine) for _ in range(W)]
    dist.all_gather(got, mine, group=group)
    a = torch.stack(got).numpy()
    if (a[:, -3:] != a[0, -3:]).any():
        desc = [f"rank {h}: B_local {r[-3]}, pooling {'mean' if r[-2] else 'sum'}, {'weighted' if r[-1] else 'unweighted'}"
                for h, r in enumerate(a)]
        raise ValueError("the ranks' jagged batches disagree on B_local, pooling or weighting: " + "; ".join(desc))
    return a[:, :-3].copy()


def exchange_indices_jagged(jag_local, counts: np.ndarray, sh: TableSharding, rank: int, group=None):
    """Jagged bags: ``jag_local`` (:class:`~dlrm_jl_b200.embedding.JaggedIndices` of this rank's B_local bags per
    table, every table) -> this rank's tables in the owner layout, a JaggedIndices at B_global = world * B_local of the
    owned tables in ascending id: table j's entries after those of the owned tables before it, rank h's entries inside
    them after those of the ranks before h, in their own order; bag j * B_global + h * B_local + b is rank h's bag b;
    weights beside their values.  ``counts`` is :func:`exchange_jagged_counts`'s [world][ntab].  Values, bag lengths
    and weights travel with three all-to-alls; the owner rebuilds its offsets by a cumulative sum.  The owner's jagged
    lookup, sort and update read the result as is."""
    from .embedding import JaggedIndices
    W = sh.world
    if W == 1:
        return jag_local
    Bl, L = jag_local.B, jag_local.L
    counts = np.asarray(counts, dtype=np.int64)
    mine = sh.local[rank]
    t = len(mine)
    dev = jag_local.values.device
    starts = np.concatenate([[0], np.cumsum(L)]).tolist()
    order = [k for r in range(W) for k in sh.local[r]]                                  # grouped by owner
    lengths = (jag_local.offsets[1:] - jag_local.offsets[:-1]).view(len(L), Bl)
    in_splits = [int(sum(L[k] for k in sh.local[r])) for r in range(W)]
    out_splits = [int(counts[h, mine].sum()) for h in range(W)]

    def values_a2a(flat):
        send = torch.cat([flat[starts[k]:starts[k + 1]] for k in order]) if order else flat[:0]
        recv = torch.empty((sum(out_splits),), dtype=flat.dtype, device=dev)
        _a2a(recv, send.contiguous(), out_splits, in_splits, group)
        # [h][j][entries] -> [j][h][entries]
        parts, base = [], np.concatenate([[0], np.cumsum(out_splits)]).tolist()
        inner = np.concatenate([np.zeros((W, 1), np.int64), np.cumsum(counts[:, mine], axis=1)], axis=1)
        for j in range(t):
            parts.extend(recv[base[h] + inner[h, j]:base[h] + inner[h, j + 1]] for h in range(W))
        return torch.cat(parts) if parts else recv[:0]

    values = values_a2a(jag_local.values)
    weights = None if jag_local.weights is None else values_a2a(jag_local.weights)
    send_n = lengths.index_select(0, sh.owner_order(dev)).reshape(-1).contiguous()
    recv_n = torch.empty((W * t * Bl,), dtype=lengths.dtype, device=dev)
    _a2a(recv_n, send_n, [t * Bl] * W, [len(sh.local[r]) * Bl for r in range(W)], group)
    n_own = recv_n.view(W, t, Bl).permute(1, 0, 2).reshape(-1)
    offsets = torch.zeros((t * W * Bl + 1,), dtype=jag_local.offsets.dtype, device=dev)
    offsets[1:] = torch.cumsum(n_own, 0).to(offsets.dtype)
    L_own = tuple(int(counts[:, k].sum()) for k in mine)
    return JaggedIndices(values.contiguous(), offsets, L_own, Bl * W, jag_local.pooling, weights)


def exchange_pooled(pooled: torch.Tensor, T: torch.Tensor, sh: TableSharding, rank: int, group=None) -> None:
    """pooled [B_global][t_mine][D] (owner side) -> T[:, 1 + k, :] for every table k, on the rank
    that owns the samples.  T is [B_local][1 + ntab][D]; slot 0 is left for x."""
    W = sh.world
    Bg, t_mine, D = pooled.shape
    Bl = Bg // W
    if W == 1:
        T[:, 1:, :] = pooled
        return
    counts = sh.counts()
    recv = torch.empty((Bl * sum(counts) * D,), dtype=pooled.dtype, device=pooled.device)
    in_splits = [Bl * t_mine * D] * W
    out_splits = [Bl * counts[r] * D for r in range(W)]
    _a2a(recv, pooled.reshape(-1), out_splits, in_splits, group)
    off = 0
    for r in range(W):
        if counts[r] == 0:
            continue
        chunk = recv[off:off + Bl * counts[r] * D].view(Bl, counts[r], D)
        T.index_copy_(1, sh.slot_index(r, T.device), chunk)
        off += Bl * counts[r] * D


def exchange_grads(dT: torch.Tensor, sh: TableSharding, rank: int, group=None) -> torch.Tensor:
    """dT [B_local][1 + ntab][D] -> [B_global][t_mine][D] on each owner (mirror of exchange_pooled)."""
    W = sh.world
    Bl, S, D = dT.shape
    if W == 1:
        return dT[:, 1:, :].contiguous()
    counts = sh.counts()
    t_mine = counts[rank]
    send = torch.cat([dT.index_select(1, sh.slot_index(r, dT.device)).reshape(-1) for r in range(W)])
    recv = torch.empty((W * Bl, t_mine, D), dtype=dT.dtype, device=dT.device)
    in_splits = [Bl * counts[r] * D for r in range(W)]
    out_splits = [Bl * t_mine * D] * W
    _a2a(recv.view(-1), send, out_splits, in_splits, group)
    return recv


def exchange_indices_cw(packed, sh: TableSharding, rank: int, group=None) -> list:
    """Column-wise plan: ``packed`` (PackedIndices of this rank's B_local samples, every table) -> one PackedIndices
    per width group of this rank (:meth:`TableSharding.groups`), each the owner layout of its tables at B_global as
    :func:`exchange_indices_mp` builds it.  A split table's block goes to every holder of one of its slices."""
    from .embedding import PackedIndices
    W = sh.world
    P, Bl, flat = packed.P, packed.B, packed.flat
    offs = np.concatenate([[0], np.cumsum([Bl * p for p in P])]).tolist()
    order = [k for r in range(W) for _c, ks in sh.groups(r) for k in ks]          # grouped by holder
    send = torch.cat([flat[offs[k]:offs[k + 1]] for k in order]) if order else flat[:0]
    in_splits = [Bl * sum(P[k] for _c, ks in sh.groups(r) for k in ks) for r in range(W)]
    groups = sh.groups(rank)
    per_rank = Bl * sum(P[k] for _c, ks in groups for k in ks)
    recv = torch.empty((W * per_rank,), dtype=flat.dtype, device=flat.device)
    _a2a(recv, send.contiguous(), [per_rank] * W, in_splits, group)
    # [h][unit][B_local][P_k] -> per group [unit][h][B_local][P_k]
    rv = recv.view(W, per_rank)
    out, o = [], 0
    for _c, ks in groups:
        parts = []
        for k in ks:
            n = Bl * P[k]
            parts.append(rv[:, o:o + n].reshape(-1))
            o += n
        out.append(PackedIndices(torch.cat(parts).contiguous() if parts else recv[:0], tuple(P[k] for k in ks), Bl * W))
    return out


def exchange_pooled_cw(pooled: Sequence[torch.Tensor], T: torch.Tensor, sh: TableSharding, rank: int,
                       group=None) -> None:
    """Column-wise plan: pooled[g] [B_global][t_g][D / c_g] of this rank's width groups -> the column range of every
    slice in T[:, 1 + k, :] on the rank that owns the samples.  T is [B_local][1 + ntab][D]."""
    W = sh.world
    Bl, F, D = T.shape
    send = torch.cat([p[h * Bl:(h + 1) * Bl].reshape(-1) for h in range(W) for p in pooled]) if pooled else T.new_empty(0)
    n_mine = Bl * sum(len(ks) * (D // c) for c, ks in sh.groups(rank))
    out_splits = [Bl * sum(len(ks) * (D // c) for c, ks in sh.groups(r)) for r in range(W)]
    recv = torch.empty((sum(out_splits),), dtype=T.dtype, device=T.device)
    _a2a(recv, send, out_splits, [n_mine] * W, group)
    off = 0
    for r in range(W):
        for c, ks in sh.groups(r):
            if not ks:
                continue
            w = D // c
            n = Bl * len(ks) * w
            slots, js = sh._unit_index(r, c, ks, T.device)
            T.view(Bl, F, c, w)[:, slots, js, :] = recv[off:off + n].view(Bl, len(ks), w)
            off += n


def exchange_grads_cw(dT: torch.Tensor, sh: TableSharding, rank: int, group=None) -> List[torch.Tensor]:
    """Column-wise plan, mirror of :func:`exchange_pooled_cw`: dT [B_local][1 + ntab][D] -> one gradient
    [B_global][t_g][D / c_g] per width group of this rank."""
    W = sh.world
    Bl, F, D = dT.shape
    parts, in_splits = [], []
    for r in range(W):
        n = 0
        for c, ks in sh.groups(r):
            if not ks:
                continue
            slots, js = sh._unit_index(r, c, ks, dT.device)
            parts.append(dT.view(Bl, F, c, D // c)[:, slots, js, :].reshape(-1))
            n += Bl * len(ks) * (D // c)
        in_splits.append(n)
    groups = sh.groups(rank)
    per_rank = Bl * sum(len(ks) * (D // c) for c, ks in groups)
    recv = torch.empty((W * per_rank,), dtype=dT.dtype, device=dT.device)
    _a2a(recv, torch.cat(parts) if parts else dT.new_empty(0), [per_rank] * W, in_splits, group)
    rv = recv.view(W, per_rank)
    out, o = [], 0
    for c, ks in groups:
        n = Bl * len(ks) * (D // c)
        out.append(rv[:, o:o + n].reshape(W * Bl, len(ks), D // c))
        o += n
    return out


class PeerExchange:
    """The interaction input buffer T [B_local][1 + ntab][D] of every rank, allocated by the
    library and mapped into every other rank's address space through CUDA IPC, so the owner of a
    table can store pooled rows straight into the buffer of the rank that owns the sample
    (`EmbeddingTables.lookup_p2p`).  `barrier` is the stream-ordered collective that orders the
    peer stores against the consumers (a one-element NCCL all-reduce by default)."""

    def __init__(self, B_local: int, ntab: int, D: int, rank: int, world: int, device, group=None,
                 barrier: Optional[Callable] = None, flag_barrier: bool = True):
        import ctypes as C

        from . import _lib
        from .embedding import _DevicePtrView
        self.lib = _lib.load()
        self.rank, self.world, self.group = rank, world, group
        self.device = torch.device(device)
        self.shape = (B_local, 1 + ntab, D)
        nbytes = B_local * (1 + ntab) * D * 4
        h = C.c_void_p()
        _lib.check(self.lib.dlrmb_xbuf_create(self.device.index or 0, nbytes, C.byref(h)))
        self._xbuf = h
        p = C.c_void_p()
        _lib.check(self.lib.dlrmb_xbuf_ptr(h, C.byref(p)))
        handle = (C.c_uint8 * 64)()
        _lib.check(self.lib.dlrmb_xbuf_ipc_handle(h, handle))
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle), group=group)
        self.peer_ptrs = []
        self._owned, self._mapped = [], [self.peer_ptrs]      # exchange buffers / peer mappings to release in close()
        for r in range(world):
            if r == rank:
                self.peer_ptrs.append(p.value)
                continue
            buf = (C.c_uint8 * 64).from_buffer_copy(handles[r])
            q = C.c_void_p()
            _lib.check(self.lib.dlrmb_xbuf_open(self.device.index or 0, buf, C.byref(q)))
            self.peer_ptrs.append(q.value)
        self.T = torch.as_tensor(_DevicePtrView(p.value, self.shape, self), device=self.device)
        self._flag = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._barrier = barrier
        self.G = None
        self.peer_G_ptrs = None
        self._gbuf = None
        self._closed = False
        self._fbuf = None
        self.peer_flag_ptrs = None
        self._ibuf = None
        self.idx_owned = None
        self._idx_dests = None
        self._jag = None
        if barrier is None and flag_barrier:
            # ordering without NCCL: a flag array per rank, mapped by every peer (dlrmb_peer_barrier)
            self._fbuf, _own, self.peer_flag_ptrs = self._share(int(self.lib.dlrmb_peer_barrier_flag_bytes()))
            self._bstate = torch.zeros(int(self.lib.dlrmb_peer_barrier_state_bytes()) // 4, dtype=torch.int32, device=self.device)
            self._flag_arr = (C.c_void_p * world)(*[int(q) for q in self.peer_flag_ptrs])
            torch.cuda.synchronize(self.device)
            dist.barrier(group=group)           # every rank's flag array exists and is zero before anyone signals

    def enable_index_exchange(self, sharding: "TableSharding", B_local: int, P: Union[int, Sequence[int]],
                              idx_bytes: int = 4):
        """Index exchange by peer stores: an index buffer [t_mine][B_global][P] on every rank, mapped
        everywhere; each rank stores its samples' index columns straight into the owners' buffers.
        ``P`` a sequence (one pooling factor per table): the buffer holds the owner layout of
        :func:`exchange_indices_mp` (sum over the owned tables of B_global * P_k indices) and ``idx_owned``
        is a :class:`~dlrm_jl_b200.embedding.PackedIndices`."""
        from .embedding import _DevicePtrView
        if sharding.split:
            Pt = (int(P),) * len(sharding.rows) if isinstance(P, (int, np.integer)) else tuple(int(p) for p in P)
            return self._enable_index_exchange_cw(sharding, B_local, Pt, idx_bytes)
        if not isinstance(P, (int, np.integer)):
            return self._enable_index_exchange_mp(sharding, B_local, tuple(int(p) for p in P), idx_bytes)
        counts = sharding.counts()
        t_mine = counts[self.rank]
        Bg = B_local * self.world
        per_table = Bg * P * idx_bytes
        self._ibuf, own, peer_idx = self._share(max(1, t_mine) * per_table)
        dt, ts = (torch.int32, "<i4") if idx_bytes == 4 else (torch.int64, "<i8")
        self.idx_owned = torch.as_tensor(_DevicePtrView(own, (max(1, t_mine), Bg, P), self, ts), device=self.device)
        assert self.idx_owned.dtype == dt
        dests = [peer_idx[sharding.owner[k]] + sharding.local[sharding.owner[k]].index(k) * per_table
                 for k in range(len(sharding.rows))]
        self._idx_dests = torch.tensor(dests, dtype=torch.int64, device=self.device)
        self._idx_geom = (len(sharding.rows), B_local, P, idx_bytes)

    def _enable_index_exchange_mp(self, sharding: "TableSharding", B_local: int, P: Tuple[int, ...], idx_bytes: int):
        import ctypes as C

        from .embedding import PackedIndices, _DevicePtrView
        if len(P) != len(sharding.rows) or min(P) < 1:
            raise ValueError(f"P must hold one pooling factor >= 1 per table ({len(sharding.rows)} tables), got {list(P)}")
        Bg = B_local * self.world
        mine = sharding.local[self.rank]
        n_owned = sum(Bg * P[k] for k in mine)
        self._ibuf, own, peer_idx = self._share(max(1, n_owned) * idx_bytes)
        ts = "<i4" if idx_bytes == 4 else "<i8"
        flat = torch.as_tensor(_DevicePtrView(own, (max(1, n_owned),), self, ts), device=self.device)
        self.idx_owned = PackedIndices(flat[:n_owned], tuple(P[k] for k in mine), Bg)
        dests = []
        for k in range(len(sharding.rows)):        # owner's block of table k: after its owned tables below k
            o = sharding.owner[k]
            dests.append(peer_idx[o] + sum(Bg * P[i] for i in sharding.local[o] if i < k) * idx_bytes)
        self._idx_dests = torch.tensor(dests, dtype=torch.int64, device=self.device)
        self._idx_geom = (len(sharding.rows), B_local, P, idx_bytes)
        self._idx_P = (C.c_int32 * len(P))(*P)

    def _enable_index_exchange_cw(self, sharding: "TableSharding", B_local: int, P: Tuple[int, ...], idx_bytes: int):
        """Column-wise plan: the index buffer holds the owner layout of every width group of this rank, group after
        group; ``idx_owned`` is a list of PackedIndices (one per group) and every holder of a slice of table k is a
        destination of k's block (dlrmb_indices_scatter_p2p_mp_list)."""
        import ctypes as C

        from .embedding import PackedIndices, _DevicePtrView
        if len(P) != len(sharding.rows) or min(P) < 1:
            raise ValueError(f"P must hold one pooling factor >= 1 per table ({len(sharding.rows)} tables), got {list(P)}")
        Bg = B_local * self.world

        def layout(r):       # element offset of every table's block in rank r's buffer
            off, o = {}, 0
            for _c, ks in sharding.groups(r):
                for k in ks:
                    off[k] = o
                    o += Bg * P[k]
            return off, o
        mine, n_owned = layout(self.rank)
        self._ibuf, own, peer_idx = self._share(max(1, n_owned) * idx_bytes)
        ts = "<i4" if idx_bytes == 4 else "<i8"
        flat = torch.as_tensor(_DevicePtrView(own, (max(1, n_owned),), self, ts), device=self.device)
        self.idx_owned = []
        for _c, ks in sharding.groups(self.rank):
            o = mine[ks[0]] if ks else 0
            n = sum(Bg * P[k] for k in ks)
            self.idx_owned.append(PackedIndices(flat[o:o + n], tuple(P[k] for k in ks), Bg))
        dest_table, dests = [], []
        for r in range(self.world):
            off, _n = layout(r)
            for k in sorted(off):
                dest_table.append(k)
                dests.append(peer_idx[r] + off[k] * idx_bytes)
        self._idx_dests = torch.tensor(dests, dtype=torch.int64, device=self.device)
        self._idx_list = (C.c_int32 * len(dest_table))(*dest_table)
        self._idx_geom = (len(sharding.rows), B_local, P, idx_bytes)
        self._idx_P = (C.c_int32 * len(P))(*P)

    def enable_jagged_index_exchange(self, sharding: "TableSharding", B_local: int, cap: Sequence[int],
                                     idx_bytes: int = 4, weighted: bool = False) -> None:
        """Index exchange of jagged batches by peer stores (:meth:`scatter_jagged`).  ``cap[k]`` is the most lookups of
        table k in one rank's local batch.  Every rank allocates, and maps on every peer, the buffers of its owner
        batch: values of world * (sum of cap over its tables) entries, offsets of t * B_global + 1 entries (t tables,
        the width of the indices) and, with ``weighted``, one f32 weight per value."""
        import ctypes as C

        from .embedding import _DevicePtrView
        if sharding.split:
            raise ValueError("jagged batches support table-wise plans only (a column-wise plan splits a table)")
        ntab, W = len(sharding.rows), self.world
        cap = tuple(int(c) for c in cap)
        if len(cap) != ntab or min(cap) < 0:
            raise ValueError(f"cap must hold one lookup count >= 0 per table ({ntab} tables), got {list(cap)}")
        Bg = B_local * W
        cap_own = [W * sum(cap[k] for k in sharding.local[o]) for o in range(W)]
        n_val, n_off = cap_own[self.rank], len(sharding.local[self.rank]) * Bg + 1
        ts = "<i4" if idx_bytes == 4 else "<i8"
        _h, own_v, peer_v = self._share(max(1, n_val) * idx_bytes)
        _h, own_o, peer_o = self._share(n_off * idx_bytes)
        self._jag_values = torch.as_tensor(_DevicePtrView(own_v, (max(1, n_val),), self, ts), device=self.device)
        self._jag_offsets = torch.as_tensor(_DevicePtrView(own_o, (n_off,), self, ts), device=self.device)
        self._jag_weights, peer_w = None, None
        if weighted:
            _h, own_w, peer_w = self._share(max(1, n_val) * 4)
            self._jag_weights = torch.as_tensor(_DevicePtrView(own_w, (max(1, n_val),), self), device=self.device)
            peer_w = (C.c_void_p * W)(*peer_w)
        self._jag = {"ntab": ntab, "B_local": B_local, "idx_bytes": idx_bytes, "cap": np.array(cap, dtype=np.int64),
                     "mine": list(sharding.local[self.rank]), "owner": (C.c_int32 * ntab)(*sharding.owner),
                     "peer_values": (C.c_void_p * W)(*peer_v), "peer_offsets": (C.c_void_p * W)(*peer_o),
                     "peer_weights": peer_w, "cap_values": (C.c_int64 * W)(*cap_own),
                     "empty": torch.zeros(4, dtype=torch.float32, device=self.device)}

    def scatter_jagged(self, jag_local, counts: np.ndarray):
        """This rank's :class:`~dlrm_jl_b200.embedding.JaggedIndices` -> the owners' buffers (peer stores, one launch)
        + barrier; returns this rank's owner batch, the layout of :func:`exchange_indices_jagged`, as a JaggedIndices
        view of its buffers.  ``counts``: :func:`exchange_jagged_counts`.  A batch over ``cap`` on any rank raises
        ValueError on every rank, before any launch."""
        import ctypes as C

        from . import _lib, _prof
        from .embedding import JaggedIndices
        j = self._jag
        counts = np.asarray(counts, dtype=np.int64)
        if jag_local.B != j["B_local"] or jag_local.element_size() != j["idx_bytes"] or len(jag_local) != j["ntab"]:
            raise ValueError(f"a jagged batch of {len(jag_local)} tables, B = {jag_local.B} and {jag_local.element_size()}-"
                             f"byte indices, the exchange was set up for {j['ntab']} tables, B_local = {j['B_local']} "
                             f"and {j['idx_bytes']}-byte indices")
        if (jag_local.weights is not None) != (j["peer_weights"] is not None):
            raise ValueError("the batch's per-sample weights do not match the exchange (enable_jagged_index_exchange("
                             "weighted=...))")
        over = np.argwhere(counts > j["cap"][None, :])
        if len(over):
            h, k = (int(x) for x in over[0])
            raise ValueError(f"rank {h} has {int(counts[h, k])} lookups of table {k}, more than cap[{k}] = "
                             f"{int(j['cap'][k])}")
        W, ntab = self.world, j["ntab"]
        L_all = (C.c_int64 * (W * ntab))(*counts.reshape(-1).tolist())
        w = None
        if jag_local.weights is not None:
            w = jag_local.weights.data_ptr() or j["empty"].data_ptr()
        with _prof.range("indices_scatter"):
            _lib.check(self.lib.dlrmb_indices_scatter_p2p_jagged(
                self.device.index or 0, jag_local.values.data_ptr() or None, jag_local.offsets.data_ptr(), w,
                j["idx_bytes"], ntab, j["B_local"], j["owner"], L_all, W, self.rank, j["peer_values"],
                j["peer_offsets"], j["peer_weights"], j["cap_values"], int(torch.cuda.current_stream(self.device).cuda_stream)))
        self.barrier(0)
        L_own = tuple(int(counts[:, k].sum()) for k in j["mine"])
        n = sum(L_own)
        return JaggedIndices(self._jag_values[:n], self._jag_offsets, L_own, j["B_local"] * W, jag_local.pooling,
                             None if self._jag_weights is None else self._jag_weights[:n])

    def enable_small_allreduce(self, n: int) -> None:
        """Exchange buffer [2][world][n] floats for `allreduce_small` (dlrmb_peer_allreduce_f32)."""
        import ctypes as C
        assert self.peer_flag_ptrs is not None, "the one-shot all-reduce is ordered by the flag barrier"
        self._ar_n = int(n)
        self._arbuf, _own, ptrs = self._share(2 * self.world * self._ar_n * 4)
        self._ar_arr = (C.c_void_p * self.world)(*[int(q) for q in ptrs])

    def allreduce_small(self, t: torch.Tensor) -> None:
        """In-place sum of `t` (contiguous f32, numel == the enabled n, a multiple of 4) over all ranks: every
        rank pushes its copy into every rank's buffer over NVLink, flag barrier, rank-ordered local sum."""
        from . import _lib, _prof
        assert t.is_contiguous() and t.dtype == torch.float32 and t.numel() == self._ar_n
        with _prof.range("peer_allreduce"):
            _lib.check(self.lib.dlrmb_peer_allreduce_f32(
                self.device.index or 0, self._ar_arr, self._flag_arr, self.world, self.rank, 3, self._bstate.data_ptr(),
                t.data_ptr(), t.numel(), int(torch.cuda.current_stream(self.device).cuda_stream)))

    def scatter_indices(self, idx_local: torch.Tensor) -> torch.Tensor:
        """idx_local [ntab][B_local][P] -> the owners' buffers (peer stores) + barrier; returns this rank's
        idx_owned [t_mine][B_global][P] (PackedIndices in, PackedIndices in the owner layout out when the
        exchange was enabled with per-table pooling factors)."""
        from . import _lib
        ntab, Bl, P, ib = self._idx_geom
        if isinstance(P, tuple) and getattr(self, "_idx_list", None) is not None:
            from . import _prof
            assert tuple(idx_local.P) == P and idx_local.B == Bl and idx_local.element_size() == ib
            with _prof.range("indices_scatter"):
                _lib.check(self.lib.dlrmb_indices_scatter_p2p_mp_list(
                    self.device.index or 0, idx_local.data_ptr(), ib, ntab, Bl, self._idx_P, len(self._idx_list),
                    self._idx_list, self._idx_dests.data_ptr(), self.rank,
                    int(torch.cuda.current_stream(self.device).cuda_stream)))
            self.barrier(0)
            return self.idx_owned
        if isinstance(P, tuple):
            from . import _prof
            assert tuple(idx_local.P) == P and idx_local.B == Bl and idx_local.element_size() == ib
            with _prof.range("indices_scatter"):
                _lib.check(self.lib.dlrmb_indices_scatter_p2p_mp(
                    self.device.index or 0, idx_local.data_ptr(), ib, ntab, Bl, self._idx_P, self._idx_dests.data_ptr(),
                    self.rank, int(torch.cuda.current_stream(self.device).cuda_stream)))
            self.barrier(0)
            return self.idx_owned
        assert tuple(idx_local.shape) == (ntab, Bl, P) and idx_local.element_size() == ib and idx_local.is_contiguous()
        from . import _prof
        with _prof.range("indices_scatter"):
            _lib.check(self.lib.dlrmb_indices_scatter_p2p(
                self.device.index or 0, idx_local.data_ptr(), ib, ntab, Bl, P, self._idx_dests.data_ptr(), self.rank,
                int(torch.cuda.current_stream(self.device).cuda_stream)))
        self.barrier(0)
        return self.idx_owned

    def close(self) -> None:
        """Unmap the peers' buffers (cudaIpcCloseMemHandle) and free this rank's exchange buffers.  Every
        rank must have finished using the mappings (call after a barrier); views of T / G are dead after."""
        if getattr(self, "_closed", True):
            return
        self._closed = True
        dev = self.device.index or 0
        for ptrs in self._mapped:
            for r, q in enumerate(ptrs):
                if r != self.rank and q:
                    self.lib.dlrmb_xbuf_close(dev, q)
        self.T = self.G = self.idx_owned = None
        self._jag = self._jag_values = self._jag_offsets = self._jag_weights = None
        for h in [self._xbuf] + self._owned:
            if h is not None:
                self.lib.dlrmb_xbuf_destroy(h)
        self._xbuf = self._gbuf = self._fbuf = self._ibuf = None
        self._owned, self._mapped = [], []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _share(self, nbytes: int):
        """Allocate an exchange buffer and map every rank's copy: returns (own ptr, [ptr per rank])."""
        import ctypes as C

        from . import _lib
        h = C.c_void_p()
        _lib.check(self.lib.dlrmb_xbuf_create(self.device.index or 0, max(256, nbytes), C.byref(h)))
        p = C.c_void_p()
        _lib.check(self.lib.dlrmb_xbuf_ptr(h, C.byref(p)))
        handle = (C.c_uint8 * 64)()
        _lib.check(self.lib.dlrmb_xbuf_ipc_handle(h, handle))
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle), group=self.group)
        ptrs = []
        for r in range(self.world):
            if r == self.rank:
                ptrs.append(p.value)
                continue
            q = C.c_void_p()
            _lib.check(self.lib.dlrmb_xbuf_open(self.device.index or 0, (C.c_uint8 * 64).from_buffer_copy(handles[r]), C.byref(q)))
            ptrs.append(q.value)
        self._owned.append(h)
        self._mapped.append(ptrs)
        return h, p.value, ptrs

    def enable_gradient_exchange(self, sharding: "TableSharding", B_local: int, D: int, split_dx: bool = False):
        """Gradient buffer G [B_global][tables of this rank][D] on every rank, mapped everywhere, and
        the per-slot destination table the scattered interaction backward reads."""
        from .embedding import _DevicePtrView
        from .interact import ScatterPlan
        if sharding.split:
            return self._enable_gradient_exchange_cw(sharding, B_local, D, split_dx)
        counts = sharding.counts()
        t_mine = counts[self.rank]
        Bg = B_local * self.world
        self._gbuf, own, self.peer_G_ptrs = self._share(Bg * max(1, t_mine) * D * 4)
        self.G = torch.as_tensor(_DevicePtrView(own, (Bg, max(1, t_mine), D), self), device=self.device)
        rows = [[0, 0, 0]]                                    # slot 0 (x) has no destination
        for k in range(len(sharding.rows)):
            o = sharding.owner[k]
            rows.append([self.peer_G_ptrs[o], counts[o] * D, sharding.local[o].index(k) * D])
        dests = torch.tensor(rows, dtype=torch.int64, device=self.device)
        return ScatterPlan(dests, self.rank * B_local, torch.cuda.Stream(self.device) if split_dx else None)

    def _enable_gradient_exchange_cw(self, sharding: "TableSharding", B_local: int, D: int, split_dx: bool):
        """Column-wise plan: one gradient buffer G [B_global][tables of the group][D / c] per width group, mapped
        everywhere (``self.G`` is the list of this rank's, in group order), and a scatter plan of Q = max c_k column
        pieces per slot (dlrmb_interaction_bwd_scatter_cols)."""
        from .embedding import _DevicePtrView
        from .interact import ScatterPlan
        Bg = B_local * self.world
        widths = sorted(set(sharding.shards))
        grp = [dict(sharding.groups(r)) for r in range(self.world)]       # rank -> {c: tables}
        peer_G = {}
        mine = dict(sharding.groups(self.rank))
        G = {}
        for c in widths:      # collective: every rank maps one buffer per width of the plan, in the same order
            t = len(mine.get(c, []))
            _h, own, peer_G[c] = self._share(Bg * max(1, t) * (D // c) * 4)
            G[c] = torch.as_tensor(_DevicePtrView(own, (Bg, max(1, t), D // c), self), device=self.device)
        self.G = [G[c] for c, _ks in sharding.groups(self.rank)]
        self.peer_G_ptrs = peer_G
        Q = max(sharding.shards)
        pw = D // Q
        rows = [[0, 0, 0]] * Q                                # slot 0 (x) has no destination
        for k in range(len(sharding.rows)):
            c = sharding.shards[k]
            for q in range(Q):
                j, sub = divmod(q, Q // c)
                h = sharding.holders[k][j]
                ks = grp[h][c]
                rows.append([peer_G[c][h], len(ks) * (D // c), ks.index(k) * (D // c) + sub * pw])
        dests = torch.tensor(rows, dtype=torch.int64, device=self.device)
        return ScatterPlan(dests, self.rank * B_local, torch.cuda.Stream(self.device) if split_dx else None, Q=Q)

    def barrier(self, channel: int = 0) -> None:
        """Order this rank's earlier peer stores before every rank's later reads (stream-ordered).
        Flag barrier over the mapped buffers (one tiny kernel, dlrmb_peer_barrier) when available; a
        caller-supplied callable (tests: host-side barrier) or a one-element NCCL all-reduce otherwise."""
        if self._barrier is not None:
            self._barrier()
        elif self.peer_flag_ptrs is not None:
            from . import _lib, _prof
            with _prof.range(f"peer_barrier_{channel}"):
                _lib.check(self.lib.dlrmb_peer_barrier(
                    self.device.index or 0, self._flag_arr, self.world, self.rank, channel, self._bstate.data_ptr(),
                    int(torch.cuda.current_stream(self.device).cuda_stream)))
        else:
            dist.all_reduce(self._flag, group=self.group)

    def barrier_timeouts(self) -> int:
        """Number of flag-barrier waits that gave up (a peer died); 0 in a healthy run."""
        if self.peer_flag_ptrs is None:
            return 0
        return int(self._bstate[-1].item())


class _ShardedLookupFn(torch.autograd.Function):
    """lookup (owner side) + pooled all-to-all forward; gradient all-to-all backward.  The
    owner-side gradient [B_global][t_mine][D] is parked on ``ctx_obj.owned_grad`` for the sparse
    update (the tables are not torch parameters, as in the reference where the lookup pullback
    yields SparseEmbeddingUpdate objects rather than dense gradients)."""

    @staticmethod
    def forward(ctx, anchor: torch.Tensor, se: "ShardedEmbedding", idx_local: torch.Tensor):
        from .embedding import _batch
        ctx.se = se
        D = se.D
        Bl = _batch(idx_local)
        if se.world == 1:
            # no exchange: pool straight into the interaction input (slot 0 is filled with x by
            # the interaction kernel's fused fast_vcat); the same launch sorts the indices for the update
            se.idx_owned = idx_local
            T = torch.empty((Bl, 1 + se.ntab, D), dtype=torch.float32, device=idx_local.device)
            se.lookup_fn(idx_local, T, 1)
            se.presorted = se.lookup_sorts
            return T
        if se.split:
            return se._forward_cw(idx_local, Bl)
        idx_owned = se._exchange_indices(idx_local)
        se.idx_owned = idx_owned
        se.presorted = False
        Bg = _batch(idx_owned)
        if se.peer is not None:
            # fused path: pooled rows go straight into the owners' T over NVLink; the barrier
            # orders every rank's stores before anyone reads its own T
            if len(se.local_ids):
                fuse = se._fuse_sort(idx_owned)
                se.tables.lookup_p2p(idx_owned, se.peer.peer_ptrs, Bl, 1 + se.ntab, se.idx_base, sort=fuse)
                se.presorted = fuse
            se.peer.barrier(1)
            # a fresh alias every step: the persistent buffer tensor itself must never pick up
            # autograd history (a stale grad_fn from an earlier step would chain the graphs)
            return se.peer.T.detach()
        pooled = torch.empty((Bg, len(se.local_ids), D), dtype=torch.float32, device=idx_local.device)
        if len(se.local_ids):
            se.lookup_fn(idx_owned, pooled, 0)
        # slot 0 needs no clearing: the interaction kernel writes x there (fused fast_vcat)
        T = torch.empty((Bl, 1 + se.ntab, D), dtype=torch.float32, device=idx_local.device)
        exchange_pooled(pooled, T, se.sharding, se.rank, se.group)
        return T

    @staticmethod
    def backward(ctx, dT: torch.Tensor):
        se = ctx.se
        if se.world == 1:
            se.owned_grad = dT.contiguous()      # [B][1 + ntab][D], consumed with slot0 = 1
        elif se.split:
            se.owned_grad = exchange_grads_cw(dT.contiguous(), se.sharding, se.rank, se.group)
        else:
            se.owned_grad = exchange_grads(dT.contiguous(), se.sharding, se.rank, se.group)
        se._update_from_backward(fused=False)
        return None, None, None


class ShardedEmbedding:
    """Table-wise sharded drop-in for ``maplookup`` + ``update!`` at world size W.

    ``lookup_fn(idx_owned [t][Bg][P], out [Bg][slot0 + t][D], slot0)`` and
    ``update_fn(idx_owned, grad [Bg][slot0 + t][D], lr, slot0, presorted)`` do the local compute;
    :meth:`create` wires them to an :class:`~dlrm_jl_b200.embedding.EmbeddingTables` holding this
    rank's tables.  ``slot0`` is 1 at world size 1 (the buffers ARE the interaction input) else 0.

    When the plan splits a table by columns (``max_col_shards`` > 1), the rank's units form width groups
    (:meth:`TableSharding.groups`, ``self.groups``) and the injected functions take the group's position as one
    more argument: ``lookup_fn(idx_g, out [Bg][t_g][D / c_g], 0, g)``, ``update_fn(idx_g, grad_g, lr, 0, presorted,
    g)``, ``sort_fn(idx_g, g)``; :meth:`create` gives each group an EmbeddingTables of its width.
    """

    def __init__(self, rows: Sequence[int], D: int, rank: int, world: int, lookup_fn: Callable,
                 update_fn: Callable, group=None, sort_fn: Optional[Callable] = None, idx_base: int = 0,
                 lookup_sorts: bool = False, P: Optional[Sequence[int]] = None, max_col_shards: int = 1,
                 jagged_cap: Optional[Sequence[int]] = None, count_group=None):
        """``idx_base``: 1 for reference-format (1-based) ids, 0 for PyTorch-style ids; it is handed to
        every kernel that reads the indices.  ``lookup_sorts``: `lookup_fn` also prepares the sort /
        dedup of the step's update (the fused launch), so `sort_async` has nothing left to do.
        ``P``: per-table pooling factors (one per table).  Then the tables are placed by
        ``TableSharding.build(rows, world, P)``, batches are :class:`~dlrm_jl_b200.embedding.PackedIndices`
        (or anything ``_as_index_tensor`` turns into one) and the owners receive theirs in the owner layout
        of :func:`exchange_indices_mp`.  Without it every table has the same P and mixed widths are refused.
        ``max_col_shards``: split hot tables by columns into up to that many slices (a power of two, D divisible into
        slices of a multiple of 4 columns); see :meth:`TableSharding.build`.
        ``jagged_cap``: the handle takes :class:`~dlrm_jl_b200.embedding.JaggedIndices` (variable-length bags, sum,
        mean or weighted pooling), ``jagged_cap[k]`` being the most lookups of table k in one rank's local batch.  ``P``
        then only weighs the tables in the plan: pass each table's expected bag length (at least 1), for instance the
        MLPerf hotness list.  Every step starts with a host all-gather of the ranks' lookup counts
        (:func:`exchange_jagged_counts`) over ``count_group`` if given, else over ``group`` when it runs on gloo, else
        over a gloo group made here across the whole job (:func:`gloo_group`; a non-gloo proper subgroup needs
        ``count_group``).  Column-wise plans of jagged tables are not supported."""
        self.P = None if P is None else tuple(int(p) for p in P)
        self.jagged_cap = None if jagged_cap is None else tuple(int(c) for c in jagged_cap)
        if self.jagged_cap is not None and len(self.jagged_cap) != len(rows):
            raise ValueError(f"jagged_cap must hold one lookup count per table ({len(rows)} tables), got "
                             f"{list(self.jagged_cap)}")
        if int(max_col_shards) == 1:
            self.sharding = TableSharding.build(rows, world, self.P)
        else:
            self.sharding = TableSharding.build(rows, world, self.P, D=D, max_col_shards=max_col_shards)
        self.split = self.sharding.split
        if self.split and self.jagged_cap is not None:
            raise ValueError("jagged_cap: jagged batches support table-wise plans only, and this column-wise plan "
                             f"(max_col_shards = {max_col_shards}) splits a table")
        self.groups = self.sharding.groups(rank)
        self.rank, self.world, self.group = rank, world, group
        self.idx_base = int(idx_base)
        self.lookup_sorts = bool(lookup_sorts)
        self.presorted = False
        self.D = D
        self.ntab = len(rows)
        self.local_ids = self.sharding.local[rank]
        self.lookup_fn, self.update_fn, self.sort_fn = lookup_fn, update_fn, sort_fn
        self.idx_owned: Optional[torch.Tensor] = None
        self.owned_grad: Optional[torch.Tensor] = None
        self.slot0 = 1 if world == 1 else 0
        self.peer: Optional[PeerExchange] = None
        self.scatter_plan = None
        self._auto_update = None
        self._count_group = None
        if self.jagged_cap is not None and world > 1:
            self._count_group = count_group if count_group is not None else gloo_group(group)

    # ---- column-wise plans: one handle / index block / gradient per width group -------------------------
    def _forward_cw(self, idx_local, Bl: int) -> torch.Tensor:
        idx_groups = self._exchange_indices(idx_local)
        self.idx_owned = idx_groups
        self.presorted = [False] * len(self.groups)
        if self.peer is not None:
            self._lookup_p2p_cw(idx_groups, Bl)
            self.peer.barrier(1)
            return self.peer.T.detach()
        dev = idx_groups[0].flat.device if idx_groups else torch.device("cpu")
        pooled = []
        for g, (c, ks) in enumerate(self.groups):
            out = torch.empty((Bl * self.world, len(ks), self.D // c), dtype=torch.float32, device=dev)
            self.lookup_fn(idx_groups[g], out, 0, g)
            pooled.append(out)
        T = torch.empty((Bl, 1 + self.ntab, self.D), dtype=torch.float32, device=self._device(idx_local))
        exchange_pooled_cw(pooled, T, self.sharding, self.rank, self.group)
        return T

    def _lookup_p2p_cw(self, idx_groups, Bl: int) -> None:
        for g, tables in enumerate(self.group_tables):
            fuse = self._fuse_sort(idx_groups[g])
            tables.lookup_p2p(idx_groups[g], self.peer.peer_ptrs, Bl, 1 + self.ntab, self.idx_base, sort=fuse)
            self.presorted[g] = fuse

    @staticmethod
    def _device(idx):
        from .embedding import PackedIndices
        return idx.flat.device if isinstance(idx, PackedIndices) else idx.device

    def download(self, k: int) -> List[Tuple[int, np.ndarray]]:
        """Read back what this rank holds of global table k: [(first column, [rows_k][width] array)] for every
        slice (one entry, column 0, for a whole table; none when the rank holds nothing of k).  Needs :meth:`create`."""
        out = []
        for (c, ks), tables in zip(self.groups, self.group_tables):
            if k in ks:
                out.append((self.sharding.slice_of(k, self.rank) * (self.D // c), tables.download(ks.index(k))))
        return out

    def update_inside_backward(self, lr: float, stream: "torch.cuda.Stream") -> None:
        """Launch the sparse update from INSIDE the backward pass, on ``stream``, as soon as the pooled-embedding
        gradient exists (the lookup's pullback, or the scattering interaction backward on the fused path)
        instead of after ``loss.backward()`` has returned.  The update touches the tables only, so it then runs
        beside the bottom MLP's backward (autograd joins every backward stream before ``backward()`` returns, so
        a call placed after it starts a whole bottom-MLP backward later).  The caller joins ``stream`` at the
        end of the step; do not call :meth:`update` / :meth:`finish_backward` yourself in this mode."""
        self._auto_update = (float(lr), stream)
        if self.scatter_plan is not None:
            self.scatter_plan.on_launched = lambda: self._update_from_backward(fused=True)

    def _update_from_backward(self, fused: bool) -> None:
        if self._auto_update is None:
            return
        lr, stream = self._auto_update
        cur = torch.cuda.current_stream(self.tables.device)
        stream.wait_stream(cur)
        with torch.cuda.stream(stream):
            if fused:
                self.finish_backward()
            self.update(lr)

    def enable_fused_backward(self, B_local: int, split_dx: bool = False) -> None:
        """Also fuse the backward exchange: the interaction backward stores dT rows into the owners'
        gradient buffers (pass `self.scatter_plan` to DotInteraction), `finish_backward()` orders the
        stores before the sparse update.  Needs enable_peer_exchange first.  ``split_dx``: dx is computed
        by a small kernel of its own ahead of the scattering pullback, which then runs on a side stream
        beside the bottom MLP's backward."""
        assert self.peer is not None
        self.scatter_plan = self.peer.enable_gradient_exchange(self.sharding, B_local, self.D, split_dx)
        if self._auto_update is not None:
            self.scatter_plan.on_launched = lambda: self._update_from_backward(fused=True)

    def lookup_fused(self, idx_local: torch.Tensor) -> torch.Tensor:
        """Forward of the fully fused path: no autograd node (the gradient never comes back through
        T; it is scattered to the owners by the interaction backward)."""
        from .embedding import _batch
        idx_local = self._indices(idx_local)
        with torch.no_grad():
            idx_owned = self._exchange_indices(idx_local)
            self.idx_owned = idx_owned
            if self.split:
                self.presorted = [False] * len(self.groups)
                self._lookup_p2p_cw(idx_owned, _batch(idx_local))
                self.peer.barrier(1)
                return self.peer.T.detach()
            self.presorted = False
            if len(self.local_ids):
                # up to 4096 lookups per table the sort of the coming update rides in the lookup launch
                fuse = self._fuse_sort(idx_owned)
                self.tables.lookup_p2p(idx_owned, self.peer.peer_ptrs, _batch(idx_local), 1 + self.ntab, self.idx_base,
                                       sort=fuse)
                self.presorted = fuse
            self.peer.barrier(1)
            return self.peer.T.detach()

    def _fuse_sort(self, idx_owned) -> bool:
        """Whether every owned table's sort fits the lookup launch (B_global * P_k <= FUSED_SORT_MAX); otherwise
        the large sorts go to the side stream (`sort_async`), off the critical path."""
        from .embedding import JaggedIndices, PackedIndices
        if isinstance(idx_owned, JaggedIndices):
            # no jagged sort rides inside the lookup launch.  With the fused backward the sort goes to the side stream
            # and finish_backward joins it before barrier(2); without it the _sort_ form sorts on this stream ahead of
            # barrier(1), so no peer's next index scatter can overwrite the owner batch while the sort reads it
            return self.scatter_plan is None
        if isinstance(idx_owned, PackedIndices):
            return max(idx_owned.P) * idx_owned.B <= self.tables.FUSED_SORT_MAX
        return idx_owned.shape[1] * idx_owned.shape[2] <= self.tables.FUSED_SORT_MAX

    def _indices(self, idx_local):
        """A handle with one P refuses mixed widths; one with per-table P takes PackedIndices or anything
        `_as_index_tensor` normalises (the reference's mixed list, or a [ntab][B][P] tensor when every P_k
        is equal) and checks the widths against its P.  A handle created with ``jagged_cap`` takes JaggedIndices
        only, every other handle refuses them."""
        from .embedding import JaggedIndices
        if isinstance(idx_local, JaggedIndices) or self.jagged_cap is not None:
            return self._jagged_indices(idx_local)
        if self.P is None:
            _require_uniform_pooling(idx_local)
            if self.split:       # column-wise plans exchange through the per-table-P machinery
                from .embedding import PackedIndices
                ntab, B, P = idx_local.shape
                return PackedIndices(idx_local.contiguous().reshape(-1), (int(P),) * ntab, int(B))
            return idx_local
        from .embedding import PackedIndices, _as_index_tensor
        tables = getattr(self, "tables", None)
        if tables is not None:
            device = tables.device
        else:
            device = idx_local.flat.device if isinstance(idx_local, PackedIndices) else (
                idx_local.device if isinstance(idx_local, torch.Tensor) else torch.device("cpu"))
        idx = _as_index_tensor(idx_local, self.ntab, device)
        if not isinstance(idx, PackedIndices):
            if tuple(int(idx.shape[2]) for _ in range(self.ntab)) != self.P:
                raise ValueError(f"batch widths {[int(idx.shape[2])] * self.ntab} differ from the handle's P {list(self.P)}")
            idx = PackedIndices(idx.reshape(-1), self.P, int(idx.shape[1]))
        if tuple(idx.P) != self.P:
            raise ValueError(f"batch widths {list(idx.P)} differ from the handle's P {list(self.P)}")
        return idx

    def _jagged_indices(self, idx_local):
        from .embedding import JaggedIndices
        if self.jagged_cap is None:
            raise ValueError("jagged batches need a handle created with jagged_cap (the most lookups of each table in "
                             "one rank's batch)")
        if not isinstance(idx_local, JaggedIndices):
            raise ValueError(f"a handle created with jagged_cap takes JaggedIndices, got {type(idx_local).__name__}")
        if len(idx_local) != self.ntab:
            raise ValueError(f"indices must hold one table per table of the handle: {self.ntab} tables, got "
                             f"{len(idx_local)}")
        over = [k for k in range(self.ntab) if idx_local.L[k] > self.jagged_cap[k]]
        if over:
            k = over[0]
            raise ValueError(f"table {k} has {idx_local.L[k]} lookups, more than jagged_cap[{k}] = {self.jagged_cap[k]}")
        tables = getattr(self, "tables", None)
        return idx_local if tables is None else idx_local.to(tables.device, non_blocking=True)

    def _exchange_indices(self, idx_local: torch.Tensor) -> torch.Tensor:
        """Index columns to the tables' owners: peer stores + flag barrier when the index buffers are
        mapped (`enable_index_exchange`), NCCL all-to-all otherwise.  Jagged batches first gather every rank's
        lookup counts on the host."""
        if self.jagged_cap is not None:
            counts = exchange_jagged_counts(idx_local, self._count_group)
            if self.peer is not None and self.peer._jag is not None:
                return self.peer.scatter_jagged(idx_local, counts)
            return exchange_indices_jagged(idx_local, counts, self.sharding, self.rank, self.group)
        if self.split:
            if self.peer is not None and self.peer._idx_dests is not None:
                return self.peer.scatter_indices(idx_local)
            return exchange_indices_cw(idx_local, self.sharding, self.rank, self.group)
        if self.P is not None:
            if self.peer is not None and self.peer._idx_dests is not None:
                return self.peer.scatter_indices(idx_local)
            return exchange_indices_mp(idx_local, self.sharding, self.rank, self.group)
        if self.peer is not None and self.peer._idx_dests is not None:
            owned = self.peer.scatter_indices(idx_local)
            return owned[:len(self.local_ids)] if len(self.local_ids) else owned[:0]
        return exchange_indices(idx_local, self.sharding, self.rank, self.group)

    def finish_backward(self) -> None:
        """After loss.backward() on the fused path: every rank's gradient rows have landed.  The index
        sort of this step (side stream) is joined first: once a rank passes this barrier its peers may
        start the next step and overwrite the index buffer the sort reads."""
        for tables in (self.group_tables if self.split else [self.tables] if len(self.local_ids) else []):
            if getattr(tables, "_pending_side", False):
                torch.cuda.current_stream(tables.device).wait_event(tables._sorted_event)
                tables._pending_side = False
        plan = self.scatter_plan
        if plan is not None and plan.stream is not None and plan._keep is not None:
            torch.cuda.current_stream(self.tables.device).wait_event(plan.done)     # this rank's peer stores are issued
            plan._keep = None
        self.peer.barrier(2)
        self.owned_grad = self.peer.G

    def enable_peer_exchange(self, B_local: int, barrier: Optional[Callable] = None, flag_barrier: bool = True,
                             P: Optional[Union[int, Sequence[int]]] = None, idx_bytes: int = 4,
                             weighted: bool = False) -> None:
        """Switch the forward exchange to the fused lookup + NVLink peer-store kernel.  Safe with
        one buffer per rank when every step also runs the backward exchange (a barrier all ranks
        reach only after they have finished reading T).  With ``P`` (lookups per sample, or the handle's
        per-table pooling factors) given, the index exchange also goes over peer stores instead of an NCCL
        all-to-all; for a handle created with ``jagged_cap`` that is the jagged exchange
        (:meth:`PeerExchange.enable_jagged_index_exchange`), ``weighted`` saying whether its batches carry per-sample
        weights."""
        if self.P is not None and P is not None and tuple(int(p) for p in P) != self.P:
            raise ValueError(f"P {list(P)} differs from the handle's per-table P {list(self.P)}")
        if self.world == 1:
            return
        if self.split:
            for (c, ks), tables in zip(self.groups, self.group_tables):
                tables.set_dest_map([1 + k for k in ks], [self.sharding.slice_of(k, self.rank) * (self.D // c) for k in ks],
                                    self.D)
        else:
            self.tables.set_slot_map([1 + k for k in self.local_ids] or [1])
        self.peer = PeerExchange(B_local, self.ntab, self.D, self.rank, self.world, self.tables.device,
                                 self.group, barrier, flag_barrier)
        if P is not None and self.jagged_cap is not None:
            self.peer.enable_jagged_index_exchange(self.sharding, B_local, self.jagged_cap, idx_bytes, weighted)
        elif P is not None:
            self.peer.enable_index_exchange(self.sharding, B_local, P, idx_bytes)

    @classmethod
    def create(cls, rows: Sequence[int], D: int, B_local: int, P: Union[int, Sequence[int]], rank: int, world: int,
               device, group=None, seed: int = 51234, idx_base: int = 0, dtype=None,
               max_col_shards: int = 1, jagged_cap: Optional[Sequence[int]] = None,
               count_group=None) -> "ShardedEmbedding":
        """``P``: lookups per sample of every table, or a sequence of one pooling factor per table (mixed
        multi-hot; the plan then weighs each table by its P_k, see :class:`TableSharding`).  ``max_col_shards``:
        split hot tables by columns (one EmbeddingTables per width group of this rank).  ``jagged_cap``: the handle
        takes JaggedIndices (see :class:`ShardedEmbedding`); ``P`` are then the plan's weights, each table's expected
        bag length, and the tables are sized for world * max(jagged_cap[k]) lookups of an owned table."""
        from .embedding import EmbeddingTables
        Pseq = None if isinstance(P, (int, np.integer)) else tuple(int(p) for p in P)
        if int(max_col_shards) != 1:
            sh = TableSharding.build(rows, world, Pseq, D=D, max_col_shards=max_col_shards)
            if sh.split and jagged_cap is not None:
                raise ValueError("jagged_cap: jagged batches support table-wise plans only, and this column-wise plan "
                                 f"(max_col_shards = {max_col_shards}) splits a table")
            if sh.split:
                return cls._create_cw(rows, D, B_local, P, Pseq, rank, world, device, group, seed, idx_base, dtype,
                                      max_col_shards)
        sh = TableSharding.build(rows, world, Pseq)
        mine = sh.local[rank]
        kw = {} if dtype is None else {"dtype": dtype}
        if jagged_cap is not None:
            max_lookups = world * max([int(jagged_cap[k]) for k in mine] or [1])
        else:
            max_lookups = B_local * world * (P if Pseq is None else max([Pseq[k] for k in mine] or [1]))
        tables = EmbeddingTables([rows[k] for k in mine] or [1], D, max_lookups, device, **kw)
        tables.init_uniform(seed + 7919 * rank)
        fused_sort = world == 1      # single GPU: the sort rides in the lookup launch
        se = cls(rows, D, rank, world,
                 lookup_fn=lambda idx, out, slot0: tables.lookup(idx, out, slot0, idx_base, sort=fused_sort),
                 update_fn=lambda idx, g, lr, slot0, presorted=False: (
                     tables.update_sorted(g, slot0, lr) if presorted else tables.bwd_sgd(idx, g, slot0, lr, idx_base)),
                 group=group,
                 sort_fn=lambda idx: tables.sort(idx, idx_base, side_stream=True),
                 idx_base=idx_base, lookup_sorts=fused_sort, P=Pseq, jagged_cap=jagged_cap, count_group=count_group)
        se.tables = tables
        return se

    @classmethod
    def _create_cw(cls, rows, D, B_local, P, Pseq, rank, world, device, group, seed, idx_base, dtype,
                   max_col_shards) -> "ShardedEmbedding":
        from .embedding import EmbeddingTables
        sh = TableSharding.build(rows, world, Pseq, D=D, max_col_shards=max_col_shards)
        kw = {} if dtype is None else {"dtype": dtype}
        group_tables = []
        for g, (c, ks) in enumerate(sh.groups(rank)):
            max_lookups = B_local * world * (P if Pseq is None else max(Pseq[k] for k in ks))
            tables = EmbeddingTables([rows[k] for k in ks], D // c, max_lookups, device, **kw)
            tables.init_uniform(seed + 7919 * rank + 104729 * g)
            group_tables.append(tables)
        se = cls(rows, D, rank, world,
                 lookup_fn=lambda idx, out, slot0, g: group_tables[g].lookup(idx, out, slot0, idx_base),
                 update_fn=lambda idx, grad, lr, slot0, presorted, g: (
                     group_tables[g].update_sorted(grad, slot0, lr) if presorted
                     else group_tables[g].bwd_sgd(idx, grad, slot0, lr, idx_base)),
                 group=group,
                 sort_fn=lambda idx, g: group_tables[g].sort(idx, idx_base, side_stream=True),
                 idx_base=idx_base, P=Pseq, max_col_shards=max_col_shards)
        se.group_tables = group_tables
        se.tables = group_tables[0] if group_tables else None
        return se

    def lookup(self, idx_local: torch.Tensor, anchor: torch.Tensor) -> torch.Tensor:
        """idx_local [ntab][B_local][P] -> T [B_local][1 + ntab][D] (requires grad through `anchor`,
        any tensor that requires grad, so autograd calls the gradient exchange).  A handle with per-table
        pooling factors takes PackedIndices (or the reference's mixed list) instead."""
        return _ShardedLookupFn.apply(anchor, self, self._indices(idx_local))

    def sort_async(self) -> None:
        """Start the index sort/dedup for this step's update on the side stream (nothing to do when
        the lookup launch already produced it)."""
        if self.split:
            for g in range(len(self.groups)):
                if not self.presorted[g] and self.sort_fn is not None:
                    self.sort_fn(self.idx_owned[g], g)
                    self.presorted[g] = True
            return
        if self.presorted:
            return
        if self.sort_fn is not None and len(self.local_ids):
            self.sort_fn(self.idx_owned)
            self.presorted = True

    def update(self, lr: float, presorted: Optional[bool] = None) -> None:
        """Owner-side sparse SGD.  ``presorted`` defaults to whether this step's sort already ran
        (fused lookup launch or `sort_async`)."""
        if self.split:
            for g in range(len(self.groups)):
                self.update_fn(self.idx_owned[g], self.owned_grad[g], lr, self.slot0,
                               self.presorted[g] if presorted is None else presorted, g)
            self.presorted = [False] * len(self.groups)
            return
        if len(self.local_ids) == 0:
            return
        if presorted is None:
            presorted = self.presorted
        self.update_fn(self.idx_owned, self.owned_grad, lr, self.slot0, presorted)
        self.presorted = False

    def close(self) -> None:
        if self.peer is not None:
            self.peer.close()
            self.peer = None
            self.scatter_plan = None


class FlatGrads:
    """Dense (MLP) gradients as views of ONE flat buffer, so the data-parallel reduction is a
    single in-place all-reduce with no pack/unpack copies (NVSwitch: bucket sized for launch
    latency, not link count).  `zero()` before backward, `allreduce()` after; the 1/world mean
    factor is left to the caller's learning rate (`scale`)."""

    def __init__(self, params: Sequence[torch.nn.Parameter], world: int, group=None):
        self.params = list(params)
        self.world, self.group = world, group
        n = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(n, dtype=self.params[0].dtype, device=self.params[0].device)
        off = 0
        self.views = []
        for p in self.params:
            self.views.append(self.flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        self.scale = 1.0 / world

    def flatten_params(self) -> torch.Tensor:
        """Re-home the parameters as views of ONE flat buffer laid out like the gradient bucket, so
        the dense SGD step is a single `pflat.add_(flat, alpha=-lr)` instead of a multi-tensor pass."""
        pflat = torch.empty_like(self.flat)
        off = 0
        with torch.no_grad():
            for p in self.params:
                view = pflat[off:off + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view
                off += p.numel()
        self.pflat = pflat
        return pflat

    def zero(self) -> None:
        self.flat.zero_()
        for p, v in zip(self.params, self.views):
            p.grad = v

    def allreduce(self) -> None:
        if self.world > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)


def allreduce_dense_grads(params: Sequence[torch.nn.Parameter], world: int, group=None) -> None:
    """Sum the data-parallel MLP gradients with ONE all-reduce over a flat bucket (a few MB: sized
    for launch latency, NVSwitch gives every pair full bandwidth).  The loss is the mean over the
    local batch, so the global-batch mean needs a 1/world factor."""
    if world == 1:
        return
    grads = [p.grad for p in params if p.grad is not None]
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.mul_(1.0 / world)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(flat[off:off + n].view_as(g))
        off += n
