"""Host-side mirror of the EmbeddingTables.jl interface DLRM.jl uses, backed by HBM tables.

Reference interface (EmbeddingTables.jl v0.1.0 is an un-vendored path dependency of DLRM.jl,
``Manifest.toml:246-250``; names and argument meaning follow DLRM.jl's call sites):

===============================  =====================================================
reference                        here
===============================  =====================================================
``SimpleEmbedding{Static{D}}``   :class:`EmbeddingTables` (all tables of a model in one
(``src/data/criteo.jl:413,490``) handle so one launch covers every table)
``maplookup(strategy, tables,    :func:`maplookup`
sparse)`` (``model.jl:161``)
``PreallocationStrategy(r)``     :class:`PreallocationStrategy`
``DefaultStrategy()``            :class:`DefaultStrategy`
``SparseEmbeddingUpdate``        :class:`SparseEmbeddingUpdate`
(``src/train/train.jl:144``)
``uncompress(update, nrows)``    :func:`uncompress`
``update!(opt, tables, grads,    :func:`update_`
indexers; ...)`` (``:283-290``)
===============================  =====================================================

All compute goes through libdlrm_b200.so; torch supplies device buffers and streams only.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib, _prof


def _stream_ptr(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


@dataclass(frozen=True, eq=False)
class PackedIndices:
    """Indices of a batch whose tables have different pooling factors (multi-hot with mixed hotness):
    table k's [B][P_k] block starts at element B * (P_0 + .. + P_{k-1}) of the flat int32 / int64
    tensor ``flat`` (Julia: ``reduce(vcat, vec.(sparse))``).  ``pack[k]`` is table k's [B][P_k] view."""
    flat: torch.Tensor
    P: Tuple[int, ...]
    B: int

    def __len__(self) -> int:
        return len(self.P)

    def __getitem__(self, k: int) -> torch.Tensor:
        o = self.B * sum(self.P[:k])
        return self.flat[o:o + self.B * self.P[k]].view(self.B, self.P[k])

    def P_array(self):
        return (C.c_int32 * len(self.P))(*self.P)

    def element_size(self) -> int:
        return self.flat.element_size()

    def data_ptr(self) -> int:
        return self.flat.data_ptr()

    @property
    def is_cuda(self) -> bool:
        return self.flat.is_cuda

    @property
    def device(self) -> torch.device:
        return self.flat.device

    def to(self, device, non_blocking: bool = False) -> "PackedIndices":
        return PackedIndices(self.flat.to(device, non_blocking=non_blocking).contiguous(), self.P, self.B)


_POOLING = {"sum": 0, "mean": 1}


@dataclass(frozen=True, eq=False)
class JaggedIndices:
    """Variable-length bags (the input of ``torch.nn.EmbeddingBag(input, offsets)`` and of the PyTorch DLRM's
    ``(lS_o, lS_i)``), in TorchRec's key-major jagged layout: ``values`` holds every table's indices, table-major;
    ``offsets`` [ntab * B + 1] (same dtype, 0-based, non-decreasing, offsets[0] = 0) makes bag b of table k
    ``values[offsets[k*B + b] : offsets[k*B + b + 1]]``; the host tuple ``L`` holds each table's lookup count.
    ``pooling`` is ``"sum"`` or ``"mean"`` (w = fl(1 / n) times the fp32 sum; an empty bag pools to zero).
    ``weights`` (optional, float32, one per entry of ``values``, same device) are per-sample weights, the
    ``per_sample_weights`` of ``EmbeddingBag`` in mode ``"sum"``: a bag pools sum_j fl(w_j * row_j); they go with
    sum pooling only.  ``jag[k]`` is table k's ``(values_k, offsets_k)`` with offsets_k rebased to 0, and
    ``(values_k, offsets_k, weights_k)`` for a weighted batch."""
    values: torch.Tensor
    offsets: torch.Tensor
    L: Tuple[int, ...]
    B: int
    pooling: str = "sum"
    weights: Optional[torch.Tensor] = None

    def __post_init__(self):
        if self.pooling not in _POOLING:
            raise ValueError(f"pooling must be 'sum' or 'mean', got {self.pooling!r}")
        if self.weights is not None:
            w = self.weights
            if self.pooling != "sum":
                raise ValueError(f"per-sample weights go with pooling='sum' only, got pooling={self.pooling!r}")
            if w.dtype != torch.float32:
                raise ValueError(f"weights must be float32, got {w.dtype}")
            if w.dim() != 1 or w.numel() != self.values.numel():
                raise ValueError(f"weights must hold one float per value: {self.values.numel()} values, "
                                 f"weights of shape {tuple(w.shape)}")
            if w.device != self.values.device:
                raise ValueError(f"weights on {w.device}, values on {self.values.device}")
        if self.values.dtype not in (torch.int32, torch.int64) or self.offsets.dtype != self.values.dtype:
            raise ValueError(f"values and offsets must share one dtype, int32 or int64 (got {self.values.dtype} and "
                             f"{self.offsets.dtype})")
        if self.B <= 0 or self.offsets.dim() != 1 or self.offsets.numel() != len(self.L) * self.B + 1:
            raise ValueError(f"offsets must hold ntab * B + 1 = {len(self.L) * self.B + 1} entries "
                             f"(got {tuple(self.offsets.shape)})")
        if any(n < 0 for n in self.L):
            raise ValueError(f"lookup counts must be >= 0, got L = {self.L}")
        if sum(self.L) != self.values.numel():
            raise ValueError(f"the lookup counts sum to {sum(self.L)}, values holds {self.values.numel()}")

    @classmethod
    def from_lengths(cls, values, lengths, pooling: str = "sum", weights=None) -> "JaggedIndices":
        """``lengths[ntab][B]``: the size of every bag; ``values`` the bags' indices, table-major; ``weights`` their
        per-sample weights in the same order (a float32 tensor, or any array, converted to float32)."""
        v = values if isinstance(values, torch.Tensor) else torch.as_tensor(np.asarray(values))
        v = _index_dtype(v.reshape(-1))
        n = np.asarray(lengths.cpu() if isinstance(lengths, torch.Tensor) else lengths, dtype=np.int64)
        if n.ndim != 2:
            raise ValueError(f"lengths must be [ntab][B], got shape {n.shape}")
        if (n < 0).any():
            raise ValueError("bag lengths must be >= 0")
        if int(n.sum()) != v.numel():
            raise ValueError(f"the bag lengths sum to {int(n.sum())}, values holds {v.numel()}")
        off = np.zeros(n.size + 1, dtype=np.int64)
        np.cumsum(n.reshape(-1), out=off[1:])
        offsets = torch.from_numpy(off).to(device=v.device, dtype=v.dtype)
        if weights is not None:
            if not isinstance(weights, torch.Tensor):
                weights = torch.from_numpy(np.asarray(weights, dtype=np.float32))
            weights = weights.reshape(-1).to(v.device).contiguous()
        return cls(v.contiguous(), offsets, tuple(int(x) for x in n.sum(axis=1)), int(n.shape[1]), pooling, weights)

    @classmethod
    def from_bags(cls, bags, pooling: str = "sum", dtype: torch.dtype = torch.int64, weights=None) -> "JaggedIndices":
        """``bags[k][b]``: the indices of bag b of table k (any sequence, possibly empty); ``weights[k][b]`` their
        per-sample weights, bag for bag."""
        Bs = {len(t) for t in bags}
        if len(Bs) != 1:
            raise ValueError(f"every table must have the same number of bags, got {[len(t) for t in bags]}")
        lengths = [[len(bag) for bag in t] for t in bags]
        flat = [int(i) for t in bags for bag in t for i in bag]
        if weights is not None:
            if [[len(w) for w in t] for t in weights] != lengths:
                raise ValueError("weights must hold one weight per index, bag for bag")
            weights = np.array([float(x) for t in weights for w in t for x in w], dtype=np.float32)
        return cls.from_lengths(torch.tensor(flat, dtype=dtype), lengths, pooling, weights)

    @classmethod
    def from_dense(cls, idx, pooling: str = "sum", weights=None) -> "JaggedIndices":
        """A fixed-width batch ([ntab][B][P] tensor or :class:`PackedIndices`) as bags of constant length;
        ``weights`` in the same shape (the flat layout of :class:`PackedIndices`)."""
        if isinstance(idx, PackedIndices):
            return cls.from_lengths(idx.flat, [[p] * idx.B for p in idx.P], pooling, weights)
        t = _index_dtype(idx if isinstance(idx, torch.Tensor) else torch.as_tensor(np.asarray(idx)))
        if t.dim() == 2:
            t = t.unsqueeze(-1)
        ntab, B, P = t.shape
        return cls.from_lengths(t.reshape(-1), [[P] * B] * ntab, pooling, weights)

    def __len__(self) -> int:
        return len(self.L)

    def __getitem__(self, k: int) -> Tuple[torch.Tensor, ...]:
        o = sum(self.L[:k])
        vo = (self.values[o:o + self.L[k]], self.offsets[k * self.B:(k + 1) * self.B + 1] - o)
        return vo if self.weights is None else vo + (self.weights[o:o + self.L[k]],)

    def L_array(self):
        return (C.c_int64 * len(self.L))(*self.L)

    def element_size(self) -> int:
        return self.values.element_size()

    @property
    def pooling_code(self) -> int:
        return _POOLING[self.pooling]

    @property
    def is_cuda(self) -> bool:
        return self.values.is_cuda

    @property
    def device(self) -> torch.device:
        return self.values.device

    def to(self, device, non_blocking: bool = False) -> "JaggedIndices":
        w = None if self.weights is None else self.weights.to(device, non_blocking=non_blocking).contiguous()
        return JaggedIndices(self.values.to(device, non_blocking=non_blocking).contiguous(),
                             self.offsets.to(device, non_blocking=non_blocking).contiguous(), self.L, self.B, self.pooling,
                             w)


def _index_dtype(t: torch.Tensor) -> torch.Tensor:
    if t.dtype in (torch.uint8, torch.int8, torch.int16):
        t = t.to(torch.int32)
    if t.dtype not in (torch.int32, torch.int64):
        if hasattr(torch, "uint32") and t.dtype == torch.uint32:
            t = t.view(torch.int32)
        else:
            raise TypeError(f"index dtype {t.dtype} not supported (int32/uint32/int64)")
    return t


def _pack_mixed(parts: List[torch.Tensor], ntab: int, device: torch.device) -> PackedIndices:
    """Per-table [B][P_k] arrays of different widths -> PackedIndices (int64 if any table is int64)."""
    if len(parts) != ntab:
        raise ValueError(f"indices must hold one array per table: {ntab} tables, got {len(parts)}")
    Bs = {p.shape[0] for p in parts}
    if len(Bs) != 1:
        raise ValueError(f"every table's indices must cover the same batch, got B = {[p.shape[0] for p in parts]}")
    parts = [_index_dtype(p) for p in parts]
    dtype = torch.int64 if any(p.dtype == torch.int64 for p in parts) else torch.int32
    flat = torch.cat([p.reshape(-1).to(dtype) for p in parts])
    return PackedIndices(flat.to(device, non_blocking=True).contiguous(), tuple(int(p.shape[1]) for p in parts),
                         int(parts[0].shape[0]))


def _as_index_tensor(sparse, ntab: int, device: torch.device):
    """Normalise the index containers DLRM.jl accepts (vector of vectors, vector of P x B
    matrices given here as [B][P], or one [ntab][B] / [ntab][B][P] array) to a contiguous
    table-major device tensor [ntab][B][P] of int32 or int64.  A vector whose tables have different
    widths (the reference's load_inputs with per-table P = length / B) becomes :class:`PackedIndices`."""
    if isinstance(sparse, (PackedIndices, JaggedIndices)):
        if len(sparse) != ntab:
            raise ValueError(f"indices must hold one array per table: {ntab} tables, got {len(sparse)}")
        return sparse.to(device, non_blocking=True)
    if isinstance(sparse, torch.Tensor):
        t = sparse
    elif isinstance(sparse, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(sparse))
    else:
        parts = [torch.as_tensor(np.asarray(s) if not isinstance(s, torch.Tensor) else s) for s in sparse]
        parts = [p.reshape(p.shape[0], -1) for p in parts]
        if len({p.shape[1] for p in parts}) > 1:
            return _pack_mixed(parts, ntab, device)
        t = torch.stack(parts, dim=0)
    t = _index_dtype(t)
    if t.dim() == 2:
        t = t.unsqueeze(-1)
    if t.dim() != 3 or t.shape[0] != ntab:
        raise ValueError(f"indices must be [ntab={ntab}][B] or [ntab][B][P], got {tuple(t.shape)}")
    return t.to(device, non_blocking=True).contiguous()


def _batch(idx) -> int:
    return idx.B if isinstance(idx, (PackedIndices, JaggedIndices)) else idx.shape[1]


class _DevicePtrView:
    """Zero-copy torch view of library-owned device memory via __cuda_array_interface__."""

    def __init__(self, ptr: int, shape, owner, typestr: str = "<f4"):
        self.__cuda_array_interface__ = {
            "shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2, "strides": None,
        }
        self._owner = owner


class EmbeddingTables:
    """All embedding tables of one model, resident in HBM ([rows_k][D] f32 each).

    ``max_lookups`` is the largest B*P per table any later call will use; workspaces are
    sized from it once, so no call allocates.
    """

    def __init__(self, rows: Sequence[int], D: int, max_lookups: int, device: Union[int, torch.device] = 0,
                 dtype: torch.dtype = torch.float32):
        """``dtype``: storage type of the rows, ``torch.float32`` (default) or ``torch.bfloat16`` (the
        reference's ``embedding_eltype`` option, src/model/model.jl:187); arithmetic is fp32 either way."""
        if dtype not in (torch.float32, torch.bfloat16):
            raise _lib.DLRMB200Error(_lib.EINVAL, f"table dtype {dtype} not supported (float32 / bfloat16)")
        self.dtype = dtype
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.type != "cuda":
            raise _lib.DLRMB200Error(_lib.EINVAL, "EmbeddingTables live in HBM: a CUDA device is required")
        self.device = dev
        self.rows = [int(r) for r in rows]
        self.D = int(D)
        self.ntab = len(self.rows)
        self.max_lookups = int(max_lookups)
        self._lib = _lib.load()
        arr = (C.c_int64 * self.ntab)(*self.rows)
        handle = C.c_void_p()
        _lib.check(self._lib.dlrmb_tables_create_ex(dev.index or 0, self.ntab, arr, self.D, self.max_lookups,
                                                   4 if dtype == torch.float32 else 2, C.byref(handle)))
        self._h = handle
        self._side_stream: Optional[torch.cuda.Stream] = None
        self._sorted_event: Optional[torch.cuda.Event] = None

    # -- construction helpers -----------------------------------------------------------------
    @classmethod
    def from_arrays(cls, arrays: Sequence[np.ndarray], max_lookups: int, device=0,
                    dtype: torch.dtype = torch.float32) -> "EmbeddingTables":
        """``SimpleEmbedding{Static{D}}(data)`` for each array ([rows][D], i.e. Julia D x rows)."""
        D = int(arrays[0].shape[1])
        t = cls([a.shape[0] for a in arrays], D, max_lookups, device, dtype)
        for k, a in enumerate(arrays):
            t.upload(k, a)
        return t

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.dlrmb_tables_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self) -> int:
        return self.ntab

    # -- storage ------------------------------------------------------------------------------
    def upload(self, k: int, array: np.ndarray) -> None:
        a = np.ascontiguousarray(array, dtype=np.float32)
        if a.shape != (self.rows[k], self.D):
            raise ValueError(f"table {k}: expected {(self.rows[k], self.D)}, got {a.shape}")
        _lib.check(self._lib.dlrmb_tables_upload(self._h, k, a.ctypes.data_as(C.c_void_p)))

    def download(self, k: int) -> np.ndarray:
        """``Array(table)`` / ``table.data`` read-back (src/validation.jl:138)."""
        out = np.empty((self.rows[k], self.D), dtype=np.float32)
        _lib.check(self._lib.dlrmb_tables_download(self._h, k, out.ctypes.data_as(C.c_void_p)))
        return out

    def table(self, k: int) -> torch.Tensor:
        """Zero-copy [rows_k][D] device view of table k (float32 or bfloat16, as stored)."""
        p = C.c_void_p()
        _lib.check(self._lib.dlrmb_tables_device_ptr(self._h, k, C.byref(p)))
        if self.dtype == torch.bfloat16:
            raw = torch.as_tensor(_DevicePtrView(p.value, (self.rows[k], self.D), self, "<i2"), device=self.device)
            return raw.view(torch.bfloat16)
        return torch.as_tensor(_DevicePtrView(p.value, (self.rows[k], self.D), self), device=self.device)

    def init_uniform(self, seed: int = 51234) -> None:
        """ScaledUniform init (src/model/model.jl:61-65); seed default from model.jl:193."""
        _lib.check(self._lib.dlrmb_tables_init_uniform(self._h, seed, _stream_ptr(self.device)))

    # -- kernels ------------------------------------------------------------------------------
    def lookup(self, idx: torch.Tensor, out: torch.Tensor, slot0: int, idx_base: int = 0, sort: bool = False) -> None:
        """Gather + sum-pool into ``out``.  ``sort=True`` is the training-step form: the same launch also
        sorts / dedups the indices for the sparse update of this batch (dlrmb_embedding_fwd_sort), so
        :meth:`update_sorted` can follow the backward pass without a sort launch."""
        slots = out.shape[1]
        if isinstance(idx, JaggedIndices):   # variable-length bags
            assert out.is_contiguous() and out.dtype == torch.float32 and out.shape == (idx.B, slots, self.D)
            with _prof.range("lookup"):
                if idx.weights is not None:
                    fn = (self._lib.dlrmb_embedding_fwd_sort_jagged_weighted if sort
                          else self._lib.dlrmb_embedding_fwd_jagged_weighted)
                    _lib.check(fn(self._h, idx.values.data_ptr(), idx.offsets.data_ptr(), idx.weights.data_ptr(),
                                  idx.element_size(), idx_base, idx.B, idx.L_array(), out.data_ptr(), slots, slot0,
                                  _stream_ptr(self.device)))
                else:
                    fn = self._lib.dlrmb_embedding_fwd_sort_jagged if sort else self._lib.dlrmb_embedding_fwd_jagged
                    _lib.check(fn(self._h, idx.values.data_ptr(), idx.offsets.data_ptr(), idx.element_size(), idx_base,
                                  idx.B, idx.L_array(), idx.pooling_code, out.data_ptr(), slots, slot0,
                                  _stream_ptr(self.device)))
            if sort:
                self._pending_side = False
            return
        if isinstance(idx, PackedIndices):   # per-table pooling factors
            B, P = idx.B, idx.P_array()
            fn = self._lib.dlrmb_embedding_fwd_sort_mp if sort else self._lib.dlrmb_embedding_fwd_mp
        else:
            ntab, B, P = idx.shape
            fn = self._lib.dlrmb_embedding_fwd_sort if sort else self._lib.dlrmb_embedding_fwd
        assert out.is_contiguous() and out.dtype == torch.float32 and out.shape == (B, slots, self.D)
        with _prof.range("lookup"):
            _lib.check(fn(self._h, idx.data_ptr(), idx.element_size(), idx_base, B, P, out.data_ptr(), slots, slot0,
                          _stream_ptr(self.device)))
        if sort:
            self._pending_side = False

    def set_slot_map(self, slots: Sequence[int]) -> None:
        """Sharded use: interaction slot (1 + global table id) of each local table."""
        arr = (C.c_int32 * self.ntab)(*[int(v) for v in slots])
        _lib.check(self._lib.dlrmb_tables_set_slot_map(self._h, arr))

    def set_dest_map(self, slots: Sequence[int], col0: Sequence[int], D_dest: int) -> None:
        """Column-wise sharded use: local table k's pooled rows land at columns [col0[k], col0[k] + D) of slot
        slots[k] in destination rows of D_dest floats per slot (dlrmb_tables_set_dest_map)."""
        arr = (C.c_int32 * self.ntab)(*[int(v) for v in slots])
        cols = (C.c_int32 * self.ntab)(*[int(v) for v in col0])
        _lib.check(self._lib.dlrmb_tables_set_dest_map(self._h, arr, cols, int(D_dest)))

    FUSED_SORT_MAX = 4096    # kFusedSortMax of csrc/common.cuh: largest B*P whose sort rides in the lookup launch

    def lookup_p2p(self, idx: torch.Tensor, peer_ptrs: Sequence[int], B_local: int, slots: int, idx_base: int = 0,
                   sort: bool = False) -> None:
        """Pool this rank's tables for the global batch and store every pooled row directly into
        the owning rank's interaction buffer (NVLink peer stores): lookup + forward exchange fused.
        ``sort=True`` also sorts / dedups the indices for this batch's sparse update in the same launch
        (dlrmb_embedding_fwd_p2p_sort).  ``idx`` may be :class:`PackedIndices` at B_global (per-table
        pooling factors, dlrmb_embedding_fwd_p2p_mp / _sort_mp) or :class:`JaggedIndices` at B_global (the owner batch
        of variable-length bags, sum, mean or weighted; dlrmb_embedding_fwd_p2p_jagged / _sort_jagged)."""
        world = len(peer_ptrs)
        arr = (C.c_void_p * world)(*[int(p) for p in peer_ptrs])
        if isinstance(idx, JaggedIndices):
            fn = self._lib.dlrmb_embedding_fwd_p2p_sort_jagged if sort else self._lib.dlrmb_embedding_fwd_p2p_jagged
            w = None if idx.weights is None else idx.weights.data_ptr() or None
            with _prof.range("lookup"):
                _lib.check(fn(self._h, idx.values.data_ptr(), idx.offsets.data_ptr(), w, idx.element_size(), idx_base,
                              idx.B, idx.L_array(), idx.pooling_code, arr, world, B_local, slots, _stream_ptr(self.device)))
            if sort:
                self._pending_side = False
            return
        if isinstance(idx, PackedIndices):
            Bg, P = idx.B, idx.P_array()
            fn = self._lib.dlrmb_embedding_fwd_p2p_sort_mp if sort else self._lib.dlrmb_embedding_fwd_p2p_mp
        else:
            ntab, Bg, P = idx.shape
            fn = self._lib.dlrmb_embedding_fwd_p2p_sort if sort else self._lib.dlrmb_embedding_fwd_p2p
        with _prof.range("lookup"):
            _lib.check(fn(self._h, idx.data_ptr(), idx.element_size(), idx_base, Bg, P, arr, world, B_local, slots,
                          _stream_ptr(self.device)))
        if sort:
            self._pending_side = False

    def sort(self, idx: torch.Tensor, idx_base: int = 0, side_stream: bool = False) -> None:
        """Index sort/dedup for the next update.  With ``side_stream`` it is issued on a second
        stream (it depends on the indices only) so it overlaps the forward/backward pass."""
        if isinstance(idx, JaggedIndices):
            L, code, offs = idx.L_array(), idx.pooling_code, idx.offsets.data_ptr()
            B, P, rec = idx.B, None, (idx.values, idx.offsets)
            if idx.weights is not None:
                w, rec = idx.weights.data_ptr(), rec + (idx.weights,)
                fn = lambda h, v, ib, base, B, _P, st: self._lib.dlrmb_embedding_sort_jagged_weighted(
                    h, v, offs, w, ib, base, B, L, st)
            else:
                fn = lambda h, v, ib, base, B, _P, st: self._lib.dlrmb_embedding_sort_jagged(
                    h, v, offs, ib, base, B, L, code, st)
            idx = idx.values
        elif isinstance(idx, PackedIndices):
            B, P, fn, rec = idx.B, idx.P_array(), self._lib.dlrmb_embedding_sort_mp, idx.flat
        else:
            (ntab, B, P), fn, rec = idx.shape, self._lib.dlrmb_embedding_sort, idx
        if side_stream:
            if self._side_stream is None:
                self._side_stream = torch.cuda.Stream(self.device)
                self._sorted_event = torch.cuda.Event()
            self._side_stream.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(self._side_stream):
                with _prof.range("sort"):
                    _lib.check(fn(self._h, idx.data_ptr(), idx.element_size(), idx_base, B, P,
                                  self._side_stream.cuda_stream))
                if not torch.cuda.is_current_stream_capturing():
                    for r in rec if isinstance(rec, tuple) else (rec,):
                        r.record_stream(self._side_stream)
                self._sorted_event.record(self._side_stream)
            self._pending_side = True
        else:
            with _prof.range("sort"):
                _lib.check(fn(self._h, idx.data_ptr(), idx.element_size(), idx_base, B, P, _stream_ptr(self.device)))
            self._pending_side = False

    def update_sorted(self, dT: torch.Tensor, slot0: int, lr: float) -> None:
        if getattr(self, "_pending_side", False):
            torch.cuda.current_stream(self.device).wait_event(self._sorted_event)
            self._pending_side = False
        B, slots, D = dT.shape
        assert dT.is_contiguous() and dT.dtype == torch.float32 and D == self.D
        with _prof.range("update"):
            _lib.check(self._lib.dlrmb_embedding_update_sorted(
                self._h, dT.data_ptr(), slots, slot0, float(lr), _stream_ptr(self.device)))

    def weight_grad(self, idx: JaggedIndices, dT: torch.Tensor, slot0: int, idx_base: int = 0) -> torch.Tensor:
        """Gradient of the pooled rows with respect to per-sample weights (``per_sample_weights.grad``): a float32
        tensor of sum(L) values, dw[j] = dT[b(j), slot0 + k] . table_k[values[j]], in the order of ``idx.values``
        (zero-length bags contribute nothing).  It reads the rows as they are: call it before
        :meth:`update_sorted` of the same batch.  ``idx`` need not carry weights."""
        if not isinstance(idx, JaggedIndices):
            raise TypeError(f"weight_grad takes JaggedIndices, got {type(idx).__name__}")
        B, slots, D = dT.shape
        assert dT.is_contiguous() and dT.dtype == torch.float32 and D == self.D and B == idx.B
        dw = torch.empty(idx.values.numel(), dtype=torch.float32, device=self.device)
        with _prof.range("weight_grad"):
            _lib.check(self._lib.dlrmb_embedding_weight_grad_jagged(
                self._h, idx.values.data_ptr(), idx.offsets.data_ptr(), idx.element_size(), idx_base, idx.B,
                idx.L_array(), dT.data_ptr(), slots, slot0, dw.data_ptr(), _stream_ptr(self.device)))
        return dw

    def bwd_sgd(self, idx: torch.Tensor, dT: torch.Tensor, slot0: int, lr: float, idx_base: int = 0) -> None:
        self.sort(idx, idx_base)
        self.update_sorted(dT, slot0, lr)

    def sort_dedup_export(self, k: int, L: int):
        """(uniq, seg_offsets, perm) of the last sort for table k, as numpy arrays.  ``L`` = B * P_k, the
        table's lookups in that sort."""
        uniq = np.empty(L, dtype=np.int64)
        seg = np.empty(L + 1, dtype=np.int32)
        perm = np.empty(L, dtype=np.int32)
        n = C.c_int32()
        _lib.check(self._lib.dlrmb_sort_dedup_export(
            self._h, k, uniq.ctypes.data_as(C.c_void_p), seg.ctypes.data_as(C.c_void_p),
            perm.ctypes.data_as(C.c_void_p), C.byref(n)))
        return uniq[:n.value].copy(), seg[:n.value + 1].copy(), perm

    def check_indices(self, idx: torch.Tensor, idx_base: int = 0) -> None:
        on_host = 0 if idx.is_cuda else 1
        if isinstance(idx, JaggedIndices):
            _lib.check(self._lib.dlrmb_check_indices_jagged(
                self._h, idx.values.data_ptr(), idx.offsets.data_ptr(), idx.element_size(), idx_base, idx.B, idx.L_array(),
                on_host))
            return
        if isinstance(idx, PackedIndices):
            _lib.check(self._lib.dlrmb_check_indices_mp(
                self._h, idx.data_ptr(), idx.element_size(), idx_base, idx.B, idx.P_array(), on_host))
            return
        ntab, B, P = idx.shape
        _lib.check(self._lib.dlrmb_check_indices(
            self._h, idx.data_ptr(), idx.element_size(), idx_base, B, P, on_host))


# ---- strategies ---------------------------------------------------------------------------------
@dataclass(frozen=True)
class PreallocationStrategy:
    """``PreallocationStrategy(r)``: one (r + ntab*D) x B result with the first r rows reserved
    for the bottom-MLP output (test/integration.jl:10-13).  r must be a multiple of D."""
    prepend_rows: int = 0


@dataclass(frozen=True)
class DefaultStrategy:
    """``DefaultStrategy()``: one D x B matrix per table (test/model/model.jl:265-271)."""


def maplookup(strategy, tables: EmbeddingTables, sparse, idx_base: int = 0, requires_grad: bool = False,
              check: bool = False):
    """``maplookup(strategy, tables, sparse)`` (src/model/model.jl:161).

    Preallocation: returns T [B][slot0 + ntab][D] (slots < slot0 zero).  Default: returns a list
    of [B][D] views, one per table.  The normalised index tensor is attached as ``.indices`` on
    the returned buffer for the pullback (:func:`sparse_updates`).  With ``requires_grad`` (a training
    step) the launch also prepares the sort / dedup of the coming sparse update (``T.presorted``).
    ``check`` range-checks the indices first (the kernels, like the reference's ``@inbounds`` loops,
    do not) and raises ``DLRMB_EOOB`` naming the first offender.
    """
    idx = _as_index_tensor(sparse, tables.ntab, tables.device)
    if isinstance(strategy, PreallocationStrategy):
        if strategy.prepend_rows % tables.D != 0:
            raise ValueError("PreallocationStrategy rows must be a multiple of the embedding dim")
        slot0 = strategy.prepend_rows // tables.D
    elif isinstance(strategy, DefaultStrategy):
        slot0 = 0
    else:
        raise TypeError(f"unknown lookup strategy {strategy!r}")
    if check:
        tables.check_indices(idx, idx_base)
    B = _batch(idx)
    alloc = torch.zeros if slot0 > 0 else torch.empty
    T = alloc((B, slot0 + tables.ntab, tables.D), dtype=torch.float32, device=tables.device)
    tables.lookup(idx, T, slot0, idx_base, sort=requires_grad)
    T.indices = idx
    T.idx_base = idx_base
    T.slot0 = slot0
    T.presorted = bool(requires_grad)
    if requires_grad:
        T.requires_grad_(True)
    if isinstance(strategy, DefaultStrategy):
        views = [T[:, k, :] for k in range(tables.ntab)]
        for v in views:
            v.parent = T
        return views
    return T


# ---- sparse gradient -----------------------------------------------------------------------------
@dataclass
class SparseEmbeddingUpdate:
    """``SparseEmbeddingUpdate(delta, indices)``: delta [B][D] (a view of slot ``slot`` of the
    pooled-embedding gradient ``parent`` [B][slots][D]) and that table's [B][P] indices."""
    delta: torch.Tensor
    indices: torch.Tensor
    parent: Optional[torch.Tensor] = None
    slot: int = -1
    idx_base: int = 0
    pooling: str = "sum"        # jagged bags: ``indices`` is the table's (values_k, offsets_k[, weights_k])


def sparse_updates(dT: torch.Tensor, indices: torch.Tensor, slot0: int, idx_base: int = 0) -> List[SparseEmbeddingUpdate]:
    """The lookup pullback: slice dT per table, no arithmetic (test/model/embedding_update.jl:36-40).
    ``indices`` is the [ntab][B][P] tensor, :class:`PackedIndices` or :class:`JaggedIndices`."""
    pooling = indices.pooling if isinstance(indices, JaggedIndices) else "sum"
    return [SparseEmbeddingUpdate(dT[:, slot0 + k, :], indices[k], dT, slot0 + k, idx_base, pooling)
            for k in range(len(indices))]


def uncompress(update: SparseEmbeddingUpdate, nrows: int) -> torch.Tensor:
    """``EmbeddingTables.uncompress(update, nrows)`` (test/train/backprop.jl:156): the dense
    [nrows][D] gradient.  Debug/inspection helper (torch index_add_), not on the hot path."""
    B, D = update.delta.shape
    if isinstance(update.indices, tuple):   # jagged bags: every lookup of bag b gets delta[b] (times 1/n for mean,
        values, offsets = update.indices[:2]  # times its own weight for per-sample weights)
        n = (offsets[1:] - offsets[:-1]).to(torch.int64).to(update.delta.device)
        delta = update.delta
        if update.pooling == "mean":
            w = torch.where(n > 0, 1.0 / n.clamp(min=1).to(torch.float32), torch.zeros((), dtype=torch.float32,
                                                                                    device=delta.device))
            delta = delta * w[:, None]
        dense = torch.zeros((nrows, D), dtype=torch.float32, device=update.delta.device)
        rows = values.to(torch.int64).to(update.delta.device) - update.idx_base
        contrib = delta.repeat_interleave(n, dim=0)
        if len(update.indices) == 3:
            contrib = contrib * update.indices[2].to(update.delta.device)[:, None]
        dense.index_add_(0, rows, contrib)
        return dense
    idx = (update.indices.reshape(B, -1).to(torch.int64) - update.idx_base)
    P = idx.shape[1]
    dense = torch.zeros((nrows, D), dtype=torch.float32, device=update.delta.device)
    dense.index_add_(0, idx.reshape(-1), update.delta.repeat_interleave(P, dim=0))
    return dense


@dataclass(frozen=True)
class Descent:
    """``Flux.Descent(eta)``: ``x .-= eta .* grad``."""
    eta: float = 0.1


def update_(opt: Descent, tables: EmbeddingTables, grads: Sequence[SparseEmbeddingUpdate],
            presorted: bool = False) -> None:
    """``EmbeddingTables.update!(opt, tables, grads, indexers; num_splits, nthreads)``
    (src/train/train.jl:283-290).  In place, one fused launch for every table.
    ``presorted`` = :meth:`EmbeddingTables.sort` already ran for these indices."""
    if len(grads) != tables.ntab:
        raise ValueError(f"expected {tables.ntab} sparse updates, got {len(grads)}")
    parent = grads[0].parent
    slot0 = grads[0].slot
    same = parent is not None and all(g.parent is parent and g.slot == slot0 + k for k, g in enumerate(grads))
    if same:
        dT = parent
    else:  # updates built one by one (DefaultStrategy): pack into one [B][ntab][D] buffer
        dT = torch.stack([g.delta for g in grads], dim=1).contiguous()
        slot0 = 0
    if not presorted and isinstance(grads[0].indices, tuple):   # jagged bags
        lengths = [(g.indices[1][1:] - g.indices[1][:-1]).cpu().numpy() for g in grads]
        w = torch.cat([g.indices[2] for g in grads]) if len(grads[0].indices) == 3 else None
        idx = JaggedIndices.from_lengths(torch.cat([g.indices[0] for g in grads]), lengths, grads[0].pooling, w)
        tables.sort(idx.to(tables.device), grads[0].idx_base)
    elif not presorted:
        idx = _as_index_tensor([g.indices.reshape(g.delta.shape[0], -1) for g in grads], tables.ntab, tables.device)
        tables.sort(idx, grads[0].idx_base)
    tables.update_sorted(dT, slot0, opt.eta)
