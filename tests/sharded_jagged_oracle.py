"""NumPy restatement of the owner layout of table-sharded jagged batches (include/dlrm_b200.h,
dlrmb_indices_scatter_p2p_jagged; dlrm_jl_b200/sharded.py, exchange_indices_jagged), the reference the sharded jagged
tests compare the exchanges against.

Rank h holds a jagged batch of B_local bags per table: ``values`` table-major, ``offsets`` [ntab * B_local + 1],
optional ``weights`` beside the values.  Owner o of tables k_0 < k_1 < .. < k_{t-1} receives the jagged batch of its
tables over the rank-major global batch (B_global = world * B_local):
  * L_own[j] = sum over h of rank h's lookups of table k_j;
  * table j's block of values starts at L_own[0] + .. + L_own[j-1]; inside it rank h's entries of k_j follow those of
    the ranks before h, each rank's in its own order;
  * offsets [t * B_global + 1]: bag j * B_global + h * B_local + b is rank h's bag b of table k_j;
  * weights sit in the positions of their values.
"""
import numpy as np


def owner_layout(batches, tables, B_local: int):
    """``batches[h]`` = (values, offsets, weights or None) of rank h, every table; ``tables`` the owner's global table
    ids, ascending.  Returns (values, offsets, L_own, weights or None) of the owner batch."""
    vals, lens, wts, L_own = [], [], [], []
    weighted = batches[0][2] is not None
    for k in tables:
        n = 0
        for v, o, w in batches:
            o = np.asarray(o, dtype=np.int64)
            a, b = int(o[k * B_local]), int(o[(k + 1) * B_local])
            vals.append(np.asarray(v)[a:b])
            lens.append(np.diff(o[k * B_local:(k + 1) * B_local + 1]))
            if weighted:
                wts.append(np.asarray(w, dtype=np.float32)[a:b])
            n += b - a
        L_own.append(n)
    dtype = np.asarray(batches[0][0]).dtype
    values = np.concatenate(vals).astype(dtype) if vals else np.zeros(0, dtype)
    offsets = np.zeros(1 + sum(len(x) for x in lens), dtype=np.int64)
    if lens:
        np.cumsum(np.concatenate(lens), out=offsets[1:])
    weights = (np.concatenate(wts) if wts else np.zeros(0, np.float32)) if weighted else None
    return values, offsets.astype(dtype), L_own, weights


def random_batch(rng, rows, B_local: int, max_len, dtype=np.int64, weighted: bool = False, base: int = 0, lo: int = 0):
    """A random jagged batch: bag lengths uniform in min(lo, m) .. m for m = max_len[k] (a table with max_len 0 has no
    lookup), indices uniform in the table (plus ``base``), weights uniform in [-2, 2).  Returns (values, offsets, weights, lengths)."""
    lengths = np.stack([rng.integers(min(lo, int(m)), int(m) + 1, size=B_local) for m in max_len])
    values = np.concatenate([rng.integers(0, r, size=int(n.sum())) for r, n in zip(rows, lengths)]).astype(dtype) + base
    offsets = np.zeros(lengths.size + 1, dtype=np.int64)
    np.cumsum(lengths.reshape(-1), out=offsets[1:])
    weights = rng.uniform(-2, 2, size=len(values)).astype(np.float32) if weighted else None
    return values, offsets.astype(dtype), weights, lengths
