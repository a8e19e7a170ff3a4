"""NumPy restatement of the jagged (variable-length bag) contract of include/dlrm_b200.h, the reference the jagged
tests compare the kernels against.

Layout: ``values`` holds every table's indices, table-major; ``offsets`` [ntab * B + 1] (0-based, non-decreasing,
offsets[0] = 0) makes bag b of table k ``values[offsets[k*B + b] : offsets[k*B + b + 1]]``.
Arithmetic, exactly as the kernels do it:
  * sum:  out[b][slot0 + k] = sum of table_k[values[j]] over the bag, j ascending, sequential fp32 adds from +0.0f;
  * mean: w = fl(1.0f / n) for a bag of n lookups, out = fl(S * w);
  * an empty bag pools to +0.0f in both modes and contributes no gradient;
  * update (Flux.Descent): sorted entry j of table k contributes dT[b(j)][slot0 + k], times w(b(j)) in mean mode;
    the contributions of one row are added sequentially in ascending position, then row -= fl(lr * sum).
"""
import numpy as np

F32 = np.float32


def bag_weights(offsets_k: np.ndarray) -> np.ndarray:
    """w[b] = fl(1 / n_b) in fp32 (0 for an empty bag, which has no lookup to weigh)."""
    n = np.diff(np.asarray(offsets_k, dtype=np.int64))
    w = np.zeros(len(n), dtype=F32)
    w[n > 0] = F32(1.0) / n[n > 0].astype(F32)
    return w


def lookup_jagged(tables, values, offsets, B: int, pooling: str = "sum", slot0: int = 0) -> np.ndarray:
    """Pooled rows [B][slot0 + ntab][D]; slots below slot0 stay zero.  ``values`` are 0-based."""
    ntab, D = len(tables), tables[0].shape[1]
    values = np.asarray(values, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    out = np.zeros((B, slot0 + ntab, D), dtype=F32)
    for k in range(ntab):
        o = offsets[k * B:(k + 1) * B + 1]
        n = np.diff(o)
        acc = np.zeros((B, D), dtype=F32)
        for p in range(int(n.max()) if B else 0):      # lookup p of every bag that has one, in ascending p
            live = np.nonzero(n > p)[0]
            acc[live] = (acc[live] + tables[k][values[o[live] + p]]).astype(F32)
        if pooling == "mean":
            acc = (acc * bag_weights(o)[:, None]).astype(F32)
        out[:, slot0 + k] = acc
    return out


def sparse_sgd_update_jagged(table: np.ndarray, values_k, offsets_k, delta: np.ndarray, lr: float,
                             pooling: str = "sum", bf16_rows: bool = False) -> None:
    """In place: one table, ``values_k`` 0-based, ``offsets_k`` [B + 1] rebased to 0, ``delta`` [B][D].
    ``bf16_rows`` rounds the updated rows to bf16 (nearest even), as bf16 storage does."""
    values_k = np.asarray(values_k, dtype=np.int64)
    o = np.asarray(offsets_k, dtype=np.int64)
    if len(values_k) == 0:
        return
    bag = np.repeat(np.arange(len(o) - 1), np.diff(o))
    contrib = delta[bag].astype(F32)
    if pooling == "mean":
        contrib = (contrib * bag_weights(o)[bag][:, None]).astype(F32)
    perm = np.argsort(values_k, kind="stable")
    rows = values_k[perm]
    uniq, start, counts = np.unique(rows, return_index=True, return_counts=True)
    rank = np.arange(len(rows)) - np.repeat(start, counts)
    run = np.repeat(np.arange(len(uniq)), counts)
    acc = np.zeros((len(uniq), table.shape[1]), dtype=F32)
    for r in range(int(counts.max())):               # r-th duplicate of every row, ascending position
        sel = rank == r
        acc[run[sel]] = (acc[run[sel]] + contrib[perm[sel]]).astype(F32)
    new = (table[uniq] - (F32(lr) * acc).astype(F32)).astype(F32)
    if bf16_rows:
        from oracle.oracle import to_bf16
        new = to_bf16(new)
    table[uniq] = new
