"""NumPy restatement of the weighted jagged-bag contract of include/dlrm_b200.h (per-sample weights, the
`_jagged_weighted` entry points and dlrmb_embedding_weight_grad_jagged), the reference the weighted tests compare the
kernels against.  The layout is the jagged one of tests/jagged_oracle.py, plus ``weights``: one f32 per entry of
``values``, in the same order.
"""
import numpy as np

F32 = np.float32


# Arithmetic, exactly as the kernels do it (sum pooling only):
#   * forward: acc = +0.0f; for j ascending over the bag, acc = fl(acc + fl(w_j * row_j)); an empty bag gives +0.0f;
#   * update: sorted entry j of table k contributes fl(dT[b(j)][slot0 + k] * w_j); the contributions of one row are
#     added in ascending position, then row -= fl(lr * sum);
#   * weight gradient, in the order of include/dlrm_b200.h: V = 4 if D % 4 == 0 else 1, C = D / V chunks of V floats,
#     G = min(32, C rounded up to a power of two); partial l adds fl(g[d] * r[d]) over the floats d of chunks
#     c = l, l + G, .. in ascending d, from +0.0f; then for s = G/2 .. 1, p_l = fl(p_l + p_(l xor s)); dw = p_0.

def lookup_jagged_weighted(tables, values, offsets, weights, B: int, slot0: int = 0) -> np.ndarray:
    """Pooled rows [B][slot0 + ntab][D] of a weighted batch; ``values`` 0-based, ``weights`` one f32 per value."""
    ntab, D = len(tables), tables[0].shape[1]
    values = np.asarray(values, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    weights = np.asarray(weights, dtype=F32)
    out = np.zeros((B, slot0 + ntab, D), dtype=F32)
    for k in range(ntab):
        o = offsets[k * B:(k + 1) * B + 1]
        n = np.diff(o)
        acc = np.zeros((B, D), dtype=F32)
        for p in range(int(n.max()) if B else 0):
            live = np.nonzero(n > p)[0]
            j = o[live] + p
            acc[live] = (acc[live] + (tables[k][values[j]] * weights[j][:, None]).astype(F32)).astype(F32)
        out[:, slot0 + k] = acc
    return out


def sparse_sgd_update_jagged_weighted(table: np.ndarray, values_k, offsets_k, weights_k, delta: np.ndarray, lr: float,
                                      bf16_rows: bool = False) -> None:
    """In place, one table: as ``jagged_oracle.sparse_sgd_update_jagged`` with entry j's contribution fl(delta[b(j)] * w_j)."""
    values_k = np.asarray(values_k, dtype=np.int64)
    o = np.asarray(offsets_k, dtype=np.int64)
    if len(values_k) == 0:
        return
    bag = np.repeat(np.arange(len(o) - 1), np.diff(o))
    contrib = (delta[bag].astype(F32) * np.asarray(weights_k, dtype=F32)[:, None]).astype(F32)
    perm = np.argsort(values_k, kind="stable")
    rows = values_k[perm]
    uniq, start, counts = np.unique(rows, return_index=True, return_counts=True)
    rank = np.arange(len(rows)) - np.repeat(start, counts)
    run = np.repeat(np.arange(len(uniq)), counts)
    acc = np.zeros((len(uniq), table.shape[1]), dtype=F32)
    for r in range(int(counts.max())):
        sel = rank == r
        acc[run[sel]] = (acc[run[sel]] + contrib[perm[sel]]).astype(F32)
    new = (table[uniq] - (F32(lr) * acc).astype(F32)).astype(F32)
    if bf16_rows:
        from oracle.oracle import to_bf16
        new = to_bf16(new)
    table[uniq] = new


def dot_in_kernel_order(g: np.ndarray, r: np.ndarray) -> np.ndarray:
    """sum_d g[.., d] * r[.., d] for rows of D floats, in the weight gradient's order (f32 bits of the kernel)."""
    g = np.asarray(g, dtype=F32)
    r = np.asarray(r, dtype=F32)
    D = g.shape[-1]
    V = 4 if D % 4 == 0 else 1
    C = D // V
    G = 1
    while G < C and G < 32:
        G *= 2
    prod = (g * r).astype(F32)
    part = np.zeros(g.shape[:-1] + (G,), dtype=F32)
    for lane in range(G):
        for c in range(lane, C, G):
            for d in range(c * V, c * V + V):
                part[..., lane] = (part[..., lane] + prod[..., d]).astype(F32)
    s = G // 2
    while s >= 1:
        part = (part + part[..., np.arange(G) ^ s]).astype(F32)
        s //= 2
    return part[..., 0]


def weight_grad_jagged(tables, values, offsets, dT: np.ndarray, B: int, slot0: int = 0) -> np.ndarray:
    """dw [len(values)]: dw[j] = dT[b(j)][slot0 + k] . table_k[values[j]] in the kernel's order; ``values`` 0-based,
    ``dT`` [B][slots][D]."""
    values = np.asarray(values, dtype=np.int64)
    offsets = np.asarray(offsets, dtype=np.int64)
    dw = np.zeros(len(values), dtype=F32)
    for k in range(len(tables)):
        o = offsets[k * B:(k + 1) * B + 1]
        j = np.arange(o[0], o[-1])
        if len(j) == 0:
            continue
        bag = np.repeat(np.arange(B), np.diff(o))
        dw[j] = dot_in_kernel_order(dT[bag, slot0 + k], tables[k][values[j]])
    return dw
