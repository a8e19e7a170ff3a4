"""The run-layout constructor and the exact-data premise of tests/test_gpu_update_exact.py, without a GPU."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.sparse_update_layouts import (chained_row_ids, edge_ends, exact_grads, exact_tables, expected_exact,
                                         lengths_from_ends, mixed_ends, runs_to_indices, update_geom)


@pytest.mark.parametrize("case", ["edges", "mixed", "single_row", "tiny"])
def test_constructed_indices_sort_to_the_intended_runs(case):
    """O.sort_dedup of the shuffled indices gives exactly the intended row ids and seg_offsets."""
    rng = np.random.default_rng(len(case))
    B = 64
    if case == "edges":
        L = B * 48
        ends = edge_ends(L, 12, 3) + edge_ends(L, 4, 0)[::7]
    elif case == "mixed":
        L = B * 200
        ends = mixed_ends(L, 64, 16, 16, rng)
    elif case == "single_row":
        L, ends = B * 5, []
    else:
        B = L = 5
        ends = [1, 2, 4]
    n = lengths_from_ends(ends, L)
    assert n.sum() == L and np.array_equal(np.cumsum(n)[:-1], np.unique([e for e in ends if 0 < e < L]))
    (ids,) = chained_row_ids([len(n)], rng)
    idx = runs_to_indices(ids, n, B, rng)
    assert idx.shape == (B, L // B)
    uniq, seg, perm = O.sort_dedup(idx)
    assert np.array_equal(uniq, ids)
    assert np.array_equal(seg, np.concatenate([[0], np.cumsum(n)]))
    assert np.array_equal(idx.reshape(-1)[perm], np.repeat(ids, n))


def test_chained_row_ids_share_the_row_at_table_boundaries():
    ids = chained_row_ids([3, 1, 5, 2], np.random.default_rng(0))
    for a, b in zip(ids[:-1], ids[1:]):
        assert a[-1] == b[0]
    assert all(np.all(np.diff(i) > 0) for i in ids)


def test_mixed_layout_has_the_boundary_runs_it_promises():
    chunk, lpr, nsub, L = 64, 16, 16, 60000
    n = lengths_from_ends(mixed_ends(L, chunk, lpr, nsub, np.random.default_rng(3)), L)
    starts = np.concatenate([[0], np.cumsum(n)[:-1]])
    first_chunk, last_chunk = starts // chunk, (starts + n - 1) // chunk
    assert np.all(n[:3] == 1)
    assert np.any((n == chunk) & (starts % chunk == 0))                         # exactly one chunk
    assert np.any((starts % chunk != 0) & (last_chunk - first_chunk > nsub))   # mid-chunk, more than nsub chunks
    assert np.sum(last_chunk - first_chunk > lpr) >= 20                         # past the first probing window
    assert np.sum(last_chunk - first_chunk == 1) >= 20                          # across one chunk boundary


def test_update_geometry_restatement():
    """Spot values of the launch geometry on a 148-SM device."""
    g = update_geom(128, [26 * 2048], 0, 148)
    assert (g.vec, g.lpr, g.nch, g.threads, g.G, g.tile) == (4, 32, 1, 256, 8, 16)
    g = update_geom(1024, [4096], 0, 148)
    assert (g.vec, g.lpr, g.nch, g.threads, g.G) == (4, 32, 8, 128, 4)
    g = update_geom(250, [10], 0, 148)
    assert (g.vec, g.lpr, g.nch, g.threads, g.G) == (1, 32, 8, 128, 4)
    g = update_geom(10, [10], 0, 148)
    assert (g.vec, g.lpr, g.nch, g.G, g.nsub) == (1, 16, 1, 16, 16)
    g = update_geom(128, [32 * 1025, 10], 4, 148)
    assert g.chunks == [1025, 1] and [g.path(0), g.path(1)] == ["grouped", "smem"]
    assert update_geom(128, [1 << 17, (1 << 17) + 1]).path(0) == "two-launch"
    assert update_geom(4, [100], 0, 148, two_launches=True).path(0) == "two-launch"


@pytest.mark.parametrize("lr,bf16", [(0.5, False), (-0.25, True)])
def test_exact_data_makes_the_order_irrelevant(lr, bf16):
    """The expected table equals the fp32 oracle's (and its bf16 form), which adds in another order."""
    rng = np.random.default_rng(1)
    rows, D, B = 40, 16, 3000
    (table,) = exact_tables([rows], D, rng)
    assert np.array_equal(O.to_bf16(table), table)
    g = exact_grads(B, D, rng)
    idx = np.minimum(rng.zipf(1.3, size=(B, 2)) - 1, rows - 1)
    ref = table.copy()
    (O.sparse_sgd_update_bf16 if bf16 else O.sparse_sgd_update_fast)(ref, idx, g, lr)
    assert np.array_equal(expected_exact(table, idx, g, lr, bf16), ref)
