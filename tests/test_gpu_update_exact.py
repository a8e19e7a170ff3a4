"""Bit-exact sparse SGD update at the boundaries of its reduction tree, for every kernel variant and fix-up path.

The update sums each row's gradients in an order fixed by the tile, the chunk and the fix-up path, so a
table-wide norm cannot see one lost or doubled contribution.  Most tests here use exact data (table entries
k / 32, gradient entries k / 16, lr a power of two; tests/sparse_update_layouts.py): the expected table is then
the same in any summation order, and every row must match it bit for bit.  The run layouts are built, not
drawn: runs end next to tile and chunk edges, cross chunks and the fix-up's probing windows, and the same row
ends one table and starts the next.  The float test pins the rounding of rows updated once or twice and bounds
the others row by row.  Which fix-up ran is checked by the launch count (two-launch: one more launch) and by
the restated geometry (shared-memory fix-up up to 1024 chunks per table, grouped above)."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.sparse_update_layouts import (INLINE_MAX_ENTRIES, chained_row_ids, edge_ends, exact_grads,
                                         exact_tables, expected_exact, lengths_from_ends, mixed_ends,
                                         row_sums, runs_to_indices, update_geom)

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

VEC4_D = [4, 12, 128, 132, 256, 516, 1024]     # NCH 1, 1, 1, 2, 2, 8, 8 (THREADS 128 for the last two)
VEC1_D = [1, 10, 33, 99, 250]                  # NCH 1, 1, 2, 4, 8
F32, BF16 = torch.float32, torch.bfloat16


def _dev():
    return torch.device("cuda", 0)


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def lib_options():
    """Set library switches for one test and restore the defaults afterwards."""
    from dlrm_jl_b200 import _lib
    touched = {}

    def set_(name, value):
        touched.setdefault(name, _lib.get_option(name))
        _lib.set_option(name, value)
    yield set_
    for name, value in touched.items():
        _lib.set_option(name, value)


def _launches():
    from dlrm_jl_b200 import _lib
    return _lib.launch_count()


def _handle(tables, max_lookups, dtype):
    from dlrm_jl_b200.embedding import EmbeddingTables
    t = EmbeddingTables.from_arrays(tables, max_lookups, 0, dtype)
    for k, a in enumerate(tables):             # exact data is representable in bf16: nothing is rounded on upload
        assert np.array_equal(t.download(k), a), k
    return t


def _device_indices(idx, grid):
    """[ntab] x [B][P_k] numpy -> the uniform [ntab][B][P] tensor or PackedIndices (even for equal P_k)."""
    from dlrm_jl_b200.embedding import PackedIndices
    if grid == "uniform":
        return torch.from_numpy(np.stack(idx)).to(_dev())
    flat = torch.from_numpy(np.concatenate([a.reshape(-1) for a in idx])).to(_dev())
    return PackedIndices(flat, tuple(int(a.shape[1]) for a in idx), int(idx[0].shape[0]))


def _dT(grads, slot0, pad, B, D):
    """[B][slot0 + ntab + pad][D] with table k's gradient in slot slot0 + k and NaN in every other slot."""
    dT = np.full((B, slot0 + len(grads) + pad, D), np.nan, dtype=np.float32)
    for k, g in enumerate(grads):
        dT[:, slot0 + k] = g
    return dT


def _layout_batch(Ls, B, ends_of, rng, extra_rows=3):
    """Indices for tables with L_k = Ls[k] entries and run ends ends_of(k, L_k); table k's first row id is
    table k-1's last.  Returns (idx list, rows list)."""
    lengths = [lengths_from_ends(ends_of(k, L), L) for k, L in enumerate(Ls)]
    ids = chained_row_ids([len(n) for n in lengths], rng)
    idx = [runs_to_indices(i, n, B, rng) for i, n in zip(ids, lengths)]
    rows = [int(i[-1]) + 1 + extra_rows for i in ids]
    return idx, rows


def _update_once(t, idx, grid, dT, slot0, lr):
    """Sort and update; returns the update's launch count."""
    t.sort(_device_indices(idx, grid))
    g = torch.from_numpy(dT).to(_dev())
    n0 = _launches()
    t.update_sorted(g, slot0, lr)
    n = _launches() - n0
    torch.cuda.synchronize()
    return n


def _check_exact(t, expected, what):
    for k, e in enumerate(expected):
        got = t.download(k)
        bad = np.argwhere(~((got == e) | (np.isnan(got) & np.isnan(e))).all(axis=1))
        assert bad.size == 0, f"{what}: table {k}, {bad.size} rows differ, first rows {bad[:8, 0].tolist()}"


def _run_exact(D, dtype, grid, idx, rows, lr, paths, rng, slot0=1, pad=0, tile=0, lib_options=None):
    """Runs one batch once per fix-up switch in `paths` ("inline" / "two"), each on a fresh handle, and
    checks every row bit for bit.  Returns the geometry of the inline run."""
    B = idx[0].shape[0]
    Ls = [a.size for a in idx]
    bf16 = dtype == BF16
    tables = exact_tables(rows, D, rng)
    grads = [exact_grads(B, D, rng) for _ in idx]
    dT = _dT(grads, slot0, pad, B, D)
    expected = [expected_exact(tb, a, g, lr, bf16) for tb, a, g in zip(tables, idx, grads)]
    geom = None
    for p in paths:
        lib_options("update_two_launches", 1 if p == "two" else 0)
        lib_options("update_tile", tile)
        gm = update_geom(D, Ls, tile, _sm_count(), two_launches=(p == "two"))
        t = _handle(tables, max(Ls), dtype)
        n = _update_once(t, idx, grid, dT, slot0, lr)
        assert n == (1 if gm.inline else 2), (p, n, gm)
        _check_exact(t, expected, f"D={D} {dtype} {grid} {p} tile={gm.tile} chunks={gm.chunks}")
        t.close()
        if p == "inline":
            geom = gm
    return geom


# ------------------------------------------------------------------------------------------------
# runs ending next to tile and chunk edges
# ------------------------------------------------------------------------------------------------
EDGE_CASES = [(128, F32, "uniform"), (12, BF16, "mp"), (33, F32, "mp"), (1024, BF16, "uniform"),
              (10, F32, "uniform"), (4, F32, "mp"), (250, BF16, "mp")]


@pytest.mark.parametrize("tile", [4, 12, 32, 0])
@pytest.mark.parametrize("D,dtype,grid", EDGE_CASES)
def test_runs_ending_at_tile_and_chunk_edges(tile, D, dtype, grid, lib_options):
    """Nine tables; in table j runs end at n*T*2^j - 1, n*T*2^j, n*T*2^j + 1 and + 2 (T the tile, j = 8..0), so
    every chunk size G*T = T*2^j has runs ending just before, on and just after its edges."""
    rng = np.random.default_rng(1000 * D + tile)
    B = 1025
    P = [24] * 9 if grid == "uniform" else [24, 20, 28, 24, 16, 32, 24, 20, 28]
    Ls = [B * p for p in P]
    T = update_geom(D, Ls, tile, _sm_count()).tile
    idx, rows = _layout_batch(Ls, B, lambda k, L: edge_ends(L, T, 8 - k), rng)
    gm = _run_exact(D, dtype, grid, idx, rows, 0.5, ("inline",), rng, tile=tile, lib_options=lib_options)
    assert gm.tile == T and gm.inline


# ------------------------------------------------------------------------------------------------
# the variant matrix: D x row type x uniform / per-table P x fix-up path
# ------------------------------------------------------------------------------------------------
def _grouped_reachable(D):
    """More than 1024 chunks in one table within 2^18 entries needs G * 4 * 1032 * 1.5 <= 2^18, i.e. G <= 16."""
    return update_geom(D, [1]).G <= 16


MATRIX = ([(D, dt, grid, path) for D in VEC4_D + VEC1_D for dt in (F32, BF16) for grid in ("uniform", "mp")
           for path in ("smem", "grouped") if path == "smem" or _grouped_reachable(D)]
          + [(D, (F32, BF16)[i % 2], ("uniform", "mp")[(i // 2) % 2], "large")
             for i, D in enumerate(VEC4_D + VEC1_D)])


@pytest.mark.parametrize("D,dtype,grid,path", MATRIX)
def test_update_variant_matrix_exact(D, dtype, grid, path, lib_options):
    """smem / grouped: the inline fix-up (asserted by the geometry) and the two-launch switch on the same
    batch; large: more than 2^18 entries, which takes two launches by itself."""
    rng = np.random.default_rng(D * 7 + len(path) + (dtype == BF16) + 2 * (grid == "mp"))
    g0 = update_geom(D, [1])
    if path == "smem":
        tile, ntab = 0, 3
        L = min(INLINE_MAX_ENTRIES // 3, max(4096, 16 * (g0.lpr + 4) * g0.G * 4)) // 16 * 16
        B, P = L // 4, ([4, 4, 4] if grid == "uniform" else [4, 2, 6])
    elif path == "grouped":
        tile, ntab = 4, 2
        L = 4 * g0.G * 1032
        B, P = L // 16, ([16, 16] if grid == "uniform" else [16, 8])
    else:
        tile, ntab = 0, 3
        B, P = 3000, ([30, 30, 30] if grid == "uniform" else [30, 20, 40])
    Ls = [B * p for p in P]
    gm = update_geom(D, Ls, tile, _sm_count())
    idx, rows = _layout_batch(Ls, B, lambda k, L: mixed_ends(L, gm.chunk, gm.lpr, gm.nsub, rng), rng)
    paths = ("inline",) if path == "large" else ("inline", "two")
    got = _run_exact(D, dtype, grid, idx, rows, -0.25 if D % 2 else 0.5, paths, rng, tile=tile,
                     lib_options=lib_options)
    if path == "large":
        assert sum(Ls) > INLINE_MAX_ENTRIES and not got.inline
    elif path == "smem":
        assert got.inline and all(got.path(k) == "smem" for k in range(ntab)), got
    else:
        assert got.inline and got.path(0) == "grouped", got


# ------------------------------------------------------------------------------------------------
# the fix-up's run-end search with several lane groups per warp (lanes per row < 32)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [4, 8, 16, 64, 1, 10])
@pytest.mark.parametrize("grid", ["uniform", "mp"])
def test_fixup_run_end_search_with_several_groups_per_warp(D, grid, lib_options):
    """Many head chunks in one table: runs longer than lpr chunks (past the first probing window of their
    lane group) alternate with runs that end in the next chunk, so neighbouring lane groups of one warp
    search for run ends at the same time.  A group must see only its own lanes' flags."""
    rng = np.random.default_rng(D + 77 * (grid == "mp"))
    g0 = update_geom(D, [1], 4)
    assert g0.lpr < 32
    B, Pu = 4096, min(32, g0.G)                 # at most 1024 chunks of 4 * G entries per table
    P = [Pu, Pu] if grid == "uniform" else [Pu, 3 * Pu // 4]
    Ls = [B * p for p in P]
    gm = update_geom(D, Ls, 4, _sm_count())
    idx, rows = _layout_batch(Ls, B, lambda k, L: mixed_ends(L, gm.chunk, gm.lpr, gm.nsub, rng, filler_runs=50,
                                                             ballot_rounds=512), rng)
    got = _run_exact(D, F32, grid, idx, rows, 0.5, ("inline", "two"), rng, tile=4, lib_options=lib_options)
    assert got.inline and all(got.path(k) == "smem" for k in range(2)), got


# ------------------------------------------------------------------------------------------------
# tiny batches, single-row tables, stale keys past L
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,dtype,grid", [(4, F32, "uniform"), (128, BF16, "mp"), (1, F32, "mp"),
                                          (33, BF16, "uniform"), (1024, F32, "uniform")])
def test_tiny_batches_after_a_long_run_on_one_handle(D, dtype, grid, lib_options):
    """L in {1, 2, 3, 5, 7, 11, 43} (the 16-byte key loads read past L) after a batch whose stream is one
    long run of the same row, so the stale keys past L continue the new batch's last run.  Table 0 has a
    single row."""
    rng = np.random.default_rng(D)
    bf16 = dtype == BF16
    rows = [1, 50, 50]
    cur = exact_tables(rows, D, rng)
    t = _handle(cur, 2048, dtype)
    batches = [(2048, "inline")] + [(L, ("inline", "two")[i % 2]) for i, L in enumerate([1, 2, 3, 5, 7, 11, 43])]
    for i, (L, fix) in enumerate(batches):
        lib_options("update_two_launches", 1 if fix == "two" else 0)
        B = L
        if i == 0:
            idx = [np.zeros((B, 1), np.int64), np.full((B, 1), 49), np.full((B, 1), 49)]
        else:
            idx = [np.zeros((B, 1), np.int64)] + [np.sort(rng.integers(45, 50, size=L))[::-1].reshape(B, 1)
                                                 for _ in range(2)]
        grads = [exact_grads(B, D, rng) for _ in rows]
        n = _update_once(t, idx, grid, _dT(grads, 1, 0, B, D), 1, 0.5)
        assert n == (1 if fix == "inline" else 2)
        cur = [expected_exact(tb, a, g, 0.5, bf16) for tb, a, g in zip(cur, idx, grads)]
        _check_exact(t, cur, f"batch {i}, L={L}")
    t.close()


# ------------------------------------------------------------------------------------------------
# dT slot layout
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("slot0", [0, 1, 3])
@pytest.mark.parametrize("D,grid", [(16, "uniform"), (10, "mp"), (132, "mp"), (99, "uniform")])
def test_update_reads_only_its_dT_slots(slot0, D, grid, lib_options):
    """slots = slot0 + ntab + 2 with NaN in every slot but slot0 .. slot0 + ntab - 1: one NaN read would
    poison a row.  Untouched rows stay bit-identical (every row is compared)."""
    rng = np.random.default_rng(slot0 * 100 + D)
    B = 600
    P = [3, 3, 3, 3] if grid == "uniform" else [3, 1, 5, 2]
    Ls = [B * p for p in P]
    gm = update_geom(D, Ls, 0, _sm_count())
    idx, rows = _layout_batch(Ls, B, lambda k, L: mixed_ends(L, gm.chunk, gm.lpr, gm.nsub, rng, filler_runs=200),
                              rng, extra_rows=40)
    _run_exact(D, F32, grid, idx, rows, 0.5, ("inline", "two"), rng, slot0=slot0, pad=2, lib_options=lib_options)


# ------------------------------------------------------------------------------------------------
# float rounding: random data
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,grid", [(4, "uniform"), (12, "mp"), (128, "uniform"), (1024, "mp"), (1, "mp"),
                                    (33, "uniform"), (250, "uniform")])
def test_update_rounding_on_random_data(D, grid, lib_options):
    """Rows updated once or twice match the fp32 oracle bit for bit: x - fl(lr * g) with two roundings (no FMA
    contraction), and g1 + g2 is commutative.  Every other row is within the per-element bound of any fp32
    summation order: |got - ref64| <= |lr| gamma_{m-1} S + u |lr| S (1 + gamma_{m-1}) + u/(1-u) |got|, with
    S = sum |g| over the row's m entries and u = 2^-24."""
    rng = np.random.default_rng(D + 5)
    lr = np.float32(0.1)
    B = 1024
    P = [4, 4, 4] if grid == "uniform" else [4, 2, 6]
    Ls = [B * p for p in P]
    gm = update_geom(D, Ls, 0, _sm_count())
    # filler runs of 1, 2 or 3 entries after the long ones
    idx, rows = _layout_batch(Ls, B, lambda k, L: mixed_ends(L, gm.chunk, gm.lpr, gm.nsub, rng, filler_runs=L,
                                                                    ballot_rounds=4),
                              rng, extra_rows=10)
    tables = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    grads = [rng.standard_normal((B, D)).astype(np.float32) for _ in rows]
    dT = _dT(grads, 1, 0, B, D)
    lib_options("update_two_launches", 0)
    t = _handle(tables, max(Ls), F32)
    _update_once(t, idx, grid, dT, 1, float(lr))
    u = 2.0 ** -24
    for k in range(len(rows)):
        got = t.download(k)
        ref32 = tables[k].copy()
        O.sparse_sgd_update_fast(ref32, idx[k], grads[k], float(lr))
        uniq, cnt, s, sa = row_sums(idx[k], grads[k])
        untouched = np.setdiff1d(np.arange(rows[k]), uniq)
        assert np.array_equal(got[untouched], tables[k][untouched])
        few = uniq[cnt <= 2]
        assert (cnt == 1).sum() > 40 and (cnt == 2).sum() > 40
        assert np.array_equal(got[few], ref32[few]), f"table {k}: rows with 1 or 2 entries"
        many = cnt > 2
        m = cnt[many][:, None].astype(np.float64)
        gam = (m - 1) * u / (1 - (m - 1) * u)
        lr64 = float(lr)
        ref64 = tables[k][uniq[many]].astype(np.float64) - lr64 * s[many]
        g64 = got[uniq[many]].astype(np.float64)
        bound = abs(lr64) * gam * sa[many] + u * abs(lr64) * sa[many] * (1 + gam) + u / (1 - u) * np.abs(g64)
        err = np.abs(g64 - ref64)
        assert np.all(err <= bound), f"table {k}: worst excess {np.max(err - bound)}"
    t.close()


# ------------------------------------------------------------------------------------------------
# state across calls on one handle
# ------------------------------------------------------------------------------------------------
STATE_STEPS = [  # (sort, grid, fix-up switch, B, P)
    ("fused", "uniform", "inline", 1024, [4, 4, 4]),
    ("radix", "mp", "two", 4096, [6, 1, 3]),
    ("smem", "uniform", "inline", 3000, [4, 4, 4]),
    ("fused", "mp", "inline", 512, [1, 8, 3]),
    ("radix", "uniform", "two", 5000, [8, 8, 8]),
    ("fused", "uniform", "inline", 5, [1, 1, 1]),
    ("smem", "mp", "two", 700, [2, 9, 1]),
    ("radix", "uniform", "inline", 20000, [1, 1, 1]),
    ("smem", "uniform", "two", 3, [1, 1, 1]),
    ("fused", "mp", "inline", 2048, [2, 1, 2]),
    ("radix", "mp", "inline", 3000, [12, 2, 7]),
]


@pytest.mark.parametrize("D,dtype", [(16, F32), (128, BF16)])
def test_update_state_across_calls_on_one_handle(D, dtype, lib_options):
    """One handle, one sequence of steps checked exactly against running expected tables: fused lookup + sort,
    shared-memory and radix sorts, uniform and per-table P, inline and two-launch fix-up, growing and
    shrinking chunk counts (per-table done counters, flags and the ping-pong half carry over)."""
    rng = np.random.default_rng(D)
    bf16 = dtype == BF16
    rows = [40000, 40000, 40000]
    cur = exact_tables(rows, D, rng)
    t = _handle(cur, 40000, dtype)
    for i, (sort, grid, fix, B, P) in enumerate(STATE_STEPS):
        Ls = [B * p for p in P]
        assert max(Ls) <= 40000
        if sort == "fused":
            assert max(Ls) <= t.FUSED_SORT_MAX or grid == "mp"
        elif sort == "smem":
            assert max(Ls) <= 16384
        else:
            assert max(Ls) > 16384
        lib_options("update_two_launches", 1 if fix == "two" else 0)
        gm = update_geom(D, Ls, 0, _sm_count(), two_launches=(fix == "two"))
        idx, _ = _layout_batch(Ls, B, lambda k, L: mixed_ends(L, gm.chunk, gm.lpr, gm.nsub, rng, filler_runs=300),
                               rng)
        assert all(int(a.max()) < r for a, r in zip(idx, rows))
        grads = [exact_grads(B, D, rng) for _ in rows]
        slot0 = 1
        dT = _dT(grads, slot0, 0, B, D)
        dev_idx = _device_indices(idx, grid)
        if sort == "fused":
            out = torch.full((B, slot0 + len(rows), D), np.nan, device=_dev())
            n0 = _launches()
            t.lookup(dev_idx, out, slot0, sort=True)
            if grid == "uniform":
                assert _launches() - n0 == 1, "the lookup and the sort must share one launch"
            ref = O.lookup(cur, idx, slot0=slot0)
            assert np.array_equal(out.cpu().numpy()[:, slot0:], ref[:, slot0:]), i
        else:
            t.sort(dev_idx)
        n0 = _launches()
        t.update_sorted(torch.from_numpy(dT).to(_dev()), slot0, 0.5)
        assert _launches() - n0 == (1 if gm.inline else 2), (i, gm)
        cur = [expected_exact(tb, a, g, 0.5, bf16) for tb, a, g in zip(cur, idx, grads)]
        _check_exact(t, cur, f"step {i} ({sort}, {grid}, {fix}, L={Ls}, chunks={gm.chunks})")
    t.close()


# ------------------------------------------------------------------------------------------------
# lookup at the update's widths
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [1, 33, 99, 250, 516, 1024])
def test_lookup_exact_at_update_widths(D):
    """Bit-exact lookup; NaN sentinels in the slots it must not write.  With D % 4 == 0, an `out` one float
    off 16-byte alignment takes the one-float fallback, and the fused lookup + sort falls back to separate
    launches that export the same sort."""
    from dlrm_jl_b200.embedding import EmbeddingTables
    rng = np.random.default_rng(D)
    rows, B, P, slot0 = [300, 7, 5000], 257, 3, 2
    slots = slot0 + len(rows) + 1
    tables = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = np.stack([rng.integers(0, r, size=(B, P)) for r in rows])
    ref = O.lookup(tables, list(idx), slot0=slot0)
    t = EmbeddingTables.from_arrays(tables, B * P, 0)
    dev_idx = torch.from_numpy(idx).to(_dev())
    for offset in ((0, 1) if D % 4 == 0 else (0,)):
        for sort in (False, True):
            buf = torch.full((B * slots * D + offset,), np.nan, device=_dev())
            out = buf[offset:].view(B, slots, D)
            assert (out.data_ptr() % 16 == 0) == (offset == 0)
            n0 = _launches()
            t.lookup(dev_idx, out, slot0, sort=sort)
            n = _launches() - n0
            o = out.cpu().numpy()
            what = (offset, sort)
            assert np.array_equal(o[:, slot0:slot0 + len(rows)], ref[:, slot0:]), what
            assert np.isnan(o[:, :slot0]).all() and np.isnan(o[:, slot0 + len(rows):]).all(), what
            assert np.isnan(buf[:offset].cpu().numpy()).all()
            if not sort:
                assert n == 1, what
                continue
            assert n == (1 if (D % 4 == 0 and offset == 0) else 2), what
            for k in range(len(rows)):
                for a, b in zip(t.sort_dedup_export(k, B * P), O.sort_dedup(idx[k])):
                    assert np.array_equal(a, b), (what, k)
    t.close()
