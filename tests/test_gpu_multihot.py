"""Per-table pooling factors (multi-hot with mixed hotness) on the GPU: lookup, sort / dedup in all three
sort regimes at once, sparse SGD, a DLRM training step with the MLPerf DLRM-DCNv2 hotness list, graph
capture, host entry points and argument errors -- against the CPU oracle and the uniform entry points."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

SGD_RTOL = 1e-4
BF16_RTOL = 1e-2
MLPERF_HOTNESS = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _dev():
    return torch.device("cuda", 0)


def _rand_tables(rng, rows, D):
    return [rng.standard_normal((r, D)).astype(np.float32) for r in rows]


def _packed(idx, dtype=np.int64, base=0):
    from dlrm_jl_b200.embedding import _as_index_tensor
    return _as_index_tensor([np.asarray(a).astype(dtype) + base for a in idx], len(idx), _dev())


def _tables(arrays, max_lookups, dtype=torch.float32):
    from dlrm_jl_b200.embedding import EmbeddingTables
    return EmbeddingTables.from_arrays(arrays, max_lookups, 0, dtype)


def _lookup(t, p, slot0=1, base=0, sort=False):
    T = torch.zeros((p.B, slot0 + t.ntab, t.D), dtype=torch.float32, device=_dev())
    t.lookup(p, T, slot0, base, sort=sort)
    return T


@pytest.mark.parametrize("D", [4, 10, 64, 128])
def test_lookup_mixed_bit_exact(D):
    rng = np.random.default_rng(D)
    rows, P = [7, 1000, 33, 5000, 64], [1, 3, 1, 100, 7]
    tables = _rand_tables(rng, rows, D)
    for B, dtype, base in [(1, np.int64, 0), (3, np.int32, 1), (257, np.int64, 1), (2048, np.int32, 0)]:
        idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
        t = _tables(tables, B * max(P))
        ref = O.lookup(tables, idx, slot0=1)
        for sort in (False, True):
            T = _lookup(t, _packed(idx, dtype, base), base=base, sort=sort).cpu().numpy()
            assert np.array_equal(T, ref), (B, dtype, base, sort)
        t.close()


def test_lookup_mixed_bf16():
    rng = np.random.default_rng(5)
    rows, P, B, D = [7, 1000, 33, 5000, 64], [1, 3, 1, 100, 7], 257, 64
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    t = _tables(tables, B * max(P), torch.bfloat16)
    stored = [t.download(k) for k in range(len(rows))]
    for sort in (False, True):
        T = _lookup(t, _packed(idx), sort=sort).cpu().numpy()
        assert O.rel_err(T, O.lookup(stored, idx, slot0=1)) < 1e-6
        assert O.rel_err(T, O.lookup(tables, idx, slot0=1)) < BF16_RTOL


@pytest.mark.parametrize("P", [1, 4, 10])
def test_equal_pooling_factors_match_uniform_bitwise(P):
    from dlrm_jl_b200.embedding import PackedIndices
    rng = np.random.default_rng(P)
    rows, B, D = [11, 3000, 70000, 5], 1024, 64
    tables = _rand_tables(rng, rows, D)
    idx = np.stack([rng.integers(0, r, size=(B, P)) for r in rows])
    u_idx = torch.from_numpy(idx).to(_dev())
    packed = PackedIndices(u_idx.reshape(-1).contiguous(), (P,) * len(rows), B)
    dT = torch.from_numpy(rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)).to(_dev())
    t_u, t_m = _tables(tables, B * P), _tables(tables, B * P)
    Tu = torch.zeros((B, 1 + len(rows), D), device=_dev())
    t_u.lookup(u_idx, Tu, 1, sort=True)
    Tm = _lookup(t_m, packed, sort=True)
    assert torch.equal(Tu, Tm)
    for k in range(len(rows)):
        for a, b in zip(t_u.sort_dedup_export(k, B * P), t_m.sort_dedup_export(k, B * P)):
            assert np.array_equal(a, b)
    t_u.update_sorted(dT, 1, 0.05)
    t_m.update_sorted(dT, 1, 0.05)
    for k in range(len(rows)):
        assert np.array_equal(t_u.download(k), t_m.download(k))


# A uniform batch on a handle with more tables than one per-table geometry holds (dlrmb_mp_max_tables):
# the uniform entry points run the per-table launchers once per group of tables.  B = 256: lookup and
# fused sort in one launch; B = 6000 with P = 3: separate lookup and radix sort.
@pytest.mark.parametrize("P,B,dtype", [(1, 256, torch.float32), (3, 256, torch.float32),
                                       (1, 256, torch.bfloat16), (3, 256, torch.bfloat16),
                                       (3, 6000, torch.float32)])
def test_uniform_more_tables_than_one_geometry(P, B, dtype):
    from dlrm_jl_b200 import _lib
    ntab, D, W, lr = 300, 16, 2, 0.05
    assert ntab > _lib.load().dlrmb_mp_max_tables()
    rng = np.random.default_rng(P + B)
    rows = [int(r) for r in rng.integers(1, 200, size=ntab)]
    t = _tables(_rand_tables(rng, rows, D), B * P, dtype)
    idx = np.stack([rng.integers(0, r, size=(B, P)) for r in rows])
    u_idx = torch.from_numpy(idx).to(_dev())
    dT = torch.from_numpy(rng.standard_normal((B, 1 + ntab, D)).astype(np.float32)).to(_dev())
    dTn = dT.cpu().numpy()

    def check_dedup():
        for k in range(ntab):
            for a, b in zip(t.sort_dedup_export(k, B * P), O.sort_dedup(idx[k])):
                assert np.array_equal(a, b), k

    def check_update(stored):
        for k in range(ntab):
            ref, got = stored[k].copy(), t.download(k)
            if dtype == torch.bfloat16:
                O.sparse_sgd_update_bf16(ref, idx[k], np.ascontiguousarray(dTn[:, 1 + k]), lr)
                assert O.rel_err(got, ref) < 2e-3, k
            else:
                O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(dTn[:, 1 + k]), lr)
                assert O.rel_err(got, ref) < SGD_RTOL, k

    stored = [t.download(k) for k in range(ntab)]
    ref = O.lookup(stored, idx, slot0=1)
    for sort in (False, True):
        T = torch.zeros((B, 1 + ntab, D), device=_dev())
        t.lookup(u_idx, T, 1, sort=sort)
        assert np.array_equal(T.cpu().numpy()[:, 1:], ref[:, 1:]), sort
    t.update_sorted(dT, 1, lr)
    check_update(stored)

    t.sort(u_idx.to(torch.int32))
    check_dedup()

    stored = [t.download(k) for k in range(ntab)]
    slotmap = [ntab - k for k in range(ntab)]          # reversed: a group must read its own part of the map
    t.set_slot_map(slotmap)
    bufs = [torch.full((B // W, 1 + ntab, D), float("nan"), device=_dev()) for _ in range(W)]
    t.lookup_p2p(u_idx, [b.data_ptr() for b in bufs], B // W, 1 + ntab, 0, sort=True)
    got = torch.cat(bufs).cpu().numpy()
    want = O.lookup(stored, idx, slot0=0)
    assert np.isnan(got[:, 0]).all()
    assert np.array_equal(got[:, slotmap], want)
    check_dedup()
    t.update_sorted(dT, 1, lr)
    check_update(stored)
    t.close()


def test_sort_dedup_all_three_regimes_in_one_batch():
    rng = np.random.default_rng(7)
    B = 2048
    P = [1, 2, 3, 5, 8, 12, 1]             # L = 2048, 4096 (fused) | 6144, 10240, 16384 (shared memory) | 24576 (radix)
    rows = [500, 40000, 7, 100000, 3, 2_000_000, 1]
    tables = _rand_tables(rng, rows, 8)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    t = _tables(tables, B * max(P))
    for sort in ("fwd", "alone"):
        if sort == "fwd":
            _lookup(t, _packed(idx), sort=True)
        else:
            t.sort(_packed(idx, np.int32))
        for k in range(len(rows)):
            u, s, perm = t.sort_dedup_export(k, B * P[k])
            ru, rs, rp = O.sort_dedup(idx[k])
            assert np.array_equal(u, ru) and np.array_equal(s, rs) and np.array_equal(perm, rp), (sort, k)


def _sgd_ref(tables, idx, dTs, lr):
    ref = [a.copy() for a in tables]
    for dT in dTs:
        for k in range(len(ref)):
            O.sparse_sgd_update_fast(ref[k], idx[k], np.ascontiguousarray(dT[:, 1 + k]), lr)
    return ref


def _run_sgd(tables, idx, dTs, lr, max_lookups):
    t = _tables(tables, max_lookups)
    p = _packed(idx)
    for dT in dTs:
        t.bwd_sgd(p, torch.from_numpy(dT).to(_dev()), 1, lr)
    out = [t.download(k) for k in range(len(tables))]
    t.close()
    return out


@pytest.mark.parametrize("case", ["uniform", "zipf", "tiny_rows"])
def test_sparse_sgd_mixed_against_oracle(case):
    rng = np.random.default_rng(11)
    B, D, lr = 512, 32, 0.05
    rows, P = [1000, 50000, 200, 3, 9000], [1, 7, 27, 27, 2]
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    if case == "zipf":
        idx[1] = np.minimum(rng.zipf(1.2, size=(B, P[1])) - 1, rows[1] - 1)
    if case == "tiny_rows":
        idx = [rng.integers(0, min(r, 3), size=(B, p)) for r, p in zip(rows, P)]
    for steps in (1, 5):
        dTs = [rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32) for _ in range(steps)]
        got = _run_sgd(tables, idx, dTs, lr, B * max(P))
        ref = _sgd_ref(tables, idx, dTs, lr)
        for k in range(len(rows)):
            assert O.rel_err(got[k], ref[k]) < SGD_RTOL, (case, steps, k)
            touched = np.zeros(rows[k], bool)
            touched[np.unique(idx[k])] = True
            assert np.array_equal(got[k][~touched], tables[k][~touched])
        again = _run_sgd(tables, idx, dTs, lr, B * max(P))
        assert all(np.array_equal(a, b) for a, b in zip(got, again))          # bitwise reproducible


def test_sparse_sgd_mixed_fixup_paths_and_tiles_agree():
    from dlrm_jl_b200 import _lib
    rng = np.random.default_rng(13)
    B, D, lr = 1024, 64, 0.1
    rows, P = [3, 20000, 5, 800], [27, 9, 1, 4]
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    idx[1] = np.minimum(rng.zipf(1.2, size=(B, P[1])) - 1, rows[1] - 1)
    dTs = [rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)]
    base = _run_sgd(tables, idx, dTs, lr, B * max(P))
    try:
        _lib.set_option("update_two_launches", 1)
        two = _run_sgd(tables, idx, dTs, lr, B * max(P))
    finally:
        _lib.set_option("update_two_launches", 0)
    assert all(np.array_equal(a, b) for a, b in zip(base, two))
    ref = _sgd_ref(tables, idx, dTs, lr)
    for tile in (4, 8, 32):
        try:
            _lib.set_option("update_tile", tile)
            got = _run_sgd(tables, idx, dTs, lr, B * max(P))
        finally:
            _lib.set_option("update_tile", 0)
        for k in range(len(rows)):
            assert O.rel_err(got[k], ref[k]) < SGD_RTOL, (tile, k)


def _mlperf_model(B, rows_cap, D=16, seed=0):
    from dlrm_jl_b200.model import dlrm
    rows = [min(r, rows_cap) for r in [39884406, 39043, 17289, 7420, 20263, 3, 7120, 1543, 63, 38532951, 2953546,
                                       403346, 10, 2208, 11938, 155, 4, 976, 14, 39979771, 25641295, 39664984,
                                       585935, 12972, 108, 36]]
    m = dlrm([13, 64, D], [64, 1], D, rows, max_lookups=B * max(MLPERF_HOTNESS), init_tables=True, seed=seed)
    return m, rows


def _np_params(mlp):
    layers = [l for l in mlp if isinstance(l, torch.nn.Linear)]
    return [(l.weight.detach().cpu().numpy().copy(), l.bias.detach().cpu().numpy().copy()) for l in layers]


def test_mlperf_hotness_training_steps_against_oracle():
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.train import train_step, wrap_loss, bce_loss
    torch.backends.cuda.matmul.allow_tf32 = False
    rng = np.random.default_rng(17)
    B, lr = 2048, 0.05
    m, rows = _mlperf_model(B, rows_cap=5000)
    tables = [m.embeddings.download(k) for k in range(len(rows))]
    bot, top = _np_params(m.bottom_mlp), _np_params(m.top_mlp)
    loss = wrap_loss(bce_loss)
    for step in range(3):
        idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, MLPERF_HOTNESS)]
        dense = rng.random((B, 13), dtype=np.float32)
        labels = rng.integers(0, 2, size=B).astype(np.float32)
        l = train_step(loss, m, Descent(lr), torch.from_numpy(labels).to(_dev()), torch.from_numpy(dense).to(_dev()),
                       idx)
        l_ref, bot, top, _fwd, _g = O.dlrm_train_step(bot, top, tables, dense, idx, labels, lr)
        assert abs(float(l) - float(l_ref)) <= 1e-4 * max(1.0, abs(float(l_ref))), step
    for k in range(len(rows)):
        assert O.rel_err(m.embeddings.download(k), tables[k]) < SGD_RTOL, k


def test_mixed_step_graph_capture_equals_eager():
    rng = np.random.default_rng(19)
    B, D, lr = 512, 64, 0.05
    rows, P = [1000, 50000, 200, 30000], [1, 7, 27, 100]
    tables = _rand_tables(rng, rows, D)
    idx = _packed([rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)])
    dT = torch.from_numpy(rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)).to(_dev())

    def step(t, T):
        t.lookup(idx, T, 1, sort=True)
        t.update_sorted(dT, 1, lr)

    t_e, t_g = _tables(tables, B * max(P)), _tables(tables, B * max(P))
    T_e = torch.zeros((B, 1 + len(rows), D), device=_dev())
    T_g = torch.zeros_like(T_e)
    step(t_e, T_e)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            step(t_g, T_g)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(T_e, T_g)
    for k in range(len(rows)):
        assert np.array_equal(t_e.download(k), t_g.download(k))


def test_host_entry_points_equal_device_entry_points():
    rng = np.random.default_rng(23)
    B, D, lr = 300, 16, 0.1
    rows, P = [50, 4000, 9], [4, 1, 13]
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    p = _packed(idx, np.int32)
    flat = p.flat.cpu().numpy()
    t_d, t_h = _tables(tables, B * max(P)), _tables(tables, B * max(P))
    T_d = _lookup(t_d, p).cpu().numpy()
    T_h = np.zeros_like(T_d)
    lib = t_h._lib
    from dlrm_jl_b200 import _lib
    _lib.check(lib.dlrmb_embedding_fwd_mp_host(t_h._h, flat.ctypes.data_as(C.c_void_p), 4, 0, B, p.P_array(),
                                               T_h.ctypes.data_as(C.c_void_p), 1 + len(rows), 1))
    assert np.array_equal(T_d, T_h)
    dT = rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)
    t_d.bwd_sgd(p, torch.from_numpy(dT).to(_dev()), 1, lr)
    _lib.check(lib.dlrmb_embedding_bwd_sgd_mp_host(t_h._h, flat.ctypes.data_as(C.c_void_p), 4, 0, B, p.P_array(),
                                                   dT.ctypes.data_as(C.c_void_p), 1 + len(rows), 1, lr))
    for k in range(len(rows)):
        assert np.array_equal(t_d.download(k), t_h.download(k))


def test_mixed_check_indices_and_argument_errors():
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.embedding import EmbeddingTables
    rng = np.random.default_rng(29)
    B, rows, P = 64, [10, 20, 30], [1, 5, 2]
    tables = _rand_tables(rng, rows, 8)
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    t = _tables(tables, B * max(P))
    t.check_indices(_packed(idx))
    bad = [a.copy() for a in idx]
    bad[1][3, 2] = 20
    with pytest.raises(_lib.DLRMB200Error, match="table 1, flat position 17, value 20") as e:
        t.check_indices(_packed(bad))
    assert e.value.status == _lib.EOOB
    lib, p = t._lib, _packed(idx)
    out = torch.zeros((B, 4, 8), device=_dev())

    def fwd(Parr, Bv=B):
        return lib.dlrmb_embedding_fwd_mp(t._h, p.data_ptr(), 8, 0, Bv, Parr, out.data_ptr(), 4, 1, None)

    assert fwd((C.c_int32 * 3)(1, 0, 2)) == _lib.EINVAL
    assert b"P[1] = 0" in lib.dlrmb_last_error()
    assert fwd(None) == _lib.EINVAL
    assert b"null" in lib.dlrmb_last_error()
    assert fwd((C.c_int32 * 3)(1, 6, 2)) == _lib.EINVAL                  # 64 * 6 > max_lookups = 320
    assert b"exceeds max_lookups" in lib.dlrmb_last_error()
    n = lib.dlrmb_mp_max_tables()
    assert n == 256
    big = EmbeddingTables([4] * (n + 1), 4, 8, _dev())
    Pb = (C.c_int32 * (n + 1))(*([1] * (n + 1)))
    zb = torch.zeros(n + 1, 2, dtype=torch.int32, device=_dev())
    ob = torch.zeros((2, n + 2, 4), device=_dev())
    assert lib.dlrmb_embedding_fwd_mp(big._h, zb.data_ptr(), 4, 0, 2, Pb, ob.data_ptr(), n + 2, 1, None) == _lib.EINVAL
    assert b"up to 256 tables" in lib.dlrmb_last_error()
    big.close()
