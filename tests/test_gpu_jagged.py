"""Jagged (variable-length) bags on the GPU: lookup, sort, position -> bag pass and update against the NumPy
reference (tests/jagged_oracle.py) and against the `_mp` path for constant lengths."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import jagged_oracle as J

pytestmark = pytest.mark.gpu

MLPERF_P = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _dev():
    return torch.device("cuda", 0)


def _tables(rows, D, max_lookups, dtype=torch.float32, seed=7):
    from dlrm_jl_b200.embedding import EmbeddingTables
    t = EmbeddingTables(rows, D, max_lookups, _dev(), dtype)
    t.init_uniform(seed)
    return t


def _jag(values, lengths, pooling="sum", dtype=torch.int64, base=0):
    from dlrm_jl_b200.embedding import JaggedIndices
    v = torch.as_tensor(np.asarray(values, dtype=np.int64) + base).to(dtype)
    return JaggedIndices.from_lengths(v, lengths, pooling).to(_dev())


def _batch(rng, rows, lengths, zipf=None):
    vals = []
    for r, n in zip(rows, lengths):
        tot = int(np.sum(n))
        if zipf is None:
            vals.append(rng.integers(0, r, size=tot))
        else:
            vals.append((rng.zipf(zipf, size=tot) - 1) % r)
    return np.concatenate(vals).astype(np.int64)


def _lookup_shapes(rng, B):
    rows = [50, 3000, 7, 100000]
    n0 = rng.integers(0, 6, size=B)
    n0[:3] = 0                                         # empty bags
    n1 = np.zeros(B, np.int64)                         # a table without lookups
    n2 = np.ones(B, np.int64)                          # bags of length 1
    n3 = rng.integers(0, 9, size=B)
    n3[5] = 4500                                       # one bag longer than 4096
    return rows, [n0, n1, n2, n3]


@pytest.mark.parametrize("D,pooling,dtype,itype,base", [
    (64, p, dt, it, b) for p in ("sum", "mean") for dt in (torch.float32, torch.bfloat16)
    for it in (torch.int32, torch.int64) for b in (0, 1)] + [
    (D, p, dt, torch.int64, 0) for D in (4, 10, 128) for p in ("sum", "mean") for dt in (torch.float32, torch.bfloat16)])
def test_lookup_bit_exact(D, pooling, dtype, itype, base):
    rng = np.random.default_rng(D + base)
    B = 96
    rows, lengths = _lookup_shapes(rng, B)
    t = _tables(rows, D, 6000, dtype)
    vals = _batch(rng, rows, lengths)
    j = _jag(vals, lengths, pooling, itype, base)
    out = torch.full((B, 2 + len(rows), D), float("nan"), device=_dev())
    out[:, :2] = 0
    t.lookup(j, out, 2, idx_base=base)
    stored = [t.download(k) for k in range(len(rows))]
    ref = J.lookup_jagged(stored, vals, j.offsets.cpu().numpy(), B, pooling, slot0=2)
    got = out.cpu().numpy()
    assert np.array_equal(got[:, 2:].view(np.uint32), ref[:, 2:].view(np.uint32))
    assert np.all(got[:, :2] == 0)


# The shared-memory sort picks one template from the longest listed table, so each regime gets a call of its own:
# 256-thread CTAs up to 1024 / 2048 / 4096 keys, 1024-thread CTAs up to 8192 / 16384, radix above; every call also
# carries a table without lookups.
@pytest.mark.parametrize("Lmax", [1000, 2000, 4000, 8000, 16000, 40000])
def test_sort_export_all_regimes(Lmax):
    rng = np.random.default_rng(Lmax)
    B = 8
    rows = [900, 2_000_000, 77]
    Ls = [Lmax // 3, Lmax, 0]
    lengths = []
    for L in Ls:
        cut = np.sort(rng.integers(0, L + 1, size=B - 1))
        lengths.append(np.diff(np.concatenate([[0], cut, [L]])))
    t = _tables(rows, 16, max(Ls))
    vals = _batch(rng, rows, lengths, zipf=1.2)
    j = _jag(vals, lengths, "mean", torch.int32)
    t.sort(j)
    o = 0
    for k, L in enumerate(Ls):
        uniq, seg, perm = t.sort_dedup_export(k, L)
        ru, rs, rp = O.sort_dedup(vals[o:o + L])
        assert np.array_equal(uniq, ru) and np.array_equal(seg, rs) and np.array_equal(perm, rp), k
        o += L


@pytest.fixture
def two_launches(request):
    """Force the update's separate fix-up launch (the path of batches above 2^18 entries) when the parameter is 1."""
    from dlrm_jl_b200 import _lib
    before = _lib.get_option("update_two_launches")
    _lib.set_option("update_two_launches", request.param)
    yield request.param
    _lib.set_option("update_two_launches", before)


@pytest.mark.parametrize("two_launches", [0, 1], indirect=True)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_constant_lengths_equal_mp_bits(dtype, two_launches):
    from dlrm_jl_b200.embedding import JaggedIndices, _as_index_tensor
    rng = np.random.default_rng(13)
    B, D, lr = 512, 128, 0.05
    rows = [int(r) for r in rng.integers(1000, 200000, size=len(MLPERF_P))]
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, MLPERF_P)]
    packed = _as_index_tensor(idx, len(rows), _dev())
    jag = JaggedIndices.from_dense(packed)
    a = _tables(rows, D, B * max(MLPERF_P), dtype)
    b = _tables(rows, D, B * max(MLPERF_P), dtype)
    S = 1 + len(rows)
    oa = torch.zeros((B, S, D), device=_dev())
    ob = torch.zeros((B, S, D), device=_dev())
    for step in range(2):
        a.lookup(packed, oa, 1, sort=True)
        b.lookup(jag, ob, 1, sort=True)
        assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), step
        if step == 0:
            for k in (0, 2, 20, 21):
                for x, y in zip(a.sort_dedup_export(k, B * MLPERF_P[k]), b.sort_dedup_export(k, B * MLPERF_P[k])):
                    assert np.array_equal(x, y), k
        dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
        a.update_sorted(dT, 1, lr)
        b.update_sorted(dT, 1, lr)
    torch.cuda.synchronize()
    for k in range(len(rows)):
        assert np.array_equal(a.download(k).view(np.uint32), b.download(k).view(np.uint32)), k


@pytest.mark.parametrize("pooling,zipf,dtype,steps", [("sum", 1.05, torch.float32, 1), ("mean", 1.05, torch.float32, 3),
                                                      ("sum", 1.2, torch.float32, 2), ("mean", 1.2, torch.bfloat16, 2),
                                                      ("sum", 1.2, torch.bfloat16, 1)])
def test_variable_lengths_against_oracle(pooling, zipf, dtype, steps):
    rng = np.random.default_rng(int(zipf * 100) + steps)
    B, D, lr = 256, 64, 0.1
    P = MLPERF_P[:12] + [100, 27]
    rows = [int(r) for r in rng.integers(50, 50000, size=len(P))]
    t = _tables(rows, D, B * 2 * max(P), dtype)
    S = 1 + len(rows)
    ref = [t.download(k) for k in range(len(rows))]
    for step in range(steps):
        lengths = [rng.integers(1, 2 * p, size=B) for p in P]
        vals = _batch(rng, rows, lengths, zipf=zipf)
        j = _jag(vals, lengths, pooling)
        out = torch.zeros((B, S, D), device=_dev())
        t.lookup(j, out, 1, sort=True)
        offs = j.offsets.cpu().numpy()
        assert np.array_equal(out.cpu().numpy()[:, 1:], J.lookup_jagged(ref, vals, offs, B, pooling, 1)[:, 1:]), step
        dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
        t.update_sorted(dT, 1, lr)
        dTn = dT.cpu().numpy()
        o = 0
        for k in range(len(rows)):
            L = int(np.sum(lengths[k]))
            J.sparse_sgd_update_jagged(ref[k], vals[o:o + L], offs[k * B:(k + 1) * B + 1] - o,
                                       np.ascontiguousarray(dTn[:, 1 + k]), lr, pooling, dtype == torch.bfloat16)
            o += L
        for k in range(len(rows)):
            got = t.download(k)
            assert O.rel_err(got, ref[k]) < (2e-3 if dtype == torch.bfloat16 else 1e-5), (step, k)
            ref[k] = got                               # the next step starts from the kernels' tables


# Mean weights in every update instance: VEC = 1 (D = 10), and 1 / 2 / 4 / 8 chunks per lane (D = 64 / 256 / 512 /
# 1024), in both fix-up paths.
@pytest.mark.parametrize("two_launches", [0, 1], indirect=True)
@pytest.mark.parametrize("D", [10, 64, 256, 512, 1024])
def test_mean_update_every_width(D, two_launches):
    rng = np.random.default_rng(D)
    B, lr = 128, 0.1
    rows = [300, 40, 5000]
    P = [3, 1, 12]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.2)
    j = _jag(vals, lengths, "mean")
    t = _tables(rows, D, 2 * B * max(P))
    ref = [t.download(k) for k in range(len(rows))]
    S = 1 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    t.sort(j)
    t.update_sorted(dT, 1, lr)
    dTn, offs, o = dT.cpu().numpy(), j.offsets.cpu().numpy(), 0
    for k in range(len(rows)):
        L = int(np.sum(lengths[k]))
        J.sparse_sgd_update_jagged(ref[k], vals[o:o + L], offs[k * B:(k + 1) * B + 1] - o,
                                   np.ascontiguousarray(dTn[:, 1 + k]), lr, "mean")
        o += L
        assert O.rel_err(t.download(k), ref[k]) < 1e-5, k


@pytest.mark.parametrize("jagged_last", [True, False])
def test_update_consumes_the_last_sort(jagged_last):
    rng = np.random.default_rng(17)
    B, D, P, lr = 64, 32, 3, 0.2
    rows = [500, 40, 3000]
    idx = np.stack([rng.integers(0, r, size=(B, P)) for r in rows])
    u = torch.from_numpy(idx).to(_dev())
    lengths = [rng.integers(0, 6, size=B) for _ in rows]
    vals = _batch(rng, rows, lengths)
    j = _jag(vals, lengths, "mean")
    t = _tables(rows, D, 6 * B)
    ref = [t.download(k) for k in range(len(rows))]
    dT = torch.from_numpy(rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)).to(_dev())
    if jagged_last:
        t.sort(u)
        t.sort(j)
    else:
        t.sort(j)
        t.sort(u)
    t.update_sorted(dT, 1, lr)
    dTn, offs = dT.cpu().numpy(), j.offsets.cpu().numpy()
    o = 0
    for k in range(len(rows)):
        L = int(np.sum(lengths[k]))
        g = np.ascontiguousarray(dTn[:, 1 + k])
        if jagged_last:
            J.sparse_sgd_update_jagged(ref[k], vals[o:o + L], offs[k * B:(k + 1) * B + 1] - o, g, lr, "mean")
        else:
            O.sparse_sgd_update(ref[k], idx[k], g, lr)
        o += L
        assert O.rel_err(t.download(k), ref[k]) < 1e-5, k


def test_graph_capture_replays_the_eager_bits():
    rng = np.random.default_rng(19)
    B, D, lr = 128, 64, 0.1
    P = [1, 3, 20, 100]
    rows = [1000, 20000, 5000, 300000]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.05)
    j = _jag(vals, lengths, "mean", torch.int32)
    S = 1 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    eager, graphed = _tables(rows, D, 2 * B * max(P)), _tables(rows, D, 2 * B * max(P))
    oe = torch.zeros((B, S, D), device=_dev())
    og = torch.zeros((B, S, D), device=_dev())
    for _ in range(2):
        eager.lookup(j, oe, 1, sort=True)
        eager.update_sorted(dT, 1, lr)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.lookup(j, og, 1, sort=True)       # warm-up outside the capture (one step)
        graphed.update_sorted(dT, 1, lr)
        torch.cuda.current_stream().synchronize()
        with torch.cuda.graph(graph, stream=s):
            graphed.lookup(j, og, 1, sort=True)
            graphed.update_sorted(dT, 1, lr)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(oe.view(torch.int32), og.view(torch.int32))
    for k in range(len(rows)):
        assert np.array_equal(eager.download(k).view(np.uint32), graphed.download(k).view(np.uint32)), k


@pytest.mark.parametrize("pooling", ["sum", "mean"])
def test_training_step_presorted_and_side_stream(pooling):
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.model import dlrm
    from dlrm_jl_b200.train import LossWrapper, bce_loss, train_step

    class SideStreamSort(LossWrapper):     # drops the lookup's sort so that train_step sorts on its side stream
        def __call__(self, *a, **kw):
            loss, T = super().__call__(*a, **kw)
            T.presorted = False
            return loss, T

    rng = np.random.default_rng(23)
    B, D = 128, 16
    rows = [100, 3000, 20, 5000]
    P = [1, 4, 2, 12]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.2)
    j = _jag(vals, lengths, pooling)
    dense = torch.from_numpy(rng.standard_normal((B, 13)).astype(np.float32)).to(_dev())
    labels = torch.from_numpy(rng.integers(0, 2, size=B).astype(np.float32)).to(_dev())
    results = []
    for wrapper in (LossWrapper(bce_loss), SideStreamSort(bce_loss)):
        model = dlrm([13, 32, D], [64, 1], D, rows, max_lookups=2 * B * max(P), device=0)
        before = [model.embeddings.download(k) for k in range(len(rows))]
        grads = {}
        orig = model.embeddings.update_sorted

        def spy(dT, slot0, lr, _orig=orig):
            grads["dT"], grads["slot0"] = dT.detach().cpu().numpy(), slot0
            _orig(dT, slot0, lr)
        model.embeddings.update_sorted = spy
        train_step(wrapper, model, Descent(0.1), labels, dense, j)
        torch.cuda.synchronize()
        after = [model.embeddings.download(k) for k in range(len(rows))]
        offs, o = j.offsets.cpu().numpy(), 0
        for k in range(len(rows)):
            L = int(np.sum(lengths[k]))
            ref = before[k].copy()
            J.sparse_sgd_update_jagged(ref, vals[o:o + L], offs[k * B:(k + 1) * B + 1] - o,
                                       np.ascontiguousarray(grads["dT"][:, grads["slot0"] + k]), 0.1, pooling)
            o += L
            assert O.rel_err(after[k], ref) < 1e-4, k
        results.append(after)
    for x, y in zip(*results):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_check_indices_jagged():
    from dlrm_jl_b200 import DLRMB200Error, _lib
    from dlrm_jl_b200.embedding import JaggedIndices
    rows = [10, 20]
    t = _tables(rows, 8, 64)
    j = JaggedIndices.from_lengths(np.array([1, 2, 3, 4, 5, 6]), [[2, 0, 1], [0, 3, 0]])
    for where in ("cpu", "cuda"):
        t.check_indices(j.to(where))
        bad = JaggedIndices(j.values.clone(), j.offsets.clone(), j.L, j.B)
        bad.values[4] = 20                                 # table 1, bag 1, position 1 of its values
        with pytest.raises(DLRMB200Error, match=r"DLRMB_EOOB.*table 1, bag 1, position 1 .*value 20"):
            t.check_indices(bad.to(where))
        off = j.offsets.clone()
        off[0] = 1
        with pytest.raises(DLRMB200Error, match=r"DLRMB_EINVAL.*offsets\[0\] = 1"):
            t.check_indices(JaggedIndices(j.values, off, j.L, j.B).to(where))
        off = j.offsets.clone()
        off[2] = 1                                          # offsets[1] = 2 > offsets[2] = 1
        with pytest.raises(DLRMB200Error, match=r"DLRMB_EINVAL.*decrease at table 0, bag 1"):
            t.check_indices(JaggedIndices(j.values, off, j.L, j.B).to(where))
        with pytest.raises(DLRMB200Error, match=r"DLRMB_EINVAL.*table 0: offsets give 3 lookups, L\[0\] = 2"):
            t.check_indices(JaggedIndices(j.values, j.offsets, (2, 4), j.B).to(where))
    with pytest.raises(DLRMB200Error, match="L\\[1\\] = 65 exceeds max_lookups = 64"):
        t.sort(JaggedIndices.from_lengths(np.zeros(66, np.int64), [[1], [65]]).to(_dev()))
    assert _lib.EOOB == 4
