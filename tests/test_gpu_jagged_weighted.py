"""Weighted jagged bags (per-sample weights) on the GPU: weighted lookup, weighted sort and update, and the weight
gradient against the NumPy reference (tests/jagged_weighted_oracle.py), against torch's per_sample_weights.grad and
against the unweighted jagged path for unit weights."""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests import jagged_oracle as J
from tests import jagged_weighted_oracle as W

pytestmark = pytest.mark.gpu

MLPERF_P = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _dev():
    return torch.device("cuda", 0)


def _tables(rows, D, max_lookups, dtype=torch.float32, seed=7):
    from dlrm_jl_b200.embedding import EmbeddingTables
    t = EmbeddingTables(rows, D, max_lookups, _dev(), dtype)
    t.init_uniform(seed)
    return t


def _weights(rng, n):
    """Random weights with zeros, negative zeros, negative values and values that are not powers of two."""
    w = (rng.standard_normal(n) * 1.7).astype(np.float32)
    if n >= 8:
        w[rng.choice(n, size=max(1, n // 50), replace=False)] = 0.0
        w[rng.choice(n, size=max(1, n // 50), replace=False)] = -0.0
        w[:4] = [0.1, -3.0, 0.0, -0.0]
    return w


def _jag(values, lengths, weights=None, dtype=torch.int64, base=0, pooling="sum"):
    from dlrm_jl_b200.embedding import JaggedIndices
    v = torch.as_tensor(np.asarray(values, dtype=np.int64) + base).to(dtype)
    return JaggedIndices.from_lengths(v, lengths, pooling, weights).to(_dev())


def _batch(rng, rows, lengths, zipf=None):
    vals = []
    for r, n in zip(rows, lengths):
        tot = int(np.sum(n))
        vals.append(rng.integers(0, r, size=tot) if zipf is None else (rng.zipf(zipf, size=tot) - 1) % r)
    return np.concatenate(vals).astype(np.int64)


def _oracle_update(ref, vals, offs, w, dTn, B, lengths, lr, slot0=1, bf16=False):
    o = 0
    for k in range(len(ref)):
        L = int(np.sum(lengths[k]))
        W.sparse_sgd_update_jagged_weighted(ref[k], vals[o:o + L], offs[k * B:(k + 1) * B + 1] - o, w[o:o + L],
                                            np.ascontiguousarray(dTn[:, slot0 + k]), lr, bf16)
        o += L


@pytest.fixture
def two_launches(request):
    """Force the update's separate fix-up launch (the path of batches above 2^18 entries) when the parameter is 1."""
    from dlrm_jl_b200 import _lib
    before = _lib.get_option("update_two_launches")
    _lib.set_option("update_two_launches", request.param)
    yield request.param
    _lib.set_option("update_two_launches", before)


def _lookup_shapes(rng, B):
    rows = [50, 3000, 7, 100000]
    n0 = rng.integers(0, 6, size=B)
    n0[:3] = 0                                         # empty bags
    n1 = np.zeros(B, np.int64)                         # a table without lookups
    n2 = np.ones(B, np.int64)                          # bags of length 1
    n3 = rng.integers(0, 9, size=B)
    n3[5] = 4500                                       # one bag longer than 4096
    return rows, [n0, n1, n2, n3]


@pytest.mark.parametrize("D,dtype,itype,base", [
    (64, dt, it, b) for dt in (torch.float32, torch.bfloat16) for it in (torch.int32, torch.int64) for b in (0, 1)] + [
    (D, dt, torch.int64, 0) for D in (4, 10, 128) for dt in (torch.float32, torch.bfloat16)])
def test_lookup_bit_exact(D, dtype, itype, base):
    rng = np.random.default_rng(100 + D + base)
    B = 96
    rows, lengths = _lookup_shapes(rng, B)
    t = _tables(rows, D, 6000, dtype)
    vals = _batch(rng, rows, lengths)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w, itype, base)
    out = torch.full((B, 2 + len(rows), D), float("nan"), device=_dev())
    out[:, :2] = 0
    t.lookup(j, out, 2, idx_base=base)
    stored = [t.download(k) for k in range(len(rows))]
    ref = W.lookup_jagged_weighted(stored, vals, j.offsets.cpu().numpy(), w, B, slot0=2)
    got = out.cpu().numpy()
    assert np.array_equal(got[:, 2:].view(np.uint32), ref[:, 2:].view(np.uint32))
    assert np.all(got[:, :2] == 0)


@pytest.mark.parametrize("two_launches", [0, 1], indirect=True)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_unit_weights_give_the_unweighted_bits(dtype, two_launches):
    rng = np.random.default_rng(211)
    B, D, lr = 256, 128, 0.05
    P = MLPERF_P
    rows = [int(r) for r in rng.integers(1000, 200000, size=len(P))]
    a = _tables(rows, D, 2 * B * max(P), dtype)
    b = _tables(rows, D, 2 * B * max(P), dtype)
    S = 1 + len(rows)
    oa = torch.zeros((B, S, D), device=_dev())
    ob = torch.zeros((B, S, D), device=_dev())
    for step in range(2):
        lengths = [rng.integers(0, 2 * p, size=B) for p in P]
        vals = _batch(rng, rows, lengths, zipf=1.1)
        plain = _jag(vals, lengths)
        ones = _jag(vals, lengths, np.ones(len(vals), np.float32))
        a.lookup(plain, oa, 1, sort=True)
        b.lookup(ones, ob, 1, sort=True)
        assert torch.equal(oa.view(torch.int32), ob.view(torch.int32)), step
        if step == 0:
            for k in (0, 2, 20, 21):
                L = int(np.sum(lengths[k]))
                for x, y in zip(a.sort_dedup_export(k, L), b.sort_dedup_export(k, L)):
                    assert np.array_equal(x, y), k
        dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
        a.update_sorted(dT, 1, lr)
        b.update_sorted(dT, 1, lr)
    torch.cuda.synchronize()
    for k in range(len(rows)):
        assert np.array_equal(a.download(k).view(np.uint32), b.download(k).view(np.uint32)), k


# Weights in every SCALE update instance: VEC = 1 (D = 10), and 1 / 2 / 4 / 8 chunks per lane (D = 64 / 256 / 512 /
# 1024), in both fix-up paths.
@pytest.mark.parametrize("two_launches", [0, 1], indirect=True)
@pytest.mark.parametrize("D", [10, 64, 256, 512, 1024])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_weighted_update_every_width(dtype, D, two_launches):
    rng = np.random.default_rng(D + 7)
    B, lr = 128, 0.1
    rows = [300, 40, 5000]
    P = [3, 1, 12]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.2)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w)
    t = _tables(rows, D, 2 * B * max(P), dtype)
    ref = [t.download(k) for k in range(len(rows))]
    S = 1 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    t.sort(j)
    t.update_sorted(dT, 1, lr)
    _oracle_update(ref, vals, j.offsets.cpu().numpy(), w, dT.cpu().numpy(), B, lengths, lr,
                   bf16=dtype == torch.bfloat16)
    for k in range(len(rows)):
        assert O.rel_err(t.download(k), ref[k]) < (2e-3 if dtype == torch.bfloat16 else 1e-5), k


# Every sort regime: 256-thread CTAs up to 1024 / 2048 / 4096 keys, 1024-thread CTAs up to 8192 / 16384, radix above;
# every call also carries a table without lookups.  The export, then the update against the reference.
@pytest.mark.parametrize("Lmax", [1000, 2000, 4000, 8000, 16000, 40000])
def test_sort_regimes_and_update(Lmax):
    rng = np.random.default_rng(Lmax + 1)
    B, D, lr = 8, 16, 0.3
    rows = [900, 2_000_000, 77]
    Ls = [Lmax // 3, Lmax, 0]
    lengths = []
    for L in Ls:
        cut = np.sort(rng.integers(0, L + 1, size=B - 1))
        lengths.append(np.diff(np.concatenate([[0], cut, [L]])))
    t = _tables(rows, D, max(Ls))
    ref = [t.download(k) for k in range(len(rows))]
    vals = _batch(rng, rows, lengths, zipf=1.2)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w, torch.int32)
    t.sort(j)
    o = 0
    for k, L in enumerate(Ls):
        uniq, seg, perm = t.sort_dedup_export(k, L)
        ru, rs, rp = O.sort_dedup(vals[o:o + L])
        assert np.array_equal(uniq, ru) and np.array_equal(seg, rs) and np.array_equal(perm, rp), k
        o += L
    S = 1 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    t.update_sorted(dT, 1, lr)
    _oracle_update(ref, vals, j.offsets.cpu().numpy(), w, dT.cpu().numpy(), B, lengths, lr)
    for k in range(len(rows)):
        assert O.rel_err(t.download(k), ref[k]) < 1e-5, k


@pytest.mark.parametrize("D,dtype,itype,base", [
    (D, dt, torch.int64, 0) for D in (4, 10, 64, 128) for dt in (torch.float32, torch.bfloat16)] + [
    (64, torch.float32, torch.int32, 1), (10, torch.bfloat16, torch.int32, 0), (256, torch.float32, torch.int64, 1)])
def test_weight_grad_bit_exact_and_against_torch(D, dtype, itype, base):
    rng = np.random.default_rng(300 + D)
    B = 96
    rows, lengths = _lookup_shapes(rng, B)
    t = _tables(rows, D, 6000, dtype)
    vals = _batch(rng, rows, lengths)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w, itype, base)
    S = 3 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    dw = t.weight_grad(j, dT, 2, idx_base=base)
    dw2 = t.weight_grad(j, dT, 2, idx_base=base)
    torch.cuda.synchronize()
    got = dw.cpu().numpy()
    assert np.array_equal(got.view(np.uint32), dw2.cpu().numpy().view(np.uint32))     # same bits call to call
    stored = [t.download(k) for k in range(len(rows))]
    offs = j.offsets.cpu().numpy()
    dTn = dT.cpu().numpy()
    ref = W.weight_grad_jagged(stored, vals, offs, dTn, B, slot0=2)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    # torch's per_sample_weights.grad in float64, table by table: within the rounding of a D-term f32 sum
    o = 0
    for k in range(len(rows)):
        L = int(np.sum(lengths[k]))
        if L == 0:
            continue
        tab = torch.from_numpy(stored[k].astype(np.float64))
        wk = torch.from_numpy(w[o:o + L].astype(np.float64)).requires_grad_(True)
        out = torch.nn.functional.embedding_bag(torch.from_numpy(vals[o:o + L]), tab,
                                                torch.from_numpy(offs[k * B:(k + 1) * B] - o), mode="sum",
                                                per_sample_weights=wk)
        g = torch.from_numpy(dTn[:, 2 + k].astype(np.float64))
        out.backward(g)
        bag = np.repeat(np.arange(B), lengths[k])
        bound = D * np.finfo(np.float32).eps * np.einsum("jd,jd->j", np.abs(dTn[bag, 2 + k]).astype(np.float64),
                                                          np.abs(stored[k][vals[o:o + L]]).astype(np.float64))
        assert np.all(np.abs(got[o:o + L] - wk.grad.numpy()) <= bound + 1e-30), k
        o += L


def test_weight_grad_reads_the_pre_update_rows():
    rng = np.random.default_rng(401)
    B, D, lr = 128, 64, 0.5
    rows = [200, 30, 4000]
    P = [4, 2, 9]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.2)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w)
    t = _tables(rows, D, 2 * B * max(P))
    before = [t.download(k) for k in range(len(rows))]
    S = 1 + len(rows)
    out = torch.zeros((B, S, D), device=_dev())
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    t.lookup(j, out, 1, sort=True)
    dw = t.weight_grad(j, dT, 1)
    t.update_sorted(dT, 1, lr)
    torch.cuda.synchronize()
    offs = j.offsets.cpu().numpy()
    ref = W.weight_grad_jagged(before, vals, offs, dT.cpu().numpy(), B, slot0=1)
    assert np.array_equal(dw.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    after = [t.download(k) for k in range(len(rows))]
    assert any(not np.array_equal(x, y) for x, y in zip(before, after))     # the update did move rows
    _oracle_update(before, vals, offs, w, dT.cpu().numpy(), B, lengths, lr)
    for k in range(len(rows)):
        assert O.rel_err(after[k], before[k]) < 1e-5, k


@pytest.mark.parametrize("weighted_last", [True, False])
def test_update_consumes_the_last_sort(weighted_last):
    rng = np.random.default_rng(17)
    B, D, lr = 64, 32, 0.2
    rows = [500, 40, 3000]
    lengths = [rng.integers(0, 6, size=B) for _ in rows]
    vals = _batch(rng, rows, lengths)
    w = _weights(rng, len(vals))
    jw = _jag(vals, lengths, w)
    lengths2 = [rng.integers(0, 6, size=B) for _ in rows]
    vals2 = _batch(rng, rows, lengths2)
    ju = _jag(vals2, lengths2, pooling="mean")
    t = _tables(rows, D, 6 * B)
    ref = [t.download(k) for k in range(len(rows))]
    dT = torch.from_numpy(rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)).to(_dev())
    if weighted_last:
        t.sort(ju)
        t.sort(jw)
    else:
        t.sort(jw)
        t.sort(ju)
    t.update_sorted(dT, 1, lr)
    dTn = dT.cpu().numpy()
    if weighted_last:
        _oracle_update(ref, vals, jw.offsets.cpu().numpy(), w, dTn, B, lengths, lr)
    else:
        offs, o = ju.offsets.cpu().numpy(), 0
        for k in range(len(rows)):
            L = int(np.sum(lengths2[k]))
            J.sparse_sgd_update_jagged(ref[k], vals2[o:o + L], offs[k * B:(k + 1) * B + 1] - o,
                                       np.ascontiguousarray(dTn[:, 1 + k]), lr, "mean")
            o += L
    for k in range(len(rows)):
        assert O.rel_err(t.download(k), ref[k]) < 1e-5, k


def test_graph_capture_replays_the_eager_bits():
    rng = np.random.default_rng(19)
    B, D, lr = 128, 64, 0.1
    P = [1, 3, 20, 100]
    rows = [1000, 20000, 5000, 300000]
    lengths = [rng.integers(0, 2 * p, size=B) for p in P]
    vals = _batch(rng, rows, lengths, zipf=1.05)
    j = _jag(vals, lengths, _weights(rng, len(vals)), torch.int32)
    S = 1 + len(rows)
    dT = torch.from_numpy(rng.standard_normal((B, S, D)).astype(np.float32)).to(_dev())
    eager, graphed = _tables(rows, D, 2 * B * max(P)), _tables(rows, D, 2 * B * max(P))
    oe = torch.zeros((B, S, D), device=_dev())
    og = torch.zeros((B, S, D), device=_dev())
    dwe = []
    for _ in range(2):
        eager.lookup(j, oe, 1, sort=True)
        dwe.append(eager.weight_grad(j, dT, 1))
        eager.update_sorted(dT, 1, lr)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.lookup(j, og, 1, sort=True)       # warm-up outside the capture (one step)
        graphed.weight_grad(j, dT, 1)
        graphed.update_sorted(dT, 1, lr)
        torch.cuda.current_stream().synchronize()
        with torch.cuda.graph(graph, stream=s):
            graphed.lookup(j, og, 1, sort=True)
            dwg = graphed.weight_grad(j, dT, 1)
            graphed.update_sorted(dT, 1, lr)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(oe.view(torch.int32), og.view(torch.int32))
    assert torch.equal(dwe[1].view(torch.int32), dwg.view(torch.int32))
    for k in range(len(rows)):
        assert np.array_equal(eager.download(k).view(np.uint32), graphed.download(k).view(np.uint32)), k


def test_training_step_presorted_and_side_stream():
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
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w)
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
        ref = [x.copy() for x in before]
        _oracle_update(ref, vals, j.offsets.cpu().numpy(), w, grads["dT"], B, lengths, 0.1, slot0=grads["slot0"])
        for k in range(len(rows)):
            assert O.rel_err(after[k], ref[k]) < 1e-4, k
        results.append(after)
    for x, y in zip(*results):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_update_rebuilds_a_weighted_batch_from_the_updates():
    from dlrm_jl_b200.embedding import Descent, sparse_updates, update_
    rng = np.random.default_rng(29)
    B, D, lr = 64, 32, 0.2
    rows = [500, 40, 3000]
    lengths = [rng.integers(0, 6, size=B) for _ in rows]
    vals = _batch(rng, rows, lengths)
    w = _weights(rng, len(vals))
    j = _jag(vals, lengths, w)
    t = _tables(rows, D, 6 * B)
    ref = [t.download(k) for k in range(len(rows))]
    dT = torch.from_numpy(rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)).to(_dev())
    update_(Descent(lr), t, sparse_updates(dT, j, 1))       # not presorted: update_ sorts the rebuilt batch
    _oracle_update(ref, vals, j.offsets.cpu().numpy(), w, dT.cpu().numpy(), B, lengths, lr)
    for k in range(len(rows)):
        assert O.rel_err(t.download(k), ref[k]) < 1e-5, k


def test_check_indices_serves_weighted_batches():
    from dlrm_jl_b200 import DLRMB200Error
    from dlrm_jl_b200.embedding import JaggedIndices
    t = _tables([10, 20], 8, 64)
    j = JaggedIndices.from_lengths(np.array([1, 2, 3, 4, 5, 6]), [[2, 0, 1], [0, 3, 0]], weights=np.ones(6))
    for where in ("cpu", "cuda"):
        t.check_indices(j.to(where))
        bad = JaggedIndices(j.values.clone(), j.offsets.clone(), j.L, j.B, "sum", j.weights.clone())
        bad.values[4] = 20
        with pytest.raises(DLRMB200Error, match=r"DLRMB_EOOB.*table 1, bag 1, position 1 .*value 20"):
            t.check_indices(bad.to(where))
