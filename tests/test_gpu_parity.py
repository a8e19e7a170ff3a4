"""Parity of the sm_100a kernels (through the C ABI) against the CPU oracle and the goldens.

Tolerances (BASELINE.json north_star): bit-exact for index sort / dedup / segment offsets and
for the lookup (pure copies and ordered fp32 adds); rel 1e-5 (2-norm) for the interaction
forward/backward; rel 1e-4 for tables after N SGD steps.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from tests.helpers import golden_model, golden_updates, load_golden, load_known_answer

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

FWD_RTOL = 1e-5
SGD_RTOL = 1e-4


def _dev():
    return torch.device("cuda", 0)


def _tables(arrays, max_lookups):
    from dlrm_jl_b200.embedding import EmbeddingTables
    return EmbeddingTables.from_arrays(arrays, max_lookups, 0)


def _rand_tables(rng, rows, D):
    return [rng.standard_normal((r, D)).astype(np.float32) for r in rows]


# ------------------------------------------------------------------------------------------------
# lookup
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["single", "multi"])
def test_lookup_golden_concatenated_result(name):
    from dlrm_jl_b200.embedding import PreallocationStrategy, maplookup
    g = load_golden(name)
    _bot, _top, tables, _dense, idx, _labels = golden_model(g)
    t = _tables(tables, idx[0].size)
    T = maplookup(PreallocationStrategy(16), t, idx).cpu().numpy()
    ref = O.lookup(tables, idx, slot0=1)
    assert np.array_equal(T, ref)                                    # bit-exact vs oracle
    assert np.all(T[:, 0] == 0)                                      # slot 0 reserved for x
    assert O.rel_err(T[:, 1:], g["concatenated_result"][:, 1:]) < FWD_RTOL   # vs PyTorch golden


@pytest.mark.parametrize("D", [4, 10, 16, 48, 64, 128, 256])
@pytest.mark.parametrize("P", [1, 3, 10])
def test_lookup_random_bit_exact(D, P):
    from dlrm_jl_b200.embedding import PreallocationStrategy, maplookup
    rng = np.random.default_rng(D * 100 + P)
    rows = [7, 1000, 33, 5000]
    tables = _rand_tables(rng, rows, D)
    for B, dtype, base in [(1, np.int64, 0), (3, np.int32, 1), (257, np.int64, 1), (1024, np.int32, 0)]:
        idx = [rng.integers(0, r, size=(B, P)) for r in rows]
        t = _tables(tables, B * P)
        dev_idx = np.stack(idx).astype(dtype) + base
        T = maplookup(PreallocationStrategy(D), t, dev_idx, idx_base=base).cpu().numpy()
        assert np.array_equal(T, O.lookup(tables, idx, slot0=1)), (B, dtype, base)
        t.close()


def test_lookup_default_strategy_and_identity_rows():
    from dlrm_jl_b200.embedding import DefaultStrategy, maplookup
    rng = np.random.default_rng(5)
    tables = _rand_tables(rng, [64, 64], 32)
    idx = [np.arange(64), np.arange(64)[::-1].copy()]
    t = _tables(tables, 64)
    ys = maplookup(DefaultStrategy(), t, idx)
    assert len(ys) == 2
    assert np.array_equal(ys[0].cpu().numpy(), tables[0])
    assert np.array_equal(ys[1].cpu().numpy(), tables[1][::-1])


def test_lookup_host_entry_point():
    import ctypes as C
    from dlrm_jl_b200 import _lib
    rng = np.random.default_rng(6)
    tables = _rand_tables(rng, [100, 50, 9], 64)
    t = _tables(tables, 40)
    idx = [rng.integers(0, r, size=(20, 2)) for r in [100, 50, 9]]
    flat = np.ascontiguousarray(np.stack(idx).astype(np.int64) + 1)   # Julia-style 1-based Int64
    out = np.zeros((20, 4, 64), dtype=np.float32)
    out[:, 0] = 7.0
    _lib.check(_lib.load().dlrmb_embedding_fwd_host(
        t._h, flat.ctypes.data_as(C.c_void_p), 8, 1, 20, 2, out.ctypes.data_as(C.c_void_p), 4, 1))
    ref = O.lookup(tables, idx, slot0=1)
    assert np.array_equal(out[:, 1:], ref[:, 1:])
    assert np.all(out[:, 0] == 7.0)


def test_index_range_check_reports_offender():
    from dlrm_jl_b200 import DLRMB200Error
    t = _tables([np.zeros((10, 8), np.float32), np.zeros((5, 8), np.float32)], 16)
    good = torch.tensor([[0, 9, 3], [4, 0, 1]], dtype=torch.int64, device=_dev()).unsqueeze(-1)
    t.check_indices(good)
    bad = good.clone()
    bad[1, 2, 0] = 5
    with pytest.raises(DLRMB200Error, match="table 1"):
        t.check_indices(bad)


def test_errors_are_loud():
    from dlrm_jl_b200 import DLRMB200Error
    from dlrm_jl_b200.embedding import EmbeddingTables
    with pytest.raises(DLRMB200Error):
        EmbeddingTables([10], 2000, 16, 0)               # unsupported D
    t = EmbeddingTables([10], 8, 16, 0)
    idx = torch.zeros((1, 32, 1), dtype=torch.int64, device=_dev())
    out = torch.zeros((32, 1, 8), device=_dev())
    with pytest.raises(DLRMB200Error, match="max_lookups"):
        t.lookup(idx, out, 0)
    with pytest.raises(DLRMB200Error, match="without a preceding"):
        t.update_sorted(out[:16].contiguous(), 0, 0.1)


# ------------------------------------------------------------------------------------------------
# interaction
# ------------------------------------------------------------------------------------------------
SHAPES = [  # (B, F, d)
    (4, 4, 4),        # known-answer geometry (test/model/model.jl)
    (128, 8, 16),     # golden geometry
    (300, 27, 64),    # Kaggle-shaped, ragged batch
    (64, 27, 128),    # Terabyte-shaped
    (130, 11, 128),   # reference test: x 128 wide, 10 ys (test/model/interact.jl:166)
    (33, 21, 256),    # reference test: implementation 2, 256 wide, 20 ys (:244)
    (10, 6, 10),      # d not a multiple of 4 -> generic path (:196)
    (5, 1, 16),       # no pairs
    (7, 2, 8),
    (1, 100, 128),    # process_slice! test geometry (:149)
]


@pytest.mark.parametrize("B,F,d", SHAPES)
def test_interaction_forward_vs_oracle(B, F, d):
    from dlrm_jl_b200.interact import interaction_fwd
    rng = np.random.default_rng(B * 1000 + F * 10 + d)
    T = rng.standard_normal((B, F, d)).astype(np.float32)
    ref = O.interaction_fwd(T)
    out = interaction_fwd(torch.from_numpy(T).to(_dev())).cpu().numpy()
    assert out.shape == ref.shape
    assert np.array_equal(out[:, :d], T[:, 0])
    assert O.rel_err(out, ref) < FWD_RTOL
    # x handed separately: slot 0 of T is filled by the kernel (fused fast_vcat)
    Tz = T.copy()
    Tz[:, 0] = 0
    Td = torch.from_numpy(Tz).to(_dev())
    out2 = interaction_fwd(Td, torch.from_numpy(T[:, 0].copy()).to(_dev())).cpu().numpy()
    assert np.array_equal(out2, out)
    assert np.array_equal(Td.cpu().numpy(), T)


def test_interaction_forward_integer_exact_and_padding():
    from dlrm_jl_b200.interact import interaction_fwd
    rng = np.random.default_rng(11)
    T = rng.integers(-4, 5, size=(50, 27, 64)).astype(np.float32)     # integer Gram is exact in fp32
    for pad in (1, 8, 64):
        ref = O.interaction_fwd(T, pad)
        out = interaction_fwd(torch.from_numpy(T).to(_dev()), pad_to_mul=pad).cpu().numpy()
        assert out.shape == ref.shape and out.shape[1] % pad == 0
        assert np.array_equal(out, ref)


@pytest.mark.parametrize("name", ["single", "multi"])
def test_interaction_forward_golden(name):
    from dlrm_jl_b200.interact import interaction_fwd
    g = load_golden(name)
    out = interaction_fwd(torch.from_numpy(g["concatenated_result"]).to(_dev())).cpu().numpy()
    assert O.rel_err(out, g["output_interaction"]) < FWD_RTOL
    assert O.rel_err(out[:, 16:], g["zflat"]) < FWD_RTOL


@pytest.mark.parametrize("B,F,d", SHAPES)
def test_interaction_backward_vs_oracle(B, F, d):
    from dlrm_jl_b200.interact import interaction_bwd, interaction_width
    rng = np.random.default_rng(B * 7 + F * 3 + d)
    T = rng.standard_normal((B, F, d)).astype(np.float32)
    for pad in (1, 16):
        w = interaction_width(F, d, pad)
        g = rng.standard_normal((B, w)).astype(np.float32)
        dx_ref, dT_ref = O.interaction_bwd(g, T, w - d - F * (F - 1) // 2)
        dx, dT = interaction_bwd(torch.from_numpy(g).to(_dev()), torch.from_numpy(T).to(_dev()), pad)
        assert O.rel_err(dT.cpu().numpy(), dT_ref) < FWD_RTOL or F == 1
        assert O.rel_err(dx.cpu().numpy(), dx_ref) < FWD_RTOL
        if F == 1:
            assert np.all(dT.cpu().numpy() == 0)


def test_interaction_autograd_matches_reference_pullback_shape():
    """rrule contract (interact.jl:438-447): returns dx and the whole dT, slot 0 included."""
    from dlrm_jl_b200.interact import DotInteraction
    rng = np.random.default_rng(3)
    B, F, d = 64, 11, 128
    Tn = rng.standard_normal((B, F, d)).astype(np.float32)
    x = torch.from_numpy(Tn[:, 0].copy()).to(_dev()).requires_grad_(True)
    T = torch.from_numpy(Tn).to(_dev()).requires_grad_(True)
    z = DotInteraction()(x, T)
    gn = rng.standard_normal(tuple(z.shape)).astype(np.float32)
    z.backward(torch.from_numpy(gn).to(_dev()))
    dx_ref, dT_ref = O.interaction_bwd(gn, Tn)
    assert O.rel_err(x.grad.cpu().numpy(), dx_ref) < FWD_RTOL
    assert O.rel_err(T.grad.cpu().numpy(), dT_ref) < FWD_RTOL


def test_interaction_host_entry_points():
    import ctypes as C
    from dlrm_jl_b200 import _lib
    rng = np.random.default_rng(8)
    t = _tables([np.zeros((4, 16), np.float32)], 4)
    B, F, d = 37, 8, 16
    T = rng.standard_normal((B, F, d)).astype(np.float32)
    out = np.empty((B, d + 28), dtype=np.float32)
    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(lib.dlrmb_interaction_fwd_host(t._h, p(T), None, B, F, d, 1, p(out)))
    assert O.rel_err(out, O.interaction_fwd(T)) < FWD_RTOL
    g = rng.standard_normal(out.shape).astype(np.float32)
    dT = np.empty_like(T)
    dx = np.empty((B, d), dtype=np.float32)
    _lib.check(lib.dlrmb_interaction_bwd_host(t._h, p(g), p(T), B, F, d, 1, p(dT), p(dx)))
    dx_ref, dT_ref = O.interaction_bwd(g, T)
    assert O.rel_err(dT, dT_ref) < FWD_RTOL and O.rel_err(dx, dx_ref) < FWD_RTOL


WARP_SHAPES = [  # (B, F, d): every compiled warp-per-sample specialisation, ragged batches included
    (2049, 27, 128), (1, 27, 128), (301, 27, 64), (37, 27, 32), (45, 27, 16), (131, 8, 16), (3, 8, 16),
]


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


@pytest.mark.parametrize("B,F,d", WARP_SHAPES)
def test_interaction_warp_kernels_vs_oracle_and_tiled_kernels(B, F, d, lib_options):
    """The warp-per-sample kernels (csrc/interact_warp.cu: tensor-core 3xTF32 forward, FFMA2 backward)
    against the oracle and against the general tiled kernels (csrc/interact.cu) on the same inputs.
    Backward keeps the tiled kernel's summation order, so it must match bit for bit."""
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.interact import interaction_bwd, interaction_fwd, interaction_width
    assert _lib.load().dlrmb_interaction_has_warp_path(F, d) == 1
    rng = np.random.default_rng(B + 31 * F + d)
    T = rng.standard_normal((B, F, d)).astype(np.float32)
    Td = torch.from_numpy(T).to(_dev())
    res = {}
    for path in ("tiled", "warp"):
        lib_options("interact_general", 1 if path == "tiled" else 0)
        outs = []
        for pad in (1, 16):
            w = interaction_width(F, d, pad)
            out = interaction_fwd(Td, pad_to_mul=pad)
            Tz = T.copy()
            Tz[:, 0] = 0
            Tzd = torch.from_numpy(Tz).to(_dev())
            out_x = interaction_fwd(Tzd, torch.from_numpy(T[:, 0].copy()).to(_dev()), pad_to_mul=pad)
            assert torch.equal(out, out_x) and torch.equal(Tzd, Td)
            g = np.random.default_rng(pad).standard_normal((B, w)).astype(np.float32)
            dx, dT = interaction_bwd(torch.from_numpy(g).to(_dev()), Td, pad)
            outs.append((out.cpu().numpy(), dx.cpu().numpy(), dT.cpu().numpy(), g, w, pad))
        res[path] = outs
    for (o_t, dx_t, dT_t, g, w, pad), (o_w, dx_w, dT_w, _, _, _) in zip(res["tiled"], res["warp"]):
        ref = O.interaction_fwd(T, pad)
        assert ref.shape == o_t.shape and O.rel_err(o_t, ref) < FWD_RTOL and np.array_equal(o_t[:, :d], T[:, 0])
        # elementwise: the 3xTF32 tensor-core Gram stays within a few fp32 ulps of the dot products' scale
        scale = np.sqrt(float(d)) * 4.0
        assert np.max(np.abs(o_w - ref)) < 2e-6 * scale * max(1.0, float(np.max(np.abs(T))))
        assert ref.shape == o_w.shape and O.rel_err(o_w, ref) < FWD_RTOL
        assert np.array_equal(o_w[:, :d], T[:, 0])
        assert np.all(o_w[:, d + F * (F - 1) // 2:] == 0)
        assert O.rel_err(o_w, o_t) < FWD_RTOL
        dx_ref, dT_ref = O.interaction_bwd(g, T, w - d - F * (F - 1) // 2)
        assert O.rel_err(dT_w, dT_ref) < FWD_RTOL and O.rel_err(dx_w, dx_ref) < FWD_RTOL
        assert np.array_equal(dT_w, dT_t) and np.array_equal(dx_w, dx_t)


@pytest.mark.parametrize("variant", [0, 2, 3, 5, 6])
@pytest.mark.parametrize("B,F,d", [(2049, 27, 128), (1, 27, 128), (301, 27, 64), (131, 8, 16)])
def test_interaction_backward_register_variants_bit_equal(B, F, d, variant, lib_options):
    """bwd_variant: the one-sample-per-warp backward with FFMA2 at 128 registers (2), with S stored once (3), as a
    streaming kernel -- half of the output rows per pass, T rows through a cp.async ring -- with duplicated S (5) or
    S stored once and row-paired FFMA2 (6), or chosen by batch size (0).  The per-output summation order does not
    depend on it: same bits as the 144-register FFMA2 kernel (1), which is pinned to the oracle here."""
    from dlrm_jl_b200.interact import interaction_bwd, interaction_width
    rng = np.random.default_rng(B + F + d + variant)
    T = torch.from_numpy(rng.standard_normal((B, F, d)).astype(np.float32)).to(_dev())
    g = torch.from_numpy(rng.standard_normal((B, interaction_width(F, d))).astype(np.float32)).to(_dev())
    lib_options("bwd_variant", 1)
    dx0, dT0 = interaction_bwd(g, T)
    lib_options("bwd_variant", variant)
    dx1, dT1 = interaction_bwd(g, T)
    assert torch.equal(dx0, dx1) and torch.equal(dT0, dT1)
    dx_ref, dT_ref = O.interaction_bwd(g.cpu().numpy(), T.cpu().numpy())
    assert O.rel_err(dT1.cpu().numpy(), dT_ref) < FWD_RTOL and O.rel_err(dx1.cpu().numpy(), dx_ref) < FWD_RTOL


@pytest.mark.parametrize("B,F,d", [(2049, 27, 128), (77, 27, 64), (33, 8, 16), (19, 11, 128)])
def test_interaction_backward_scatter_matches_plain_backward(B, F, d, lib_options):
    """dlrmb_interaction_bwd_scatter with every destination in local memory: the rows land at
    base + (sample_offset + b) * stride + offset, bit-identical to the plain backward's dT rows
    (slot 0 is not scattered), for the warp-per-sample and the tiled kernels."""
    from dlrm_jl_b200.interact import DotInteraction, ScatterPlan, interaction_bwd, interaction_width
    rng = np.random.default_rng(B + F)
    T = torch.from_numpy(rng.standard_normal((B, F, d)).astype(np.float32)).to(_dev())
    x = T[:, 0].clone().requires_grad_(True)
    g = torch.from_numpy(rng.standard_normal((B, interaction_width(F, d))).astype(np.float32)).to(_dev())
    sample_offset = 5
    # two "owners": even tables in buffer A [B + 8][nA][d], odd tables in buffer B [B + 8][nB][d]
    owners = [[f for f in range(1, F) if f % 2 == 0], [f for f in range(1, F) if f % 2 == 1]]
    for path in ("tiled", None):
        lib_options("interact_general", 1 if path else 0)
        bufs = [torch.full((B + 8, max(1, len(o)), d), -7.0, device=_dev()) for o in owners]
        dests = torch.zeros((F, 3), dtype=torch.int64)
        for buf, own in zip(bufs, owners):
            for j, f in enumerate(own):
                dests[f, 0] = buf.data_ptr()
                dests[f, 1] = buf.shape[1] * d
                dests[f, 2] = j * d
        plan = ScatterPlan(dests.to(_dev()), sample_offset)
        x.grad = None
        DotInteraction()(x, T.clone(), scatter=plan).backward(g)
        dx_ref, dT_ref = interaction_bwd(g, T)
        assert torch.equal(x.grad, dx_ref)
        for buf, own in zip(bufs, owners):
            for j, f in enumerate(own):
                assert torch.equal(buf[sample_offset:sample_offset + B, j], dT_ref[:, f])
            assert torch.all(buf[:sample_offset] == -7.0) and torch.all(buf[sample_offset + B:] == -7.0)


def test_interaction_warp_path_coverage():
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    for F, d in [(27, 128), (27, 64), (8, 16)]:
        assert lib.dlrmb_interaction_has_warp_path(F, d) == 1
    for F, d in [(11, 128), (21, 256), (6, 10), (100, 128)]:
        assert lib.dlrmb_interaction_has_warp_path(F, d) == 0


# ------------------------------------------------------------------------------------------------
# sort / dedup (bit-exact integers)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L,rows", [(1, 5), (2, 2), (128, 1000), (1280, 1000), (2048, 3), (2048, 10131227),
                                    (4096, 50), (4097, 50), (5000, 100000), (8192, 3), (12000, 40000000), (16384, 1000), (16385, 1000), (70000, 7), (1 << 16, 1 << 20),
                                    (200000, 40000000)])
@pytest.mark.parametrize("dtype,base", [(np.int32, 0), (np.int64, 1)])
def test_sort_dedup_bit_exact(L, rows, dtype, base):
    from dlrm_jl_b200.embedding import EmbeddingTables
    rng = np.random.default_rng(L + rows)
    row_list = [rows, max(2, rows // 3)]
    t = EmbeddingTables(row_list, 4, L, 0)
    idx = np.stack([rng.integers(0, r, size=L) for r in row_list])
    dev = torch.from_numpy((idx + base).astype(dtype)).to(_dev()).reshape(2, L, 1)
    t.sort(dev, base)
    for k in range(2):
        uniq, seg, perm = t.sort_dedup_export(k, L)
        u_ref, s_ref, p_ref = O.sort_dedup(idx[k])
        assert np.array_equal(uniq, u_ref)
        assert np.array_equal(seg, s_ref)
        assert np.array_equal(perm, p_ref)
    t.close()


# ------------------------------------------------------------------------------------------------
# sparse SGD update
# ------------------------------------------------------------------------------------------------
def _run_update(tables_np, idx, dT, slot0, lr, steps=1):
    t = _tables(tables_np, idx[0].size)
    dev_idx = torch.from_numpy(np.stack([i.reshape(i.shape[0], -1) for i in idx])).to(_dev())
    g = torch.from_numpy(dT).to(_dev())
    for _ in range(steps):
        t.bwd_sgd(dev_idx, g, slot0, lr)
    out = [t.download(k) for k in range(len(tables_np))]
    t.close()
    return out


@pytest.mark.parametrize("D", [4, 10, 16, 64, 128, 256])
@pytest.mark.parametrize("B,P,rows", [(128, 1, [1000, 3, 57]), (2048, 1, [3, 10131227 // 1000, 24]),
                                      (128, 10, [1000, 5, 300]), (3000, 3, [4, 100000, 11]),
                                      (5, 1, [2, 2, 2])])
def test_sparse_sgd_vs_oracle(D, B, P, rows):
    rng = np.random.default_rng(D + B + P)
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, P)) for r in rows]
    dT = rng.standard_normal((B, 1 + len(rows), D)).astype(np.float32)
    got = _run_update(tables, idx, dT, 1, 0.1, steps=3)
    ref = [tb.copy() for tb in tables]
    for _ in range(3):
        for k in range(len(rows)):
            O.sparse_sgd_update_fast(ref[k], idx[k], np.ascontiguousarray(dT[:, 1 + k]), 0.1)
    for k in range(len(rows)):
        assert O.rel_err(got[k], ref[k]) < SGD_RTOL, k
        assert not np.array_equal(got[k], tables[k]), "update must change the table"
        untouched = np.setdiff1d(np.arange(rows[k]), np.unique(idx[k]))
        assert np.array_equal(got[k][untouched], tables[k][untouched]), "untouched rows must be bit-identical"


def test_sparse_sgd_is_deterministic_and_matches_ordered_sum():
    rng = np.random.default_rng(42)
    rows, D, B = [3, 17, 5000], 64, 4096 + 123
    tables = _rand_tables(rng, rows, D)
    # Zipf-like skew: a few very hot rows
    idx = [np.minimum((rng.pareto(1.05, size=(B, 1)) * 1.0).astype(np.int64), r - 1) for r in rows]
    dT = rng.standard_normal((B, len(rows), D)).astype(np.float32)
    a = _run_update(tables, idx, dT, 0, 0.5)
    b = _run_update(tables, idx, dT, 0, 0.5)
    for k in range(len(rows)):
        assert np.array_equal(a[k], b[k]), "run-to-run bitwise reproducibility"
        ref = tables[k].copy()
        O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(dT[:, k]), 0.5)
        assert O.rel_err(a[k], ref) < SGD_RTOL


@pytest.mark.parametrize("D", [4, 64, 128, 256, 512])
def test_sparse_sgd_inline_fixup_equals_two_launch_fixup(D, lib_options):
    """DLRM-sized batches finish the chunk-crossing runs inside the tiles launch (the last CTA of each
    table); large batches (or the "update_two_launches" switch) use the separate fix-up kernel.  Same
    arithmetic order, same bits -- over several consecutive steps, so the in-kernel per-table counters
    must re-arm correctly."""
    rng = np.random.default_rng(D)
    rows, B = [2, 3, 40, 50000, 1], 6000 + D
    tables = _rand_tables(rng, rows, D)
    idx = [np.minimum((rng.pareto(1.05, size=(B, 1)) * 1.0).astype(np.int64), r - 1) for r in rows]
    dT = (rng.standard_normal((B, len(rows), D)) * 0.01).astype(np.float32)
    lib_options("update_two_launches", 0)
    a = _run_update(tables, idx, dT, 0, 0.5, steps=4)
    lib_options("update_two_launches", 1)
    b = _run_update(tables, idx, dT, 0, 0.5, steps=4)
    ref = [tb.copy() for tb in tables]
    for _ in range(4):
        for k in range(len(rows)):
            O.sparse_sgd_update_fast(ref[k], idx[k], np.ascontiguousarray(dT[:, k]), 0.5)
    for k in range(len(rows)):
        assert np.array_equal(a[k], b[k]), k
        assert O.rel_err(a[k], ref[k]) < SGD_RTOL, k


def test_sparse_sgd_radix_path_hot_rows():
    """L above the shared-memory sort limit: radix path + runs spanning thousands of tiles."""
    rng = np.random.default_rng(9)
    rows, D, B = [2, 100000], 16, 70000
    tables = _rand_tables(rng, rows, D)
    idx = [rng.integers(0, r, size=(B, 1)) for r in rows]
    dT = (rng.standard_normal((B, 2, D)) * 0.01).astype(np.float32)
    got = _run_update(tables, idx, dT, 0, 1.0)
    for k in range(2):
        ref = tables[k].copy()
        O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(dT[:, k]), 1.0)
        assert O.rel_err(got[k], ref) < SGD_RTOL
        dense = O.uncompress(np.ascontiguousarray(dT[:, k]), idx[k], rows[k]) if rows[k] < 10 else None
        if dense is not None:
            assert np.allclose(got[k], tables[k] - dense, rtol=1e-3, atol=1e-3)


def test_uncompress_matches_dense_gradient():
    """test/train/backprop.jl:148-158: uncompress(update) == dense gradient of table[:, ids]."""
    from dlrm_jl_b200.embedding import sparse_updates, uncompress
    rng = np.random.default_rng(1234)
    B, D, nrows = 128, 64, 1000
    ids = rng.integers(0, nrows, size=(26, B))
    dT = rng.standard_normal((B, 27, D)).astype(np.float32)
    ups = sparse_updates(torch.from_numpy(dT).to(_dev()), torch.from_numpy(ids).to(_dev()).unsqueeze(-1), 1)
    for k in (0, 13, 25):
        ref = O.uncompress(np.ascontiguousarray(dT[:, 1 + k]), ids[k], nrows)
        assert O.rel_err(uncompress(ups[k], nrows).cpu().numpy(), ref) < 1e-6


def test_update_host_entry_point():
    import ctypes as C
    from dlrm_jl_b200 import _lib
    rng = np.random.default_rng(10)
    rows, D, B, P = [40, 7], 32, 50, 2
    tables = _rand_tables(rng, rows, D)
    t = _tables(tables, B * P)
    idx = [rng.integers(0, r, size=(B, P)) for r in rows]
    flat = np.ascontiguousarray(np.stack(idx).astype(np.int32))
    dT = rng.standard_normal((B, 3, D)).astype(np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _lib.check(_lib.load().dlrmb_embedding_bwd_sgd_host(t._h, p(flat), 4, 0, B, P, p(dT), 3, 1, 0.25))
    for k in range(2):
        ref = tables[k].copy()
        O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(dT[:, 1 + k]), 0.25)
        assert O.rel_err(t.download(k), ref) < SGD_RTOL


# ------------------------------------------------------------------------------------------------
# fused sigmoid + BCE (SURVEY section 8(f) row 1)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 4, 128, 2048, 100003])
def test_sigmoid_bce_fused_vs_oracle(B):
    from dlrm_jl_b200.train import SigmoidBCELoss
    rng = np.random.default_rng(B)
    z = (rng.standard_normal(B) * 3).astype(np.float32)
    z[: min(B, 2)] = [40.0, -40.0][: min(B, 2)]                     # saturated: exercises the -100 clamp
    y = rng.random(B).astype(np.float32)                            # soft labels, as in the goldens
    loss_ref, dz_ref = O.sigmoid_bce(z, y)
    fn = SigmoidBCELoss(_dev())
    zt = torch.from_numpy(z).to(_dev()).requires_grad_(True)
    for _ in range(2):                                              # second call: the block counter reset itself
        zt.grad = None
        loss = fn(zt.reshape(-1, 1), torch.from_numpy(y).to(_dev()))
        loss.backward()
    assert abs(float(loss) - float(loss_ref)) <= 2e-6 * max(1.0, abs(float(loss_ref)))
    assert O.rel_err(zt.grad.cpu().numpy().reshape(-1), dz_ref) < FWD_RTOL


@pytest.mark.parametrize("name", ["single", "multi"])
def test_sigmoid_bce_fused_golden_loss(name):
    from dlrm_jl_b200.train import SigmoidBCELoss
    g = load_golden(name)
    p = g["mlp_top"].reshape(-1).astype(np.float64)
    logits = np.log(p / (1.0 - p)).astype(np.float32)               # invert the stored sigmoid outputs
    loss = SigmoidBCELoss(_dev())(torch.from_numpy(logits).to(_dev()), torch.from_numpy(g["labels"].reshape(-1)).to(_dev()))
    assert abs(float(loss) - float(g["loss"])) < 2e-6


# ------------------------------------------------------------------------------------------------
# end to end: the reference's validate() on both goldens, and the hand-typed PyTorch case
# ------------------------------------------------------------------------------------------------
def _torch_mlp(layers, sigmoid_last):
    import torch.nn as nn
    mods = []
    for i, (W, b) in enumerate(layers):
        lin = nn.Linear(W.shape[1], W.shape[0], device=_dev())
        with torch.no_grad():
            lin.weight.copy_(torch.from_numpy(W))
            lin.bias.copy_(torch.from_numpy(b))
        mods += [lin, nn.Sigmoid() if (sigmoid_last and i == len(layers) - 1) else nn.ReLU()]
    return nn.Sequential(*mods)


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("name", ["single", "multi"])
def test_validate_golden_one_sgd_step(name, fused):
    """src/validation.jl:1-44 + test/integration.jl: loss, then one step at lr = 10.0; every
    embedding table and MLP parameter must match the PyTorch post-step values -- with the MLPs as
    nn.Linear autograd and as fused dense layers (dlrm_jl_b200.dense)."""
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.interact import DotInteraction
    from dlrm_jl_b200.model import DLRMModel
    from dlrm_jl_b200.train import bce_loss, train_step, wrap_loss
    torch.backends.cuda.matmul.allow_tf32 = False
    g = load_golden(name)
    bot, top, tables, dense, idx, labels = golden_model(g)
    t = _tables(tables, idx[0].size)
    mb, mt = _torch_mlp(bot, False), _torch_mlp(top, True)
    if fused:
        from dlrm_jl_b200.dense import FusedMLP
        mb, mt = FusedMLP(mb), FusedMLP(mt)
    model = DLRMModel(mb, t, DotInteraction(), mt)
    seen = []
    loss_fn = wrap_loss(bce_loss, cb=seen.append)
    dense_d = torch.from_numpy(dense).to(_dev())
    labels_d = torch.from_numpy(labels).to(_dev())
    with torch.no_grad():
        out, T = model(dense_d, idx)
    assert O.rel_err(T.cpu().numpy()[:, 1:], g["concatenated_result"][:, 1:]) < FWD_RTOL
    assert O.rel_err(out.cpu().numpy(), g["mlp_top"].reshape(-1)) < FWD_RTOL
    loss = train_step(loss_fn, model, Descent(10.0), labels_d, dense_d, idx)
    assert abs(float(loss) - float(g["loss"])) < 1e-5
    ubot, utop, uemb = golden_updates(g)
    for k in range(7):
        got = t.download(k)
        assert O.rel_err(got, uemb[k]) < SGD_RTOL, k
        assert not O.isapprox(tables[k], got), "update must differ from the original (validation.jl:142)"
    linears = [m for mlp in (model.bottom_mlp, model.top_mlp) for m in mlp.modules() if isinstance(m, torch.nn.Linear)]
    assert len(linears) == len(ubot) + len(utop)
    for lin, (uW, ub) in zip(linears, ubot + utop):
        assert O.rel_err(lin.weight.detach().cpu().numpy(), uW) < SGD_RTOL
        assert O.rel_err(lin.bias.detach().cpu().numpy(), ub) < SGD_RTOL
    for sym in ("start", "lookup", "bottom_mlp", "interaction", "top_mlp", "loss", "interaction_back",
                "grads_done", "weight_update_done", "embedding_update_done", "update_done"):
        assert sym in seen, sym


def test_known_answer_small_pytorch_case():
    """test/model/model.jl:80-283 (values typed to 5 decimals -> absolute gate)."""
    from dlrm_jl_b200.embedding import DefaultStrategy, PreallocationStrategy
    from dlrm_jl_b200.interact import DotInteraction
    from dlrm_jl_b200.model import DLRMModel
    ka = load_known_answer()
    tables = [ka[f"py_embedding{i}_weights"] for i in (1, 2, 3)]
    t = _tables(tables, 4)
    bot = [(ka["py_dense1_weights"], ka["py_dense1_bias"])]
    top = [(ka["py_dense2_weights"], ka["py_dense2_bias"]), (ka["py_dense3_weights"].reshape(1, -1), ka["py_dense3_bias"])]
    model = DLRMModel(_torch_mlp(bot, False), t, DotInteraction(), _torch_mlp(top, True))
    dense = torch.from_numpy(ka["py_dense_input"]).to(_dev())
    idx = [np.asarray(v) for v in ka["py_sparse_input"]]
    for strategy in (PreallocationStrategy(4), DefaultStrategy()):
        with torch.no_grad():
            out, y = model(dense, idx, strategy=strategy)
        assert np.allclose(out.cpu().numpy(), ka["py_top_mlp_output"], atol=2e-5)
    with torch.no_grad():
        out, T = model(dense, idx)
    for k in range(3):
        assert np.allclose(T[:, 1 + k].cpu().numpy(), np.asarray(ka["py_embedding_outputs"][k], np.float32), atol=1e-6)
    z = DotInteraction()(model.bottom_mlp(dense), T)
    assert np.allclose(z.detach().cpu().numpy(), ka["py_interaction_output"], atol=2e-5)


# ------------------------------------------------------------------------------------------------
# BASELINE-size runs: size-independent properties (Kaggle-shaped: 26 tables, D 64, B 2048)
# ------------------------------------------------------------------------------------------------
def test_kaggle_shaped_properties():
    from dlrm_jl_b200.embedding import EmbeddingTables, PreallocationStrategy, maplookup
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES as ROWS
    D, B = 64, 2048
    t = EmbeddingTables(ROWS, D, B, 0)
    t.init_uniform(1)
    rng = np.random.default_rng(20261018)
    idx_np = np.stack([rng.integers(0, r, size=B) for r in ROWS]).astype(np.int32)
    idx = torch.from_numpy(idx_np).to(_dev()).unsqueeze(-1)
    # init bounds: U(-1/sqrt(rows), 1/sqrt(rows))
    for k in (0, 8, 2):
        tv = t.table(k)
        bound = 1.0 / np.sqrt(ROWS[k])
        assert float(tv.abs().max()) <= bound and float(tv.abs().max()) > 0.5 * bound
    # lookup == rows of the zero-copy table views, and is idempotent
    T = maplookup(PreallocationStrategy(D), t, idx)
    T2 = maplookup(PreallocationStrategy(D), t, idx)
    assert torch.equal(T, T2)
    for k in range(26):
        assert torch.equal(T[:, 1 + k], t.table(k)[idx[k, :, 0].long()])
    # sort: keys ascending, perm a permutation, keys == idx[perm]
    t.sort(idx)
    for k in (2, 8, 25):
        uniq, seg, perm = t.sort_dedup_export(k, B)
        keys = idx_np[k][perm]
        assert np.all(np.diff(keys) >= 0) and np.array_equal(np.sort(perm), np.arange(B))
        assert np.array_equal(uniq, np.unique(idx_np[k])) and seg[-1] == B
    # update: checksum of checksums -- the total change of a table equals -lr * sum of its deltas
    dT = torch.randn((B, 27, D), device=_dev())
    before = [t.table(k).double().sum(dim=0) for k in range(26)]
    snap = {k: t.table(k).clone() for k in (0, 5, 8, 19)}
    t.update_sorted(dT, 1, 0.1)
    for k in range(26):
        delta = t.table(k).double().sum(dim=0) - before[k]
        want = -0.1 * dT[:, 1 + k].double().sum(dim=0)
        assert torch.allclose(delta, want, rtol=1e-4, atol=1e-4), k
    # linearity: the opposite step restores the tables to rounding error
    t.bwd_sgd(idx, dT, 1, -0.1)
    for k, s in snap.items():
        assert torch.allclose(t.table(k), s, rtol=0, atol=1e-5), k
    t.close()


@pytest.mark.parametrize("name", ["single", "multi"])
def test_validate_entry_point_and_table_checkpoint(name, tmp_path):
    """dlrm_jl_b200.validation.validate == the reference's DLRM.validate(path, strategy)
    (test/integration.jl:39), fed from the committed golden; plus the table export round trip."""
    from dlrm_jl_b200.validation import load_hdf5, load_tables, save_tables, validate
    path = str(tmp_path / f"pytorch_reference_{name}.npz")
    np.savez(path, **load_golden(name))      # the 58 datasets in one file, as the reference's HDF5 has them
    assert validate(path) is True
    model = load_hdf5(path)
    ck = str(tmp_path / "tables.npz")
    save_tables(model.embeddings, ck)
    again = load_tables(ck, 16)
    for k in range(7):
        assert np.array_equal(again.download(k), model.embeddings.download(k))


def test_dac_loader_device_unpack_bit_exact():
    """DACLoader + dlrmb_dac_unpack vs the reference's load! (src/data/criteo.jl:284-310)."""
    from dlrm_jl_b200.loader import DAC_DTYPE, DACLoader
    rng = np.random.default_rng(77)
    n, B = 1000, 192                               # 5 whole batches, the ragged tail is dropped
    data = np.zeros(n, dtype=DAC_DTYPE)
    data["label"] = rng.integers(0, 2, size=n)
    data["continuous"] = rng.standard_normal((n, 13)).astype(np.float32)
    data["categorical"] = rng.integers(0, 2**32 - 1, size=(n, 26), dtype=np.uint64).astype(np.uint32)
    loader = DACLoader(data, B, 0)
    assert len(loader) == n // B
    seen = 0
    for i, (labels, dense, sparse) in enumerate(loader):
        l_ref, d_ref, s_ref = O.dac_unpack(data[i * B:(i + 1) * B])
        assert np.array_equal(labels.cpu().numpy(), l_ref)
        assert np.array_equal(dense.cpu().numpy(), d_ref)
        assert np.array_equal(sparse.cpu().numpy().view(np.uint32)[:, :, 0], s_ref)
        seen += 1
    assert seen == n // B


def test_five_sgd_steps_full_model_vs_oracle():
    """north_star tolerance "1e-4 after N SGD steps": five training steps of the golden model
    (fresh random inputs each step, lr 0.1) on the GPU path vs the CPU oracle's train step."""
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.interact import DotInteraction
    from dlrm_jl_b200.model import DLRMModel
    from dlrm_jl_b200.train import bce_loss, train_step, wrap_loss
    torch.backends.cuda.matmul.allow_tf32 = False
    g = load_golden("multi")
    bot, top, tables, _dense, _idx, _labels = golden_model(g)
    t = _tables(tables, 1280)
    model = DLRMModel(_torch_mlp(bot, False), t, DotInteraction(), _torch_mlp(top, True))
    loss_fn = wrap_loss(bce_loss)
    rng = np.random.default_rng(2026)
    o_bot, o_top, o_tables = bot, top, [x.copy() for x in tables]
    for step in range(5):
        dense = rng.random((128, 13), dtype=np.float32)
        labels = (rng.random(128) < 0.3).astype(np.float32)
        idx = [rng.integers(0, 1000, size=(128, 10)) for _ in range(7)]
        loss = train_step(loss_fn, model, Descent(0.1), torch.from_numpy(labels).to(_dev()),
                          torch.from_numpy(dense).to(_dev()), idx)
        o_loss, o_bot, o_top, _f, _g = O.dlrm_train_step(o_bot, o_top, o_tables, dense, idx, labels, 0.1)
        assert abs(float(loss) - float(o_loss)) < 1e-5 * max(1.0, abs(float(o_loss))), step
    for k in range(7):
        assert O.rel_err(t.download(k), o_tables[k]) < SGD_RTOL, k
    lins = [m for m in list(model.bottom_mlp) + list(model.top_mlp) if hasattr(m, "weight")]
    for lin, (W, b) in zip(lins, o_bot + o_top):
        assert O.rel_err(lin.weight.detach().cpu().numpy(), W) < SGD_RTOL
        assert O.rel_err(lin.bias.detach().cpu().numpy(), b) < SGD_RTOL


def test_kaggle_dlrm_builder_trains():
    """Whole-pipeline smoke as test/model/model.jl:2-31: builder, forward, backward, update, and the
    `train` loop with telemetry; the loss of a fixed batch must go down."""
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.model import kaggle_dlrm
    from dlrm_jl_b200.train import bce_loss, train, wrap_loss
    rows = [100000, 3, 57, 1000, 24, 5000, 10, 7]
    model = kaggle_dlrm(feature_size=64, max_lookups=128, device=0, embedding_sizes=rows)
    assert model.top_mlp[0].in_features == 64 + 9 * 8 // 2
    rng = np.random.default_rng(3)
    dense = torch.from_numpy(rng.random((128, 13), dtype=np.float32)).to(_dev())
    labels = torch.from_numpy((rng.random(128) < 0.5).astype(np.float32)).to(_dev())
    idx = torch.from_numpy(np.stack([rng.integers(0, r, size=128) for r in rows]).astype(np.int32)).to(_dev())
    seen = []
    out = train(wrap_loss(bce_loss, cb=seen.append), model, [(labels, dense, idx)] * 6, Descent(0.5), maxiters=6)
    assert len(out["losses"]) == 6 and len(out["iteration_times"]) == 6
    assert np.isfinite(out["losses"]).all() and out["losses"][-1] < out["losses"][0]
    assert seen.count("embedding_update_done") == 6 and "lookup_back" in seen


@pytest.mark.parametrize("D", [10, 64, 128])
def test_bf16_tables_lookup_and_update(D):
    """BF16 row storage (SURVEY 8(f) row 3): upload rounds to nearest even, the lookup is bit-exact
    against the oracle on the rounded tables, the update rounds the written rows."""
    from dlrm_jl_b200.embedding import EmbeddingTables, PreallocationStrategy, maplookup
    rng = np.random.default_rng(D)
    rows, B, P = [500, 3, 40000], 2048, 2
    tables = _rand_tables(rng, rows, D)
    t = EmbeddingTables.from_arrays(tables, B * P, 0, dtype=torch.bfloat16)
    rounded = [O.to_bf16(x) for x in tables]
    for k in range(3):
        assert np.array_equal(t.download(k), rounded[k])                    # RNE upload, exact download
        assert t.table(k).dtype == torch.bfloat16
    idx = [rng.integers(0, r, size=(B, P)) for r in rows]
    T = maplookup(PreallocationStrategy(D), t, idx).cpu().numpy()
    assert np.array_equal(T, O.lookup(rounded, idx, slot0=1))               # fp32 accumulate, bit-exact
    dT = (rng.standard_normal((B, 4, D)) * 0.05).astype(np.float32)
    t.bwd_sgd(torch.from_numpy(np.stack(idx)).to(_dev()), torch.from_numpy(dT).to(_dev()), 1, 0.1)
    for k in range(3):
        ref = rounded[k].copy()
        O.sparse_sgd_update_bf16(ref, idx[k], np.ascontiguousarray(dT[:, 1 + k]), 0.1)
        got = t.download(k)
        assert np.array_equal(got, O.to_bf16(got)), "rows must hold bf16-representable values"
        # the fp32 sums are reduced in a different (fixed) order, so a few rows land one bf16 ulp apart
        assert O.rel_err(got, ref) < 2e-3
        assert np.mean(got == ref) > 0.98
        untouched = np.setdiff1d(np.arange(rows[k]), np.unique(idx[k]))
        assert np.array_equal(got[untouched], rounded[k][untouched])


# ------------------------------------------------------------------------------------------------
# fused dense layers (training-step glue around the library GEMMs)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,sizes,sig", [(2048, [13, 512, 256, 128], 0), (300, [479, 1024, 64, 1], 4),
                                         (7, [16, 8, 3], 0), (129, [44, 33, 1], 3)])
def test_fused_mlp_matches_autograd_mlp(B, sizes, sig):
    """FusedMLP (epilogue-fused forward, dlrmb_dense_bwd_act_bias backward, gradients written into caller
    buffers) against the same parameters run through nn.Linear / ReLU autograd."""
    from dlrm_jl_b200.dense import FusedMLP
    from dlrm_jl_b200.model import create_mlp
    dev = _dev()
    torch.backends.cuda.matmul.allow_tf32 = False
    gen = torch.Generator().manual_seed(B)
    seq = create_mlp(sizes, sig, dev, gen)
    with torch.no_grad():
        for p in seq.parameters():
            if p.dim() == 1:
                p.copy_(torch.randn(p.shape, generator=gen).to(dev) * 0.1)
    mods = list(seq)[:-1] if sig else list(seq)      # the final sigmoid lives in the loss kernel
    ref = torch.nn.Sequential(*mods)
    fused = FusedMLP(mods)
    x = torch.randn((B, sizes[0]), generator=gen).to(dev)
    g = torch.randn((B, sizes[-1]), generator=gen).to(dev)
    for steps in range(2):                           # twice: the kernel's counters must re-arm
        xr = x.clone().requires_grad_(True)
        xf = x.clone().requires_grad_(True)
        for p in ref.parameters():
            p.grad = None
        yr = ref(xr)
        yr.backward(g)
        yf = fused(xf)
        yf.backward(g)
        assert torch.allclose(yf, yr, rtol=1e-5, atol=1e-6)
        assert torch.allclose(xf.grad, xr.grad, rtol=1e-4, atol=1e-6)
        for p, gbuf in zip(ref.parameters(), fused.grad_buffers()):
            assert O.rel_err(gbuf.cpu().numpy(), p.grad.cpu().numpy()) < 1e-5


def test_dense_bwd_act_bias_kernel_exact():
    """dZ = dY * (Y > 0) exactly; db = column sums (fixed order -> identical on repeat); no mask when Y is NULL."""
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    dev = _dev()
    for B, N in [(2048, 1024), (33, 1), (5, 70), (1000, 479)]:
        rng = np.random.default_rng(B + N)
        dy = torch.from_numpy(rng.standard_normal((B, N)).astype(np.float32)).to(dev)
        y = torch.from_numpy(np.maximum(rng.standard_normal((B, N)), 0).astype(np.float32)).to(dev)
        scratch = torch.zeros(int(lib.dlrmb_dense_bwd_scratch_floats(N)), device=dev)
        outs = []
        for rep in range(2):
            dz = torch.empty_like(dy)
            db = torch.empty(N, device=dev)
            _lib.check(lib.dlrmb_dense_bwd_act_bias(0, dy.data_ptr(), y.data_ptr(), B, N, dz.data_ptr(), db.data_ptr(),
                                                   scratch.data_ptr(), int(torch.cuda.current_stream().cuda_stream)))
            outs.append((dz.clone(), db.clone()))
        assert torch.equal(outs[0][0], dy * (y > 0)) and torch.equal(outs[0][1], outs[1][1])
        ref = (dy * (y > 0)).double().sum(0)
        assert torch.allclose(outs[0][1].double(), ref, rtol=1e-5, atol=1e-4)
        db2 = torch.empty(N, device=dev)
        dyc = dy.clone()
        _lib.check(lib.dlrmb_dense_bwd_act_bias(0, dyc.data_ptr(), None, B, N, dyc.data_ptr(), db2.data_ptr(),
                                               scratch.data_ptr(), int(torch.cuda.current_stream().cuda_stream)))
        assert torch.equal(dyc, dy) and torch.allclose(db2.double(), dy.double().sum(0), rtol=1e-5, atol=1e-4)


# ------------------------------------------------------------------------------------------------
# round 2: fused lookup + sort launch, DefaultStrategy gradient, pooling / skew, index base,
# Terabyte geometry
# ------------------------------------------------------------------------------------------------
def zipf_indices(rng, rows, size, alpha):
    """SURVEY 8(d): inverse-CDF Zipf r = floor(((N^(1-a) - 1) u + 1)^(1/(1-a))) - 1, then a fixed
    random relabelling of the row ids (multiplicative hash) so hot rows are spread over the table."""
    u = rng.random(size)
    r = np.floor(((float(rows) ** (1.0 - alpha) - 1.0) * u + 1.0) ** (1.0 / (1.0 - alpha))).astype(np.int64) - 1
    r = np.clip(r, 0, rows - 1)
    return (r * 2654435761 + 12345) % rows


@pytest.mark.parametrize("B,P", [(1, 1), (5, 3), (2048, 1), (683, 3), (4096, 1), (100, 40), (4097, 1), (3000, 2), (333, 1)])
@pytest.mark.parametrize("dtype,base", [(np.int32, 0), (np.int64, 1)])
def test_lookup_sort_fused_launch_equals_separate_launches(B, P, dtype, base):
    """dlrmb_embedding_fwd_sort (the sort rides in extra CTAs of the lookup launch for B*P <= 4096, two
    launches above) == dlrmb_embedding_fwd + dlrmb_embedding_sort: pooled rows and the exported
    dedup, bit for bit, and against the oracle."""
    from dlrm_jl_b200.embedding import EmbeddingTables
    rng = np.random.default_rng(B * 7 + P)
    rows, D = [3, 1000, 40_000_000, 513, 70000], 32
    L = B * P
    t = EmbeddingTables(rows, D, L, 0)
    t.init_uniform(3)
    idx = np.stack([rng.integers(0, r, size=(B, P)) for r in rows])
    dev_idx = torch.from_numpy((idx + base).astype(dtype)).to(_dev())
    T1 = torch.empty((B, 1 + len(rows), D), device=_dev())
    T2 = torch.full((B, 1 + len(rows), D), -3.0, device=_dev())
    t.lookup(dev_idx, T1, 1, base)
    t.lookup(dev_idx, T2, 1, base, sort=True)
    assert torch.equal(T1[:, 1:], T2[:, 1:]) and torch.all(T2[:, 0] == -3.0)
    fused = [t.sort_dedup_export(k, L) for k in range(len(rows))]
    t.sort(dev_idx, base)
    for k in range(len(rows)):
        sep = t.sort_dedup_export(k, L)
        ref = O.sort_dedup(idx[k].reshape(-1))
        for a, b, c in zip(fused[k], sep, ref):
            assert np.array_equal(a, b) and np.array_equal(a, c)
    # the update consumes the fused launch's sort directly
    dT = torch.randn((B, 1 + len(rows), D), device=_dev())
    before = {k: t.table(k).clone() for k in (0, 1, 3)}
    t.lookup(dev_idx, T2, 1, base, sort=True)
    t.update_sorted(dT, 1, 0.25)
    for k in (0, 1, 3):
        ref = before[k].cpu().numpy()
        O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(dT[:, 1 + k].cpu().numpy()), 0.25)
        assert O.rel_err(t.table(k).cpu().numpy(), ref) < SGD_RTOL
    t.close()


def test_dot_interaction_default_strategy_gradient_reaches_x():
    """dot_interaction (src/model/interact.jl:503-513; DefaultStrategy) under autograd: the gradient of
    x is dOut[:, :d] + (S T)[0] -- Zygote differentiates concat([X, Zflat]) -- and the ys get their Gram
    rows.  Checked against the oracle pullback and against DotInteraction on the same inputs."""
    from dlrm_jl_b200.interact import DotInteraction, dot_interaction, interaction_width
    rng = np.random.default_rng(17)
    for B, F, d in [(33, 8, 16), (20, 27, 64), (9, 5, 12)]:
        Tn = rng.standard_normal((B, F, d)).astype(np.float32)
        g = rng.standard_normal((B, interaction_width(F, d))).astype(np.float32)
        x = torch.from_numpy(Tn[:, 0].copy()).to(_dev()).requires_grad_(True)
        ys = [torch.from_numpy(Tn[:, f].copy()).to(_dev()).requires_grad_(True) for f in range(1, F)]
        z = dot_interaction(x, ys)
        z.backward(torch.from_numpy(g).to(_dev()))
        dx_ref, dT_ref = O.interaction_bwd(g, Tn)
        assert O.rel_err(z.detach().cpu().numpy(), O.interaction_fwd(Tn)) < FWD_RTOL
        assert O.rel_err(x.grad.cpu().numpy(), dx_ref) < FWD_RTOL
        assert not np.allclose(x.grad.cpu().numpy(), dT_ref[:, 0], atol=1e-3), "pass-through term must be present"
        for f in range(1, F):
            assert O.rel_err(ys[f - 1].grad.cpu().numpy(), dT_ref[:, f]) < FWD_RTOL
        x2 = torch.from_numpy(Tn[:, 0].copy()).to(_dev()).requires_grad_(True)
        T2 = torch.from_numpy(Tn).to(_dev()).requires_grad_(True)
        DotInteraction()(x2, T2).backward(torch.from_numpy(g).to(_dev()))
        assert torch.equal(x2.grad, x.grad)


@pytest.mark.parametrize("D", [16, 64, 128])
@pytest.mark.parametrize("B,P,alpha", [(512, 4, 0.0), (64, 64, 0.0), (2048, 4, 1.05), (256, 64, 1.2), (2048, 1, 1.2),
                                       (6000, 16, 1.2)])
def test_sparse_sgd_pooling_and_zipf_skew_vs_oracle(D, B, P, alpha):
    """Pooling factors 4 / 16 / 64 (BASELINE config 5) and Zipf-skewed indices (alpha 1.05, 1.2): tables
    after three SGD steps against the oracle, run-to-run bit-reproducible, untouched rows untouched."""
    rng = np.random.default_rng(D * 3 + B + P)
    rows = [100000, 50, 3, 1000003]
    tables = _rand_tables(rng, rows, D)
    idx = [(zipf_indices(rng, r, (B, P), alpha) if alpha > 0 else rng.integers(0, r, size=(B, P))) for r in rows]
    dT = (rng.standard_normal((B, 1 + len(rows), D)) * 0.05).astype(np.float32)
    got = _run_update(tables, idx, dT, 1, 0.1, steps=3)
    again = _run_update(tables, idx, dT, 1, 0.1, steps=3)
    ref = [tb.copy() for tb in tables]
    for _ in range(3):
        for k in range(len(rows)):
            O.sparse_sgd_update_fast(ref[k], idx[k], np.ascontiguousarray(dT[:, 1 + k]), 0.1)
    for k in range(len(rows)):
        assert np.array_equal(got[k], again[k]), "bitwise reproducible"
        assert O.rel_err(got[k], ref[k]) < SGD_RTOL, k
        untouched = np.setdiff1d(np.arange(rows[k]), np.unique(idx[k]))
        assert np.array_equal(got[k][untouched], tables[k][untouched])


def test_lookup_pooling_64_and_zipf_bit_exact():
    from dlrm_jl_b200.embedding import PreallocationStrategy, maplookup
    rng = np.random.default_rng(64)
    rows, D = [100000, 7, 5000], 128
    tables = _rand_tables(rng, rows, D)
    for B, P, alpha in [(128, 64, 1.2), (300, 16, 1.05), (2048, 4, 1.2)]:
        idx = [zipf_indices(rng, r, (B, P), alpha) for r in rows]
        t = _tables(tables, B * P)
        T = maplookup(PreallocationStrategy(D), t, idx).cpu().numpy()
        assert np.array_equal(T, O.lookup(tables, idx, slot0=1)), (B, P, alpha)
        t.close()


def test_one_based_reference_format_batches_train_on_the_right_rows():
    """Reference-preprocessed data is 1-based (src/data/criteo.jl:249-253).  A DACLoader over such
    records carries idx_base = 1, `train` adopts it and range-checks the first batch; the resulting
    tables equal the oracle run on the 0-based ids, and a 0-based interpretation of the same file is
    refused (DLRMB_EOOB) instead of training on rows shifted by one."""
    from dlrm_jl_b200 import DLRMB200Error
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.loader import DAC_DTYPE, DACLoader
    from dlrm_jl_b200.model import kaggle_dlrm
    from dlrm_jl_b200.train import bce_loss, train, wrap_loss
    rows = [50, 3, 57, 1000, 24, 5000, 10, 7] + [11 + k for k in range(18)]
    rng = np.random.default_rng(12)
    n, B = 256, 64
    data = np.zeros(n, dtype=DAC_DTYPE)
    data["label"] = rng.integers(0, 2, size=n)
    data["continuous"] = rng.random((n, 13), dtype=np.float32)
    ids0 = np.stack([rng.integers(0, r, size=n) for r in rows], axis=1)
    ids0[0, :] = np.asarray(rows) - 1                      # the largest legal id of every table is present
    data["categorical"] = (ids0 + 1).astype(np.uint32)     # 1-based on disk
    model = kaggle_dlrm(feature_size=16, max_lookups=B, device=0, embedding_sizes=rows)
    start = [model.embeddings.download(k) for k in range(26)]
    loader = DACLoader(data, B, 0)
    assert loader.idx_base == 1
    out = train(wrap_loss(bce_loss), model, loader, Descent(0.5), maxiters=2)
    assert len(out["losses"]) == 2 and np.isfinite(out["losses"]).all()
    for k in (0, 1, 3):
        got = model.embeddings.download(k)
        touched = np.unique(ids0[:2 * B, k])
        untouched = np.setdiff1d(np.arange(rows[k]), touched)
        assert np.array_equal(got[untouched], start[k][untouched])
        assert not np.array_equal(got[touched], start[k][touched])
    model0 = kaggle_dlrm(feature_size=16, max_lookups=B, device=0, embedding_sizes=rows)
    with pytest.raises(DLRMB200Error, match="DLRMB_EOOB"):
        train(wrap_loss(bce_loss), model0, DACLoader(data, B, 0, idx_base=0), Descent(0.5), maxiters=1)


def test_terabyte_shaped_properties():
    """BASELINE config 4 geometry on one GPU: 26 tables with rows = min(TERABYTE_EMBEDDING_SIZES, 40M)
    (src/data/criteo.jl:379-406), D = 128 (104.5 GB of fp32 tables), B = 2048.  Size-independent
    properties: lookup == rows of the zero-copy views, idempotence, sortedness / permutation, the update's
    checksum of checksums, and the inverse step restoring the tables."""
    from dlrm_jl_b200.embedding import EmbeddingTables
    from dlrm_jl_b200.interact import interaction_bwd, interaction_fwd, interaction_width
    from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES
    free, _total = torch.cuda.mem_get_info()
    ROWS = [min(r, 40_000_000) for r in TERABYTE_EMBEDDING_SIZES]
    D, B = 128, 2048
    if free < sum(ROWS) * D * 4 + (8 << 30):
        pytest.skip("needs ~113 GB of free HBM")
    t = EmbeddingTables(ROWS, D, B, 0)
    t.init_uniform(7)
    rng = np.random.default_rng(20261018)
    idx_np = np.stack([rng.integers(0, r, size=B) for r in ROWS]).astype(np.int32)
    idx_np[:, 0] = np.asarray(ROWS) - 1                     # the last row of every table (40M - 1 included)
    idx_np[:, 1] = 0
    idx = torch.from_numpy(idx_np).to(_dev()).unsqueeze(-1)
    T = torch.zeros((B, 27, D), device=_dev())
    T2 = torch.zeros((B, 27, D), device=_dev())
    t.lookup(idx, T, 1, sort=True)
    t.lookup(idx, T2, 1)
    assert torch.equal(T, T2)
    for k in range(26):
        assert torch.equal(T[:, 1 + k], t.table(k)[idx[k, :, 0].long()])
    for k in (0, 5, 9, 19, 25):
        uniq, seg, perm = t.sort_dedup_export(k, B)
        keys = idx_np[k][perm]
        assert np.all(np.diff(keys) >= 0) and np.array_equal(np.sort(perm), np.arange(B))
        assert np.array_equal(uniq, np.unique(idx_np[k])) and seg[-1] == B
        u_ref, s_ref, p_ref = O.sort_dedup(idx_np[k])
        assert np.array_equal(perm, p_ref) and np.array_equal(seg, s_ref)
    # interaction at this geometry against the oracle on a slice of the batch
    T[:, 0] = torch.randn((B, D), device=_dev())
    z = interaction_fwd(T)
    g = torch.randn((B, interaction_width(27, D)), device=_dev())
    dx, dT = interaction_bwd(g, T)
    sl = slice(0, 64)
    Tn = T[sl].cpu().numpy()
    assert O.rel_err(z[sl].cpu().numpy(), O.interaction_fwd(Tn)) < FWD_RTOL
    dx_ref, dT_ref = O.interaction_bwd(g[sl].cpu().numpy(), Tn)
    assert O.rel_err(dT[sl].cpu().numpy(), dT_ref) < FWD_RTOL and O.rel_err(dx[sl].cpu().numpy(), dx_ref) < FWD_RTOL
    # update: per-table column checksums move by -lr * the column sums of the deltas
    snap_rows = {k: t.table(k)[idx[k, :, 0].long()].clone() for k in (0, 5, 20)}
    before = {k: t.table(k)[idx[k, :, 0].long().unique()].double().sum(dim=0) for k in range(26)}
    t.update_sorted(dT, 1, 0.1)
    for k in range(26):
        after = t.table(k)[idx[k, :, 0].long().unique()].double().sum(dim=0)
        want = -0.1 * dT[:, 1 + k].double().sum(dim=0)
        assert torch.allclose(after - before[k], want, rtol=1e-4, atol=1e-5), k
    # oracle on the touched rows of three tables (a 3-row table, and two 40M-row tables)
    for k in (0, 5, 20):
        rows_k, first_idx, inv = np.unique(idx_np[k], return_index=True, return_inverse=True)
        sub = t.table(k)[torch.from_numpy(rows_k).to(_dev()).long()].cpu().numpy()
        ref = snap_rows[k].cpu().numpy()[first_idx].copy()          # the touched rows before the update, compacted
        O.sparse_sgd_update_fast(ref, inv.reshape(-1, 1), np.ascontiguousarray(dT[:, 1 + k].cpu().numpy()), 0.1)
        assert O.rel_err(sub, ref) < SGD_RTOL, k
    # inverse step restores the touched rows to rounding error
    t.lookup(idx, T2, 1, sort=True)
    t.update_sorted(dT, 1, -0.1)
    for k, s in snap_rows.items():
        assert torch.allclose(t.table(k)[idx[k, :, 0].long()], s, rtol=0, atol=1e-5), k
    t.close()


def test_comm_c_abi_world_one_round_trip():
    """The dlrmb_comm_* entry points (NCCL behind the C ABI) with a one-rank communicator: the exchanges
    degenerate to sends to self, which still run the real NCCL group calls and the pack / unpack kernels.
    (The multi-rank behaviour is exercised on 2+ GPUs by tests/cabi_sharded_step.py.)"""
    import ctypes as C
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    dev = _dev()
    rows = (C.c_int64 * 5)(50, 4000, 7, 4000, 900)
    owner = (C.c_int32 * 5)()
    _lib.check(lib.dlrmb_shard_plan(5, rows, 2, owner))
    assert sorted(list(owner)) == [0, 0, 1, 1, 1] or sorted(list(owner)) == [0, 0, 0, 1, 1]
    assert owner[1] != owner[3]                                  # the two big tables on different ranks
    _lib.check(lib.dlrmb_shard_plan(5, rows, 1, owner))
    assert list(owner) == [0] * 5
    uid = (C.c_uint8 * 128)()
    _lib.check(lib.dlrmb_comm_unique_id(uid))
    h = C.c_void_p()
    _lib.check(lib.dlrmb_comm_create(0, uid, 0, 1, C.byref(h)))
    r, w = C.c_int32(-1), C.c_int32(-1)
    _lib.check(lib.dlrmb_comm_info(h, C.byref(r), C.byref(w)))
    assert (r.value, w.value) == (0, 1)
    s = int(torch.cuda.current_stream().cuda_stream)
    B, P, D, ntab = 24, 3, 32, 5
    idx = torch.randint(0, 1000, (ntab, B, P), device=dev, dtype=torch.int64)
    idx_owned = torch.zeros_like(idx)
    _lib.check(lib.dlrmb_comm_a2a_indices(h, owner, ntab, idx.data_ptr(), 8, B, P, idx_owned.data_ptr(), s))
    assert torch.equal(idx_owned, idx)
    pooled = torch.randn((B, ntab, D), device=dev)
    T = torch.full((B, 1 + ntab, D), -1.0, device=dev)
    _lib.check(lib.dlrmb_comm_a2a_fwd(h, owner, ntab, pooled.data_ptr(), B, D, T.data_ptr(), s))
    assert torch.equal(T[:, 1:], pooled) and torch.all(T[:, 0] == -1.0)
    grads = torch.zeros((B, ntab, D), device=dev)
    _lib.check(lib.dlrmb_comm_a2a_bwd(h, owner, ntab, T.data_ptr(), B, D, grads.data_ptr(), s))
    assert torch.equal(grads, pooled)
    buf = torch.arange(1000, device=dev, dtype=torch.float32)
    _lib.check(lib.dlrmb_comm_allreduce_f32(h, buf.data_ptr(), 1000, s))
    assert torch.equal(buf, torch.arange(1000, device=dev, dtype=torch.float32))
    blob = torch.arange(64, device=dev, dtype=torch.uint8)
    out = torch.zeros(64, device=dev, dtype=torch.uint8)
    _lib.check(lib.dlrmb_comm_allgather(h, blob.data_ptr(), out.data_ptr(), 64, s))
    assert torch.equal(out, blob)
    torch.cuda.synchronize()
    _lib.check(lib.dlrmb_comm_destroy(h))


@pytest.mark.parametrize("B,F,d", [(2049, 27, 128), (77, 27, 64), (33, 8, 16), (19, 11, 128), (5, 1, 16)])
def test_interaction_backward_dx_alone_and_split_scatter(B, F, d):
    """dlrmb_interaction_bwd_dx == the dx of the full pullback (same bits for the specialised shapes: same
    summation order), and a ScatterPlan with a side stream (dx first, peer stores beside whatever consumes
    dx) gives the same dx and the same scattered rows as the single-kernel scatter."""
    import ctypes as C
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.interact import DotInteraction, ScatterPlan, interaction_bwd, interaction_width
    rng = np.random.default_rng(B * 3 + F)
    T = torch.from_numpy(rng.standard_normal((B, F, d)).astype(np.float32)).to(_dev())
    g = torch.from_numpy(rng.standard_normal((B, interaction_width(F, d))).astype(np.float32)).to(_dev())
    dx_ref, dT_ref = interaction_bwd(g, T)
    dx = torch.empty((B, d), device=_dev())
    _lib.check(_lib.load().dlrmb_interaction_bwd_dx(0, g.data_ptr(), T.data_ptr(), B, F, d, 1, dx.data_ptr(),
                                                    int(torch.cuda.current_stream().cuda_stream)))
    if _lib.load().dlrmb_interaction_has_warp_path(F, d):
        assert torch.equal(dx, dx_ref)
    assert O.rel_err(dx.cpu().numpy(), dx_ref.cpu().numpy()) < 1e-6
    if F < 2:
        return
    buf = torch.full((B + 3, F - 1, d), -7.0, device=_dev())
    dests = torch.zeros((F, 3), dtype=torch.int64)
    for f in range(1, F):
        dests[f, 0], dests[f, 1], dests[f, 2] = buf.data_ptr(), (F - 1) * d, (f - 1) * d
    plan = ScatterPlan(dests.to(_dev()), 2, stream=torch.cuda.Stream())
    x = T[:, 0].clone().requires_grad_(True)
    DotInteraction()(x, T.clone(), scatter=plan).backward(g)
    torch.cuda.current_stream().wait_event(plan.done)
    assert torch.equal(x.grad, dx)
    assert torch.equal(buf[2:2 + B], dT_ref[:, 1:]) and torch.all(buf[:2] == -7.0) and torch.all(buf[2 + B:] == -7.0)


@pytest.mark.parametrize("B,F,d", [(2049, 27, 128), (1, 27, 128), (301, 27, 64), (5000, 27, 128)])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_interaction_forward_one_and_two_warps_per_sample(B, F, d, mode, lib_options):
    """The tensor-core forward with one warp per sample (mode 0), two warps per sample splitting k (mode 2) and
    the default choice by batch size (mode 1): same contract and tolerance, integer inputs exact, fused
    fast_vcat, padding."""
    from dlrm_jl_b200.interact import interaction_fwd
    rng = np.random.default_rng(B + F + d)
    T = rng.standard_normal((B, F, d)).astype(np.float32)
    lib_options("fwd_ksplit", mode)
    for pad in (1, 16):
        ref = O.interaction_fwd(T, pad)
        Tz = T.copy()
        Tz[:, 0] = 0
        Tzd = torch.from_numpy(Tz).to(_dev())
        out = interaction_fwd(Tzd, torch.from_numpy(T[:, 0].copy()).to(_dev()), pad_to_mul=pad).cpu().numpy()
        assert out.shape == ref.shape and O.rel_err(out, ref) < FWD_RTOL
        assert np.array_equal(out[:, :d], T[:, 0]) and np.array_equal(Tzd.cpu().numpy(), T)
        assert np.all(out[:, d + F * (F - 1) // 2:] == 0)
    Ti = rng.integers(-4, 5, size=(64, F, d)).astype(np.float32)
    assert np.array_equal(interaction_fwd(torch.from_numpy(Ti).to(_dev())).cpu().numpy(), O.interaction_fwd(Ti))


@pytest.mark.parametrize("tile", [4, 12, 20, 28, 32])
def test_sparse_sgd_any_tile_length_gives_the_same_tables(tile, lib_options):
    """The tile (entries per lane group) is any multiple of 4 up to 32, chosen per batch so that the update is
    one wave; every choice must give oracle-level tables, inline and two-launch fix-up bit-equal."""
    rng = np.random.default_rng(tile)
    rows, D, B = [3, 40, 50000, 7, 1000], 128, 5000 + tile
    tables = _rand_tables(rng, rows, D)
    idx = [np.minimum((rng.pareto(1.05, size=(B, 1)) * 1.0).astype(np.int64), r - 1) for r in rows]
    idx[2] = rng.integers(0, rows[2], size=(B, 1))
    dT = (rng.standard_normal((B, len(rows), D)) * 0.01).astype(np.float32)
    lib_options("update_tile", tile)
    lib_options("update_two_launches", 0)
    a = _run_update(tables, idx, dT, 0, 0.5, steps=2)
    lib_options("update_two_launches", 1)
    b = _run_update(tables, idx, dT, 0, 0.5, steps=2)
    ref = [tb.copy() for tb in tables]
    for _ in range(2):
        for k in range(len(rows)):
            O.sparse_sgd_update_fast(ref[k], idx[k], np.ascontiguousarray(dT[:, k]), 0.5)
    for k in range(len(rows)):
        assert np.array_equal(a[k], b[k]), k
        assert O.rel_err(a[k], ref[k]) < SGD_RTOL, k


def test_sparse_update_launched_inside_backward_equals_explicit_update():
    """ShardedEmbedding.update_inside_backward (the bench's form: the update is launched by the lookup's pullback
    on a side stream, beside the rest of the backward pass) gives the tables of the explicit update call."""
    from dlrm_jl_b200.interact import DotInteraction, interaction_width
    from dlrm_jl_b200.sharded import ShardedEmbedding
    rows, D, B = [50, 7, 400, 3, 1200, 33, 9] + [20 + 31 * k for k in range(19)], 64, 300
    rng = np.random.default_rng(3)
    idx = torch.from_numpy(np.stack([rng.integers(0, r, size=(B, 1)) for r in rows]).astype(np.int32)).to(_dev())
    x_np = rng.standard_normal((B, D)).astype(np.float32)
    g = torch.from_numpy(rng.standard_normal((B, interaction_width(27, D))).astype(np.float32)).to(_dev())
    got = []
    for inside in (False, True):
        se = ShardedEmbedding.create(rows, D, B, 1, 0, 1, _dev())
        side = torch.cuda.Stream()
        if inside:
            se.update_inside_backward(0.3, side)
        anchor = torch.zeros(1, device=_dev(), requires_grad=True)
        x = torch.from_numpy(x_np).to(_dev()).requires_grad_(True)
        T = se.lookup(idx, anchor)
        DotInteraction()(x, T).backward(g)
        if inside:
            torch.cuda.current_stream().wait_stream(side)
        else:
            se.update(0.3)
        got.append([se.tables.download(k) for k in range(len(rows))])
    for a, b in zip(*got):
        assert np.array_equal(a, b)


def test_tables_reserve_grows_the_workspaces_and_keeps_the_tables():
    """dlrmb_tables_reserve (what the Julia glue calls when a batch is larger than any before): the sort /
    update workspaces grow, the tables keep their bits, and the larger batch then runs."""
    import ctypes as C
    from dlrm_jl_b200 import DLRMB200Error, _lib
    from dlrm_jl_b200.embedding import EmbeddingTables
    rng = np.random.default_rng(21)
    rows, D = [300, 5, 70000], 32
    tables = _rand_tables(rng, rows, D)
    t = EmbeddingTables.from_arrays(tables, 64, 0)
    B = 5000
    idx = torch.from_numpy(np.stack([rng.integers(0, r, size=(B, 1)) for r in rows])).to(_dev())
    T = torch.empty((B, 4, D), device=_dev())
    with pytest.raises(DLRMB200Error, match="max_lookups"):
        t.lookup(idx, T, 1)
    _lib.check(_lib.load().dlrmb_tables_reserve(t._h, B))
    _lib.check(_lib.load().dlrmb_tables_reserve(t._h, 10))           # never shrinks
    ml = C.c_int64()
    _lib.check(_lib.load().dlrmb_tables_info(t._h, None, None, C.byref(ml), None))
    assert ml.value == B
    for k in range(3):
        assert np.array_equal(t.download(k), tables[k])
    t.lookup(idx, T, 1, sort=True)
    assert np.array_equal(T[:, 1:].cpu().numpy(), O.lookup(tables, list(idx.cpu().numpy()), slot0=1)[:, 1:])
    dT = torch.randn((B, 4, D), device=_dev())
    t.update_sorted(dT, 1, 0.1)
    for k in range(3):
        ref = tables[k].copy()
        O.sparse_sgd_update_fast(ref, idx[k].cpu().numpy(), np.ascontiguousarray(dT[:, 1 + k].cpu().numpy()), 0.1)
        assert O.rel_err(t.download(k), ref) < SGD_RTOL


@pytest.mark.gpu
@pytest.mark.parametrize("B", [2048, 20000])
def test_device_clock_stamps_cover_every_cta_of_a_large_grid(B):
    """dlrmb_clock_enable: the kernels' own %globaltimer stamps (bench.py's in-step clock) must span the WHOLE
    launch whatever the grid size -- CTAs fold into 4096 slots (earliest entry, latest exit).  At B = 20000 the
    interaction kernels launch more CTAs than slots: the stamped window has to stay within the CUDA-event time
    of the same launch and well above the share a truncated window would show."""
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.interact import interaction_bwd, interaction_fwd, interaction_width
    lib = _lib.load()
    F, d = 27, 128
    nk = int(lib.dlrmb_clock_kernels())
    buf = torch.empty(int(lib.dlrmb_clock_buffer_bytes()) // 8, dtype=torch.int64, device=_dev())
    view = buf.view(nk, -1, 2)
    T = torch.randn(B, F, d, device=_dev())
    dOut = torch.randn(B, interaction_width(F, d), device=_dev())
    IFWD, IBWD = 4, 5       # kernel order of include/dlrm_b200.h
    for which, fn in ((IFWD, lambda: interaction_fwd(T)), (IBWD, lambda: interaction_bwd(dOut, T))):
        fn()                # warm-up without stamps
        torch.cuda.synchronize()
        view[:, :, 0] = 1 << 62
        view[:, :, 1] = 0
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _lib.check(lib.dlrmb_clock_enable(buf.data_ptr()))
        try:
            torch.cuda._sleep(4_000_000)      # ~2 ms of device spin: the host is ahead, the events time the device only
            a.record()
            fn()
            b.record()
        finally:
            _lib.check(lib.dlrmb_clock_enable(None))
        torch.cuda.synchronize()
        event_us = 1e3 * a.elapsed_time(b)
        t0 = int(view[which, :, 0].min().item())
        t1 = int(view[which, :, 1].max().item())
        assert t0 < (1 << 62) and t1 > 0, "no stamps written"
        stamped_us = (t1 - t0) * 1e-3
        assert stamped_us <= event_us + 1.0, (stamped_us, event_us)
        # the event pair adds launch latency and an allocation on top of the kernel; a window truncated to the
        # first 4096 of ~10000 CTAs would be below 0.45 of it at B = 20000
        if B >= 20000:
            assert stamped_us > 0.6 * event_us, (stamped_us, event_us)
        others = [k for k in range(nk) if k != which]
        assert int(view[others, :, 1].max().item()) == 0, "stamps of a kernel that did not run"
