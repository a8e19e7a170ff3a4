"""Weighted jagged bags (per-sample weights) without a GPU: the NumPy reference against
torch.nn.functional.embedding_bag(..., mode="sum", per_sample_weights=w) (forward, table gradient and weight gradient),
the JaggedIndices container's weights, and the weighted C entry points' refusal of bad arguments before any CUDA call."""
import os
import subprocess

import numpy as np
import pytest
import torch

from tests import jagged_oracle as J
from tests import jagged_weighted_oracle as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torch_reference(table, values, offsets, weights, g):
    t = torch.from_numpy(table).requires_grad_(True)
    w = torch.from_numpy(weights).requires_grad_(True)
    out = torch.nn.functional.embedding_bag(torch.from_numpy(values), t, torch.from_numpy(offsets[:-1]), mode="sum",
                                            per_sample_weights=w)
    out.backward(torch.from_numpy(g))
    return out.detach().numpy(), t.grad.numpy(), w.grad.numpy()


@pytest.mark.parametrize("D", [4, 10, 16])
def test_oracle_against_torch_embedding_bag(D):
    rng = np.random.default_rng(30 + D)
    rows, B = 40, 33
    table = rng.standard_normal((rows, D)).astype(np.float32)
    n = rng.integers(0, 7, size=B)
    n[[0, 5, B - 1]] = 0                                   # empty bags, the last one included
    n[7] = 1
    offsets = np.zeros(B + 1, np.int64)
    np.cumsum(n, out=offsets[1:])
    values = rng.integers(0, rows, size=int(n.sum())).astype(np.int64)
    values[:3] = 11                                        # duplicates across bags
    w = rng.standard_normal(len(values)).astype(np.float32)
    w[[1, 4]] = 0.0
    w[2] = -0.0
    w[6] = -3.0
    g = rng.standard_normal((B, D)).astype(np.float32)
    ref_out, ref_grad, ref_wgrad = _torch_reference(table, values, offsets, w, g)
    out = W.lookup_jagged_weighted([table], values, offsets, w, B)[:, 0]
    assert np.allclose(out, ref_out, rtol=1e-5, atol=1e-6)
    assert np.all(out[n == 0] == 0) and not np.signbit(out[n == 0]).any()
    lr = 0.5
    got = table.copy()
    W.sparse_sgd_update_jagged_weighted(got, values, offsets, w, g, lr)
    assert np.allclose(got, table - lr * ref_grad, rtol=1e-5, atol=1e-6)
    untouched = np.setdiff1d(np.arange(rows), values)
    assert np.array_equal(got[untouched], table[untouched])
    dw = W.weight_grad_jagged([table], values, offsets, g[:, None, :], B)
    bag = np.repeat(np.arange(B), n)
    exact = np.einsum("jd,jd->j", g[bag].astype(np.float64), table[values].astype(np.float64))
    assert np.allclose(dw, ref_wgrad, rtol=1e-5, atol=1e-5)
    assert np.all(np.abs(dw - exact) <= 4 * D * np.finfo(np.float32).eps * np.einsum(
        "jd,jd->j", np.abs(g[bag]).astype(np.float64), np.abs(table[values]).astype(np.float64)))


def test_oracle_unit_weights_are_the_unweighted_sum():
    rng = np.random.default_rng(41)
    tables = [rng.standard_normal((50, 12)).astype(np.float32) for _ in range(2)]
    B = 9
    n = rng.integers(0, 6, size=2 * B)
    offsets = np.zeros(2 * B + 1, np.int64)
    np.cumsum(n, out=offsets[1:])
    values = np.concatenate([rng.integers(0, 50, size=int(n[:B].sum())), rng.integers(0, 50, size=int(n[B:].sum()))])
    ones = np.ones(len(values), np.float32)
    a = W.lookup_jagged_weighted(tables, values, offsets, ones, B, slot0=1)
    b = J.lookup_jagged(tables, values, offsets, B, "sum", slot0=1)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_weight_grad_order_is_the_stated_butterfly():
    # D = 8 (two chunks of four floats, G = 2): p_0 = g0 r0 + .. + g3 r3, p_1 = g4 r4 + .. + g7 r7, dw = p_0 + p_1
    g = np.array([1e8, 1.0, -1e8, 1.0, 3.0, 0.5, 0.25, 2.0], np.float32)
    r = np.ones(8, np.float32)
    p0 = np.float32(np.float32(np.float32(np.float32(1e8) + np.float32(1.0)) - np.float32(1e8)) + np.float32(1.0))
    p1 = np.float32(3.0 + 0.5 + 0.25 + 2.0)
    assert W.dot_in_kernel_order(g, r) == np.float32(p0 + p1)
    # D = 10: ten chunks of one float, G = 16: lane l < 10 holds product l, the rest zero
    g = np.arange(1, 11, dtype=np.float32) / np.float32(3)
    r = np.full(10, 1.5, np.float32)
    p = np.zeros(16, np.float32)
    p[:10] = g * r
    for s in (8, 4, 2, 1):
        p = (p + p[np.arange(16) ^ s]).astype(np.float32)
    assert W.dot_in_kernel_order(g, r) == p[0]


def test_container_weights():
    from dlrm_jl_b200.embedding import JaggedIndices, PackedIndices, _as_index_tensor
    j = JaggedIndices.from_bags([[[1, 2], [], [3]], [[4], [5, 6, 7], []]],
                                weights=[[[0.5, -1.0], [], [2.0]], [[0.0], [1.0, 1.5, -0.0], []]])
    assert j.weights.dtype == torch.float32 and j.weights.tolist() == [0.5, -1.0, 2.0, 0.0, 1.0, 1.5, -0.0]
    v1, o1, w1 = j[1]
    assert v1.tolist() == [4, 5, 6, 7] and o1.tolist() == [0, 1, 4, 4] and w1.tolist() == [0.0, 1.0, 1.5, -0.0]
    assert len(JaggedIndices.from_bags([[[1]]])[0]) == 2          # unweighted: (values_k, offsets_k) as before
    k = j.to("cpu")
    assert k.weights is not None and torch.equal(k.weights, j.weights)
    idx = torch.arange(24, dtype=torch.int32).reshape(2, 4, 3)
    d = JaggedIndices.from_dense(idx, weights=np.full((2, 4, 3), 0.25))
    assert d.weights.tolist() == [0.25] * 24
    p = _as_index_tensor([np.zeros((4, 1), np.int64), np.ones((4, 5), np.int64)], 2, torch.device("cpu"))
    assert isinstance(p, PackedIndices)
    dp = JaggedIndices.from_dense(p, weights=torch.arange(24, dtype=torch.float32))
    assert dp.L == (4, 20) and dp[1][2].tolist() == list(range(4, 24))
    lw = JaggedIndices.from_lengths(np.arange(3), [[2, 1]], weights=[1, 2, 3])
    assert lw.weights.dtype == torch.float32 and lw.weights.tolist() == [1.0, 2.0, 3.0]


def test_container_weight_errors():
    from dlrm_jl_b200.embedding import JaggedIndices
    v, o = torch.arange(3), torch.tensor([0, 2, 3])
    with pytest.raises(ValueError, match="one float per value"):
        JaggedIndices(v, o, (3,), 2, "sum", torch.ones(2))
    with pytest.raises(ValueError, match="one float per value"):
        JaggedIndices(v, o, (3,), 2, "sum", torch.ones(3, 1))
    with pytest.raises(ValueError, match="float32"):
        JaggedIndices(v, o, (3,), 2, "sum", torch.ones(3, dtype=torch.float64))
    with pytest.raises(ValueError, match="pooling='sum' only"):
        JaggedIndices(v, o, (3,), 2, "mean", torch.ones(3))
    with pytest.raises(ValueError, match="pooling='sum' only"):
        JaggedIndices.from_lengths(np.arange(3), [[2, 1]], "mean", weights=np.ones(3))
    with pytest.raises(ValueError, match="one weight per index"):
        JaggedIndices.from_bags([[[1, 2], [3]]], weights=[[[1.0], [1.0]]])
    with pytest.raises(ValueError, match="one float per value"):
        JaggedIndices.from_lengths(np.arange(3), [[2, 1]], weights=np.ones(4))


def test_uncompress_weighted_matches_oracle_gradient():
    from dlrm_jl_b200.embedding import JaggedIndices, sparse_updates, uncompress
    rng = np.random.default_rng(43)
    rows, D, B = 9, 4, 6
    w = rng.standard_normal(10).astype(np.float32)
    j = JaggedIndices.from_lengths(rng.integers(0, rows, size=10), [[2, 0, 3, 1, 4, 0]], weights=w)
    dT = torch.from_numpy(rng.standard_normal((B, 2, D)).astype(np.float32))
    u = sparse_updates(dT, j, 1)[0]
    table = np.zeros((rows, D), np.float32)
    W.sparse_sgd_update_jagged_weighted(table, j.values.numpy(), j.offsets.numpy(), w, dT[:, 1].numpy(), -1.0)
    assert np.allclose(uncompress(u, rows).numpy(), table, rtol=1e-6, atol=1e-6)


_ARGS_PROGRAM = r"""
#include <stdio.h>
#include "common.cuh"
// Handles built on the host only: every check below runs before the entry point touches the device.
int main() {
    dlrmb_tables t;
    t.ntab = 2;
    t.max_lookups = 100;
    t.D = 8;
    int64_t L[300];
    for (int i = 0; i < 300; ++i) L[i] = 1;
    int64_t Lz[2] = {0, 0};
    int64_t off[1] = {0};
    int32_t v[1] = {0};
    float out[8], w[2] = {1.f, 1.f};
    float dT[16] __attribute__((aligned(16)));
    auto show = [](const char* what, int rc) { printf("%s %d %s\n", what, rc, dlrmb_last_error()); };
    show("weights", dlrmb_embedding_fwd_jagged_weighted(&t, v, off, nullptr, 8, 0, 1, L, out, 3, 1, nullptr));
    show("weights_sort", dlrmb_embedding_sort_jagged_weighted(&t, v, off, nullptr, 8, 0, 1, L, nullptr));
    show("weights_fwd_sort", dlrmb_embedding_fwd_sort_jagged_weighted(&t, v, off, nullptr, 4, 0, 1, L, out, 3, 1, nullptr));
    show("dw", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, L, dT, 3, 1, nullptr, nullptr));
    show("dT", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, L, nullptr, 3, 1, out, nullptr));
    show("slots", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, L, dT, 2, 1, out, nullptr));
    show("align", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, L, dT + 1, 3, 1, out, nullptr));
    show("out", dlrmb_embedding_fwd_jagged_weighted(&t, v, off, w, 8, 0, 1, L, nullptr, 3, 1, nullptr));
    show("offsets", dlrmb_embedding_sort_jagged_weighted(&t, v, nullptr, w, 8, 0, 1, L, nullptr));
    show("values", dlrmb_embedding_fwd_sort_jagged_weighted(&t, nullptr, off, w, 8, 0, 1, L, out, 3, 1, nullptr));
    show("lengths", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, nullptr, dT, 3, 1, out, nullptr));
    show("handle", dlrmb_embedding_sort_jagged_weighted(nullptr, v, off, w, 8, 0, 1, L, nullptr));
    show("idx_bytes", dlrmb_embedding_weight_grad_jagged(&t, v, off, 2, 0, 1, L, dT, 3, 1, out, nullptr));
    show("base", dlrmb_embedding_fwd_jagged_weighted(&t, v, off, w, 8, 2, 1, L, out, 3, 1, nullptr));
    L[1] = 101;
    show("max_lookups", dlrmb_embedding_fwd_jagged_weighted(&t, v, off, w, 8, 0, 1, L, out, 3, 1, nullptr));
    L[1] = -1;
    show("negative", dlrmb_embedding_weight_grad_jagged(&t, v, off, 8, 0, 1, L, dT, 3, 1, out, nullptr));
    L[1] = 1;
    // no lookup at all: null weights / dw are allowed, so the next check to fail is the last argument's
    show("empty_weights", dlrmb_embedding_fwd_jagged_weighted(&t, nullptr, off, nullptr, 8, 0, 1, Lz, nullptr, 3, 1, nullptr));
    show("empty_dw", dlrmb_embedding_weight_grad_jagged(&t, nullptr, off, 8, 0, 1, Lz, nullptr, 3, 1, nullptr, nullptr));
    t.ntab = 257;
    show("ntab", dlrmb_embedding_sort_jagged_weighted(&t, v, off, w, 8, 0, 1, L, nullptr));
    return 0;
}
"""


def test_c_entry_points_refuse_bad_arguments(tmp_path):
    from dlrm_jl_b200.csrc import build
    lib = build.build()
    src = tmp_path / "jagged_weighted_args.cu"
    src.write_text(_ARGS_PROGRAM)
    exe = tmp_path / "jagged_weighted_args"
    subprocess.run([build._nvcc(), "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", build.HERE, str(src),
                    "-o", str(exe), "-L", os.path.dirname(lib), "-ldlrm_b200", "-Xlinker", "-rpath=" + os.path.dirname(lib)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = {line.split(" ", 1)[0]: line.split(" ", 2)[1:] for line in out.splitlines()}
    want = {"weights": "weights is null", "weights_sort": "weights is null", "weights_fwd_sort": "weights is null",
            "dw": "dw is null", "dT": "dT is null", "slots": "slots = 2 too small for slot0 = 1 + 2 tables",
            "align": "dT must be 16-byte aligned", "out": "out is null", "offsets": "offsets is null",
            "values": "values is null", "lengths": "L (per-table lookup counts) is null", "handle": "null tables handle",
            "idx_bytes": "idx_bytes must be 4 or 8", "base": "idx_base must be 0 or 1",
            "max_lookups": "L[1] = 101 exceeds max_lookups = 100", "negative": "L[1] = -1",
            "empty_weights": "out is null", "empty_dw": "dT is null", "ntab": "up to 256 tables (handle has 257)"}
    assert set(got) == set(want)
    for what, msg in want.items():
        rc, text = got[what]
        assert int(rc) == 1, (what, rc, text)        # DLRMB_EINVAL
        assert msg in text, (what, text)
