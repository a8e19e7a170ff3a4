"""Jagged (variable-length) bags without a GPU: the JaggedIndices container, the NumPy reference against
torch.nn.functional.embedding_bag (forward and autograd gradient, sum and mean, empty bags), and the C entry
points' refusal of bad arguments before any CUDA call."""
import os
import subprocess

import numpy as np
import pytest
import torch

from tests import jagged_oracle as J

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_constructors_and_rebasing():
    from dlrm_jl_b200.embedding import JaggedIndices
    j = JaggedIndices.from_bags([[[1, 2], [], [3]], [[4], [5, 6, 7], []]], pooling="mean")
    assert j.L == (3, 4) and j.B == 3 and len(j) == 2 and j.pooling == "mean" and j.pooling_code == 1
    assert j.offsets.tolist() == [0, 2, 2, 3, 4, 7, 7] and j.values.dtype == torch.int64
    v1, o1 = j[1]
    assert v1.tolist() == [4, 5, 6, 7] and o1.tolist() == [0, 1, 4, 4]
    v0, o0 = j[0]
    assert v0.tolist() == [1, 2, 3] and o0.tolist() == [0, 2, 2, 3]
    assert list(j.L_array()) == [3, 4]
    k = JaggedIndices.from_lengths(np.arange(5, dtype=np.int32), [[2, 0], [0, 3]])
    assert k.values.dtype == torch.int32 and k.offsets.dtype == torch.int32 and k.offsets.tolist() == [0, 2, 2, 2, 5]
    assert k.L == (2, 3) and k.pooling == "sum"


def test_from_dense_is_constant_lengths():
    from dlrm_jl_b200.embedding import JaggedIndices, _as_index_tensor
    idx = torch.arange(24, dtype=torch.int32).reshape(2, 4, 3)
    j = JaggedIndices.from_dense(idx)
    assert j.L == (12, 12) and j.B == 4 and j.offsets.tolist() == list(range(0, 25, 3))
    assert torch.equal(j.values, idx.reshape(-1))
    p = _as_index_tensor([np.zeros((4, 1), np.int64), np.ones((4, 5), np.int64)], 2, torch.device("cpu"))
    jp = JaggedIndices.from_dense(p, pooling="mean")
    assert jp.L == (4, 20) and jp.offsets.tolist() == [0, 1, 2, 3, 4, 9, 14, 19, 24] and jp.pooling == "mean"
    assert _as_index_tensor(jp, 2, torch.device("cpu")).L == (4, 20)


def test_container_errors():
    from dlrm_jl_b200.embedding import JaggedIndices, _as_index_tensor
    j = JaggedIndices.from_bags([[[1], [2]], [[3], []]])
    with pytest.raises(ValueError, match="3 tables, got 2"):
        _as_index_tensor(j, 3, torch.device("cpu"))
    with pytest.raises(ValueError, match="sum to 3, values holds 4"):
        JaggedIndices.from_lengths(np.arange(4), [[1, 2]])
    with pytest.raises(ValueError, match=">= 0"):
        JaggedIndices.from_lengths(np.arange(1), [[2, -1]])
    with pytest.raises(ValueError, match="share one dtype"):
        JaggedIndices(torch.zeros(2, dtype=torch.int32), torch.tensor([0, 1, 2]), (2,), 2)
    with pytest.raises(ValueError, match="same number of bags"):
        JaggedIndices.from_bags([[[1], [2]], [[3]]])
    with pytest.raises(ValueError, match="pooling"):
        JaggedIndices.from_bags([[[1]]], pooling="max")
    with pytest.raises(ValueError, match="ntab \\* B \\+ 1"):
        JaggedIndices(torch.zeros(2, dtype=torch.int64), torch.tensor([0, 2]), (2,), 2)


def _torch_reference(table, values, offsets, mode, g):
    w = torch.from_numpy(table).requires_grad_(True)
    out = torch.nn.functional.embedding_bag(torch.from_numpy(values), w, torch.from_numpy(offsets[:-1]), mode=mode,
                                            include_last_offset=False)
    out.backward(torch.from_numpy(g))
    return out.detach().numpy(), w.grad.numpy()


@pytest.mark.parametrize("mode", ["sum", "mean"])
def test_oracle_against_torch_embedding_bag(mode):
    rng = np.random.default_rng(3 if mode == "sum" else 4)
    rows, D, B = 40, 8, 33
    table = rng.standard_normal((rows, D)).astype(np.float32)
    n = rng.integers(0, 7, size=B)
    n[[0, 5, B - 1]] = 0                                   # empty bags, the last one included
    n[7] = 1
    offsets = np.zeros(B + 1, np.int64)
    np.cumsum(n, out=offsets[1:])
    values = rng.integers(0, rows, size=int(n.sum())).astype(np.int64)
    values[:3] = 11                                        # duplicates across bags
    out = J.lookup_jagged([table], values, offsets, B, mode)[:, 0]
    g = rng.standard_normal((B, D)).astype(np.float32)
    ref_out, ref_grad = _torch_reference(table, values, offsets, mode, g)
    assert np.allclose(out, ref_out, rtol=1e-6, atol=1e-6)
    assert np.all(out[n == 0] == 0) and not np.signbit(out[n == 0]).any()
    if mode == "sum":
        assert np.array_equal(out, ref_out)                # sequential fp32 adds, as torch on the CPU
    lr = 0.5
    got = table.copy()
    J.sparse_sgd_update_jagged(got, values, offsets, g, lr, mode)
    assert np.allclose(got, table - lr * ref_grad, rtol=1e-5, atol=1e-6)
    untouched = np.setdiff1d(np.arange(rows), values)
    assert np.array_equal(got[untouched], table[untouched])


def test_oracle_mean_uses_rounded_reciprocal():
    table = np.array([[1.0], [2.0], [4.0]], np.float32)
    out = J.lookup_jagged([table], np.array([0, 1, 2]), np.array([0, 3]), 1, "mean")
    assert out[0, 0, 0] == np.float32(7.0) * (np.float32(1.0) / np.float32(3.0))


def test_uncompress_jagged_matches_oracle_gradient():
    from dlrm_jl_b200.embedding import JaggedIndices, sparse_updates, uncompress
    rng = np.random.default_rng(5)
    rows, D, B = 9, 4, 6
    for pooling in ("sum", "mean"):
        j = JaggedIndices.from_lengths(rng.integers(0, rows, size=10), [[2, 0, 3, 1, 4, 0]], pooling)
        dT = torch.from_numpy(rng.standard_normal((B, 2, D)).astype(np.float32))
        u = sparse_updates(dT, j, 1)[0]
        table = np.zeros((rows, D), np.float32)
        J.sparse_sgd_update_jagged(table, j.values.numpy(), j.offsets.numpy(), dT[:, 1].numpy(), -1.0, pooling)
        assert np.allclose(uncompress(u, rows).numpy(), table, rtol=1e-6, atol=1e-6)


_ARGS_PROGRAM = r"""
#include <stdio.h>
#include "common.cuh"
// Handles built on the host only: every check below runs before the entry point touches the device.
int main() {
    dlrmb_tables t;
    t.ntab = 2;
    t.max_lookups = 100;
    int64_t L[300];
    for (int i = 0; i < 300; ++i) L[i] = 1;
    int64_t off[1] = {0};
    int32_t v[1] = {0};
    float out[1];
    auto show = [](const char* what, int rc) { printf("%s %d %s\n", what, rc, dlrmb_last_error()); };
    show("pooling", dlrmb_embedding_fwd_jagged(&t, v, off, 8, 0, 1, L, 2, out, 3, 1, nullptr));
    show("offsets", dlrmb_embedding_sort_jagged(&t, v, nullptr, 8, 0, 1, L, 0, nullptr));
    show("values", dlrmb_embedding_fwd_sort_jagged(&t, nullptr, off, 8, 0, 1, L, 0, out, 3, 1, nullptr));
    show("lengths", dlrmb_check_indices_jagged(&t, v, off, 8, 0, 1, nullptr, 1));
    show("handle", dlrmb_embedding_sort_jagged(nullptr, v, off, 8, 0, 1, L, 0, nullptr));
    L[1] = 101;
    show("max_lookups", dlrmb_embedding_fwd_jagged(&t, v, off, 8, 0, 1, L, 0, out, 3, 1, nullptr));
    L[1] = -1;
    show("negative", dlrmb_embedding_sort_jagged(&t, v, off, 8, 0, 1, L, 0, nullptr));
    L[1] = 1;
    t.ntab = 257;
    show("ntab", dlrmb_check_indices_jagged(&t, v, off, 8, 0, 1, L, 1));
    return 0;
}
"""


def test_c_entry_points_refuse_bad_arguments(tmp_path):
    from dlrm_jl_b200.csrc import build
    lib = build.build()
    src = tmp_path / "jagged_args.cu"
    src.write_text(_ARGS_PROGRAM)
    exe = tmp_path / "jagged_args"
    subprocess.run([build._nvcc(), "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", build.HERE, str(src),
                    "-o", str(exe), "-L", os.path.dirname(lib), "-ldlrm_b200", "-Xlinker", "-rpath=" + os.path.dirname(lib)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = {line.split(" ", 1)[0]: line.split(" ", 2)[1:] for line in out.splitlines()}
    want = {"pooling": "pooling must be 0 (sum) or 1 (mean)", "offsets": "offsets is null", "values": "values is null",
            "lengths": "L (per-table lookup counts) is null", "handle": "null tables handle",
            "max_lookups": "L[1] = 101 exceeds max_lookups = 100", "negative": "L[1] = -1",
            "ntab": "up to 256 tables (handle has 257)"}
    for what, msg in want.items():
        rc, text = got[what]
        assert int(rc) == 1, (what, rc, text)        # DLRMB_EINVAL
        assert msg in text, (what, text)
