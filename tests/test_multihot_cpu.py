"""Per-table pooling factors (multi-hot with mixed hotness) without a GPU: packing of the reference's
mixed index containers, argument errors, the sharded path's refusal, and the oracle on mixed P."""
import numpy as np
import pytest
import torch

from oracle import oracle as O


def _cpu():
    return torch.device("cpu")


def test_mixed_container_packs_table_major():
    from dlrm_jl_b200.embedding import PackedIndices, _as_index_tensor
    rng = np.random.default_rng(0)
    B = 5
    vec = rng.integers(0, 9, size=B)                                # one-hot table given as a vector
    m3 = rng.integers(0, 9, size=(B, 3)).astype(np.int32)
    m7 = torch.from_numpy(rng.integers(0, 9, size=(B, 7)))         # int64
    p = _as_index_tensor([vec, m3, m7], 3, _cpu())
    assert isinstance(p, PackedIndices)
    assert p.P == (1, 3, 7) and p.B == B and len(p) == 3
    assert p.flat.dtype == torch.int64 and p.flat.numel() == B * 11
    ref = np.concatenate([vec.reshape(-1), m3.reshape(-1), m7.numpy().reshape(-1)])
    assert np.array_equal(p.flat.numpy(), ref)                      # reduce(vcat, vec.(sparse))
    for k, a in enumerate([vec.reshape(B, 1), m3, m7.numpy()]):
        assert np.array_equal(p[k].numpy(), a)
    assert list(p.P_array()) == [1, 3, 7]


def test_mixed_int32_stays_int32_and_uniform_keeps_tensor():
    from dlrm_jl_b200.embedding import PackedIndices, _as_index_tensor
    B = 4
    p = _as_index_tensor([np.zeros((B, 2), np.int32), np.ones((B, 1), np.uint32)], 2, _cpu())
    assert isinstance(p, PackedIndices) and p.flat.dtype == torch.int32 and p.P == (2, 1)
    u = _as_index_tensor([np.zeros((B, 2), np.int64), np.ones((B, 2), np.int64)], 2, _cpu())
    assert isinstance(u, torch.Tensor) and tuple(u.shape) == (2, B, 2)


def test_mixed_container_errors():
    from dlrm_jl_b200.embedding import _as_index_tensor
    with pytest.raises(ValueError, match="3 tables, got 2"):
        _as_index_tensor([np.zeros((4, 1), np.int64), np.zeros((4, 2), np.int64)], 3, _cpu())
    with pytest.raises(ValueError, match="same batch"):
        _as_index_tensor([np.zeros((4, 1), np.int64), np.zeros((5, 2), np.int64)], 2, _cpu())


def test_sparse_updates_slice_packed_indices():
    from dlrm_jl_b200.embedding import _as_index_tensor, sparse_updates, uncompress
    rng = np.random.default_rng(1)
    B, D, rows = 6, 3, [5, 8]
    idx = [rng.integers(0, rows[0], size=(B, 1)), rng.integers(0, rows[1], size=(B, 4))]
    p = _as_index_tensor(idx, 2, _cpu())
    dT = torch.from_numpy(rng.standard_normal((B, 3, D)).astype(np.float32))
    ups = sparse_updates(dT, p, 1)
    assert len(ups) == 2
    for k, u in enumerate(ups):
        assert np.array_equal(u.indices.numpy(), idx[k])
        ref = O.uncompress(dT[:, 1 + k].numpy(), idx[k], rows[k])
        assert np.allclose(uncompress(u, rows[k]).numpy(), ref, rtol=1e-6, atol=1e-6)


def test_sharded_path_rejects_mixed_pooling():
    from dlrm_jl_b200.embedding import _as_index_tensor
    from dlrm_jl_b200.sharded import TableSharding, exchange_indices
    sh = TableSharding.build([10, 20, 30], 2)
    mixed = [np.zeros((4, 1), np.int64), np.zeros((4, 3), np.int64), np.zeros((4, 1), np.int64)]
    with pytest.raises(ValueError, match="per-table pooling factors"):
        exchange_indices(mixed, sh, 0)
    with pytest.raises(ValueError, match="table-sharded"):
        exchange_indices(_as_index_tensor(mixed, 3, _cpu()), sh, 0)


def test_oracle_mixed_pooling_against_naive_loops():
    rng = np.random.default_rng(2)
    B, D, rows, P = 7, 4, [3, 50, 9], [1, 5, 27]
    tables = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = [rng.integers(0, r, size=(B, p)) for r, p in zip(rows, P)]
    T = O.lookup(tables, idx, slot0=1)
    for k in range(3):
        for b in range(B):
            acc = np.float32(0) * tables[k][0]
            for p in range(P[k]):
                acc = (acc + tables[k][idx[k][b, p]]).astype(np.float32)
            assert np.array_equal(T[b, 1 + k], acc)
    dT = rng.standard_normal((B, 4, D)).astype(np.float32)
    for k in range(3):
        got = tables[k].copy()
        O.sparse_sgd_update(got, idx[k], np.ascontiguousarray(dT[:, 1 + k]), 0.1)
        ref = tables[k].copy()
        for r in range(rows[k]):
            acc = np.zeros(D, np.float32)
            for b in range(B):
                for p in range(P[k]):
                    if idx[k][b, p] == r:
                        acc = (acc + dT[b, 1 + k]).astype(np.float32)
            if any(idx[k].reshape(-1) == r):
                ref[r] = (ref[r] - (np.float32(0.1) * acc).astype(np.float32)).astype(np.float32)
        assert np.array_equal(got, ref)
