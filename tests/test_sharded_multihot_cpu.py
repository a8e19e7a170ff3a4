"""Table-sharded embeddings with per-table pooling factors (mixed multi-hot) without a GPU: the
lookup-weighted shard plan (C ABI and Python), and world-size-2/3 gloo runs of the index exchange and
of a whole ShardedEmbedding step with the CPU oracle as the injected compute."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dlrm_jl_b200.sharded import ShardedEmbedding, TableSharding, exchange_indices_mp

MLPERF_HOTNESS = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _c_plan(rows, P, world):
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    n = len(rows)
    owner = (C.c_int32 * n)()
    _lib.check(lib.dlrmb_shard_plan_mp(n, (C.c_int64 * n)(*[int(r) for r in rows]), (C.c_int32 * n)(*[int(p) for p in P]),
                                       world, owner))
    return list(owner)


def _terabyte_rows(cap=40_000_000):
    from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES
    return [min(r, cap) for r in TERABYTE_EMBEDDING_SIZES]


def test_plan_mp_matches_python_plan():
    """dlrmb_shard_plan_mp deals the tables exactly as TableSharding.build(rows, world, P) does: the MLPerf
    hotness list on Terabyte-shaped tables, Kaggle sizes with random P, ties, and more ranks than tables."""
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES
    rng = np.random.default_rng(11)
    kaggle = list(KAGGLE_EMBEDDING_SIZES)
    cases = [(_terabyte_rows(), MLPERF_HOTNESS),
             (kaggle, list(rng.integers(1, 30, size=len(kaggle)))),
             (kaggle, list(rng.integers(1, 4, size=len(kaggle)))),
             ([7, 7, 7, 7, 7], [2, 1, 2, 1, 2]),                          # ties in P and rows
             ([5, 1000, 5, 1000, 3], [4, 4, 1, 1, 4]),
             ([9, 9, 9], [1, 2, 3]),                                      # world > ntab below
             ([1], [5])]
    cases += [(list(rng.integers(1, 10 ** 7, size=int(n))), list(rng.integers(1, 120, size=int(n))))
              for n in rng.integers(2, 40, size=6)]
    for rows, P in cases:
        for world in (1, 2, 3, 4, 8, 16):
            sh = TableSharding.build(rows, world, P)
            assert _c_plan(rows, P, world) == sh.owner, (rows, P, world)
            assert sorted(k for l in sh.local for k in l) == list(range(len(rows)))


def test_plan_mp_equal_P_is_the_snake_plan():
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES
    lib = _lib.load()
    for rows in (list(KAGGLE_EMBEDDING_SIZES), _terabyte_rows(), [7, 7, 7], [5, 1000, 5, 1000, 3]):
        for world in (1, 2, 3, 4, 8, 16):
            n = len(rows)
            snake = (C.c_int32 * n)()
            _lib.check(lib.dlrmb_shard_plan(n, (C.c_int64 * n)(*rows), world, snake))
            for p in (1, 3, 100):
                assert _c_plan(rows, [p] * n, world) == list(snake)
                assert TableSharding.build(rows, world, [p] * n).owner == list(snake)
            assert TableSharding.build(rows, world).owner == list(snake)


def test_plan_mp_reproduces_mlperf_loads():
    """Sum of P_k per rank on Terabyte-shaped tables (capped at 40M rows) with the MLPerf hotness list:
    107 / 107 at 2 GPUs, the hotness-100 table alone on its rank at 4 and 8 (the best table-wise
    placement can do: that table is 100 of the 214 lookups per sample)."""
    rows = _terabyte_rows()
    assert sum(MLPERF_HOTNESS) == 214
    loads = {w: TableSharding.build(rows, w, MLPERF_HOTNESS).lookups_per_rank() for w in (2, 4, 8)}
    assert loads[2] == [107, 107]
    assert loads[4] == [100, 38, 38, 38]
    assert max(loads[8]) == 100
    for w in (4, 8):
        sh = TableSharding.build(rows, w, MLPERF_HOTNESS)
        big = MLPERF_HOTNESS.index(100)
        assert sh.local[sh.owner[big]] == [big]
    # the snake plan, for comparison: the busiest rank carries 163, 141 and 110 lookups per sample
    snake = {w: TableSharding.build(rows, w) for w in (2, 4, 8)}
    snake_load = {w: [sum(MLPERF_HOTNESS[k] for k in l) for l in s.local] for w, s in snake.items()}
    assert snake_load[2] == [163, 51] and snake_load[4] == [22, 27, 24, 141]
    assert snake_load[8] == [10, 9, 19, 110, 31, 5, 18, 12]
    for w in (2, 4, 8):
        assert _c_plan(rows, MLPERF_HOTNESS, w) == TableSharding.build(rows, w, MLPERF_HOTNESS).owner


def test_plan_mp_errors():
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    rows = (C.c_int64 * 3)(1, 2, 3)
    P = (C.c_int32 * 3)(1, 2, 3)
    out = (C.c_int32 * 3)()
    assert lib.dlrmb_shard_plan_mp(3, rows, None, 2, out) == _lib.EINVAL
    assert b"P" in lib.dlrmb_last_error()
    assert lib.dlrmb_shard_plan_mp(3, rows, (C.c_int32 * 3)(1, 0, 3), 2, out) == _lib.EINVAL
    assert b"P[1] = 0" in lib.dlrmb_last_error()
    assert lib.dlrmb_shard_plan_mp(3, rows, P, 0, out) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_mp(0, rows, P, 2, out) == _lib.EINVAL
    with pytest.raises(ValueError):
        TableSharding.build([1, 2, 3], 2, [1, 0, 3])
    with pytest.raises(ValueError):
        TableSharding.build([1, 2, 3], 2, [1, 2])


def test_int_P_handle_keeps_refusing_mixed_widths():
    se = ShardedEmbedding([5, 6], 4, 0, 2, lambda *a: None, lambda *a, **k: None)
    with pytest.raises(ValueError, match="per-table pooling factors"):
        se.lookup([np.zeros((3, 1), np.int64), np.zeros((3, 2), np.int64)], torch.zeros(1, requires_grad=True))


def test_mixed_handle_checks_batch_widths():
    se = ShardedEmbedding([5, 6], 4, 0, 2, lambda *a: None, lambda *a, **k: None, P=[1, 2])
    with pytest.raises(ValueError, match="differ from the handle's P"):
        se._indices([np.zeros((3, 2), np.int64), np.zeros((3, 1), np.int64)])
    p = se._indices([np.zeros((3, 1), np.int64), np.ones((3, 2), np.int64)])
    assert p.P == (1, 2) and p.B == 3


# ---- gloo runs ----------------------------------------------------------------------------------
ROWS = [50, 7, 400, 3, 120, 33, 9, 61]
HOT = [3, 1, 7, 2, 1, 12, 1, 5]
D, BL = 8, 6


def _owner_layout(idx_all, sh, rank):
    """numpy restatement of the owner layout: owned tables ascending, each [B_global][P_k], rank-major."""
    parts = [np.concatenate([idx_all[h][k] for h in range(sh.world)], axis=0).reshape(-1) for k in sh.local[rank]]
    return np.concatenate(parts) if parts else np.zeros(0, np.int64)


def _worker(rank, world, port, q):
    from dlrm_jl_b200.embedding import PackedIndices, _as_index_tensor
    from oracle import oracle as O
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rng = np.random.default_rng(17)                      # same tables / batches on every rank
        tables = [rng.standard_normal((r, D)).astype(np.float32) for r in ROWS]
        idx_all = [[rng.integers(0, r, size=(BL, p)) for r, p in zip(ROWS, HOT)] for _ in range(world)]
        x_all = [rng.standard_normal((BL, D)).astype(np.float32) for _ in range(world)]
        F = 1 + len(ROWS)
        gz_all = [rng.standard_normal((BL, D + F * (F - 1) // 2)).astype(np.float32) for _ in range(world)]
        sh = TableSharding.build(ROWS, world, HOT)
        mine = sh.local[rank]

        # index exchange alone, int32 and int64
        ok_x = True
        for dt in (np.int32, np.int64):
            packed = _as_index_tensor([a.astype(dt) for a in idx_all[rank]], len(ROWS), torch.device("cpu"))
            owned = exchange_indices_mp(packed, sh, rank)
            ok_x = ok_x and isinstance(owned, PackedIndices) and owned.P == tuple(HOT[k] for k in mine)
            ok_x = ok_x and owned.B == BL * world and owned.flat.dtype == packed.flat.dtype
            ok_x = ok_x and np.array_equal(owned.flat.numpy(), _owner_layout(idx_all, sh, rank).astype(dt))

        # a whole step with the oracle as the injected compute
        local_tables = [tables[k].copy() for k in mine]

        def lookup_fn(idx, out, slot0):
            out.copy_(torch.from_numpy(O.lookup(local_tables, [idx[j].numpy() for j in range(len(idx))], slot0=slot0)))

        def update_fn(idx, g, lr, slot0, presorted=False):
            for j in range(len(mine)):
                O.sparse_sgd_update_fast(local_tables[j], idx[j].numpy(), np.ascontiguousarray(g[:, slot0 + j].numpy()), lr)

        se = ShardedEmbedding(ROWS, D, rank, world, lookup_fn, update_fn, P=HOT)
        assert se.sharding.owner == sh.owner
        anchor = torch.zeros(1, requires_grad=True)
        T = se.lookup(idx_all[rank], anchor)                 # the reference's mixed list
        ref_T = O.lookup(tables, idx_all[rank], slot0=1)
        ok_fwd = np.array_equal(T.detach().numpy()[:, 1:], ref_T[:, 1:])
        Tn = T.detach().numpy().copy()
        Tn[:, 0] = x_all[rank]
        _dx, dT = O.interaction_bwd(gz_all[rank], Tn)
        T.backward(torch.from_numpy(dT))
        se.update(0.5)
        ref = [t.copy() for t in tables]
        dT_glob = []
        for r in range(world):
            Tr = O.lookup(tables, idx_all[r], slot0=1)
            Tr[:, 0] = x_all[r]
            dT_glob.append(O.interaction_bwd(gz_all[r], Tr)[1])
        dT_glob = np.concatenate(dT_glob, axis=0)
        for k in range(len(ROWS)):
            idx_glob = np.concatenate([idx_all[r][k] for r in range(world)], axis=0)
            O.sparse_sgd_update_fast(ref[k], idx_glob, np.ascontiguousarray(dT_glob[:, 1 + k]), 0.5)
        ok_upd = all(np.array_equal(local_tables[j], ref[k]) for j, k in enumerate(mine))
        q.put((rank, bool(ok_x), bool(ok_fwd), bool(ok_upd), ""))
    except Exception as exc:  # noqa: BLE001
        import traceback
        q.put((rank, False, False, False, repr(exc) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_mixed_pooling_matches_unsharded_oracle(world):
    """exchange_indices_mp equals a numpy packing of the owner layout; a ShardedEmbedding with per-table P
    gives the unsharded oracle's pooled rows and updated tables bit for bit."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, ok_x, ok_fwd, ok_upd, err in res:
        assert not err, f"rank {rank}: {err}"
        assert ok_x, f"rank {rank}: exchange_indices_mp differs from the owner layout"
        assert ok_fwd, f"rank {rank}: forward exchange mismatch"
        assert ok_upd, f"rank {rank}: sharded update differs from unsharded oracle"
