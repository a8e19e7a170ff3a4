"""Column-wise sharding of hot embedding tables without a GPU: the plan (C ABI and Python, same rule and same
result), its coverage and balance on the MLPerf hotness list, argument errors, and gloo runs of a whole
ShardedEmbedding step with a split table against the unsharded oracle, bit for bit."""
import ctypes as C
import os
import socket
from fractions import Fraction

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dlrm_jl_b200.sharded import ShardedEmbedding, TableSharding, exchange_indices_cw

MLPERF_HOTNESS = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _c_plan_cw(rows, P, world, D, S):
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    n = len(rows)
    shards, owner = (C.c_int32 * n)(), (C.c_int32 * (n * S))()
    _lib.check(lib.dlrmb_shard_plan_cw(n, (C.c_int64 * n)(*[int(r) for r in rows]), (C.c_int32 * n)(*[int(p) for p in P]),
                                       world, D, S, shards, owner))
    return list(shards), [list(owner[k * S:(k + 1) * S]) for k in range(n)]


def _c_plan_mp(rows, P, world):
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


def _cases():
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES
    rng = np.random.default_rng(23)
    kaggle = list(KAGGLE_EMBEDDING_SIZES)
    cases = [(_terabyte_rows(), MLPERF_HOTNESS),
             (kaggle, list(rng.integers(1, 30, size=len(kaggle)))),
             (kaggle, [1] * len(kaggle)),                                   # equal P
             ([7, 7, 7, 7, 7], [2, 1, 2, 1, 2]),                            # ties in P and rows
             ([5, 1000, 5, 1000, 3], [40, 40, 1, 1, 4]),
             ([9, 9, 9], [1, 2, 30]),                                       # world > ntab below
             ([1], [5])]
    cases += [(list(rng.integers(1, 10 ** 7, size=int(n))), list(rng.integers(1, 120, size=int(n))))
              for n in rng.integers(2, 40, size=8)]
    return cases


def _check_plan(sh, rows, P, world, D):
    """Every column of every table covered exactly once, no rank with two slices of a table, slices contiguous."""
    for k in range(len(rows)):
        c = sh.shards[k] if sh.split else 1
        holders = sh.holders[k] if sh.split else [sh.owner[k]]
        assert c & (c - 1) == 0 and len(holders) == c and len(set(holders)) == c
        assert all(0 <= h < world for h in holders)
        cols = np.zeros(D, np.int32)
        for j in range(c):
            cols[j * D // c:(j + 1) * D // c] += 1
        assert (cols == 1).all()
        for r in range(world):
            assert (k in sh.local[r]) == (r in holders)
    for r in range(world):
        ks = [k for _c, g in sh.groups(r) for k in g]
        assert sorted(ks) == sh.local[r] and len(set(ks)) == len(ks)


@pytest.mark.parametrize("S", [1, 2, 4, 8])
def test_plan_cw_matches_python_plan(S):
    """dlrmb_shard_plan_cw gives exactly TableSharding.build(rows, world, P, D=D, max_col_shards=S)."""
    D = 128
    for rows, P in _cases():
        for world in (1, 2, 3, 4, 8, 16):
            sh = TableSharding.build(rows, world, P, D=D, max_col_shards=S)
            shards, owner = _c_plan_cw(rows, P, world, D, S)
            if sh.split:
                assert shards == list(sh.shards), (rows, P, world, S)
                assert owner == [h + [-1] * (S - len(h)) for h in sh.holders], (rows, P, world, S)
            else:
                assert shards == [1] * len(rows)
                assert owner == [[o] + [-1] * (S - 1) for o in sh.owner], (rows, P, world, S)
            _check_plan(sh, rows, P, world, D)


def test_plan_cw_without_split_is_the_table_wise_plan():
    D = 64
    for rows, P in _cases():
        for world in (1, 2, 3, 4, 8, 16):
            base = TableSharding.build(rows, world, P)
            assert _c_plan_mp(rows, P, world) == base.owner
            one = TableSharding.build(rows, world, P, D=D, max_col_shards=1)
            assert one.owner == base.owner and not one.split
            assert _c_plan_cw(rows, P, world, D, 1) == ([1] * len(rows), [[o] for o in base.owner])
            for S in (2, 4, 8):
                sh = TableSharding.build(rows, world, P, D=D, max_col_shards=S)
                if not sh.split:
                    assert sh.owner == base.owner and sh.local == base.local
    # equal P with at least as many tables as ranks never splits: the snake plan
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES
    rows = list(KAGGLE_EMBEDDING_SIZES)
    for world in (2, 4, 8, 16):
        sh = TableSharding.build(rows, world, None, D=D, max_col_shards=8)
        assert not sh.split and sh.owner == TableSharding.build(rows, world).owner


def test_plan_cw_reproduces_mlperf_loads():
    """Busiest rank in lookups per sample weighted by width (Terabyte rows capped at 40M, MLPerf hotness, S = 8):
    107 / 72 / 54 / 27 at 2 / 3 / 4 / 8 GPUs against the table-wise 107 / 100 / 100 / 100."""
    rows = _terabyte_rows()
    want = {2: (107, {}), 3: (72, {20: 2}), 4: (54, {20: 2}), 8: (27, {20: 4, 21: 2})}
    for world, (busiest, splits) in want.items():
        sh = TableSharding.build(rows, world, MLPERF_HOTNESS, D=128, max_col_shards=8)
        loads = sh.lookups_per_rank()
        assert max(loads) == busiest, (world, loads)
        assert sum(loads) == 214
        got = {k: c for k, c in enumerate(sh.shards)} if sh.split else {}
        assert {k: c for k, c in got.items() if c > 1} == splits
        assert max(TableSharding.build(rows, world, MLPERF_HOTNESS).lookups_per_rank()) == (107 if world == 2 else 100)
    sh = TableSharding.build(rows, 8, MLPERF_HOTNESS, D=128, max_col_shards=8)
    assert all(isinstance(v, Fraction) for v in sh.lookups_per_rank())
    assert sum(sh.bytes_per_rank(128)) == sum(rows) * 128 * 4


def test_plan_cw_errors():
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    rows = (C.c_int64 * 3)(1, 2, 3)
    P = (C.c_int32 * 3)(1, 2, 3)
    shards, owner = (C.c_int32 * 3)(), (C.c_int32 * 24)()
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 2, 128, 3, shards, owner) == _lib.EINVAL
    assert b"power of two" in lib.dlrmb_last_error()
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 2, 24, 8, shards, owner) == _lib.EINVAL
    assert b"multiple of 4" in lib.dlrmb_last_error()
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 2, 128, 0, shards, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, rows, None, 2, 128, 2, shards, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, None, P, 2, 128, 2, shards, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 2, 128, 2, None, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 2, 128, 2, shards, None) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, rows, (C.c_int32 * 3)(1, 0, 3), 2, 128, 2, shards, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(0, rows, P, 2, 128, 2, shards, owner) == _lib.EINVAL
    assert lib.dlrmb_shard_plan_cw(3, rows, P, 0, 128, 2, shards, owner) == _lib.EINVAL
    for kw in ({"D": 128, "max_col_shards": 3}, {"D": 24, "max_col_shards": 8}, {"D": None, "max_col_shards": 2},
               {"D": 128, "max_col_shards": 0}):
        with pytest.raises(ValueError):
            TableSharding.build([1, 2, 3], 2, [1, 2, 3], **kw)
    with pytest.raises(ValueError):
        ShardedEmbedding([5, 6], 8, 0, 2, lambda *a: None, lambda *a: None, P=[1, 9], max_col_shards=4)


# ---- gloo runs ----------------------------------------------------------------------------------
ROWS = [50, 7, 400, 3, 120, 33, 9, 61]
HOT = [3, 1, 40, 2, 1, 12, 1, 5]          # table 2 is split at world >= 2
D, BL = 16, 6


def _worker(rank, world, port, uniform, q):
    from dlrm_jl_b200.embedding import PackedIndices, _as_index_tensor
    from oracle import oracle as O
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rng = np.random.default_rng(29)                      # same tables / batches on every rank
        rows = [5, 7, 9] if uniform else ROWS            # one P: more ranks than tables, so every table splits
        hot = [2, 2, 2] if uniform else HOT
        tables = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
        idx_all = [[rng.integers(0, r, size=(BL, p)) for r, p in zip(rows, hot)] for _ in range(world)]
        x_all = [rng.standard_normal((BL, D)).astype(np.float32) for _ in range(world)]
        F = 1 + len(rows)
        gz = [[rng.standard_normal((BL, D + F * (F - 1) // 2)).astype(np.float32) for _ in range(world)] for _ in range(2)]
        se_kw = {"max_col_shards": 4}
        sh = TableSharding.build(rows, world, None if uniform else hot, D=D, **se_kw)
        assert sh.split, "the test plan must split a table"
        groups = sh.groups(rank)

        # index exchange alone: each group's owner layout
        ok_x = True
        packed = _as_index_tensor([a.astype(np.int64) for a in idx_all[rank]], len(rows), torch.device("cpu"))
        if not isinstance(packed, PackedIndices):
            packed = PackedIndices(packed.reshape(-1), tuple(hot), BL)
        owned = exchange_indices_cw(packed, sh, rank)
        for (c, ks), o in zip(groups, owned):
            want = np.concatenate([np.concatenate([idx_all[h][k] for h in range(world)], 0).reshape(-1) for k in ks])
            ok_x = ok_x and o.P == tuple(hot[k] for k in ks) and o.B == BL * world and np.array_equal(o.flat.numpy(), want)

        # slices of the tables this rank holds, per group
        local = [[np.ascontiguousarray(tables[k][:, sh.slice_of(k, rank) * (D // c):(sh.slice_of(k, rank) + 1) * (D // c)])
                  for k in ks] for c, ks in groups]

        def lookup_fn(idx, out, slot0, g):
            out.copy_(torch.from_numpy(O.lookup(local[g], [idx[j].numpy() for j in range(len(idx))], slot0=slot0)))

        def update_fn(idx, grad, lr, slot0, presorted, g):
            for j in range(len(local[g])):
                O.sparse_sgd_update_fast(local[g][j], idx[j].numpy(), np.ascontiguousarray(grad[:, slot0 + j].numpy()), lr)

        se = ShardedEmbedding(rows, D, rank, world, lookup_fn, update_fn, P=None if uniform else hot, **se_kw)
        assert se.split and se.groups == groups
        ref = [t.copy() for t in tables]
        ok_fwd = ok_upd = True
        for step in range(2):
            anchor = torch.zeros(1, requires_grad=True)
            batch = (torch.from_numpy(np.stack(idx_all[rank])) if uniform else idx_all[rank])
            T = se.lookup(batch, anchor)
            ref_T = O.lookup(ref, idx_all[rank], slot0=1)
            ok_fwd = ok_fwd and np.array_equal(T.detach().numpy()[:, 1:], ref_T[:, 1:])
            Tn = T.detach().numpy().copy()
            Tn[:, 0] = x_all[rank]
            T.backward(torch.from_numpy(O.interaction_bwd(gz[step][rank], Tn)[1]))
            se.update(0.5)
            dT_glob = []
            for r in range(world):
                Tr = O.lookup(ref, idx_all[r], slot0=1)
                Tr[:, 0] = x_all[r]
                dT_glob.append(O.interaction_bwd(gz[step][r], Tr)[1])
            dT_glob = np.concatenate(dT_glob, axis=0)
            for k in range(len(rows)):
                idx_glob = np.concatenate([idx_all[r][k] for r in range(world)], axis=0)
                O.sparse_sgd_update_fast(ref[k], idx_glob, np.ascontiguousarray(dT_glob[:, 1 + k]), 0.5)
            for g, (c, ks) in enumerate(groups):
                for j, k in enumerate(ks):
                    c0 = sh.slice_of(k, rank) * (D // c)
                    ok_upd = ok_upd and np.array_equal(local[g][j], ref[k][:, c0:c0 + D // c])
        q.put((rank, bool(ok_x), bool(ok_fwd), bool(ok_upd), ""))
    except Exception as exc:  # noqa: BLE001
        import traceback
        q.put((rank, False, False, False, repr(exc) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,uniform", [(2, False), (3, False), (4, False), (4, True)])
def test_column_sharded_step_matches_unsharded_oracle(world, uniform):
    """Two steps of a ShardedEmbedding whose plan splits a table by columns (per-table P, and one P with more
    ranks than tables): the pooled rows and the updated tables are the unsharded oracle's, bit for bit."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, uniform, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, ok_x, ok_fwd, ok_upd, err in res:
        assert not err, f"rank {rank}: {err}"
        assert ok_x, f"rank {rank}: exchange_indices_cw differs from the owner layout"
        assert ok_fwd, f"rank {rank}: pooled rows differ from the unsharded oracle"
        assert ok_upd, f"rank {rank}: table slices differ from the unsharded oracle"
