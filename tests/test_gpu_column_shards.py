"""Column-wise sharding of hot embedding tables on the GPU.

Single process, local buffers standing in for the peers: the fused lookup with a destination map
(dlrmb_tables_set_dest_map) stores a column slice's pooled rows bit-exact into its column range and nothing
else, and leaves the same sort as an undivided handle; the scattering interaction backward by column pieces
(dlrmb_interaction_bwd_scatter_cols) reproduces dT; the list index scatter fills every holder; graph replay
equals eager; argument errors.

Two to four ranks sharing cuda:0 through CUDA IPC: the whole fused step with a split table against the
UNSHARDED oracle, with the slices read back through ShardedEmbedding.download.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O
from tests.test_gpu_sharded_multihot import (SGD_RTOL, _arm_watchdog, _collect, _dev, _free_port, _packed,
                                             _peer_buffers, _tables)

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

# rows, P, B_local, world: at B_global = 2048 the sorts are fused (L <= 4096), shared-memory and radix
BIG = ([7, 1000, 33, 50000, 64, 3, 40000], [1, 2, 3, 100, 7, 1, 12], 1024, 2)
SMALL = ([50, 7, 400, 3, 1200], [4, 1, 9, 2, 1], 85, 3)


@pytest.mark.parametrize("case,D,c,tdtype,idt,base,misaligned", [
    ("big", 128, 2, torch.float32, np.int64, 0, False),
    ("big", 128, 4, torch.bfloat16, np.int32, 1, False),
    ("big", 64, 2, torch.float32, np.int32, 1, True),         # peer buffers 4 bytes off 16: the VEC 1 path
    ("small", 32, 4, torch.float32, np.int64, 1, False),
    ("small", 64, 8, torch.bfloat16, np.int64, 0, True),
])
def test_fwd_p2p_dest_map_matches_whole_table_columns(case, D, c, tdtype, idt, base, misaligned):
    """A handle of column slices (width D / c, slice j_k of table k) pools into columns [j_k D / c, (j_k + 1) D / c)
    of its slots: bit-equal to those columns of dlrmb_embedding_fwd_mp over the whole tables, every other element
    untouched (NaN), and the sort it leaves equals the whole handle's."""
    rows, P, BL, W = BIG if case == "big" else SMALL
    Bg, w = BL * W, D // c
    rng = np.random.default_rng(D + c)
    arrays = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = [rng.integers(0, r, size=(Bg, p)) for r, p in zip(rows, P)]
    js = [(3 * k + 1) % c for k in range(len(rows))]
    slotmap = [2 + k for k in range(len(rows))]
    slots = slotmap[-1] + 1
    whole = _tables(arrays, Bg * max(P), tdtype)
    ref = torch.empty((Bg, len(rows), D), dtype=torch.float32, device=_dev())
    whole.lookup(_packed(idx, idt, base), ref, 0, base, sort=True)
    torch.cuda.synchronize()
    ref = ref.cpu().numpy()
    stored = [whole.download(k) for k in range(len(rows))]
    part = _tables([np.ascontiguousarray(stored[k][:, j * w:(j + 1) * w]) for k, j in enumerate(js)], Bg * max(P), tdtype)
    part.set_dest_map(slotmap, [j * w for j in js], D)
    bufs = _peer_buffers(W, BL, slots, D, misaligned)
    part.lookup_p2p(_packed(idx, idt, base), [b.data_ptr() for b in bufs], BL, slots, base, sort=True)
    torch.cuda.synchronize()
    for h, buf in enumerate(bufs):
        got = buf.cpu().numpy()
        want = np.full_like(got, np.nan)
        for k, j in enumerate(js):
            want[:, slotmap[k], j * w:(j + 1) * w] = ref[h * BL:(h + 1) * BL, k, j * w:(j + 1) * w]
        assert np.array_equal(got, want, equal_nan=True), h
    for k in range(len(rows)):
        a, b = whole.sort_dedup_export(k, Bg * P[k]), part.sort_dedup_export(k, Bg * P[k])
        assert all(np.array_equal(x, y) for x, y in zip(a, b)), k
    whole.close()
    part.close()


def _plain_bwd(F, d, B, seed):
    from dlrm_jl_b200.interact import interaction_bwd, interaction_width
    rng = np.random.default_rng(seed)
    T = torch.from_numpy(rng.standard_normal((B, F, d)).astype(np.float32)).to(_dev())
    dOut = torch.from_numpy(rng.standard_normal((B, interaction_width(F, d))).astype(np.float32)).to(_dev())
    dx, dT = interaction_bwd(dOut, T)
    return T, dOut, dx, dT


@pytest.mark.parametrize("F,d,general", [(27, 128, False), (27, 128, True), (5, 32, False), (8, 16, False)])
@pytest.mark.parametrize("Q", [1, 2, 4])
def test_interaction_bwd_scatter_cols_matches_dT_columns(F, d, general, Q):
    """Entry (f, q) receives columns [q d / Q, (q + 1) d / Q) of slot f's row: stored at a permuted place, every
    piece equals those columns of the plain backward's dT bit for bit, and dx is the plain dx."""
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    B, off = 300, 7
    T, dOut, dx_ref, dT_ref = _plain_bwd(F, d, B, F * d + Q)
    pw = d // Q
    G = torch.full((B + off, F, d), float("nan"), dtype=torch.float32, device=_dev())
    rows = [[0, 0, 0]] * Q
    for f in range(1, F):
        for q in range(Q):                       # piece q lands where piece (q + 1) % Q would sit
            rows.append([G.data_ptr(), F * d, f * d + ((q + 1) % Q) * pw])
    dests = torch.tensor(rows, dtype=torch.int64, device=_dev())
    dx = torch.empty_like(dx_ref)
    if general:
        _lib.set_option("interact_general", 1)
    try:
        _lib.check(lib.dlrmb_interaction_bwd_scatter_cols(0, dOut.data_ptr(), T.data_ptr(), B, F, d, 1, dests.data_ptr(),
                                                          Q, off, dx.data_ptr(), int(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
    finally:
        if general:
            _lib.set_option("interact_general", 0)
    got = G.cpu().numpy()[off:]
    want = dT_ref.cpu().numpy()
    for q in range(Q):
        p = (q + 1) % Q
        assert np.array_equal(got[:, 1:, p * pw:(p + 1) * pw], want[:, 1:, q * pw:(q + 1) * pw]), q
    assert np.isnan(got[:, 0]).all() and np.isnan(G.cpu().numpy()[:off]).all()
    assert torch.equal(dx, dx_ref)


@pytest.mark.parametrize("idt", [np.int32, np.int64])
def test_indices_scatter_list_fills_every_holder(idt):
    """A split table's block goes to every holder: each holder's buffer equals the numpy owner layout of its
    width groups."""
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.sharded import TableSharding
    lib = _lib.load()
    rows, P, BL, W = [50, 7, 400, 3, 1200, 33, 9], [3, 1, 70, 100, 1, 12, 2], 37, 4
    Bg, ib = BL * W, np.dtype(idt).itemsize
    sh = TableSharding.build(rows, W, P, D=64, max_col_shards=4)
    assert sh.split
    rng = np.random.default_rng(5)
    idx_all = [[rng.integers(0, r, size=(BL, p)).astype(idt) for r, p in zip(rows, P)] for _ in range(W)]
    order = [[k for _c, ks in sh.groups(r) for k in ks] for r in range(W)]
    owned = [torch.full((max(1, sum(Bg * P[k] for k in order[r])),), -7, dtype=torch.int32 if ib == 4 else torch.int64,
                        device=_dev()) for r in range(W)]
    dest_table, dests = [], []
    for r in range(W):
        o = 0
        for k in order[r]:
            dest_table.append(k)
            dests.append(owned[r].data_ptr() + o * ib)
            o += Bg * P[k]
    dests = torch.tensor(dests, dtype=torch.int64, device=_dev())
    s = int(torch.cuda.current_stream().cuda_stream)
    for h in range(W):
        loc = _packed(idx_all[h], idt)
        _lib.check(lib.dlrmb_indices_scatter_p2p_mp_list(0, loc.data_ptr(), ib, len(rows), BL, (C.c_int32 * len(P))(*P),
                                                        len(dest_table), (C.c_int32 * len(dest_table))(*dest_table),
                                                        dests.data_ptr(), h, s))
    torch.cuda.synchronize()
    for r in range(W):
        parts = [np.concatenate([idx_all[h][k] for h in range(W)], axis=0).reshape(-1) for k in order[r]]
        want = np.concatenate(parts) if parts else np.full(1, -7, idt)
        assert np.array_equal(owned[r].cpu().numpy(), want), r


def test_graph_capture_replay_matches_eager():
    """The dest-mapped lookup with its sort, the list scatter and the column-piece backward captured into one graph
    and replayed give the eager results."""
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    rows, P, BL, W, D, c = [50, 7, 400, 3], [3, 1, 40, 2], 64, 2, 128, 2
    Bg, w = BL * W, D // c
    rng = np.random.default_rng(9)
    arrays = [rng.standard_normal((r, w)).astype(np.float32) for r in rows]
    idx = _packed([rng.integers(0, r, size=(Bg, p)) for r, p in zip(rows, P)], np.int64)
    loc = _packed([rng.integers(0, r, size=(BL, p)) for r, p in zip(rows, P)], np.int64)
    t = _tables(arrays, Bg * max(P))
    t.set_dest_map([1, 2, 3, 4], [w, 0, w, 0], D)
    bufs = _peer_buffers(W, BL, 5, D)
    ibuf = torch.zeros(2 * sum(Bg * p for p in P), dtype=torch.int64, device=_dev())
    dest_table = [0, 1, 2, 3, 2]
    offs = [0, Bg * 3, Bg * 4, Bg * 44, Bg * 46]
    dests = torch.tensor([ibuf.data_ptr() + 8 * o for o in offs], dtype=torch.int64, device=_dev())
    T, dOut, _dx, _dT = _plain_bwd(27, 128, BL, 3)
    G = torch.zeros((BL, 27, 128), dtype=torch.float32, device=_dev())
    pd = torch.tensor([[0, 0, 0]] * 2 + [[G.data_ptr(), 27 * 128, f * 128 + q * 64] for f in range(1, 27) for q in range(2)],
                      dtype=torch.int64, device=_dev())
    dx = torch.empty((BL, 128), dtype=torch.float32, device=_dev())

    def run(stream):
        t.lookup_p2p(idx, [b.data_ptr() for b in bufs], BL, 5, 0, sort=True)
        _lib.check(lib.dlrmb_indices_scatter_p2p_mp_list(0, loc.data_ptr(), 8, 4, BL, (C.c_int32 * 4)(*P), 5,
                                                        (C.c_int32 * 5)(*dest_table), dests.data_ptr(), 1, stream))
        _lib.check(lib.dlrmb_interaction_bwd_scatter_cols(0, dOut.data_ptr(), T.data_ptr(), BL, 27, 128, 1, pd.data_ptr(),
                                                          2, 0, dx.data_ptr(), stream))

    run(int(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    eager = [b.clone() for b in bufs] + [ibuf.clone(), G.clone(), dx.clone()]
    for b in bufs:
        b.fill_(float("nan"))
    ibuf.zero_()
    G.zero_()
    dx.zero_()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            run(int(s.cuda_stream))
    g.replay()
    torch.cuda.synchronize()
    replay = [b for b in bufs] + [ibuf, G, dx]
    for a, b in zip(eager, replay):
        assert torch.equal(torch.nan_to_num(a, nan=-1.0), torch.nan_to_num(b, nan=-1.0)) if a.is_floating_point() \
            else torch.equal(a, b)
    t.close()


def test_argument_errors():
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    t = _tables([np.zeros((5, 32), np.float32), np.zeros((6, 32), np.float32)], 64)
    with pytest.raises(_lib.DLRMB200Error, match="leave the destination row"):
        t.set_dest_map([1, 2], [0, 100], 128)
    with pytest.raises(_lib.DLRMB200Error, match="narrower"):
        t.set_dest_map([1, 2], [0, 0], 16)
    with pytest.raises(_lib.DLRMB200Error):
        t.set_dest_map([1, -1], [0, 0], 64)
    assert lib.dlrmb_tables_set_dest_map(t._h, (C.c_int32 * 2)(1, 2), None, 64) == _lib.EINVAL
    T, dOut, _dx, _dT = _plain_bwd(27, 128, 8, 1)
    d = torch.zeros((27 * 4, 3), dtype=torch.int64, device=_dev())
    s = int(torch.cuda.current_stream().cuda_stream)
    for Q in (3, 64, 0):
        assert lib.dlrmb_interaction_bwd_scatter_cols(0, dOut.data_ptr(), T.data_ptr(), 8, 27, 128, 1, d.data_ptr(), Q, 0,
                                                      dOut.data_ptr(), s) == _lib.EINVAL
    idx = torch.zeros(64, dtype=torch.int32, device=_dev())
    P = (C.c_int32 * 2)(1, 1)
    assert lib.dlrmb_indices_scatter_p2p_mp_list(0, idx.data_ptr(), 4, 2, 4, P, 0, (C.c_int32 * 1)(0), d.data_ptr(), 0,
                                                 s) == _lib.EINVAL
    assert lib.dlrmb_indices_scatter_p2p_mp_list(0, idx.data_ptr(), 4, 2, 4, P, 1, (C.c_int32 * 1)(2), d.data_ptr(), 0,
                                                 s) == _lib.EINVAL
    assert lib.dlrmb_indices_scatter_p2p_mp_list(0, idx.data_ptr(), 4, 2, 4, P, 1, None, d.data_ptr(), 0, s) == _lib.EINVAL
    t.close()


# ---- two to four ranks sharing cuda:0 -------------------------------------------------------------
def _step_worker(rank, world, port, q, D, BL, P, rows, S, steps, bf16):
    _arm_watchdog()
    try:
        from dlrm_jl_b200.interact import DotInteraction, interaction_width
        from dlrm_jl_b200.sharded import ShardedEmbedding
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        torch.cuda.set_device(0)
        dev = torch.device("cuda", 0)
        ntab, F = len(rows), len(rows) + 1
        se = ShardedEmbedding.create(rows, D, BL, P, rank, world, dev, dtype=torch.bfloat16 if bf16 else None,
                                     max_col_shards=S)
        assert se.split

        def barrier():
            torch.cuda.synchronize()
            dist.barrier()

        se.enable_peer_exchange(BL, barrier=barrier, P=P, idx_bytes=8)
        se.enable_fused_backward(BL, split_dx=(D == 128))

        def gather_tables():        # reassemble every table from its slices
            mine = {k: se.download(k) for k in se.local_ids}
            gathered = [None] * world
            dist.all_gather_object(gathered, mine)
            out = [np.full((r, D), np.nan, np.float32) for r in rows]
            for part in gathered:
                for k, slices in part.items():
                    for c0, a in slices:
                        out[k][:, c0:c0 + a.shape[1]] = a
            assert not any(np.isnan(t).any() for t in out), "a column of a table is held by nobody"
            return out

        dot = DotInteraction()
        w = interaction_width(F, D)
        worst = {"z": 0.0, "dx": 0.0, "tables": 0.0, "bf16_equal": 1.0}
        ok_T = True
        lr = 0.25
        def run_step(seed):
            rng = np.random.default_rng(seed)                  # same stream on every rank
            idx_all = [[rng.integers(0, r, size=(BL, p)) for r, p in zip(rows, P)] for _ in range(world)]
            x_all = [rng.standard_normal((BL, D)).astype(np.float32) for _ in range(world)]
            gz_all = [rng.standard_normal((BL, w)).astype(np.float32) for _ in range(world)]
            x = torch.from_numpy(x_all[rank]).to(dev).requires_grad_(True)
            T = se.lookup_fused(idx_all[rank])
            se.sort_async()
            z = dot(x, T, scatter=se.scatter_plan)
            side = torch.cuda.Stream()
            se.update_inside_backward(lr, side)
            z.backward(torch.from_numpy(gz_all[rank]).to(dev))
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            return idx_all, x_all, gz_all, x, T, z

        for step in range(steps):
            ref_tables = gather_tables()
            idx_all, x_all, gz_all, x, T, z = run_step(100 + step)
            T_ref = O.lookup(ref_tables, idx_all[rank], slot0=1)
            ok_T = ok_T and bool(np.array_equal(T.cpu().numpy()[:, 1:], T_ref[:, 1:]))
            T_ref[:, 0] = x_all[rank]
            worst["z"] = max(worst["z"], O.rel_err(z.detach().cpu().numpy(), O.interaction_fwd(T_ref)))
            dT_glob = []
            for r in range(world):
                Tr = O.lookup(ref_tables, idx_all[r], slot0=1)
                Tr[:, 0] = x_all[r]
                dx_r, dT_r = O.interaction_bwd(gz_all[r], Tr)
                dT_glob.append(dT_r)
                if r == rank:
                    worst["dx"] = max(worst["dx"], O.rel_err(x.grad.cpu().numpy(), dx_r))
            dT_glob = np.concatenate(dT_glob, axis=0)
            upd = O.sparse_sgd_update_bf16 if bf16 else O.sparse_sgd_update_fast
            for k in range(ntab):
                idx_glob = np.concatenate([idx_all[r][k] for r in range(world)], axis=0)
                upd(ref_tables[k], idx_glob, np.ascontiguousarray(dT_glob[:, 1 + k]), lr)
            got_tables = gather_tables()
            for k in range(ntab):
                worst["tables"] = max(worst["tables"], O.rel_err(got_tables[k], ref_tables[k]))
                if bf16:
                    worst["bf16_equal"] = min(worst["bf16_equal"], float(np.mean(got_tables[k] == ref_tables[k])))
            barrier()
        # the same step twice from the same state: bit-identical tables
        state = [[t.download(j) for j in range(t.ntab)] for t in se.group_tables]
        run_step(7)
        first = [[t.download(j) for j in range(t.ntab)] for t in se.group_tables]
        for t, arrs in zip(se.group_tables, state):
            for j, a in enumerate(arrs):
                t.upload(j, a)
        barrier()
        run_step(7)
        second = [[t.download(j) for j in range(t.ntab)] for t in se.group_tables]
        worst["repeat_equal"] = all(np.array_equal(a, b) for ga, gb in zip(first, second) for a, b in zip(ga, gb))
        barrier()
        se.close()
        q.put((rank, ok_T, worst, ""))
    except Exception as exc:  # noqa: BLE001
        import traceback
        q.put((rank, False, {}, repr(exc) + traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


_ROWS27 = [50, 7, 400, 3, 1200, 33, 9, 20000] + [20 + 31 * k for k in range(18)]
_HOT27 = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


@pytest.mark.parametrize("world,D,BL,P,rows,S,bf16", [
    (3, 128, 64, _HOT27, _ROWS27, 8, False),          # F = 27, d = 128: the warp kernels; table 20 in 2
    (2, 64, 48, [3, 1, 70, 2, 1, 12, 5], [50, 7, 400, 3, 1200, 33, 9], 2, False),   # general kernel, Q = 2
    (4, 128, 48, _HOT27, _ROWS27, 8, True),           # table 20 in 2, bf16 storage
    (3, 32, 40, [3, 1, 70, 2, 1, 12, 5], [50, 7, 400, 3, 1200, 33, 9], 4, False),   # general interaction kernel
])
def test_column_sharded_step_matches_unsharded_oracle(world, D, BL, P, rows, S, bf16):
    """Fused step with a split table: list index scatter, dest-mapped lookups per width group, column-piece
    scattering backward, per-group updates inside the backward -- pooled rows bit-exact, z / dx rel 1e-5, tables
    (reassembled from the slices) rel 1e-4 (bf16: 2e-3 and >= 98 % bit-equal) after two steps; the same step run
    twice from the same state leaves bit-identical tables."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_step_worker, args=(r, world, port, q, D, BL, P, rows, S, 2, bf16)) for r in range(world)]
    for p in procs:
        p.start()
    res = _collect(procs, q, world, 300)
    for rank, ok_T, worst, err in res:
        assert not err, f"rank {rank}: {err}"
        assert ok_T, f"rank {rank}: pooled rows differ from the oracle"
        assert worst["z"] < 1e-5 and worst["dx"] < 1e-5, (rank, worst)
        assert worst["repeat_equal"], f"rank {rank}: the same step from the same state gave different tables"
        if bf16:
            assert worst["tables"] < 2e-3 and worst["bf16_equal"] >= 0.98, (rank, worst)
        else:
            assert worst["tables"] < SGD_RTOL, (rank, worst)
