"""Table-sharded embeddings with per-table pooling factors (mixed multi-hot) on the GPU.

Single process: the fused lookup + peer-store kernel (dlrmb_embedding_fwd_p2p_mp / _sort_mp) is given
`world` peer pointers that are all buffers of this process, which checks everything the kernel computes
and where it stores it: pooled rows bit-exact against the oracle with NaN in every slot it must not
touch, the sort it leaves for the update, the update itself, equal P_k against the uniform entry points,
graph capture, argument errors and the index scatter.

Two or three ranks sharing cuda:0 through CUDA IPC (ordered by a host barrier, as in test_gpu_p2p.py:
the flag barrier needs one GPU per rank): the whole mixed-P sharded training step against the
UNSHARDED oracle.  The C-ABI-only step on two GPUs is tests/cabi_sharded_step_mp.py.
"""
import ctypes as C
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import oracle as O

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SGD_RTOL = 1e-4
MLPERF_HOTNESS = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def _dev():
    return torch.device("cuda", 0)


def _packed(idx, dtype=np.int64, base=0):
    from dlrm_jl_b200.embedding import _as_index_tensor
    return _as_index_tensor([np.asarray(a).astype(dtype) + base for a in idx], len(idx), _dev())


def _tables(arrays, max_lookups, dtype=torch.float32):
    from dlrm_jl_b200.embedding import EmbeddingTables
    return EmbeddingTables.from_arrays(arrays, max_lookups, 0, dtype)


def _peer_buffers(world, BL, slots, D, misaligned=False):
    """`world` NaN-filled [B_local][slots][D] buffers of this process; misaligned: 4 bytes off 16."""
    bufs = []
    for _ in range(world):
        n = BL * slots * D
        raw = torch.full((n + 1,), float("nan"), dtype=torch.float32, device=_dev())
        bufs.append((raw[1:] if misaligned else raw[:n]).view(BL, slots, D))
    return bufs


def _check_peer_rows(bufs, ref, slotmap, BL):
    """ref [B_global][ntab][D]: sample b of table j must sit in bufs[b // BL][b % BL][slotmap[j]], every
    other slot must still be NaN."""
    slots = bufs[0].shape[1]
    other = [s for s in range(slots) if s not in slotmap]
    for h, buf in enumerate(bufs):
        got = buf.cpu().numpy()
        want = ref[h * BL:(h + 1) * BL]
        for j, s in enumerate(slotmap):
            if not np.array_equal(got[:, s], want[:, j]):
                return f"rank {h}, table {j}"
        if other and not np.isnan(got[:, other]).all():
            return f"rank {h}: a slot outside the slot map was written"
    return ""


# rows, P, B_local, world: P = 1 tables, hotness up to 100, and all three sort regimes at B_global = 2048
# (L = 2048 and 4096 fused into the lookup launch, 6144 and 14336 shared memory, 24576 and 204800 radix)
BIG = ([7, 1000, 33, 50000, 64, 3, 40000], [1, 2, 3, 100, 7, 1, 12], 1024, 2)
SMALL = ([50, 7, 400, 3, 1200], [4, 1, 9, 2, 1], 85, 3)


@pytest.mark.parametrize("case,D,tdtype,idt,base,misaligned", [
    ("big", 128, torch.float32, np.int64, 0, False),
    ("big", 64, torch.bfloat16, np.int32, 1, False),
    ("big", 64, torch.float32, np.int32, 1, True),          # peer buffers 4 bytes off 16: the VEC 1 path
    ("small", 16, torch.float32, np.int64, 1, False),
    ("small", 10, torch.float32, np.int32, 0, False),        # D % 4 != 0: VEC 1
    ("small", 32, torch.bfloat16, np.int64, 0, True),
])
def test_fwd_p2p_mp_bit_exact_and_sort_and_update(case, D, tdtype, idt, base, misaligned):
    rows, P, BL, W = BIG if case == "big" else SMALL
    Bg = BL * W
    rng = np.random.default_rng(D + len(rows))
    arrays = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = [rng.integers(0, r, size=(Bg, p)) for r, p in zip(rows, P)]
    slotmap = [3 + 2 * j for j in range(len(rows))]           # owner's slots spread inside the receivers' T
    slots = slotmap[-1] + 2
    G = torch.from_numpy(rng.standard_normal((Bg, len(rows), D)).astype(np.float32)).to(_dev())
    for sort in (False, True):
        t = _tables(arrays, Bg * max(P), tdtype)
        t.set_slot_map(slotmap)
        stored = [t.download(k) for k in range(len(rows))]   # the bf16-rounded rows for bf16 storage
        bufs = _peer_buffers(W, BL, slots, D, misaligned)
        t.lookup_p2p(_packed(idx, idt, base), [b.data_ptr() for b in bufs], BL, slots, base, sort=sort)
        torch.cuda.synchronize()
        err = _check_peer_rows(bufs, O.lookup(stored, idx, slot0=0), slotmap, BL)
        assert not err, (sort, err)
        if not sort:
            t.close()
            continue
        for k in range(len(rows)):
            u, s, perm = t.sort_dedup_export(k, Bg * P[k])
            ru, rs, rp = O.sort_dedup(idx[k])
            assert np.array_equal(u, ru) and np.array_equal(s, rs) and np.array_equal(perm, rp), k
        t.update_sorted(G, 0, 0.05)
        torch.cuda.synchronize()
        Gn = G.cpu().numpy()
        for k in range(len(rows)):
            ref = stored[k].copy()
            got = t.download(k)
            if tdtype == torch.bfloat16:
                O.sparse_sgd_update_bf16(ref, idx[k], np.ascontiguousarray(Gn[:, k]), 0.05)
                assert O.rel_err(got, ref) < 2e-3, k
                assert np.mean(got == ref) >= 0.98, k
            else:
                O.sparse_sgd_update_fast(ref, idx[k], np.ascontiguousarray(Gn[:, k]), 0.05)
                assert O.rel_err(got, ref) < SGD_RTOL, k
        t.close()


@pytest.mark.parametrize("P,B_local", [(1, 512), (3, 700), (9, 1024)])
def test_equal_P_matches_uniform_p2p_bitwise(P, B_local):
    from dlrm_jl_b200.embedding import PackedIndices
    rng = np.random.default_rng(P)
    rows, D, W = [11, 3000, 70000, 5], 64, 2
    Bg = B_local * W
    arrays = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = np.stack([rng.integers(0, r, size=(Bg, P)) for r in rows])
    u_idx = torch.from_numpy(idx).to(_dev())
    packed = PackedIndices(u_idx.reshape(-1).contiguous(), (P,) * len(rows), Bg)
    slotmap = [1, 4, 2, 3]
    G = torch.from_numpy(rng.standard_normal((Bg, len(rows), D)).astype(np.float32)).to(_dev())
    res = []
    for ix in (u_idx, packed):
        t = _tables(arrays, Bg * P)
        t.set_slot_map(slotmap)
        bufs = _peer_buffers(W, B_local, 5, D)
        t.lookup_p2p(ix, [b.data_ptr() for b in bufs], B_local, 5, 0, sort=True)
        t.update_sorted(G, 0, 0.05)
        torch.cuda.synchronize()
        res.append(([b.cpu().numpy() for b in bufs], [t.download(k) for k in range(len(rows))]))
        t.close()
    for a, b in zip(res[0][0], res[1][0]):
        assert np.array_equal(a, b, equal_nan=True)
    for a, b in zip(res[0][1], res[1][1]):
        assert np.array_equal(a, b)


def test_graph_capture_replay_matches_eager():
    rows, P, BL, W = BIG
    D, Bg = 64, BL * W
    rng = np.random.default_rng(21)
    arrays = [rng.standard_normal((r, D)).astype(np.float32) for r in rows]
    idx = _packed([rng.integers(0, r, size=(Bg, p)) for r, p in zip(rows, P)])
    G = torch.from_numpy(rng.standard_normal((Bg, len(rows), D)).astype(np.float32)).to(_dev())
    slotmap = list(range(1, 1 + len(rows)))
    slots = 1 + len(rows)
    out = {}
    for mode in ("eager", "graph"):
        t = _tables(arrays, Bg * max(P))
        t.set_slot_map(slotmap)
        bufs = _peer_buffers(W, BL, slots, D)
        ptrs = [b.data_ptr() for b in bufs]
        if mode == "eager":
            t.lookup_p2p(idx, ptrs, BL, slots, 0, sort=True)
            t.update_sorted(G, 0, 0.05)
        else:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(s):
                with torch.cuda.graph(g, stream=s):
                    t.lookup_p2p(idx, ptrs, BL, slots, 0, sort=True)
                    t.update_sorted(G, 0, 0.05)
            torch.cuda.current_stream().wait_stream(s)
            g.replay()
        torch.cuda.synchronize()
        out[mode] = ([b.cpu().numpy() for b in bufs], [t.download(k) for k in range(len(rows))])
        t.close()
    for a, b in zip(out["eager"][0], out["graph"][0]):
        assert np.array_equal(a, b, equal_nan=True)
    for a, b in zip(out["eager"][1], out["graph"][1]):
        assert np.array_equal(a, b)


def test_argument_errors():
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    rows, P, BL, W, D = [10, 20, 30], [1, 4, 2], 8, 2, 16
    Bg = BL * W
    arrays = [np.zeros((r, D), np.float32) for r in rows]
    t = _tables(arrays, Bg * max(P))
    idx = _packed([np.zeros((Bg, p), np.int64) for p in P])
    bufs = _peer_buffers(W, BL, 4, D)
    ptrs = (C.c_void_p * W)(*[b.data_ptr() for b in bufs])
    s = int(torch.cuda.current_stream().cuda_stream)

    def call(Parr, Bg_=Bg, BL_=BL, slots=4, ptrs_=ptrs, fn=lib.dlrmb_embedding_fwd_p2p_sort_mp):
        return fn(t._h, idx.data_ptr(), 8, 0, Bg_, Parr, ptrs_, W, BL_, slots, s)

    Pok = (C.c_int32 * 3)(*P)
    for fn in (lib.dlrmb_embedding_fwd_p2p_mp, lib.dlrmb_embedding_fwd_p2p_sort_mp):
        assert call(Pok, fn=fn) == _lib.ESTATE                                # no slot map yet
        assert b"slot_map" in lib.dlrmb_last_error()
    t.set_slot_map([1, 2, 3])
    assert call(None) == _lib.EINVAL
    assert call((C.c_int32 * 3)(1, 0, 2)) == _lib.EINVAL
    assert b"P[1] = 0" in lib.dlrmb_last_error()
    assert call((C.c_int32 * 3)(1, 5, 2)) == _lib.EINVAL                       # B_global * 5 > max_lookups
    assert b"max_lookups" in lib.dlrmb_last_error()
    assert call(Pok, BL_=BL + 1) == _lib.EINVAL                                 # B_global != B_local * world
    assert call(Pok, slots=3) == _lib.EINVAL                                    # slot 3 not covered
    assert call(Pok, ptrs_=(C.c_void_p * W)(ptrs[0], None)) == _lib.EINVAL
    assert call(Pok) == _lib.OK
    torch.cuda.synchronize()
    scatter = lib.dlrmb_indices_scatter_p2p_mp
    dests = torch.zeros(3, dtype=torch.int64, device=_dev())
    assert scatter(0, idx.data_ptr(), 8, 3, BL, None, dests.data_ptr(), 0, s) == _lib.EINVAL
    assert scatter(0, idx.data_ptr(), 8, 3, BL, (C.c_int32 * 3)(1, -1, 2), dests.data_ptr(), 0, s) == _lib.EINVAL
    t.close()


@pytest.mark.parametrize("idt", [np.int32, np.int64])
def test_indices_scatter_mp_fills_owner_layout(idt):
    """Every "rank" stores its local batch into the owners' buffers (all in this process); each owner's
    buffer then equals the numpy packing of the owner layout."""
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.sharded import TableSharding
    lib = _lib.load()
    rows, P, BL, W = [50, 7, 400, 3, 1200, 33, 9], [3, 1, 7, 100, 1, 12, 2], 37, 3
    Bg = BL * W
    rng = np.random.default_rng(3)
    sh = TableSharding.build(rows, W, P)
    idx_all = [[rng.integers(0, r, size=(BL, p)).astype(idt) for r, p in zip(rows, P)] for _ in range(W)]
    ib = np.dtype(idt).itemsize
    owned = [torch.full((max(1, sum(Bg * P[k] for k in sh.local[o])),), -7, dtype=torch.int32 if ib == 4 else torch.int64,
                        device=_dev()) for o in range(W)]
    dests = torch.tensor([owned[sh.owner[k]].data_ptr() + sum(Bg * P[i] for i in sh.local[sh.owner[k]] if i < k) * ib
                          for k in range(len(rows))], dtype=torch.int64, device=_dev())
    s = int(torch.cuda.current_stream().cuda_stream)
    for h in range(W):
        loc = _packed(idx_all[h], idt)
        _lib.check(lib.dlrmb_indices_scatter_p2p_mp(0, loc.data_ptr(), ib, len(rows), BL, (C.c_int32 * len(P))(*P),
                                                   dests.data_ptr(), h, s))
    torch.cuda.synchronize()
    for o in range(W):
        parts = [np.concatenate([idx_all[h][k] for h in range(W)], axis=0).reshape(-1) for k in sh.local[o]]
        want = np.concatenate(parts) if parts else np.full(1, -7, idt)
        assert np.array_equal(owned[o].cpu().numpy(), want), o


# ---- two or three ranks sharing cuda:0 ------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _arm_watchdog(seconds: int = 200) -> None:
    """A worker that is stuck dumps every thread's stack to stderr and exits instead of hanging the suite."""
    import faulthandler
    faulthandler.enable()
    faulthandler.dump_traceback_later(seconds, exit=True)


def _collect(procs, q, world, timeout):
    """Results of the workers; whatever happens, no worker survives the test."""
    import queue
    res = []
    try:
        for _ in range(world):
            try:
                res.append(q.get(timeout=timeout))
            except queue.Empty:
                res.append((-1, False, {}, "a worker did not answer within %d s (see its stack dump on stderr)" % timeout))
                break
    finally:
        for p in procs:
            p.join(timeout=20)
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
    return res


def _step_worker(rank, world, port, q, D, BL, P, rows, steps, bf16):
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
        se = ShardedEmbedding.create(rows, D, BL, P, rank, world, dev, dtype=torch.bfloat16 if bf16 else None)

        def barrier():
            torch.cuda.synchronize()
            dist.barrier()

        se.enable_peer_exchange(BL, barrier=barrier, P=P, idx_bytes=8)
        se.enable_fused_backward(BL, split_dx=(D == 128))
        mine = se.local_ids

        def gather_tables():
            gathered = [None] * world
            dist.all_gather_object(gathered, {k: se.tables.download(j) for j, k in enumerate(mine)})
            out = [None] * ntab
            for part in gathered:
                for k, v in part.items():
                    out[k] = v
            return out

        dot = DotInteraction()
        w = interaction_width(F, D)
        worst = {"z": 0.0, "dx": 0.0, "tables": 0.0, "bf16_equal": 1.0}
        ok_T = True
        lr = 0.25
        for step in range(steps):
            ref_tables = gather_tables()
            rng = np.random.default_rng(100 + step)            # same stream on every rank
            idx_all = [[rng.integers(0, r, size=(BL, p)) for r, p in zip(rows, P)] for _ in range(world)]
            x_all = [rng.standard_normal((BL, D)).astype(np.float32) for _ in range(world)]
            gz_all = [rng.standard_normal((BL, w)).astype(np.float32) for _ in range(world)]
            x = torch.from_numpy(x_all[rank]).to(dev).requires_grad_(True)
            T = se.lookup_fused(idx_all[rank])                  # the reference's mixed list
            se.sort_async()
            z = dot(x, T, scatter=se.scatter_plan)
            side = torch.cuda.Stream()
            se.update_inside_backward(lr, side)                 # update launched from inside the backward
            z.backward(torch.from_numpy(gz_all[rank]).to(dev))
            torch.cuda.current_stream().wait_stream(side)
            barrier()
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
            for j, k in enumerate(mine):
                got = se.tables.download(j)
                worst["tables"] = max(worst["tables"], O.rel_err(got, ref_tables[k]))
                if bf16:
                    worst["bf16_equal"] = min(worst["bf16_equal"], float(np.mean(got == ref_tables[k])))
            barrier()
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


@pytest.mark.parametrize("world,D,BL,P,rows,bf16", [
    # F = 27, d = 128 (the bench's interaction kernels); B_global * 100 and 2 * 96 * 100 > 16384: radix sorts
    (2, 128, 96, MLPERF_HOTNESS, _ROWS27, False),
    (3, 16, 40, [3, 1, 7, 2, 1, 12, 5], [50, 7, 400, 3, 1200, 33, 9], False),
    (2, 64, 48, [2, 1, 30, 4, 1], [50, 7, 400, 3, 1200], True),
])
def test_sharded_mixed_pooling_step_matches_unsharded_oracle(world, D, BL, P, rows, bf16):
    """Full mixed-P sharded step on CUDA: peer-store index exchange (int64), fused lookup, scattering
    backward, update launched inside the backward -- pooled rows bit-exact, z / dx rel 1e-5, tables rel
    1e-4 (bf16 storage: rel 2e-3 and >= 98 % of the elements bit-equal) after two steps."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_step_worker, args=(r, world, port, q, D, BL, P, rows, 2, bf16)) for r in range(world)]
    for p in procs:
        p.start()
    res = _collect(procs, q, world, 240)
    for rank, ok_T, worst, err in res:
        assert not err, f"rank {rank}: {err}"
        assert ok_T, f"rank {rank}: pooled rows differ from the oracle"
        assert worst["z"] < 1e-5 and worst["dx"] < 1e-5, (rank, worst)
        if bf16:
            assert worst["tables"] < 2e-3 and worst["bf16_equal"] >= 0.98, (rank, worst)
        else:
            assert worst["tables"] < SGD_RTOL, (rank, worst)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("mode", ["nccl", "p2p"])
def test_mixed_pooling_sharded_step_through_the_c_abi_alone(mode):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "cabi_sharded_step_mp.py"), "--gpus", "2", "--mode", mode,
                          "--B", "128", "--steps", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res["ok"] and res["pooled_rows_bit_exact"]
    assert res["interaction_fwd_rel_err"] < 1e-5 and res["dx_rel_err"] < 1e-5 and res["tables_rel_err"] < 1e-4
