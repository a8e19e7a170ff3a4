#!/usr/bin/env python
"""BASELINE config 4 (table-wise sharded training step) with PER-TABLE POOLING FACTORS (the MLPerf
DLRM-DCNv2 hotness list) driven ONLY through the C ABI -- the calls a non-Python host (DLRM.jl via ccall)
would make -- on N GPUs, one process per GPU, checked against the unsharded CPU oracle.

    python tests/cabi_sharded_step_mp.py --gpus 2 [--mode nccl|p2p] [--B 256] [--D 128] [--steps 2]

No torch.distributed: the NCCL unique id of dlrmb_comm_unique_id travels from rank 0 to the others
through a multiprocessing queue (a Julia host would use a file or a socket), every collective is a
dlrmb_comm_* call, every kernel a dlrmb_* call.  torch is used for device buffers only.

  plan:      dlrmb_shard_plan_mp (tables weighed by their P_k)
  mode nccl: dlrmb_comm_a2a_indices_mp -> dlrmb_embedding_fwd_mp (slot0 = 0) -> dlrmb_comm_a2a_fwd ->
             dlrmb_interaction_fwd / _bwd -> dlrmb_comm_a2a_bwd -> dlrmb_embedding_bwd_sgd_mp
  mode p2p:  exchange buffers (dlrmb_xbuf_*) whose IPC handles are all-gathered with
             dlrmb_comm_allgather, then dlrmb_embedding_fwd_p2p_sort_mp and dlrmb_interaction_bwd_scatter
             store straight into the peers' buffers; a one-float dlrmb_comm_allreduce_f32 is the ordering
             point; dlrmb_embedding_update_sorted consumes the sort the lookup launch left.
Prints one JSON line per run with the worst errors over ranks and steps.  It lives under tests/ because the
oracle is its checker; `tests/test_gpu_sharded_multihot.py` runs it when the box has two or more GPUs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MLPERF_HOTNESS = [3, 2, 1, 2, 6, 1, 1, 1, 1, 7, 3, 8, 1, 6, 9, 5, 1, 1, 1, 12, 100, 27, 10, 3, 1, 1]


def worker(rank, world, uid_q, res_q, args):
    try:
        import torch
        from dlrm_jl_b200 import _lib
        from oracle import oracle as O
        lib = _lib.load()
        chk = _lib.check
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        # ---- communicator: unique id from rank 0, carried by the host program
        uid = (C.c_uint8 * 128)()
        if rank == 0:
            chk(lib.dlrmb_comm_unique_id(uid))
            for _ in range(world - 1):
                uid_q.put(bytes(uid))
        else:
            uid = (C.c_uint8 * 128).from_buffer_copy(uid_q.get(timeout=120))
        comm = C.c_void_p()
        chk(lib.dlrmb_comm_create(rank, uid, rank, world, C.byref(comm)))
        # ---- geometry and partition
        rows = [50, 7, 400, 3, 1200, 33, 9] + [20 + 31 * k for k in range(19)]     # 26 tables: F = 27
        ntab, F, D, Bl, P = len(rows), len(rows) + 1, args.D, args.B, MLPERF_HOTNESS
        Bg = Bl * world
        Pg = (C.c_int32 * ntab)(*P)
        owner = (C.c_int32 * ntab)()
        chk(lib.dlrmb_shard_plan_mp(ntab, (C.c_int64 * ntab)(*rows), Pg, world, owner))
        owner_l = list(owner)
        mine = [k for k in range(ntab) if owner_l[k] == rank]
        counts = [owner_l.count(r) for r in range(world)]
        t_mine = len(mine)
        Pm = (C.c_int32 * max(1, t_mine))(*[P[k] for k in mine])
        n_owned = sum(Bg * P[k] for k in mine)
        # ---- this rank's tables (every rank can rebuild every table for the oracle)
        rng_t = np.random.default_rng(7)
        all_tables = [rng_t.standard_normal((r, D)).astype(np.float32) for r in rows]
        th = C.c_void_p()
        chk(lib.dlrmb_tables_create(rank, t_mine, (C.c_int64 * t_mine)(*[rows[k] for k in mine]), D,
                                    Bg * max([P[k] for k in mine] or [1]), C.byref(th)))
        for j, k in enumerate(mine):
            chk(lib.dlrmb_tables_upload(th, j, all_tables[k].ctypes.data_as(C.c_void_p)))
        s = int(torch.cuda.current_stream().cuda_stream)
        width = D + F * (F - 1) // 2
        flag = torch.zeros(1, device=dev)

        def barrier():
            chk(lib.dlrmb_comm_allreduce_f32(comm, flag.data_ptr(), 1, s))

        if args.mode == "p2p":
            def shared(nbytes):
                xb = C.c_void_p()
                chk(lib.dlrmb_xbuf_create(rank, max(256, nbytes), C.byref(xb)))
                own = C.c_void_p()
                chk(lib.dlrmb_xbuf_ptr(xb, C.byref(own)))
                hnd = (C.c_uint8 * 64)()
                chk(lib.dlrmb_xbuf_ipc_handle(xb, hnd))
                send = torch.frombuffer(bytearray(bytes(hnd)), dtype=torch.uint8).to(dev)
                recv = torch.empty(64 * world, dtype=torch.uint8, device=dev)
                chk(lib.dlrmb_comm_allgather(comm, send.data_ptr(), recv.data_ptr(), 64, s))
                torch.cuda.synchronize()
                blobs = recv.cpu().numpy().tobytes()
                ptrs = []
                for r in range(world):
                    if r == rank:
                        ptrs.append(own.value)
                        continue
                    q = C.c_void_p()
                    chk(lib.dlrmb_xbuf_open(rank, (C.c_uint8 * 64).from_buffer_copy(blobs[64 * r:64 * r + 64]), C.byref(q)))
                    ptrs.append(q.value)
                return xb, own.value, ptrs

            from dlrm_jl_b200.embedding import _DevicePtrView
            xT, T_ptr, T_peers = shared(Bl * F * D * 4)
            xG, G_ptr, G_peers = shared(Bg * max(1, t_mine) * D * 4)
            keep = object()
            T = torch.as_tensor(_DevicePtrView(T_ptr, (Bl, F, D), keep), device=dev)
            G = torch.as_tensor(_DevicePtrView(G_ptr, (Bg, max(1, t_mine), D), keep), device=dev)
            chk(lib.dlrmb_tables_set_slot_map(th, (C.c_int32 * t_mine)(*[1 + k for k in mine])))
            dests = [[0, 0, 0]] + [[G_peers[owner_l[k]], counts[owner_l[k]] * D,
                                    [kk for kk in range(ntab) if owner_l[kk] == owner_l[k]].index(k) * D] for k in range(ntab)]
            dests_d = torch.tensor(dests, dtype=torch.int64, device=dev)
        else:
            T = torch.zeros((Bl, F, D), device=dev)
            G = torch.zeros((Bg, max(1, t_mine), D), device=dev)
        pooled = torch.zeros((Bg, max(1, t_mine), D), device=dev)
        idx_owned = torch.zeros((max(1, n_owned),), dtype=torch.int32, device=dev)
        out = torch.empty((Bl, width), device=dev)
        dT = torch.empty((Bl, F, D), device=dev)
        dx = torch.empty((Bl, D), device=dev)
        worst = {"z": 0.0, "dx": 0.0, "tables": 0.0}
        bit_exact = True
        lr = 0.25
        ref_tables = [t.copy() for t in all_tables]
        for step in range(args.steps):
            rng = np.random.default_rng(100 + step)
            idx_all = [[rng.integers(0, r, size=(Bl, p)).astype(np.int32) for r, p in zip(rows, P)] for _ in range(world)]
            x_all = [rng.standard_normal((Bl, D)).astype(np.float32) for _ in range(world)]
            gz_all = [rng.standard_normal((Bl, width)).astype(np.float32) for _ in range(world)]
            idx_local = torch.from_numpy(np.concatenate([a.reshape(-1) for a in idx_all[rank]])).to(dev)
            x = torch.from_numpy(x_all[rank]).to(dev)
            gz = torch.from_numpy(gz_all[rank]).to(dev)
            chk(lib.dlrmb_comm_a2a_indices_mp(comm, owner, ntab, idx_local.data_ptr(), 4, Bl, Pg, idx_owned.data_ptr(), s))
            if args.mode == "p2p":
                peers = (C.c_void_p * world)(*T_peers)
                if t_mine:
                    chk(lib.dlrmb_embedding_fwd_p2p_sort_mp(th, idx_owned.data_ptr(), 4, 0, Bg, Pm, peers, world, Bl, F, s))
                barrier()
            else:
                if t_mine:
                    chk(lib.dlrmb_embedding_fwd_mp(th, idx_owned.data_ptr(), 4, 0, Bg, Pm, pooled.data_ptr(), t_mine, 0, s))
                chk(lib.dlrmb_comm_a2a_fwd(comm, owner, ntab, pooled.data_ptr(), Bl, D, T.data_ptr(), s))
            chk(lib.dlrmb_interaction_fwd(rank, T.data_ptr(), x.data_ptr(), Bl, F, D, 1, out.data_ptr(), s))
            if args.mode == "p2p":
                chk(lib.dlrmb_interaction_bwd_scatter(rank, gz.data_ptr(), T.data_ptr(), Bl, F, D, 1, dests_d.data_ptr(),
                                                      rank * Bl, dx.data_ptr(), s))
                barrier()
            else:
                chk(lib.dlrmb_interaction_bwd(rank, gz.data_ptr(), T.data_ptr(), Bl, F, D, 1, dT.data_ptr(), dx.data_ptr(), s))
                chk(lib.dlrmb_comm_a2a_bwd(comm, owner, ntab, dT.data_ptr(), Bl, D, G.data_ptr(), s))
            if t_mine and args.mode == "p2p":
                chk(lib.dlrmb_embedding_update_sorted(th, G.data_ptr(), t_mine, 0, lr, s))
            elif t_mine:
                chk(lib.dlrmb_embedding_bwd_sgd_mp(th, idx_owned.data_ptr(), 4, 0, Bg, Pm, G.data_ptr(), t_mine, 0, lr, s))
            barrier()
            torch.cuda.synchronize()
            # ---- unsharded oracle on the same inputs
            T_ref = O.lookup(ref_tables, idx_all[rank], slot0=1)
            bit_exact = bit_exact and bool(np.array_equal(T.cpu().numpy()[:, 1:], T_ref[:, 1:]))
            T_ref[:, 0] = x_all[rank]
            worst["z"] = max(worst["z"], float(O.rel_err(out.cpu().numpy(), O.interaction_fwd(T_ref))))
            dT_glob = []
            for r in range(world):
                Tr = O.lookup(ref_tables, idx_all[r], slot0=1)
                Tr[:, 0] = x_all[r]
                dx_r, dT_r = O.interaction_bwd(gz_all[r], Tr)
                dT_glob.append(dT_r)
                if r == rank:
                    worst["dx"] = max(worst["dx"], float(O.rel_err(dx.cpu().numpy(), dx_r)))
            dT_glob = np.concatenate(dT_glob, axis=0)
            for k in range(ntab):
                idx_glob = np.concatenate([idx_all[r][k] for r in range(world)], axis=0)
                O.sparse_sgd_update_fast(ref_tables[k], idx_glob, np.ascontiguousarray(dT_glob[:, 1 + k]), lr)
            for j, k in enumerate(mine):
                got = np.empty((rows[k], D), dtype=np.float32)
                chk(lib.dlrmb_tables_download(th, j, got.ctypes.data_as(C.c_void_p)))
                worst["tables"] = max(worst["tables"], float(O.rel_err(got, ref_tables[k])))
                ref_tables[k] = got                 # next step starts from the GPU's own bits
            # every rank needs every table's current bits for the next step's oracle: rebuild from the owners
            if args.steps > 1 and step + 1 < args.steps:
                res_q.put(("tables", rank, {k: ref_tables[k] for k in mine}))
                merged = uid_q.get(timeout=300)
                for k, v in merged.items():
                    ref_tables[k] = v
        res_q.put(("done", rank, {"pooled_rows_bit_exact": bit_exact, **worst}))
        chk(lib.dlrmb_tables_destroy(th))
        chk(lib.dlrmb_comm_destroy(comm))
    except Exception as exc:  # noqa: BLE001
        import traceback
        res_q.put(("error", rank, repr(exc) + "\n" + traceback.format_exc()))


def main():
    import torch.multiprocessing as mp
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=2)
    ap.add_argument("--mode", default="nccl", choices=["nccl", "p2p"])
    ap.add_argument("--B", type=int, default=256)
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--steps", type=int, default=2)
    args = ap.parse_args()
    ctx = mp.get_context("spawn")
    world = args.gpus
    uid_q, res_q = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, world, uid_q, res_q, args)) for r in range(world)]
    for p in procs:
        p.start()
    done, errors = {}, []
    pending_tables = {}
    while len(done) + len(errors) < world:
        kind, rank, payload = res_q.get(timeout=600)
        if kind == "done":
            done[rank] = payload
        elif kind == "error":
            errors.append((rank, payload))
            break
        else:   # a step's updated tables from one owner: once all ranks reported, hand everyone the merged set
            pending_tables[rank] = payload
            if len(pending_tables) == world:
                merged = {}
                for part in pending_tables.values():
                    merged.update(part)
                for _ in range(world):
                    uid_q.put(merged)
                pending_tables = {}
    for p in procs:
        p.join(timeout=30)
        if p.is_alive():
            p.terminate()
    if errors:
        print(json.dumps({"ok": False, "errors": errors}))
        sys.exit(1)
    worst = {k: max(d[k] for d in done.values()) for k in ("z", "dx", "tables")}
    ok = all(d["pooled_rows_bit_exact"] for d in done.values()) and worst["z"] < 1e-5 and worst["dx"] < 1e-5 and worst["tables"] < 1e-4
    print(json.dumps({"ok": bool(ok), "what": "mixed-P sharded training step through the C ABI only vs the unsharded CPU oracle",
                      "gpus": world, "mode": args.mode, "B_local": args.B, "D": args.D, "steps": args.steps,
                      "pooled_rows_bit_exact": all(d["pooled_rows_bit_exact"] for d in done.values()),
                      "interaction_fwd_rel_err": worst["z"], "dx_rel_err": worst["dx"], "tables_rel_err": worst["tables"]}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
