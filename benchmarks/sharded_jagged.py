#!/usr/bin/env python
"""Table-sharded jagged bags (variable length) on the B200: the owner's work and the exchange's host and device costs.

Workload (DESIGN.md §4c): the MLPerf hotness list on Terabyte-shaped tables with rows capped at --rows-cap (20M), D 128,
B_local 2048, bag lengths uniform in 1 .. 2 P_k - 1, uniform indices.  Method of multihot.py: a CUDA graph of --nb
launches over --nb pre-generated batches, replay timed with CUDA events.  One JSON line per record, each with the GPU
name and power limit read in the same process.

    python benchmarks/sharded_jagged.py --mode owner --out profiles/r09_sharded_jagged_owner.jsonl
    torchrun --nproc-per-node 8 benchmarks/sharded_jagged.py --mode step

--mode owner, one GPU, for W = 2, 4, 8 under the plan TableSharding.build(rows, W, P) (P = the hotness list, the
  tables' expected bag lengths):
    owner    the busiest owner's tables in one handle, fed its jagged owner batch at B_global = W * B_local:
             dlrmb_embedding_fwd_p2p_jagged into W local [B_local][1 + ntab][D] buffers (lookup), the _sort_ form
             (lookup + sort), and that plus update_sorted (lookup + sort + update); beside it, in the same process,
             the `_mp` path on constant lengths P_k (the same expected lookups) as the A/B, and the one-GPU jagged
             lookup (dlrmb_embedding_fwd_jagged into one [B_global][t][D] buffer) on the same batches: the cost of the
             peer-store epilogue
    scatter  dlrmb_indices_scatter_p2p_jagged of one rank's local batch (all tables) into local stand-ins of the
             owners' buffers: µs and bytes moved (read + write) over the copy bandwidth measured in the same process
    counts   the per-step host all-gather of the lookup counts (exchange_jagged_counts) on gloo with W processes
             on this machine's CPUs: wall µs per call
--mode step (torchrun, one process per GPU, >= 2 GPUs; with fewer it prints measured: false): ms per step and
  samples/s of the embedding part of the jagged sharded step -- the host count all-gather, the peer-store index
  scatter, the fused lookup + peer stores, the side-stream sort, the gradient all-to-all (NCCL) and the owner's
  sparse SGD -- under the plan TableSharding.build(rows, W, P), jagged_cap[k] = (2 P_k - 1) * B_local.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import socket
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from dlrm_jl_b200 import _lib  # noqa: E402
from dlrm_jl_b200.embedding import EmbeddingTables, JaggedIndices  # noqa: E402
from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES  # noqa: E402
from dlrm_jl_b200.sharded import TableSharding  # noqa: E402
from multihot import MLPERF_HOTNESS, copy_bandwidth_gbs, gpu_info, make_batches, timed  # noqa: E402


def jagged_lengths(rng, P, B):
    return [rng.integers(1, 2 * p, size=B) for p in P]


def jagged_batch(rng, rows, P, B, dev):
    lengths = jagged_lengths(rng, P, B)
    vals = np.concatenate([rng.integers(0, r, size=int(n.sum())) for r, n in zip(rows, lengths)]).astype(np.int32)
    return JaggedIndices.from_lengths(torch.from_numpy(vals), lengths).to(dev)


def owner(a, rows, P, W, dev):
    sh = TableSharding.build(rows, W, P)
    loads = sh.lookups_per_rank()
    o = int(np.argmax(loads))
    mine = sh.local[o]
    r_rows, r_P = [rows[k] for k in mine], [P[k] for k in mine]
    Bl, D, ntab = a.batch, a.D, len(rows)
    Bg = Bl * W
    rng = np.random.default_rng(1234 + W)
    jag = [jagged_batch(rng, r_rows, r_P, Bg, dev) for _ in range(a.nb)]
    mp = make_batches(rng, r_rows, r_P, Bg, a.nb, 0.0, dev)
    t = EmbeddingTables(r_rows, D, Bg * (2 * max(r_P) - 1), dev)
    t.init_uniform(1 + o)
    t.set_slot_map([1 + k for k in mine])
    bufs = [torch.empty((Bl, 1 + ntab, D), device=dev) for _ in range(W)]
    ptrs = [b.data_ptr() for b in bufs]
    G = torch.randn((Bg, len(mine), D), device=dev) * 0.01
    out = torch.empty((Bg, len(mine), D), device=dev)

    def three(batches):
        def chain(i):
            t.lookup_p2p(batches[i], ptrs, Bl, 1 + ntab, 0, sort=True)
            t.update_sorted(G, 0, 0.01)
        return {"lookup_us": timed(lambda i: t.lookup_p2p(batches[i], ptrs, Bl, 1 + ntab, 0), a.nb, a.iters),
                "lookup_sort_us": timed(lambda i: t.lookup_p2p(batches[i], ptrs, Bl, 1 + ntab, 0, sort=True), a.nb,
                                        a.iters),
                "lookup_sort_update_us": timed(chain, a.nb, a.iters)}
    t.lookup_p2p(jag[0], ptrs, Bl, 1 + ntab, 0)             # the same pooled rows either way
    t.lookup(jag[0], out, 0)
    torch.cuda.synchronize()
    equal = bool(torch.equal(torch.cat([b[:, [1 + k for k in mine]] for b in bufs], dim=0), out))
    rj, rm, rl = [], [], []
    for _ in range(a.repeats):                # alternate the paths
        rj.append(three(jag))
        rm.append(three(mp))
        rl.append(timed(lambda i: t.lookup(jag[i], out, 0), a.nb, a.iters))
    t.close()
    del bufs, G, jag, mp, out
    torch.cuda.empty_cache()
    med = lambda rs, key: float(np.median([r[key] for r in rs]))  # noqa: E731
    keys = ("lookup_us", "lookup_sort_us", "lookup_sort_update_us")
    return {"busiest_owner": o, "tables": mine, "expected_lookups_per_sample": int(loads[o]),
            "jagged_p2p": {k: med(rj, k) for k in keys}, "mp_p2p_constant_lengths": {k: med(rm, k) for k in keys},
            "jagged_over_mp": {k: med(rj, k) / med(rm, k) for k in keys},
            "jagged_one_gpu_lookup_us": float(np.median(rl)), "pooled_rows_bit_equal": equal,
            "p2p_over_one_gpu_lookup": med(rj, "lookup_us") / float(np.median(rl)),
            "all_repeats": {"jagged": rj, "mp": rm, "jagged_one_gpu_lookup_us": rl}}


def scatter(a, rows, P, W, dev, bw):
    """One rank's local batch (all tables, B_local bags each) into local stand-ins of the owners' buffers."""
    sh = TableSharding.build(rows, W, P)
    ntab, Bl = len(rows), a.batch
    rng = np.random.default_rng(77 + W)
    loc = [jagged_batch(rng, rows, P, Bl, dev) for _ in range(a.nb)]
    cap = [(2 * p - 1) * Bl for p in P]
    cap_own = [W * sum(cap[k] for k in sh.local[o]) for o in range(W)]
    vals = [torch.empty(max(1, c), dtype=torch.int32, device=dev) for c in cap_own]
    offs = [torch.empty(len(sh.local[o]) * Bl * W + 1, dtype=torch.int32, device=dev) for o in range(W)]
    lib = _lib.load()
    owner_arr = (C.c_int32 * ntab)(*sh.owner)
    pv = (C.c_void_p * W)(*[v.data_ptr() for v in vals])
    po = (C.c_void_p * W)(*[x.data_ptr() for x in offs])
    capa = (C.c_int64 * W)(*cap_own)
    L_alls = [(C.c_int64 * (W * ntab))(*(list(b.L) * W)) for b in loc]     # every rank sends a batch like this one

    def one(i):
        b = loc[i]
        _lib.check(lib.dlrmb_indices_scatter_p2p_jagged(
            dev.index or 0, b.values.data_ptr(), b.offsets.data_ptr(), None, 4, ntab, Bl, owner_arr, L_alls[i], W, 0,
            pv, po, None, capa, int(torch.cuda.current_stream(dev).cuda_stream)))
    us = [timed(one, a.nb, a.iters) for _ in range(a.repeats)]
    moved = float(np.mean([2 * 4 * (sum(b.L) + ntab * Bl) for b in loc]))       # values + offsets, read + write
    return {"scatter_us": float(np.median(us)), "all": us, "bytes_read_plus_written": moved,
            "frac_copy_bw": moved / float(np.median(us)) / 1e3 / bw}


def _counts_worker(rank, W, port, iters, q):
    import torch.distributed as dist

    from dlrm_jl_b200.sharded import exchange_jagged_counts
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=W)
    rng = np.random.default_rng(rank)
    P = [int(p) for p in MLPERF_HOTNESS.split(",")]
    lengths = [rng.integers(1, 2 * p, size=64) for p in P]
    jag = JaggedIndices.from_lengths(torch.zeros(int(sum(n.sum() for n in lengths)), dtype=torch.int32), lengths)
    for _ in range(20):
        exchange_jagged_counts(jag)
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(iters):
        exchange_jagged_counts(jag)
    us = (time.perf_counter() - t0) / iters * 1e6
    q.put((rank, us))
    dist.destroy_process_group()


def counts(W, iters=500):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_counts_worker, args=(r, W, port, iters, q)) for r in range(W)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(W)]
    for p in procs:
        p.join(timeout=60)
    return {"counts_allgather_us_per_step": max(u for _r, u in res), "per_rank_us": sorted(res),
            "where": "gloo over loopback, W processes on the CPUs of the machine that holds the GPU"}


def mode_step(a, rows, P):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world < 2 or torch.cuda.device_count() < 2:
        print(json.dumps(dict(gpu_info(), mode="step", measured=False,
                              reason=f"needs torchrun with >= 2 GPUs (WORLD_SIZE {world}, "
                                     f"{torch.cuda.device_count()} visible GPUs)")))
        return
    import torch.distributed as dist

    from dlrm_jl_b200.sharded import ShardedEmbedding
    rank = int(os.environ["RANK"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    Bl, D, ntab = a.batch, a.D, len(rows)
    cap = [(2 * p - 1) * Bl for p in P]
    se = ShardedEmbedding.create(rows, D, Bl, P, rank, world, dev, jagged_cap=cap)   # the counts go over a gloo group
    se.enable_peer_exchange(Bl, P=P, idx_bytes=4)     # peer-store index scatter, fused lookup + peer stores
    rng = np.random.default_rng(77 + rank)
    batches = [jagged_batch(rng, rows, P, Bl, dev) for _ in range(a.nb)]
    anchor = torch.zeros(1, device=dev, requires_grad=True)
    dT = torch.randn((Bl, 1 + ntab, D), device=dev) * 0.01

    def step(i):
        T = se.lookup(batches[i], anchor)
        se.sort_async()
        T.backward(dT)
        se.update(0.01)

    for i in range(3):
        step(i % a.nb)
    torch.cuda.synchronize()
    dist.barrier()
    steps = a.iters * a.nb
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i % a.nb)
    e1.record()
    e1.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3 / steps
    ms = e0.elapsed_time(e1) / steps
    if rank == 0:
        print(json.dumps(dict(gpu_info(), mode="step", measured=True, world=world, rows_cap=a.rows_cap, D=D, B_local=Bl,
                              hotness=list(P), lengths="uniform in 1 .. 2 P_k - 1", steps=steps, ms_per_step=ms,
                              wall_ms_per_step=wall_ms, samples_per_s=Bl * world / ms * 1e3,
                              barrier_timeouts=se.peer.barrier_timeouts(),
                              what="embedding part of the jagged sharded step: host count all-gather (gloo), "
                                   "peer-store index scatter, fused lookup + peer stores, side-stream sort, gradient "
                                   "all-to-all (NCCL), owner-side sparse SGD")), flush=True)
    dist.barrier()
    se.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["owner", "step"], default="owner")
    ap.add_argument("--worlds", default="2,4,8")
    ap.add_argument("--rows-cap", type=int, default=20_000_000)
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--nb", type=int, default=4)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sharded_jagged.py measures on a CUDA device; none is visible")
    P = [int(p) for p in MLPERF_HOTNESS.split(",")]
    rows = [min(r, a.rows_cap) for r in TERABYTE_EMBEDDING_SIZES]
    if a.mode == "step":
        mode_step(a, rows, P)
        return
    info = gpu_info()
    dev = torch.device("cuda", 0)
    bw = copy_bandwidth_gbs(dev)
    info = dict(info, copy_gbs=bw, rows_cap=a.rows_cap, D=a.D, B_local=a.batch, hotness=P,
                lengths="uniform in 1 .. 2 P_k - 1")
    out = open(a.out, "w") if a.out else None
    for W in [int(w) for w in a.worlds.split(",")]:
        for name, fn in (("owner", lambda: owner(a, rows, P, W, dev)), ("scatter", lambda: scatter(a, rows, P, W, dev, bw)),
                         ("counts", lambda: counts(W))):
            rec = dict(info, mode=name, world=W, **fn())
            line = json.dumps(rec)
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()


if __name__ == "__main__":
    main()
