#!/usr/bin/env python
"""Table-sharded embeddings with per-table pooling factors (the MLPerf DLRM-DCNv2 hotness list), B200.

Workload: MLPerf hotness list (214 lookups per sample) on Terabyte-shaped tables with rows capped at
--rows-cap (20M, as multihot.py --mode ab), D 128, B_local 2048.  Same timing method as multihot.py (a CUDA
graph of --nb launches over --nb pre-generated batches, replay timed with CUDA events); one JSON line per
mode with the GPU name and power limit read in the same process.

    python benchmarks/sharded_multihot.py --mode owner      # one GPU: every rank's owner-side work
    torchrun --nproc-per-node 8 benchmarks/sharded_multihot.py --mode step

--mode owner: for W = 2, 4, 8 and for the lookup-weighted plan (TableSharding.build(rows, W, P)) and the
  snake plan (TableSharding.build(rows, W)), each rank's owned tables in one handle at B_global = W * B_local:
    p2p   dlrmb_embedding_fwd_p2p_sort_mp into W local [B_local][1 + ntab][D] buffers + update_sorted on
          G [B_global][t][D] -- what the owner runs in the fused sharded step, minus the NVLink hop
    local dlrmb_embedding_fwd_sort_mp into one [B_global][t][D] buffer + update_sorted -- same bytes
  µs per step (median, min-max of --repeats), the fraction of the device-to-device copy bandwidth measured
  in the same process, and the busiest rank in µs under each plan.
--plan column (with --mode owner): the column-wise plan (TableSharding.build(rows, W, P, D=D, max_col_shards=8))
  beside the lookup-weighted one: every rank's owner-side µs -- for each of its width groups (one handle each),
  dlrmb_embedding_fwd_p2p_sort_mp with the destination map + update_sorted, all groups in one timed step -- the
  busiest rank under both plans, and, for the groups of split tables, the stand-alone sort of their indices
  (every holder of a split table sorts its whole index stream; column sharding cannot shrink that part).
--mode step: samples/s of the mixed-P sharded training step of the embeddings (NCCL index exchange,
  fused lookup + peer stores, gradient all-to-all, owner-side sparse SGD) under torchrun with >= 2 GPUs.
  With fewer GPUs it prints that nothing was measured.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from fractions import Fraction

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from dlrm_jl_b200.embedding import EmbeddingTables  # noqa: E402
from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES  # noqa: E402
from dlrm_jl_b200.sharded import ShardedEmbedding, TableSharding  # noqa: E402
from multihot import MLPERF_HOTNESS, copy_bandwidth_gbs, distinct, gpu_info, make_batches, timed, traffic  # noqa: E402


def _stats(xs):
    return {"median": float(np.median(xs)), "min": float(min(xs)), "max": float(max(xs)), "all": [float(x) for x in xs]}


def owner_rank(a, rows, P, sh, rank, dev, bw, with_local):
    """One rank's owned tables: p2p and (optionally) single-buffer step times, and the bit-equality check."""
    W, Bl, D, ntab = sh.world, a.batch, a.D, len(rows)
    Bg = Bl * W
    mine = sh.local[rank]
    if not mine:
        return {"rank": rank, "tables": [], "lookups_per_sample": 0, "p2p_us": None}
    r_rows, r_P = [rows[k] for k in mine], [P[k] for k in mine]
    t = EmbeddingTables(r_rows, D, Bg * max(r_P), dev)
    t.init_uniform(1 + rank)
    t.set_slot_map([1 + k for k in mine])
    rng = np.random.default_rng(1234 + rank)
    batches = make_batches(rng, r_rows, r_P, Bg, a.nb, 0.0, dev)
    bufs = [torch.empty((Bl, 1 + ntab, D), device=dev) for _ in range(W)]
    ptrs = [b.data_ptr() for b in bufs]
    out = torch.empty((Bg, len(mine), D), device=dev)
    G = torch.randn((Bg, len(mine), D), device=dev) * 0.01

    def step_p2p(i):
        t.lookup_p2p(batches[i], ptrs, Bl, 1 + ntab, 0, sort=True)
        t.update_sorted(G, 0, 0.01)

    def step_local(i):
        t.lookup(batches[i], out, 0, 0, sort=True)
        t.update_sorted(G, 0, 0.01)

    # same pooled rows either way (checked on batch 0 before timing; lr 0 leaves the tables as they are)
    t.lookup_p2p(batches[0], ptrs, Bl, 1 + ntab, 0, sort=False)
    t.lookup(batches[0], out, 0, 0, sort=False)
    torch.cuda.synchronize()
    via_peers = torch.cat([b[:, [1 + k for k in mine]] for b in bufs], dim=0)
    equal = bool(torch.equal(via_peers, out))
    res_p, res_l = [], []
    for _ in range(a.repeats):
        res_p.append(timed(step_p2p, a.nb, a.iters))
        if with_local:
            res_l.append(timed(step_local, a.nb, a.iters))
    U = distinct(batches, Bg)
    look, upd, _ = traffic(r_rows, r_P, Bg, D, U)
    r = {"rank": rank, "tables": mine, "lookups_per_sample": sum(r_P), "pooled_rows_bit_equal": equal,
         "p2p_us": _stats(res_p), "algorithmic_bytes": look + upd,
         "p2p_frac_copy_bw": (look + upd) / float(np.median(res_p)) / 1e3 / bw}
    if with_local:
        r["local_us"] = _stats(res_l)
        r["p2p_over_local"] = float(np.median(res_p) / np.median(res_l))
    t.close()
    del bufs, out, G, batches
    torch.cuda.empty_cache()
    return r


def owner_rank_cw(a, rows, P, sh, rank, dev):
    """One rank's units under a column-wise plan: one handle per width group, all groups in one timed step."""
    W, Bl, D, ntab = sh.world, a.batch, a.D, len(rows)
    Bg = Bl * W
    groups = sh.groups(rank)
    if not groups:
        return {"rank": rank, "groups": [], "lookups_per_sample": 0, "p2p_us": None}
    bufs = [torch.empty((Bl, 1 + ntab, D), device=dev) for _ in range(W)]
    ptrs = [b.data_ptr() for b in bufs]
    rng = np.random.default_rng(1234 + rank)
    hs, bats, Gs = [], [], []
    for c, ks in groups:
        r_rows, r_P = [rows[k] for k in ks], [P[k] for k in ks]
        t = EmbeddingTables(r_rows, D // c, Bg * max(r_P), dev)
        t.init_uniform(1 + rank + 97 * c)
        t.set_dest_map([1 + k for k in ks], [sh.slice_of(k, rank) * (D // c) for k in ks], D)
        hs.append(t)
        bats.append(make_batches(rng, r_rows, r_P, Bg, a.nb, 0.0, dev))
        Gs.append(torch.randn((Bg, len(ks), D // c), device=dev) * 0.01)

    def step(i):
        for t, b, G in zip(hs, bats, Gs):
            t.lookup_p2p(b[i], ptrs, Bl, 1 + ntab, 0, sort=True)
            t.update_sorted(G, 0, 0.01)

    res = [timed(step, a.nb, a.iters) for _ in range(a.repeats)]
    r = {"rank": rank, "groups": [{"shards": c, "tables": ks, "slices": [sh.slice_of(k, rank) for k in ks]} for c, ks in groups],
         "lookups_per_sample": float(sum(Fraction(P[k], c) for c, ks in groups for k in ks)), "p2p_us": _stats(res)}
    split = [(t, b) for (c, _ks), t, b in zip(groups, hs, bats) if c > 1]
    if split:
        r["split_sort_us"] = _stats([timed(lambda i: [t.sort(b[i]) for t, b in split], a.nb, a.iters)
                                     for _ in range(a.repeats)])
    for t in hs:
        t.close()
    del bufs, bats, Gs
    torch.cuda.empty_cache()
    return r


def mode_owner_column(a, rows, P, dev, info):
    lines = []
    for W in (2, 4, 8):
        res = {}
        for plan in ("lookup_weighted", "column"):
            if plan == "column":
                sh = TableSharding.build(rows, W, P, D=a.D, max_col_shards=8)
                ranks = [owner_rank_cw(a, rows, P, sh, r, dev) for r in range(W)]
            else:
                sh = TableSharding.build(rows, W, P)
                ranks = [owner_rank(a, rows, P, sh, r, dev, info["copy_gbs"], False) for r in range(W)]
            busiest = max((x for x in ranks if x["p2p_us"]), key=lambda x: x["p2p_us"]["median"])
            res[plan] = {"shards": list(sh.shards) if sh.split else None,
                         "holders": sh.holders if sh.split else [[o] for o in sh.owner],
                         "lookups_per_rank": [float(x) for x in sh.lookups_per_rank()],
                         "ranks": ranks, "busiest_rank": busiest["rank"],
                         "busiest_rank_p2p_us": busiest["p2p_us"]["median"]}
        r = dict(info, mode="owner", plan="column", world=W, rows_cap=a.rows_cap, D=a.D, B_local=a.batch,
                 B_global=W * a.batch, hotness=list(P), max_col_shards=8, nb=a.nb, iters=a.iters, repeats=a.repeats,
                 **res, busiest_rank_us={p: res[p]["busiest_rank_p2p_us"] for p in res})
        print(json.dumps(r), flush=True)
        lines.append(r)
    return lines


def mode_owner(a, rows, P, dev, info):
    lines = []
    for W in (2, 4, 8):
        res = {}
        for plan in ("lookup_weighted", "snake"):
            sh = TableSharding.build(rows, W, P) if plan == "lookup_weighted" else TableSharding.build(rows, W)
            ranks = [owner_rank(a, rows, P, sh, r, dev, info["copy_gbs"], plan == "lookup_weighted") for r in range(W)]
            busiest = max((x for x in ranks if x["p2p_us"]), key=lambda x: x["p2p_us"]["median"])
            res[plan] = {"owner": sh.owner, "lookups_per_rank": [x["lookups_per_sample"] for x in ranks], "ranks": ranks,
                         "busiest_rank": busiest["rank"], "busiest_rank_p2p_us": busiest["p2p_us"]["median"]}
        r = dict(info, mode="owner", world=W, rows_cap=a.rows_cap, D=a.D, B_local=a.batch, B_global=W * a.batch,
                 hotness=list(P), nb=a.nb, iters=a.iters, repeats=a.repeats, **res,
                 busiest_rank_us={"snake": res["snake"]["busiest_rank_p2p_us"],
                                  "lookup_weighted": res["lookup_weighted"]["busiest_rank_p2p_us"]})
        print(json.dumps(r), flush=True)
        lines.append(r)
    return lines


def mode_step(a, rows, P):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world < 2 or torch.cuda.device_count() < 2:
        print(json.dumps({"mode": "step", "measured": False,
                          "reason": f"needs torchrun with >= 2 GPUs (WORLD_SIZE {world}, {torch.cuda.device_count()} visible GPUs)"}))
        return
    import torch.distributed as dist
    rank = int(os.environ["RANK"])
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    Bl, D = a.batch, a.D
    se = ShardedEmbedding.create(rows, D, Bl, P, rank, world, dev)
    se.enable_peer_exchange(Bl)             # fused lookup + peer stores; indices over NCCL
    rng = np.random.default_rng(77 + rank)
    batches = [[torch.from_numpy(rng.integers(0, r, size=(Bl, p)).astype(np.int32)) for r, p in zip(rows, P)]
               for _ in range(a.nb)]
    from dlrm_jl_b200.embedding import _as_index_tensor
    batches = [_as_index_tensor(b, len(rows), dev) for b in batches]
    anchor = torch.zeros(1, device=dev, requires_grad=True)
    dT = torch.randn((Bl, 1 + len(rows), D), device=dev) * 0.01

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
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i % a.nb)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if rank == 0:
        print(json.dumps(dict(gpu_info(), mode="step", measured=True, world=world, rows_cap=a.rows_cap, D=D, B_local=Bl,
                              hotness=list(P), steps=steps, ms_per_step=ms, samples_per_s=Bl * world / ms * 1e3,
                              what="embedding part of the mixed-P sharded step: forward exchange, fused lookup, "
                                   "gradient all-to-all, owner-side sparse SGD")))
    se.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="owner", choices=["owner", "step"])
    ap.add_argument("--plan", default="table", choices=["table", "column"],
                    help="owner mode: table-wise plans (lookup-weighted and snake) or the column-wise plan")
    ap.add_argument("--hotness", default=MLPERF_HOTNESS)
    ap.add_argument("--rows-cap", type=int, default=20_000_000)
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--batch", type=int, default=2048, help="B_local")
    ap.add_argument("--nb", type=int, default=4)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    a = ap.parse_args()
    P = [int(x) for x in a.hotness.split(",")]
    rows = [min(r, a.rows_cap) for r in TERABYTE_EMBEDDING_SIZES]
    assert len(P) == len(rows)
    if a.mode == "step":
        mode_step(a, rows, P)
        return
    if not torch.cuda.is_available():
        raise SystemExit("--mode owner measures on a GPU; none is visible (nothing measured)")
    dev = torch.device("cuda", 0)
    info = dict(gpu_info(), copy_gbs=copy_bandwidth_gbs(dev))
    lines = (mode_owner_column if a.plan == "column" else mode_owner)(a, rows, P, dev, info)
    if a.out:
        with open(a.out, "a") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
