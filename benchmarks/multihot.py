#!/usr/bin/env python
"""Multi-hot embeddings with per-table pooling factors (the `_mp` entry points), B200.

Default workload: the MLPerf DLRM-DCNv2 hotness list (214 lookups per sample over 26 tables) on
Terabyte-shaped tables (rows capped at --rows-cap), D 128, B 2048, uniform indices (--zipf for skew).
Same method as hotpath.py: a CUDA graph of --nb launches over --nb pre-generated batches, replay timed
with CUDA events; one JSON line per mode, with the GPU name and power limit read in the same process.

    python benchmarks/multihot.py --mode ab --rows-cap 20000000     # mixed vs one handle per hotness group
    python benchmarks/multihot.py --mode full                        # mixed only, rows capped at 40M
    python benchmarks/multihot.py --mode step                        # DLRMModel training step, samples/s
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from dlrm_jl_b200 import _prof  # noqa: E402
from dlrm_jl_b200.embedding import EmbeddingTables, PackedIndices  # noqa: E402
from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES  # noqa: E402
from hotpath import zipf_indices  # noqa: E402

MLPERF_HOTNESS = "3,2,1,2,6,1,1,1,1,7,3,8,1,6,9,5,1,1,1,12,100,27,10,3,1,1"
SGD_RTOL = 1e-4


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def copy_bandwidth_gbs(dev) -> float:
    """Device-to-device copy of 4 GB (read + write bytes / time): the HBM rate the fractions refer to."""
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    gbs = 10 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def make_batches(rng, rows, P, B, nb, zipf, dev):
    out = []
    for _ in range(nb):
        parts = [(zipf_indices(rng, r, B * p, zipf) if zipf else rng.integers(0, r, size=B * p)).astype(np.int32)
                 for r, p in zip(rows, P)]
        out.append(PackedIndices(torch.from_numpy(np.concatenate(parts)).to(dev), tuple(P), B))
    return out


def distinct(batches, B):
    return [float(np.mean([len(np.unique(b[k].cpu().numpy())) for b in batches])) for k in range(len(batches[0]))]


def traffic(rows, P, B, D, U, eb=4):
    L = [B * p for p in P]
    look = sum(l * D * eb + B * D * 4 + l * 4 for l in L)                     # SURVEY 8(d), per table
    upd = sum(B * D * 4 + l * 4 for l in L) + 2 * sum(U) * D * eb
    return look, upd, sum(l * D * 4 for l in L)                               # last: gradient rows read per entry


def timed(fn, nb, iters):
    return _prof.time_launches(fn, nb, iters, True)


def mode_full(a, rows, P, dev, info):
    D, B = a.D, a.batch
    t = EmbeddingTables(rows, D, B * max(P), dev)
    t.init_uniform(1)
    rng = np.random.default_rng(1234)
    batches = make_batches(rng, rows, P, B, a.nb, a.zipf, dev)
    T = torch.empty((B, 1 + len(rows), D), device=dev)
    dT = torch.randn((B, 1 + len(rows), D), device=dev) * 0.01
    us_l = timed(lambda i: t.lookup(batches[i], T, 1), a.nb, a.iters)
    us_ls = timed(lambda i: t.lookup(batches[i], T, 1, sort=True), a.nb, a.iters)

    def chain(i):
        t.lookup(batches[i], T, 1, sort=True)
        t.update_sorted(dT, 1, 0.01)
    us_c = timed(chain, a.nb, a.iters)
    U = distinct(batches, B)
    look, upd, grad_entries = traffic(rows, P, B, D, U)
    bw = info["copy_gbs"]
    us_u = us_c - us_ls
    r = dict(info, mode="full", rows_cap=a.rows_cap, D=D, B=B, hotness=list(P), zipf=a.zipf,
             lookups_per_step=B * sum(P), distinct_rows=sum(U),
             lookup={"us": us_l, "algorithmic_bytes": look, "frac_copy_bw": look / us_l / 1e3 / bw},
             lookup_sort={"us": us_ls},
             update={"us": us_u, "algorithmic_bytes": upd, "frac_copy_bw": upd / us_u / 1e3 / bw,
                     "gradient_rows_per_entry_bytes": grad_entries,
                     "frac_copy_bw_with_entry_gradient_rows": (upd - sum(B * D * 4 for _ in P) + grad_entries) / us_u / 1e3 / bw},
             chain={"us": us_c})
    t.close()
    return r


def mode_ab(a, rows, P, dev, info):
    D, B = a.D, a.batch
    ntab = len(rows)
    mixed = EmbeddingTables(rows, D, B * max(P), dev)
    mixed.init_uniform(1)
    groups = {}
    for k, p in enumerate(P):
        groups.setdefault(p, []).append(k)
    handles = []
    for p, ks in sorted(groups.items()):
        h = EmbeddingTables([rows[k] for k in ks], D, B * p, dev)
        for j, k in enumerate(ks):
            h.table(j).copy_(mixed.table(k))
        handles.append((p, ks, h))
    rng = np.random.default_rng(1234)
    batches = make_batches(rng, rows, P, B, a.nb, a.zipf, dev)
    gb = [[torch.stack([b[k] for k in ks]).contiguous() for (_p, ks, _h) in handles] for b in batches]
    T = torch.empty((B, 1 + ntab, D), device=dev)
    dT = torch.randn((B, 1 + ntab, D), device=dev) * 0.01
    Tg = [torch.empty((B, 1 + len(ks), D), device=dev) for (_p, ks, _h) in handles]
    dTg = []
    for (_p, ks, _h) in handles:
        g = torch.empty((B, 1 + len(ks), D), device=dev)
        g[:, 1:] = dT[:, [1 + k for k in ks]]
        dTg.append(g)

    def step_mixed(i):
        mixed.lookup(batches[i], T, 1, sort=True)
        mixed.update_sorted(dT, 1, 0.01)

    def step_grouped(i):
        for j, (_p, _ks, h) in enumerate(handles):
            h.lookup(gb[i][j], Tg[j], 1, sort=True)
            h.update_sorted(dTg[j], 1, 0.01)

    # equality check on batch 0 before timing: pooled rows bit-equal, tables within SGD_RTOL
    step_mixed(0)
    step_grouped(0)
    torch.cuda.synchronize()
    pooled_equal = all(torch.equal(T[:, [1 + k for k in ks]], Tg[j][:, 1:]) for j, (_p, ks, _h) in enumerate(handles))
    worst = 0.0
    for (_p, ks, h) in handles:
        for j, k in enumerate(ks):
            a_, b_ = mixed.table(k), h.table(j)
            worst = max(worst, float(torch.linalg.norm(a_ - b_) / torch.linalg.norm(b_)))
    res_m, res_g = [], []
    for _ in range(a.repeats):
        res_m.append(timed(step_mixed, a.nb, a.iters))
        res_g.append(timed(step_grouped, a.nb, a.iters))
    r = dict(info, mode="ab", rows_cap=a.rows_cap, D=D, B=B, hotness=list(P), zipf=a.zipf, groups=len(handles),
             pooled_rows_bit_equal=bool(pooled_equal), tables_max_rel_err=worst, tables_within_rtol=worst < SGD_RTOL,
             mixed_step_us={"median": float(np.median(res_m)), "min": min(res_m), "max": max(res_m), "all": res_m},
             grouped_step_us={"median": float(np.median(res_g)), "min": min(res_g), "max": max(res_g), "all": res_g},
             launches_per_step={"mixed": None, "grouped": None})
    from dlrm_jl_b200 import _lib
    for name, fn in (("mixed", step_mixed), ("grouped", step_grouped)):
        n0 = _lib.launch_count()
        fn(0)
        r["launches_per_step"][name] = _lib.launch_count() - n0
    torch.cuda.synchronize()
    mixed.close()
    for (_p, _ks, h) in handles:
        h.close()
    return r


def mode_step(a, rows, P, dev, info):
    from dlrm_jl_b200.embedding import Descent
    from dlrm_jl_b200.model import dlrm
    from dlrm_jl_b200.train import bce_loss, train_step, wrap_loss
    D, B = a.D, a.batch
    m = dlrm([13, 512, 256, D], [1024, 1024, 512, 256, 1], D, rows, max_lookups=B * max(P), device=dev)
    rng = np.random.default_rng(7)
    batches = make_batches(rng, rows, P, B, a.nb, a.zipf, dev)
    dense = [torch.rand((B, 13), device=dev) for _ in range(a.nb)]
    labels = [(torch.rand(B, device=dev) < 0.25).float() for _ in range(a.nb)]
    loss, opt = wrap_loss(bce_loss), Descent(0.01)
    for i in range(3):
        train_step(loss, m, opt, labels[i % a.nb], dense[i % a.nb], batches[i % a.nb])
    torch.cuda.synchronize()
    steps = a.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        l = train_step(loss, m, opt, labels[i % a.nb], dense[i % a.nb], batches[i % a.nb])
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / steps
    m.embeddings.close()
    return dict(info, mode="step", rows_cap=a.rows_cap, D=D, B=B, hotness=list(P), steps=steps, ms_per_step=ms,
                samples_per_s=B / ms * 1e3, last_loss=float(l))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["ab", "full", "step"], nargs="+", default=["full"])
    ap.add_argument("--hotness", default=MLPERF_HOTNESS)
    ap.add_argument("--zipf", type=float, default=0.0)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--rows-cap", type=int, default=40_000_000)
    ap.add_argument("--ab-rows-cap", type=int, default=20_000_000, help="rows cap of --mode ab (two copies of the tables)")
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--nb", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multihot.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda", 0)
    P = [int(x) for x in a.hotness.split(",")]
    info = gpu_info()
    info["copy_gbs"] = copy_bandwidth_gbs(dev)
    full_cap = a.rows_cap
    for mode in a.mode:
        a.rows_cap = a.ab_rows_cap if mode == "ab" else full_cap
        rows = [min(r, a.rows_cap) for r in TERABYTE_EMBEDDING_SIZES][:len(P)]
        if mode == "full":
            r = mode_full(a, rows, P, dev, info)
        elif mode == "ab":
            r = mode_ab(a, rows, P, dev, info)
        else:
            r = mode_step(a, rows, P, dev, info)
        torch.cuda.empty_cache()
        line = json.dumps(r)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(line + "\n")


if __name__ == "__main__":
    main()
