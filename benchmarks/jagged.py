"""Variable-length bags (the `_jagged` entry points) against the `_mp` path, B200.

Workload: the MLPerf DLRM-DCNv2 hotness list on Terabyte-shaped tables (rows capped at --rows-cap), D 128, B 2048,
uniform indices.  Method of multihot.py: a CUDA graph of --nb launches over --nb pre-generated batches, replay timed
with CUDA events; lookup, lookup + sort, and lookup + sort + update, in µs and as a share of the measured copy
bandwidth; one JSON line per mode, with the GPU name and power limit read in the same process.
  const  bags of exactly P_k lookups through the jagged path, against the `_mp` path on the same batch: the same
         work, so the gap is the cost of the jagged path
  var    bag lengths uniform in 1 .. 2 P_k - 1 (the same expected total) through the jagged path, against `_mp` at P_k
  mean   mean against sum pooling on the var batches
  weighted  per-sample weights (random, f32) against the unweighted sum on the var batches, and the weight
         gradient (dw = dT . row per entry) on its own, with its algorithmic bytes over the copy bandwidth

    python benchmarks/jagged.py --out profiles/r07_jagged_b200.jsonl
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from dlrm_jl_b200.embedding import EmbeddingTables, JaggedIndices  # noqa: E402
from dlrm_jl_b200.model import TERABYTE_EMBEDDING_SIZES  # noqa: E402
from multihot import MLPERF_HOTNESS, copy_bandwidth_gbs, gpu_info, make_batches, timed  # noqa: E402


def jagged_batches(rng, rows, P, B, nb, pooling, dev):
    out = []
    for _ in range(nb):
        lengths = [rng.integers(1, 2 * p, size=B) for p in P]
        vals = np.concatenate([rng.integers(0, r, size=int(n.sum())) for r, n in zip(rows, lengths)]).astype(np.int32)
        out.append(JaggedIndices.from_lengths(torch.from_numpy(vals), lengths, pooling).to(dev))
    return out


def lookup_bytes(L, B, D, ntab, offsets_bytes=0):
    """Rows read + pooled rows written + indices read (+ the jagged path's offsets)."""
    return sum(L) * D * 4 + ntab * B * D * 4 + sum(L) * 4 + offsets_bytes


def measure(t, batches, T, dT, a):
    us_l = timed(lambda i: t.lookup(batches[i], T, 1), a.nb, a.iters)
    us_ls = timed(lambda i: t.lookup(batches[i], T, 1, sort=True), a.nb, a.iters)

    def chain(i):
        t.lookup(batches[i], T, 1, sort=True)
        t.update_sorted(dT, 1, 0.01)
    us_c = timed(chain, a.nb, a.iters)
    return {"lookup_us": us_l, "lookup_sort_us": us_ls, "lookup_sort_update_us": us_c}


def weight_grad_bytes(L, B, D, ntab, offsets_bytes):
    """Rows read + indices read + dw written + one dT row read per bag + the offsets."""
    return sum(L) * D * 4 + sum(L) * 4 + sum(L) * 4 + ntab * B * D * 4 + offsets_bytes


def with_bw(r, nbytes, bw):
    r = dict(r)
    r["lookup_algorithmic_bytes"] = nbytes
    r["lookup_frac_copy_bw"] = nbytes / r["lookup_us"] / 1e3 / bw
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", choices=["const", "var", "mean", "weighted"], nargs="+", default=["const", "var", "mean"])
    ap.add_argument("--hotness", default=MLPERF_HOTNESS)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--rows-cap", type=int, default=20_000_000)
    ap.add_argument("--D", type=int, default=128)
    ap.add_argument("--nb", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("benchmarks/jagged.py measures the GPU: no CUDA device")
    dev = torch.device("cuda", 0)
    P = [int(x) for x in a.hotness.split(",")]
    B, D = a.batch, a.D
    rows = [min(r, a.rows_cap) for r in TERABYTE_EMBEDDING_SIZES][:len(P)]
    info = gpu_info()
    info["copy_gbs"] = copy_bandwidth_gbs(dev)
    bw = info["copy_gbs"]
    t = EmbeddingTables(rows, D, 2 * B * max(P), dev)
    t.init_uniform(1)
    T = torch.empty((B, 1 + len(rows), D), device=dev)
    dT = torch.randn((B, 1 + len(rows), D), device=dev) * 0.01
    rng = np.random.default_rng(1234)
    packed = make_batches(rng, rows, P, B, a.nb, 0.0, dev)
    const = [JaggedIndices.from_dense(p) for p in packed]
    var_sum = jagged_batches(np.random.default_rng(99), rows, P, B, a.nb, "sum", dev)
    var_mean = [JaggedIndices(j.values, j.offsets, j.L, j.B, "mean") for j in var_sum]
    wrng = np.random.default_rng(7)
    var_weighted = [JaggedIndices(j.values, j.offsets, j.L, j.B, "sum",
                                  torch.from_numpy(wrng.uniform(0.0, 2.0, j.values.numel()).astype(np.float32)).to(dev))
                    for j in var_sum]
    ntab = len(rows)
    off_bytes = (ntab * B + 1) * 4
    L_mp = [B * p for p in P]
    L_var = [float(np.mean([j.L[k] for j in var_sum])) for k in range(ntab)]
    for mode in a.mode:
        for rep in range(a.repeats):
            if mode == "const":
                base = with_bw(measure(t, packed, T, dT, a), lookup_bytes(L_mp, B, D, ntab), bw)
                new = with_bw(measure(t, const, T, dT, a), lookup_bytes(L_mp, B, D, ntab, off_bytes), bw)
                names = ("mp", "jagged_const")
            elif mode == "var":
                base = with_bw(measure(t, packed, T, dT, a), lookup_bytes(L_mp, B, D, ntab), bw)
                new = with_bw(measure(t, var_sum, T, dT, a), lookup_bytes(L_var, B, D, ntab, off_bytes), bw)
                names = ("mp", "jagged_var")
            elif mode == "mean":
                base = with_bw(measure(t, var_sum, T, dT, a), lookup_bytes(L_var, B, D, ntab, off_bytes), bw)
                new = with_bw(measure(t, var_mean, T, dT, a), lookup_bytes(L_var, B, D, ntab, off_bytes), bw)
                names = ("jagged_var_sum", "jagged_var_mean")
            else:
                base = with_bw(measure(t, var_sum, T, dT, a), lookup_bytes(L_var, B, D, ntab, off_bytes), bw)
                # the weights are read once per gathered row: 4 bytes more per lookup
                new = with_bw(measure(t, var_weighted, T, dT, a),
                              lookup_bytes(L_var, B, D, ntab, off_bytes + 4 * sum(L_var)), bw)
                names = ("jagged_var_sum", "jagged_var_weighted")
            r = dict(info, mode=mode, repeat=rep, rows_cap=a.rows_cap, D=D, B=B, hotness=P,
                     lookups_per_step_mp=sum(L_mp), lookups_per_step_var_mean=sum(L_var),
                     **{names[0]: base, names[1]: new},
                     ratio={k: new[k] / base[k] for k in ("lookup_us", "lookup_sort_us", "lookup_sort_update_us")})
            if mode == "weighted":
                us_dw = timed(lambda i: t.weight_grad(var_weighted[i], dT, 1), a.nb, a.iters)
                nbytes = weight_grad_bytes(L_var, B, D, ntab, off_bytes)
                r["weight_grad"] = {"us": us_dw, "algorithmic_bytes": nbytes, "frac_copy_bw": nbytes / us_dw / 1e3 / bw}
            line = json.dumps(r)
            print(line, flush=True)
            if a.out:
                with open(a.out, "a") as f:
                    f.write(line + "\n")
    t.close()


if __name__ == "__main__":
    main()
