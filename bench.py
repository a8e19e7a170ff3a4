#!/usr/bin/env python
"""bench.py -- DLRM training samples/s on synthetic Criteo-shaped data (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload terabyte|kaggle|sweep] [--batch B] [--no-cpu-baseline] [--dump-outputs DIR]

A "step" is one DLRM training step on one batch: embedding lookup -> bottom MLP -> dot
interaction -> top MLP -> BCE -> backward (interaction pullback) -> dense SGD -> sparse
gradient scatter-add + in-place SGD.  The lookup, interaction and sparse update are this
repo's sm_100a kernels (libdlrm_b200.so through the C ABI); the MLPs are library GEMMs
(torch/cuBLAS, fp32, TF32 off), as the reference keeps them in oneDNN.

Default workload (all N): Terabyte-shaped -- 26 tables, rows = min(TERABYTE_EMBEDDING_SIZES,
40M), D = 128 (104.5 GB of fp32 tables, fits one B200), batch 2048 PER GPU (weak scaling).
N > 1: tables sharded table-wise, pooled embeddings / gradients exchanged by all-to-all, MLPs
data-parallel.  `--workload kaggle` = 26 Kaggle tables, D = 64, B = 2048 (BASELINE config 3).

`--impl reference`: the reference's CPU algorithm for the same step (C restatement of the
Julia path for lookup / interaction / sparse SGD + torch-CPU (oneDNN) MLPs) on the host cores.
`--workload sweep`: BASELINE config 5, the single-table embedding microbenchmark grid (rows 1e5-1e8,
D 16-256, pooling 1-64, uniform / Zipf 1.05 / Zipf 1.2), gather + sort + update GB/s per case.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TERABYTE_CAP = 40_000_000
LR = 0.1  # script.jl:14
# arithmetic type of the path: fp32 everywhere; the interaction forward computes its Gram matrix on the
# tensor cores in 3xTF32 form (error-compensated, measured 1.2e-6 relative against float64, tolerance 1e-5)
DTYPE_LABEL = "f32 (3xTF32 interaction forward)"


def workload(name: str, batch: int):
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES, TERABYTE_EMBEDDING_SIZES
    if name == "terabyte":
        rows = [min(r, TERABYTE_CAP) for r in TERABYTE_EMBEDDING_SIZES]
        D = 128
    elif name == "kaggle":
        rows = list(KAGGLE_EMBEDDING_SIZES)
        D = 64
    else:
        raise SystemExit(f"unknown workload {name}")
    F = len(rows) + 1
    return dict(name=name, rows=rows, D=D, B=batch, P=1, F=F,
                bottom=[13, 512, 256, D], top=[D + F * (F - 1) // 2, 1024, 1024, 512, 256, 1])


def synth_batch(wl, step: int, rank: int = 0, rows_cap: int | None = None):
    """SURVEY section 8(d): rng = default_rng(20261018 + step); dense U[0,1); labels Bernoulli(0.25);
    indices uniform over [0, rows_k)."""
    rng = np.random.default_rng(20261018 + step * 1009 + rank)
    B = wl["B"]
    dense = rng.random((B, 13), dtype=np.float32)
    labels = (rng.random(B) < 0.25).astype(np.float32)
    rows = wl["rows"] if rows_cap is None else [min(r, rows_cap) for r in wl["rows"]]
    idx = np.stack([rng.integers(0, r, size=B, dtype=np.int64) for r in rows]).astype(np.int32)
    return dense, labels, idx[:, :, None]


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed regions: an NVML polling thread (5 ms period;
    `nvidia-smi -lms` as the fallback) whose samples are kept only if they fall inside a window
    opened with `begin()` and closed with `end()`."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []      # (time, sm_mhz, max_mhz, reasons)
        self.windows = []
        self._open = None
        self._stop = threading.Event()
        self.thread = None
        self.proc = None
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.index
            if vis:
                try:
                    phys = int(vis.split(",")[self.index])
                except (ValueError, IndexError):
                    phys = self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop.is_set():
                    try:
                        mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        r = int(get_reasons(h))
                        self.samples.append((time.perf_counter(), mhz, mx, {n for n, b in bits.items() if r & b}))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            self.source = "nvml, 5 ms period"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            self.source = "nvidia-smi -lms 20"
        except Exception:
            self.proc = None

    def _pump(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                self.samples.append((time.perf_counter(), float(parts[0]), float(parts[1]),
                                     {n for n, v in zip(names, parts[3:7]) if v.lower().startswith("active")}))
            except ValueError:
                continue

    def begin(self):
        self._open = time.perf_counter()

    def end(self):
        if self._open is not None:
            self.windows.append((self._open, time.perf_counter()))
            self._open = None

    def stop(self):
        if self.thread is None:
            return None
        time.sleep(0.03)
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in self.windows)]
        used = inside or self.samples
        if not used:
            return None
        reasons = set()
        for s_ in used:
            reasons |= s_[3]
        return {"sm_mhz": float(np.median([s_[1] for s_ in used])), "sm_max_mhz": float(max(s_[2] for s_ in used)),
                "reasons": sorted(reasons), "samples": len(used),
                "window": "inside the timed regions (value + e2e)" if inside else "whole run (no sample fell inside the timed regions)",
                "source": self.source}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm on the host cores
# ----------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Host cores this process may use.  Not omp_get_max_threads(): torch.distributed.run exports
    OMP_NUM_THREADS=1 to its workers, which would pin the CPU arm to one core.  DLRMB_CPU_THREADS overrides."""
    env = os.environ.get("DLRMB_CPU_THREADS")
    if env:
        return max(1, int(env))
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def host_ram_bytes():
    """(total, available) host memory in bytes (/proc/meminfo), (0, 0) if unknown."""
    try:
        info = {}
        with open("/proc/meminfo") as fh:
            for line in fh:
                k, v = line.split(":")
                info[k] = int(v.split()[0]) * 1024
        return info.get("MemTotal", 0), info.get("MemAvailable", 0)
    except Exception:
        return 0, 0


def auto_rows_cap(wl, budget_bytes: int) -> int:
    """Largest per-table row cap (a power of two, or no cap) whose tables fit `budget_bytes`."""
    full = sum(wl["rows"]) * wl["D"] * 4
    if full <= budget_bytes:
        return max(wl["rows"])
    cap = 1 << 26
    while cap > 1024 and sum(min(r, cap) for r in wl["rows"]) * wl["D"] * 4 > budget_bytes:
        cap >>= 1
    return cap


def cpu_arm(wl, steps: int, warmup: int, rows_cap: int, budget_s: float = 25.0):
    """Full training step on the CPU.  Tables capped at `rows_cap` rows each (0 = the largest cap that fits
    55 % of the available host RAM, at most 112 GiB: the full-size Terabyte-shaped tables, 97 GiB, on a box with
    ~180 GiB free); everything else (batch, D, MLP sizes, step structure) is the workload's."""
    import torch
    from oracle import c_oracle as CO
    threads = host_threads()
    torch.set_num_threads(threads)
    ram_total, ram_avail = host_ram_bytes()
    if rows_cap <= 0:
        budget = min(int(0.55 * ram_avail) if ram_avail else (4 << 30), 112 << 30)
        rows_cap = auto_rows_cap(wl, budget)
    rows = [min(r, rows_cap) for r in wl["rows"]]
    D, B, F = wl["D"], wl["B"], wl["F"]
    tables = [CO.init_uniform(r, D, 1 + k, threads) for k, r in enumerate(rows)]

    def mlp(sizes, sigmoid_last):
        mods = []
        for i in range(1, len(sizes)):
            mods.append(torch.nn.Linear(sizes[i - 1], sizes[i]))
            mods.append(torch.nn.Sigmoid() if (sigmoid_last and i == len(sizes) - 1) else torch.nn.ReLU())
        return torch.nn.Sequential(*mods)

    torch.manual_seed(0)
    bottom, top = mlp(wl["bottom"], False), mlp(wl["top"], True)
    params = list(bottom.parameters()) + list(top.parameters())
    T = np.zeros((B, F, D), dtype=np.float32)
    z = np.empty((B, wl["top"][0]), dtype=np.float32)
    dT = np.empty_like(T)
    dx = np.empty((B, D), dtype=np.float32)

    def step(i):
        dense, labels, idx = synth_batch(wl, 10_000 + i, rows_cap=rows_cap)
        idx64 = np.ascontiguousarray(idx, dtype=np.int64)
        t0 = time.perf_counter()
        for p in params:
            p.grad = None
        CO.lookup(tables, idx64, slot0=1, out=T, nthreads=threads)     # maplookup (model.jl:161)
        x = bottom(torch.from_numpy(dense))                            # bottom MLP (oneDNN)
        T[:, 0, :] = x.detach().numpy()                                # fast_vcat (interact.jl:271-281)
        CO.interaction_fwd(T, out=z, nthreads=threads)                 # DotInteraction (:394-411)
        zt = torch.from_numpy(z).requires_grad_(True)
        out = top(zt).reshape(-1)
        loss = torch.nn.functional.binary_cross_entropy(out, torch.from_numpy(labels))
        loss.backward()
        CO.interaction_bwd(zt.grad.numpy(), T, dT=dT, dx=dx, nthreads=threads)   # dot_back (:424-436)
        x.backward(torch.from_numpy(dx))
        with torch.no_grad():
            torch._foreach_add_(params, [p.grad for p in params], alpha=-LR)
        CO.sparse_sgd(tables, idx64, dT, 1, LR, nthreads=threads)      # EmbeddingTables.update!
        _ = float(loss.detach())
        return time.perf_counter() - t0

    for i in range(warmup):
        step(i)
    times = []
    t_start = time.perf_counter()
    for i in range(steps):
        times.append(step(warmup + i))
        if time.perf_counter() - t_start > budget_s and len(times) >= 3:
            break
    total = float(sum(times))
    capped = rows_cap < max(wl["rows"])
    return dict(value=B * len(times) / total, ms_per_step=1e3 * total / len(times), steps=len(times),
                cores=threads, rows_cap=(rows_cap if capped else None), host_ram_gb=round(ram_total / 2**30, 1),
                sample=(f"{len(times)} full training steps (after {warmup} warm-up), batch {B}, 26 tables, D {D}, "
                        + (f"rows capped at {rows_cap} per table to fit host RAM" if capped else "full-size tables")
                        + f" ({sum(rows) * D * 4 / 2**30:.1f} GiB of tables; host RAM {ram_total / 2**30:.0f} GiB, "
                        f"{ram_avail / 2**30:.0f} GiB available); {threads} host threads; "
                        "C restatement of the Julia lookup/interaction/sparse-SGD path (OpenMP) + torch-CPU "
                        "(oneDNN) MLPs; batch generation excluded"))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "sweep":
        print(json.dumps({"impl": "reference", "unavailable": "the sweep workload has no CPU arm (run terabyte / kaggle)"}), flush=True)
        return
    wl = workload(args.workload, args.batch)
    r = cpu_arm(wl, args.steps, args.warmup, args.cpu_rows_cap, budget_s=float("inf"))   # exactly --steps timed steps
    line = {
        "impl": "reference", "metric": "dlrm_train_samples_per_sec", "value": r["value"], "unit": "samples/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_LABEL, "data": "synthetic",
        "config": bench_config(wl, 1, note="CPU arm: one process on the host cores, no GPU",
                               rows_cap=r["rows_cap"], host_ram_gb=r["host_ram_gb"]),
        "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def library_options():
    """The library's tuning switches as this run had them (dlrmb_get_option): defaults unless --opt changed them."""
    from dlrm_jl_b200 import _lib
    return {k: _lib.get_option(k) for k in ("interact_general", "update_two_launches", "update_tile", "bwd_variant", "fwd_ksplit")}


def bench_config(wl, world, note="", rows_cap=None, host_ram_gb=None):
    return {
        "rows_cap": rows_cap, "host_ram_gb": host_ram_gb,
        "workload": f"criteo_{wl['name']}_synthetic: 26 tables, D {wl['D']}, batch {wl['B']} per GPU, P 1, "
                    f"{sum(wl['rows']) * wl['D'] * 4 / 1e9:.1f} GB fp32 tables",
        "tables": len(wl["rows"]), "embedding_dim": wl["D"], "batch_per_gpu": wl["B"],
        "global_batch": wl["B"] * world, "pooling": wl["P"],
        "bottom_mlp": wl["bottom"], "top_mlp": wl["top"], "lr": LR,
        "parallelism": ("single GPU" if world == 1 else
                        f"table-wise sharded embeddings over {world} GPUs (all-to-all) + data-parallel MLP/interaction"),
        "l2": ("inputs larger than L2: fresh random indices every step; the tables that hold 99.9 % of the bytes (16 of the 26 "
               "Terabyte-shaped, 104 GB) are far larger than the 126 MB L2, so their rows come from HBM; the 10 tables with fewer "
               "than 2048 rows stay L2-resident and their lookups show up as L2 hits (fractions above the DRAM traffic ncu reports)"),
        "note": note,
    }


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from dlrm_jl_b200 import _prof, launch_count
    from dlrm_jl_b200.interact import DotInteraction
    from dlrm_jl_b200.model import create_mlp
    from dlrm_jl_b200.sharded import FlatGrads, ShardedEmbedding
    from dlrm_jl_b200.train import SigmoidBCELoss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything a library prints there meanwhile (NCCL's version
    # banner, for one) is sent to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    wl = workload(args.workload, args.batch)
    B, D, F = wl["B"], wl["D"], wl["F"]
    K, W = args.steps, args.warmup

    gen = torch.Generator().manual_seed(51234)
    bottom = create_mlp(wl["bottom"], 0, dev, gen)
    top = create_mlp(wl["top"], len(wl["top"]), dev, gen)
    top_logits = torch.nn.Sequential(*list(top)[:-1])   # the final sigmoid is fused into the loss kernel
    sigmoid_bce = SigmoidBCELoss(dev)
    params = list(bottom.parameters()) + list(top.parameters())
    se = ShardedEmbedding.create(wl["rows"], D, B, wl["P"], rank, world, dev)
    exchange = "none (single GPU)"
    exchange_check = None
    if world > 1:
        exchange = "nccl all-to-all"
        if args.exchange == "p2p":
            ok, why = 1.0, ""
            try:
                se.enable_peer_exchange(B, flag_barrier=(args.barrier == "flags"), P=wl["P"], idx_bytes=4)
                se.enable_fused_backward(B, split_dx=args.split_dx)
            except Exception as exc:  # noqa: BLE001 - e.g. CUDA IPC not permitted in this container
                ok, why = 0.0, f"{type(exc).__name__}: {exc}"
            flag = torch.tensor([ok], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)      # every rank takes the same decision
            if float(flag.item()) == 1.0:
                exchange = ("fused over NVLink peer stores: index columns -> owners' index buffers, lookup -> peers' "
                            "interaction inputs (forward), interaction backward -> owners' gradient buffers (backward); ordering: "
                            + ("flag barrier over the mapped buffers (dlrmb_peer_barrier, one tiny kernel per exchange)"
                               if args.barrier == "flags" else "one-element NCCL all-reduce per exchange"))
            else:
                se.peer = None
                se.scatter_plan = None
                exchange = f"nccl all-to-all (peer mapping unavailable: {why or 'on another rank'})"
        # one sharded step on a batch whose ids fall in the first CHECK_ROWS rows of every table, compared
        # with the UNSHARDED CPU oracle run on a downloaded copy of those rows
        exchange_check = sharded_oracle_check(se, wl, dev, rank, world)
        if rank == 0:
            print(f"[bench] sharded step vs unsharded oracle: {exchange_check}", file=sys.stderr)
        if not exchange_check["ok"]:
            raise SystemExit(f"sharded path disagrees with the oracle: {exchange_check}")
    dot = DotInteraction()
    anchor = torch.zeros(1, device=dev, requires_grad=True)

    flat = FlatGrads(params, world)
    pflat = flat.flatten_params()       # dense SGD = one axpy over the flat parameter buffer
    mlp_stream_ = torch.cuda.Stream()
    upd_stream_ = torch.cuda.Stream()
    # Dense layers as the reference has them (OneDNN.Dense: GEMM + bias + relu in one primitive): library
    # GEMMs, epilogue-fused activations, one launch of this repo's kernel per layer for relu mask +
    # bias gradient, weight gradients written straight into the flat all-reduce bucket.
    fused_mlp = not args.unfused_mlp
    if fused_mlp:
        from dlrm_jl_b200.dense import FusedMLP
        nbp = len(list(bottom.parameters()))
        bottom_f = FusedMLP(bottom, flat.views[:nbp])
        top_f = FusedMLP(list(top)[:-1], flat.views[nbp:])
    else:
        bottom_f, top_f = bottom, top_logits

    serial = {"on": False}      # profiling pass: every kernel of the step on ONE stream (no overlap between streams)
    n_bottom = sum(p.numel() for p in bottom.parameters())
    comm_stream_ = torch.cuda.Stream()
    early = world > 1 and not args.late_allreduce
    # the bottom MLP's gradients (0.7 MB) end the step on the critical path: one-shot all-reduce over the
    # IPC-mapped buffers (push + flag barrier + rank-ordered sum) instead of a latency-bound NCCL call
    small_ar = (early and se.peer is not None and se.peer.peer_flag_ptrs is not None and n_bottom % 4 == 0
                and not args.nccl_bottom_allreduce)
    if small_ar:
        se.peer.enable_small_allreduce(n_bottom)

    def allreduce_top_grads(g):
        """Gradient hook on the interaction output: the top MLP's backward has been launched, so its 93 % of
        the dense gradient bytes start their all-reduce now, beside the interaction backward, the gradient
        exchange, the bottom MLP's backward and the sparse update."""
        main = torch.cuda.current_stream()
        comm = main if serial["on"] else comm_stream_
        comm.wait_stream(main)
        with torch.cuda.stream(comm):
            with _prof.range("allreduce_top_mlp"):
                dist.all_reduce(flat.flat[n_bottom:], op=dist.ReduceOp.SUM)
        return g

    def train_step(dense, labels, idx):
        main = torch.cuda.current_stream()
        mlp_stream = main if serial["on"] else mlp_stream_
        se.update_inside_backward(LR * flat.scale, main if serial["on"] else upd_stream_)
        if not fused_mlp:
            flat.zero()        # autograd accumulates into the bucket; the fused layers overwrite it
        # bottom MLP on a second stream: it is independent of the embedding exchange until the
        # interaction, so its GEMMs hide the index / pooled-embedding all-to-alls (and, because
        # autograd replays backward ops on their forward stream, its backward hides the gradient
        # all-to-all and the sparse update)
        mlp_stream.wait_stream(main)
        with torch.cuda.stream(mlp_stream), _prof.range("bottom_mlp_fwd"):
            x = bottom_f(dense)
        fused = se.scatter_plan is not None
        T = se.lookup_fused(idx) if fused else se.lookup(idx, anchor)
        se.sort_async()
        main.wait_stream(mlp_stream)
        z = dot(x, T, scatter=se.scatter_plan) if fused else dot(x, T)
        if early:
            z.register_hook(allreduce_top_grads)
        with _prof.range("top_mlp_fwd"):
            logits = top_f(z)
        loss = sigmoid_bce(logits, labels)
        # the sparse update is launched from inside the backward pass (se.update_inside_backward below): it
        # touches the tables only and runs on upd_stream beside the bottom MLP's backward and the dense reduction
        loss.backward()
        main.wait_stream(mlp_stream)
        if early:      # the bottom MLP's share now; the top MLP's has been in flight since its backward
            if small_ar:
                se.peer.allreduce_small(flat.flat[:n_bottom])
            else:
                with _prof.range("allreduce_bottom_mlp"):
                    dist.all_reduce(flat.flat[:n_bottom], op=dist.ReduceOp.SUM)
            main.wait_stream(main if serial["on"] else comm_stream_)
        elif world > 1:
            with _prof.range("allreduce_dense"):
                flat.allreduce()
        with torch.no_grad(), _prof.range("dense_sgd"):
            pflat.add_(flat.flat, alpha=-LR * flat.scale)      # Flux.update!: x .-= eta * grad
        main.wait_stream(main if serial["on"] else upd_stream_)
        return loss.detach()

    # synthetic batches: host-pinned copies (e2e) and device copies (value)
    nb = K + W
    host = []
    for i in range(nb):
        dense, labels, idx = synth_batch(wl, i, rank)
        host.append((torch.from_numpy(dense).pin_memory(), torch.from_numpy(labels).pin_memory(),
                     torch.from_numpy(idx).pin_memory()))
    devb = [(a.to(dev), b.to(dev), c.to(dev)) for a, b, c in host]
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the step as ONE CUDA graph (kernels of this repo, cuBLAS GEMMs, NCCL collectives):
    # inputs are copied into static device buffers, then the graph is replayed.  Falls back to
    # eager launches if capture is unavailable; the mode is reported in config.step_launch.
    s_dense, s_labels, s_idx = (t.clone() for t in devb[0])
    s_loss = None
    graph = None
    mode = "eager"
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    train_step(s_dense, s_labels, s_idx)
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                s_loss = train_step(s_dense, s_labels, s_idx)
            barrier()
            mode = "cuda_graph"
        except Exception as exc:  # noqa: BLE001
            if rank == 0:
                import traceback
                print(f"[bench] CUDA graph capture failed ({type(exc).__name__}: {exc}); running eager", file=sys.stderr)
                traceback.print_exc()
            graph = None
            torch.cuda.synchronize()

    def run_step(dense, labels, idx, non_blocking=False):
        if graph is None:
            return train_step(dense.to(dev, non_blocking=non_blocking), labels.to(dev, non_blocking=non_blocking),
                              idx.to(dev, non_blocking=non_blocking))
        s_dense.copy_(dense, non_blocking=non_blocking)
        s_labels.copy_(labels, non_blocking=non_blocking)
        s_idx.copy_(idx, non_blocking=non_blocking)
        graph.replay()
        return s_loss

    # ---- value: inputs resident in HBM ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(W):
        run_step(*devb[i])
    barrier()
    n0 = launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.begin()
    e0.record()
    for i in range(K):
        last_loss_d = run_step(*devb[W + i])
    e1.record()
    barrier()
    sampler.end()
    launches = launch_count() - n0
    if args.dump_outputs and rank == 0:     # now: the launch count and the timing passes below train further
        dump_outputs(args.dump_outputs, last_loss_d, pflat, flat.flat, se, devb[W + K - 1][2])
    if graph is not None:   # replays do not pass through the host-side counter: count per captured step
        n1 = launch_count()
        train_step(*devb[0])
        torch.cuda.synchronize()
        launches = (launch_count() - n1) * K
    ms_total = max_over_ranks(e0.elapsed_time(e1))

    # ---- per-kernel device time of this repo's kernels over the same K batches.  Preferred: the
    # step captured a second time with an event-record node on either side of every library call
    # (cudaEventRecordExternal), replayed per batch -- the kernels run back to back exactly as in the
    # timed graph.  Fallback (no graph / no external events): eager launches with an event pair
    # around every call, each step queued behind a device-side spin so the host runs ahead.
    prof, prof_mode, graph_map = None, None, None
    if graph is not None:
        try:
            _prof.enable(True, external=True)
            pgraph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(pgraph):
                train_step(s_dense, s_labels, s_idx)
            _prof.enable(False)
            acc = {}
            for i in range(K):
                s_dense.copy_(devb[W + i][0])
                s_labels.copy_(devb[W + i][1])
                s_idx.copy_(devb[W + i][2])
                pgraph.replay()
                torch.cuda.synchronize()
                for name, ms in _prof.read_replay().items():
                    acc.setdefault(name, []).extend(ms)
                if i == K - 1:
                    graph_map = {n: [round(v[0][0], 1), round(v[0][1], 1)] for n, v in _prof.read_replay_timeline().items() if v}
            barrier()
            prof = {n: {"count": len(v), "total_ms": float(sum(v)), "avg_ms": float(sum(v) / max(1, len(v)))}
                    for n, v in acc.items()}
            prof_mode = "event-record nodes inside a CUDA graph of the step, replayed over the timed batches"
            del pgraph
        except Exception as exc:  # noqa: BLE001
            _prof.enable(False)
            if rank == 0:
                print(f"[bench] in-graph kernel timing unavailable ({type(exc).__name__}: {exc}); eager event pairs", file=sys.stderr)
            torch.cuda.synchronize()
            prof = None
    in_graph = prof
    # The clock the rooflines use: the step's own launch sequence on its real data, every kernel on ONE
    # stream (serialised like an ncu launch list, so a kernel is not timed while the bottom MLP or the
    # dense all-reduce shares the SMs with it), launched eagerly behind a device-side spin so the host
    # stays ahead, one CUDA-event pair per library call.
    serial["on"] = True
    for i in range(min(3, K)):
        train_step(*devb[W + i])
    torch.cuda.synchronize()
    _prof.enable(True)
    for i in range(K):
        torch.cuda._sleep(6_000_000)
        train_step(*devb[W + i])
    barrier()
    _prof.enable(False)
    serial["on"] = False
    prof = _prof.summary()
    prof_mode = ("the step's launch sequence on the timed batches, all kernels on one stream, eager launches queued behind a "
                 "device-side spin, one CUDA-event pair per library call")
    if in_graph:
        for n, st in in_graph.items():
            if n in prof:
                prof[n]["in_graph_avg_ms"] = st["avg_ms"]
    # The most faithful clock: %globaltimer stamps taken by the kernels themselves (dlrmb_clock_enable) inside
    # a capture of the REAL multi-stream step graph, replayed over the timed batches: min(CTA entry) to
    # max(CTA exit) of each kernel, no event nodes, no serialisation.
    dev_clock, timeline = None, None
    if graph is not None:
        try:
            dev_clock = device_clock_pass(train_step, (s_dense, s_labels, s_idx), devb[W:W + K], dev)
            timeline = dev_clock.pop("_timeline", None)
            for n, us in dev_clock.items():
                if n in prof:
                    prof[n]["device_clock_us"] = us
                elif n in OWN_KERNELS:
                    # a kernel launched inside another call's event pair (the separate index sort of
                    # dlrmb_embedding_fwd_sort above kFusedSortMax keys, the update's fix-up launch for large
                    # batches): it has no event pair of its own, only its own stamps
                    prof[n] = {"count": K, "avg_ms": us * 1e-3, "total_ms": us * 1e-3 * K, "device_clock_us": us,
                               "device_clock_only": True}
        except Exception as exc:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] device-clock pass failed ({type(exc).__name__}: {exc})", file=sys.stderr)
        barrier()

    # ---- e2e: host inputs in, loss out, every step.  Graph mode runs it as a two-slot pipeline, the way
    # a training loop with a prefetching loader does (DACLoader, SURVEY 8(f) row 2): the pinned-host ->
    # device copy of step i+1's inputs is issued on a copy stream before step i is launched, and step
    # i's loss is copied to pinned host memory behind the step and read while step i+1 runs.  Every
    # step's inputs cross PCIe and every step's loss is read on the host inside the timed region.
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def e2e_step(i):
        a, b, c = host[i]
        l = run_step(a, b, c, non_blocking=True)
        loss_host.copy_(l.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(loss_host[0])

    def e2e_pipelined(first, count):
        main = torch.cuda.current_stream()
        for slot in (0, 1):                     # staging buffers are free at the start
            stage_free[slot].record(main)
        losses = []

        def prefetch(i, slot):
            copy_stream.wait_event(stage_free[slot])
            with torch.cuda.stream(copy_stream):
                for dst, src in zip(stage[slot], host[i]):
                    dst.copy_(src, non_blocking=True)
                stage_ready[slot].record(copy_stream)

        prefetch(first, 0)
        for j in range(count):
            slot = j & 1
            if j + 1 < count:
                prefetch(first + j + 1, 1 - slot)
            main.wait_event(stage_ready[slot])
            s_dense.copy_(stage[slot][0], non_blocking=True)
            s_labels.copy_(stage[slot][1], non_blocking=True)
            s_idx.copy_(stage[slot][2], non_blocking=True)
            stage_free[slot].record(main)
            graph.replay()
            loss_pinned[slot].copy_(s_loss.reshape(1), non_blocking=True)
            loss_done[slot].record(main)
            if j >= 1:                          # read the previous step's loss while this one runs
                loss_done[1 - slot].synchronize()
                losses.append(float(loss_pinned[1 - slot][0]))
        last = (count - 1) & 1
        loss_done[last].synchronize()
        losses.append(float(loss_pinned[last][0]))
        return losses

    pipelined = graph is not None and not args.e2e_sync
    if pipelined:
        copy_stream = torch.cuda.Stream()
        stage = [tuple(torch.empty_like(t) for t in (s_dense, s_labels, s_idx)) for _ in range(2)]
        stage_ready = [torch.cuda.Event() for _ in range(2)]
        stage_free = [torch.cuda.Event() for _ in range(2)]
        loss_pinned = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_done = [torch.cuda.Event() for _ in range(2)]
        e2e_pipelined(0, min(W, 3))
    else:
        for i in range(min(W, 3)):
            e2e_step(i)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.begin()
    f0.record()
    last_loss = 0.0
    if pipelined:
        e2e_losses = e2e_pipelined(W, K)
        assert len(e2e_losses) == K
        last_loss = e2e_losses[-1]
    else:
        for i in range(K):
            last_loss = e2e_step(W + i)
    f1.record()
    barrier()
    sampler.end()
    e2e_ms = max_over_ranks(f0.elapsed_time(f1))
    clocks = sampler.stop() if rank == 0 else None
    e2e_mode = ("two-slot pipeline: inputs of step i+1 copied (pinned host -> device) while step i runs, loss of step i "
                "read on the host while step i+1 runs" if pipelined else
                "synchronous: copy inputs, run the step, read the loss, every step")

    # ---- per-launch device time of each kernel of this repo, launched back to back over the timed
    # batches (one CUDA graph of nb launches per kernel, every launch on a different batch; the
    # interaction inputs of the nb batches together exceed the L2).  This is the figure the roofline
    # uses: an event-record node on either side of a kernel inside the step graph adds several
    # microseconds of graph-dependency latency to a 10-20 us kernel.
    replay = None
    if world == 1:
        try:
            replay = kernel_replays(se, devb[W:W + K], wl, dev)
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] kernel replays failed ({type(exc).__name__}: {exc})", file=sys.stderr)

    if world > 1:
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())

    if rank == 0:
        ms_step = ms_total / K
        Bg = B * world
        line = {
            "metric": "dlrm_train_samples_per_sec", "value": Bg * K / (ms_total * 1e-3), "unit": "samples/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE_LABEL, "data": "synthetic",
            "config": dict(bench_config(wl, world), library_options=library_options(), step_launch=mode, exchange=exchange, exchange_check=exchange_check,
                           barrier_timeouts=(se.peer.barrier_timeouts() if se.peer is not None else 0),
                           dense_allreduce=("none (single GPU)" if world == 1 else
                                            ("top MLP gradients: NCCL all-reduce started from a gradient hook as soon as the top MLP's backward is "
                                             "launched; bottom MLP gradients: " + ("one-shot all-reduce over NVLink peer stores (dlrmb_peer_allreduce_f32)"
                                                                                  if small_ar else "NCCL all-reduce") if early else "one NCCL all-reduce after backward")),
                           mlp=("fused dense layers (library fp32 GEMMs, epilogue bias+relu, dlrmb_dense_bwd_act_bias)" if fused_mlp
                                else "nn.Linear + ReLU autograd")),
            "e2e": {"value": Bg * K / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": 4 * world, "ms_per_step": e2e_ms / K, "last_loss": last_loss,
                    "mode": e2e_mode},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        line.update(hot_path_report(wl, world, rank, se, prof, ms_step, replay))
        line["hot_path"]["kernel_timing"] = prof_mode
        if graph_map:
            line["hot_path"]["step_map_us"] = dict(graph_map, note="[start, end] of every bracketed call of the step (this repo's kernels, "
                                                   "the MLP blocks, the NCCL all-reduces, the dense SGD), microseconds from the first stamp, from "
                                                   "CUDA event-record nodes inside a capture of the step graph, last timed batch, rank 0; each node "
                                                   "adds a few microseconds, so this is a map of the step, not a stopwatch")
        if timeline:
            line["hot_path"]["timeline_us"] = dict(timeline, note="[first CTA in, last CTA out] of each kernel, microseconds from the "
                                                   "first stamp of the step, from the kernels' own %globaltimer stamps inside the step graph "
                                                   f"(rank 0; step = {ms_step * 1e3:.0f} us)")
        if world == 1 and not args.no_host_leg:
            try:
                line["e2e_host"] = e2e_host_leg(se, wl, host[W:W + min(K, 10)], dev)
            except Exception as exc:  # noqa: BLE001
                line["e2e_host"] = {"error": f"{type(exc).__name__}: {exc}"}
        if world == 1 and not args.no_cpu_baseline:
            r = cpu_arm(wl, 20, 3, args.cpu_rows_cap, budget_s=20.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"]}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    # Leave without tearing NCCL down: destroying a communicator that captured CUDA graphs still
    # reference can block for minutes.  Everything measured is already printed and flushed.
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


DUMP_SAMPLES = 2048
DUMP_BYTES = 64 << 20


def dump_outputs(path, loss, params, grads, se, idx):
    """--dump-outputs: what the last timed step computed, as float32 .npy files: its loss, the MLP parameters
    after its dense SGD, their gradients, and the embedding rows it looked up, read after its sparse SGD
    ([tables of this rank][samples][D]; at most DUMP_SAMPLES of the batch's samples, a fixed seeded choice).
    The batches and the initial weights are seeded, so two builds run with the same arguments can be
    compared file for file."""
    import torch
    B = idx.shape[1]
    pick = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_SAMPLES), replace=False))
    sel = torch.from_numpy(pick).to(idx.device)
    rows = torch.stack([se.tables.table(j)[idx[k, sel, 0].long()] for j, k in enumerate(se.local_ids)])
    out = {"loss": loss.reshape(1), "dense_params": params, "dense_grads": grads, "embedding_rows": rows}
    out = {n: t.detach().float().cpu().numpy() for n, t in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for n, a in out.items():
        np.save(os.path.join(path, f"{n}.npy"), a)
    print(f"[bench] outputs of the last timed step -> {path}: "
          + ", ".join(f"{n}{list(a.shape)}" for n, a in out.items()), file=sys.stderr)


OWN_KERNELS = {"lookup", "sort", "update", "update_fixup", "interaction_fwd", "interaction_bwd", "bce", "indices_scatter"}
CLOCK_NAMES = ["lookup", "sort", "update", "update_fixup", "interaction_fwd", "interaction_bwd", "bce"]


def device_clock_pass(train_step, statics, batches, dev):
    """name -> microseconds per launch from the kernels' own %globaltimer stamps, inside the step graph."""
    import torch
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    nk = int(lib.dlrmb_clock_kernels())
    n = int(lib.dlrmb_clock_buffer_bytes()) // 8
    buf = torch.empty(n, dtype=torch.int64, device=dev)
    view = buf.view(nk, -1, 2)
    _lib.check(lib.dlrmb_clock_enable(buf.data_ptr()))
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            train_step(*statics)
    finally:
        _lib.check(lib.dlrmb_clock_enable(None))
    acc, starts, ends = {}, {}, {}
    for b in batches:
        for dst, src in zip(statics, b):
            dst.copy_(src)
        view[:, :, 0] = 1 << 62
        view[:, :, 1] = 0
        g.replay()
        torch.cuda.synchronize()
        t0 = view[:, :, 0].min(dim=1).values.cpu().tolist()
        t1 = view[:, :, 1].max(dim=1).values.cpu().tolist()
        live = [k for k in range(nk) if t1[k] > 0 and t0[k] < (1 << 62)]
        origin = min(t0[k] for k in live) if live else 0
        for k in live:
            acc.setdefault(CLOCK_NAMES[k], []).append((t1[k] - t0[k]) * 1e-3)
            starts.setdefault(CLOCK_NAMES[k], []).append((t0[k] - origin) * 1e-3)
            ends.setdefault(CLOCK_NAMES[k], []).append((t1[k] - origin) * 1e-3)
    del g
    out = {k: float(np.mean(v)) for k, v in acc.items()}
    # where the kernels sit in the step: microseconds from the first stamp of the step (the lookup's first CTA)
    out["_timeline"] = {k: [round(float(np.mean(starts[k])), 1), round(float(np.mean(ends[k])), 1)] for k in acc}
    return out


CHECK_ROWS = 64


def sharded_oracle_check(se, wl, dev, rank, world):
    """One sharded training step of the hot path on this run's GPUs -- index exchange, owner-side pooling
    with the forward exchange, interaction forward / backward with the gradient exchange, owner-side sort
    + sparse SGD -- against the unsharded CPU oracle (the checker; tolerances of tests/test_gpu_parity.py:
    pooled rows bit-exact, interaction 1e-5, tables 1e-4).  Ids are drawn from the first CHECK_ROWS rows
    of every table so that the oracle only needs a small downloaded sample of the 100 GB of tables."""
    import torch
    import torch.distributed as dist
    from dlrm_jl_b200.interact import DotInteraction, interaction_width
    from oracle import oracle as O
    B, D, F = wl["B"], wl["D"], wl["F"]
    rows = wl["rows"]
    ntab = len(rows)
    mine = se.local_ids
    sample = {k: se.tables.table(j)[:min(rows[k], CHECK_ROWS)].float().cpu().numpy().copy() for j, k in enumerate(mine)}
    parts = [None] * world
    dist.all_gather_object(parts, sample)
    ref_tables = [None] * ntab
    for part in parts:
        for k, v in part.items():
            ref_tables[k] = v
    w = interaction_width(F, D)
    rngs = [np.random.default_rng(4242 + r) for r in range(world)]          # every rank can rebuild every rank's batch
    idx_all = [np.stack([g.integers(0, min(r_, CHECK_ROWS), size=(B, 1)) for r_ in rows]) for g in rngs]
    x_all = [g.standard_normal((B, D)).astype(np.float32) for g in rngs]
    gz_all = [(g.standard_normal((B, w)) * 0.1).astype(np.float32) for g in rngs]
    lr = 0.05
    x = torch.from_numpy(x_all[rank]).to(dev).requires_grad_(True)
    idx_local = torch.from_numpy(idx_all[rank].astype(np.int32)).to(dev)
    dot = DotInteraction()
    fused = se.scatter_plan is not None
    anchor = torch.zeros(1, device=dev, requires_grad=True)
    T = se.lookup_fused(idx_local) if fused else se.lookup(idx_local, anchor)
    se.sort_async()
    z = dot(x, T, scatter=se.scatter_plan) if fused else dot(x, T)
    z.backward(torch.from_numpy(gz_all[rank]).to(dev))
    if fused:
        se.finish_backward()
    se.update(lr)
    torch.cuda.synchronize()
    dist.barrier()
    # ---- oracle
    T_ref = O.lookup(ref_tables, list(idx_all[rank]), slot0=1)
    T_got = T.detach().cpu().numpy()
    res = {"pooled_rows_bit_exact": bool(np.array_equal(T_got[:, 1:], T_ref[:, 1:]))}
    T_ref[:, 0] = x_all[rank]
    res["interaction_fwd_rel_err"] = float(O.rel_err(z.detach().cpu().numpy(), O.interaction_fwd(T_ref)))
    dT_glob = []
    for r in range(world):
        Tr = O.lookup(ref_tables, list(idx_all[r]), slot0=1)
        Tr[:, 0] = x_all[r]
        dx_r, dT_r = O.interaction_bwd(gz_all[r], Tr)
        dT_glob.append(dT_r)
        if r == rank:
            res["dx_rel_err"] = float(O.rel_err(x.grad.cpu().numpy(), dx_r))
    dT_glob = np.concatenate(dT_glob, axis=0)
    terr = 0.0
    for j, k in enumerate(mine):
        idx_glob = np.concatenate([idx_all[r][k] for r in range(world)], axis=0)
        O.sparse_sgd_update_fast(ref_tables[k], idx_glob, np.ascontiguousarray(dT_glob[:, 1 + k]), lr)
        got = se.tables.table(j)[:min(rows[k], CHECK_ROWS)].float().cpu().numpy()
        terr = max(terr, float(O.rel_err(got, ref_tables[k])))
    res["tables_rel_err_after_update"] = terr
    ok = (res["pooled_rows_bit_exact"] and res["interaction_fwd_rel_err"] < 1e-5 and res["dx_rel_err"] < 1e-5
          and terr < 1e-4)
    flag = torch.tensor([1.0 if ok else 0.0, -res["interaction_fwd_rel_err"], -res["dx_rel_err"], -terr], device=dev,
                        dtype=torch.float64)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)          # worst rank
    v = flag.cpu().tolist()
    return {"ok": bool(v[0] == 1.0), "against": "unsharded CPU oracle (oracle/oracle.py) on the first "
            f"{CHECK_ROWS} rows of every table, batch {B} per rank, one full sharded step, worst rank",
            "pooled_rows_bit_exact": bool(v[0] == 1.0 or res["pooled_rows_bit_exact"]),
            "interaction_fwd_rel_err": -v[1], "dx_rel_err": -v[2], "tables_rel_err_after_update": -v[3]}


def e2e_host_leg(se, wl, batches, dev):
    """The hot path through the HOST-buffer C entry points (the form a CPU-resident DLRM.jl calls today:
    Julia arrays in and out, copies inside each call): dlrmb_embedding_fwd_host -> dlrmb_interaction_fwd_host
    -> dlrmb_interaction_bwd_host -> dlrmb_embedding_bwd_sgd_host on numpy buffers, wall clock per step
    (every call returns synchronised).  MLPs are not part of this leg (they stay on the host in that set-up)."""
    import ctypes as C
    from dlrm_jl_b200 import _lib
    from dlrm_jl_b200.interact import interaction_width
    lib = _lib.load()
    t = se.tables
    B, D, F = wl["B"], wl["D"], wl["F"]
    w = interaction_width(F, D)
    T = np.zeros((B, F, D), dtype=np.float32)
    x = np.random.default_rng(3).standard_normal((B, D)).astype(np.float32)
    out = np.empty((B, w), dtype=np.float32)
    g = (np.random.default_rng(4).standard_normal((B, w)) * 1e-3).astype(np.float32)
    dT = np.empty_like(T)
    dx = np.empty((B, D), dtype=np.float32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731

    def step(idx):
        _lib.check(lib.dlrmb_embedding_fwd_host(t._h, p(idx), 4, 0, B, 1, p(T), F, 1))
        _lib.check(lib.dlrmb_interaction_fwd_host(t._h, p(T), p(x), B, F, D, 1, p(out)))
        _lib.check(lib.dlrmb_interaction_bwd_host(t._h, p(g), p(T), B, F, D, 1, p(dT), p(dx)))
        _lib.check(lib.dlrmb_embedding_bwd_sgd_host(t._h, p(idx), 4, 0, B, 1, p(dT), F, 1, 1e-6))

    idxs = [np.ascontiguousarray(b[2].numpy().reshape(F - 1, B)) for b in batches]
    for i in range(min(3, len(idxs))):
        step(idxs[i])
    t0 = time.perf_counter()
    for idx in idxs:
        step(idx)
    dt = (time.perf_counter() - t0) / len(idxs)
    h2d = idxs[0].nbytes * 2 + T.nbytes * 3 + x.nbytes + g.nbytes      # idx (twice), T (fwd slot-0 fill, interaction, bwd), x, dOut, dT
    h2d += dT.nbytes
    d2h = T.nbytes * 2 + out.nbytes + dT.nbytes + dx.nbytes
    return {"value": B / dt, "unit": "samples/s", "ms_per_step": 1e3 * dt, "steps": len(idxs),
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "what": "hot path only (lookup, interaction fwd/bwd, sparse SGD) through the dlrmb_*_host entry points on "
                    "pageable numpy buffers; every call copies its operands in and out and returns synchronised"}


def run_sweep(args):
    """BASELINE config 5 (SURVEY 8(d)): one table, 2^20 lookups per launch, rows x D x pooling x skew grid."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
    import hotpath
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    cases = []
    rows_list = (100_000, 1_000_000, 10_000_000, 100_000_000)
    dims = (16, 32, 64, 128, 256)
    pools = (1, 4, 16, 64)
    alphas = (0.0, 1.05, 1.2)
    if args.sweep_quick:
        rows_list, dims, pools, alphas = (1_000_000, 100_000_000), (64, 128), (1, 16), (0.0, 1.2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for rows in rows_list:
        for D in dims:
            if rows * D * 4 > 120e9:
                continue
            for P in pools:
                for alpha in alphas:
                    r = hotpath.run_case([rows], D, (1 << 20) // P, P, alpha, 3, True, 3, interaction=False,
                                         label=f"rows={rows} D={D} P={P} zipf={alpha}")
                    cases.append({"rows": rows, "D": D, "P": P, "zipf": alpha,
                                  "lookup_us": r["lookup"]["us"], "lookup_frac": r["lookup"]["frac_hbm"],
                                  "sort_us": r["sort"]["us"],
                                  "update_us": r["update_only"]["us"], "update_frac": r["update_only"]["frac_hbm"],
                                  "total_us": r["embedding_lookup_plus_update"]["us"],
                                  "gbs": r["embedding_lookup_plus_update"]["gbs"],
                                  "frac_hbm": r["embedding_lookup_plus_update"]["frac_hbm"],
                                  "algorithmic_bytes": r["embedding_lookup_plus_update"]["algorithmic_bytes"]})
                    print(json.dumps(cases[-1]), file=sys.stderr, flush=True)
    e1.record()
    torch.cuda.synchronize()
    big = [c for c in cases if c["D"] >= 64]
    gm = float(np.exp(np.mean([np.log(c["gbs"]) for c in cases])))
    peak, peak_src = hotpath.hbm_peak()
    line = {"metric": "embedding_lookup_plus_update_gbs", "value": gm, "unit": "GB/s", "n_gpus": 1,
            "steps": len(cases), "warmup": 3, "ms_per_step": e0.elapsed_time(e1) / max(1, len(cases)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "embedding microbench sweep (BASELINE config 5): one table, 2^20 lookups per launch, "
                                   "rows 1e5-1e8 x D 16-256 x pooling 1/4/16/64 x uniform / Zipf 1.05 / Zipf 1.2; value = "
                                   "geometric mean over the cases of (lookup + sort + update algorithmic bytes) / time",
                       "l2": "fresh index batch every launch; tables of 1e5 rows fit L2 and are reported as such"},
            "summary": {"cases": len(cases), "hbm_peak_gbs": peak, "peak_source": peak_src,
                        "frac_hbm_geomean": gm / peak,
                        "frac_hbm_geomean_D_ge_64": float(np.exp(np.mean([np.log(c["frac_hbm"]) for c in big]))) if big else None,
                        "cases_at_or_above_70pct": sum(1 for c in cases if c["frac_hbm"] >= 0.70),
                        "cases_below_50pct": sum(1 for c in cases if c["frac_hbm"] < 0.50)},
            "sweep": cases}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def kernel_replays(se, batches, wl, dev):
    """name -> microseconds per launch, kernels launched back to back (dlrm_jl_b200._prof.time_launches).
    "lookup" is the launch the step uses: gather + the index sort of the coming update in one kernel;
    "embedding_chain" is that launch followed by the update launch, per batch (the BASELINE metric)."""
    import torch
    from dlrm_jl_b200 import _lib, _prof
    from dlrm_jl_b200.interact import interaction_bwd, interaction_fwd, interaction_width
    t = se.tables
    B, D, F = wl["B"], wl["D"], wl["F"]
    nb = min(len(batches), 16)
    idx = [b[2] for b in batches[:nb]]
    w = interaction_width(F, D)
    Ts, gs = [], []
    for i in range(nb):
        Ti = torch.empty((B, F, D), device=dev)
        t.lookup(idx[i], Ti, 1)
        Ti[:, 0] = torch.randn((B, D), device=dev)
        Ts.append(Ti)
        gs.append(torch.randn((B, w), device=dev) * 1e-3)
    dT = torch.randn((B, F, D), device=dev) * 1e-3
    out = {}
    out["lookup"] = _prof.time_launches(lambda i: t.lookup(idx[i], Ts[i], 1, sort=True), nb)
    out["lookup_without_sort"] = _prof.time_launches(lambda i: t.lookup(idx[i], Ts[i], 1), nb)
    out["sort_alone"] = _prof.time_launches(lambda i: t.sort(idx[i]), nb)

    def chain(i):
        t.lookup(idx[i], Ts[i], 1, sort=True)
        t.update_sorted(dT, 1, 1e-6)
    out["embedding_chain"] = _prof.time_launches(chain, nb)
    out["update"] = max(out["embedding_chain"] - out["lookup"], 1e-3)
    out["interaction_fwd"] = _prof.time_launches(lambda i: interaction_fwd(Ts[i]), nb)
    out["interaction_bwd"] = _prof.time_launches(lambda i: interaction_bwd(gs[i], Ts[i]), nb)
    z = torch.randn((B,), device=dev)
    y = (torch.rand((B,), device=dev) < 0.25).float()
    prob, dz, loss, scratch = torch.empty_like(z), torch.empty_like(z), torch.zeros(1, device=dev), torch.zeros(128, device=dev)
    lib = _lib.load()
    s_ptr = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
    try:
        out["bce"] = _prof.time_launches(lambda i: _lib.check(lib.dlrmb_bce_sigmoid_fwd_bwd(
            dev.index or 0, z.data_ptr(), y.data_ptr(), B, prob.data_ptr(), dz.data_ptr(), loss.data_ptr(),
            scratch.data_ptr(), s_ptr())), nb)
    except Exception:  # noqa: BLE001 - signature drift must not cost the bench line
        pass
    out["_nb"] = nb
    out["_interaction_inputs_mb"] = nb * B * F * D * 4 / 1e6
    return out


def hot_path_report(wl, world, rank, se, prof, ms_step, replay):
    """Per-kernel device time and rooflines.  Algorithmic bytes per SURVEY.md section 8(d), rank 0's share.

    Clocks per kernel, all reported:
      * in_step_us -- when the step runs as a CUDA graph: the kernel's own %globaltimer stamps (first CTA in
        to last CTA out, dlrmb_clock_enable) inside a capture of the real multi-stream step graph, replayed
        over the timed batches -- the kernel exactly where and how it runs in the step, no event nodes;
        otherwise (and always as event_pair_us): the step's own launch sequence serialised on one stream,
        eager launches, a CUDA-event pair around the call (adds ~5 us per pair: the 2.7 us BCE kernel reads 8);
      * in_graph_us -- an event-record node on either side of the call inside a second capture of the
        multi-stream step graph: includes the kernels of other streams sharing the SMs and a few
        microseconds of graph-dependency latency per event pair;
      * back_to_back_us -- the kernel launched back to back over the same batches (1 GPU only).
    `roofline` and `embedding` use in_step_us; the other figures are printed beside them."""
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    D, B, F = wl["D"], wl["B"], wl["F"]
    Bg = B * world
    t_mine = len(se.local_ids)
    L = Bg * wl["P"]
    # distinct rows touched per step on this rank's tables (U), expectation for L uniform draws
    rows = [wl["rows"][k] for k in se.local_ids]
    U = sum(r * (1.0 - (1.0 - 1.0 / r) ** L) for r in rows)
    lookup_bytes = t_mine * (L * D * 4 + Bg * D * 4 + L * 4)
    update_bytes = t_mine * (Bg * D * 4 + L * 8) + 2 * U * D * 4
    width = D + F * (F - 1) // 2
    ifwd_bytes = B * (F * D + D + width - D) * 4
    ibwd_bytes = B * (width + 2 * F * D + D) * 4
    alg = {"lookup": lookup_bytes, "update": update_bytes, "interaction_fwd": ifwd_bytes, "interaction_bwd": ibwd_bytes}
    kernels = {}
    others = {}     # bracketed calls that are not this repo's kernels (MLP blocks, NCCL, dense SGD): event-pair time only
    for name, st in prof.items():
        if not (name in OWN_KERNELS or name.startswith("peer_barrier")):
            others[name] = round(1e3 * st["avg_ms"], 2)
            continue
        k = {"launches": st["count"], "in_step_us": 1e3 * st["avg_ms"], "in_step_clock": "serialised eager step, CUDA-event pair"}
        if "device_clock_us" in st:      # the kernel's own %globaltimer stamps inside the real step graph
            if not st.get("device_clock_only"):
                k["event_pair_us"] = k["in_step_us"]
            k["in_step_us"] = float(st["device_clock_us"])
            k["in_step_clock"] = "device %globaltimer stamps (first CTA in .. last CTA out) inside the step graph"
        if "in_graph_avg_ms" in st:      # event-record nodes inside the multi-stream step graph (adds graph-dependency latency)
            k["in_graph_us"] = 1e3 * st["in_graph_avg_ms"]
        if replay and name in replay:
            k["back_to_back_us"] = float(replay[name])
        if name in alg and k["in_step_us"] > 0:
            k["algorithmic_bytes"] = int(alg[name])
            k["gbs"] = alg[name] / (k["in_step_us"] * 1e-6) / 1e9
            k["frac_hbm"] = k["gbs"] / hbm_peak
            if "back_to_back_us" in k:
                k["frac_hbm_back_to_back"] = alg[name] / (k["back_to_back_us"] * 1e-6) / 1e9 / hbm_peak
        kernels[name] = k
    if replay:
        for extra in ("lookup_without_sort", "sort_alone", "embedding_chain"):
            if extra in replay:
                kernels.setdefault("_replays", {})[extra + "_us"] = float(replay[extra])
    own_ms = sum(k["in_step_us"] for n, k in kernels.items() if not n.startswith("_")) * 1e-3
    cand = [n for n in ("update", "lookup", "interaction_fwd", "interaction_bwd") if n in kernels]
    dom = max(cand, key=lambda n: kernels[n]["in_step_us"]) if cand else None
    out = {"kernels": kernels,
           "hot_path": {"other_calls_event_pair_us": others, "own_kernels_us_per_step": 1e3 * own_ms, "share_of_step": own_ms / ms_step if ms_step else None,
                        "samples_per_s_own_kernels_only": (B / (own_ms * 1e-3)) if own_ms else None}}
    emb_names = [n for n in ("lookup", "sort", "update", "update_fixup") if n in kernels]
    emb_us = sum(kernels[n]["in_step_us"] for n in emb_names)
    if emb_us:
        emb_bytes = lookup_bytes + update_bytes
        out["embedding"] = {"algorithmic_bytes": int(emb_bytes), "us": emb_us,
                            "gbs": emb_bytes / (emb_us * 1e-6) / 1e9,
                            "frac_hbm": emb_bytes / (emb_us * 1e-6) / 1e9 / hbm_peak,
                            "clock": "in_step_us (kernels.<name>.in_step_clock: the kernels' own %globaltimer stamps inside the replayed step graph; CUDA-event pairs of the serialised eager step when the step does not run as a graph), summed over the launches below",
                            "includes": " + ".join(emb_names) + " launches (gather, index sort / dedup, scatter-add + SGD)"}
        if replay and "embedding_chain" in replay:
            out["embedding"]["back_to_back_us"] = float(replay["embedding_chain"])
            out["embedding"]["frac_hbm_back_to_back"] = emb_bytes / (replay["embedding_chain"] * 1e-6) / 1e9 / hbm_peak
    if dom:
        traffic, traffic_src = None, None
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of that kernel, one ncu --set full capture
            for tag in ("r02", "r01"):
                path = os.path.join(ROOT, "profiles", f"{tag}_ncu_traffic_{wl['name']}.json")
                if os.path.exists(path):
                    with open(path) as fh:
                        tj = json.load(fh)
                    if world == 1 and dom in tj["kernels"] and tj.get("batch_per_gpu", 2048) == wl["B"]:
                        traffic = tj["kernels"][dom]["dram_bytes_read"] + tj["kernels"][dom]["dram_bytes_write"]
                        traffic_src = (f"constant: profiles/{tag}_ncu_traffic_{wl['name']}.json ({tj['report']}): "
                                       + tj.get("note", "an ncu --set full capture of this command") + "; not measured in this run")
                    break
        except Exception:
            pass
        kd = kernels[dom]
        out["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": kd["gbs"], "peak": hbm_peak,
                           "unit": "GB/s", "frac": kd["gbs"] / hbm_peak, "traffic": traffic,
                           "traffic_source": traffic_src, "peak_source": peak_src,
                           "achieved_back_to_back": (kd["algorithmic_bytes"] / (kd["back_to_back_us"] * 1e-6) / 1e9
                                                     if "back_to_back_us" in kd else None),
                           "note": ("dominant kernel of this repo by in-step time; achieved = algorithmic bytes per launch / "
                                    "in-step device time (kernels.<name>.in_step_us and its in_step_clock: the kernel's own "
                                    "%globaltimer stamps inside the replayed step graph, averaged over the timed batches); "
                                    "achieved_back_to_back = same bytes / back-to-back launch time")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="terabyte", choices=["terabyte", "kaggle", "sweep"])
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--cpu-rows-cap", type=int, default=0,
                    help="CPU arm: rows per table (0 = as many as 55 %% of the available host RAM holds, 112 GiB at most)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU forward exchange: fused lookup + NVLink peer stores, or NCCL all-to-all")
    ap.add_argument("--split-dx", action="store_true",
                    help="multi-GPU: dx from a kernel of its own ahead of the scattering interaction backward, which then runs on a "
                         "side stream beside the bottom MLP's backward (measured: no gain at 2 and 8 GPUs, off by default)")
    ap.add_argument("--nccl-bottom-allreduce", action="store_true",
                    help="multi-GPU: NCCL for the bottom MLP's gradient all-reduce instead of the one-shot peer-store all-reduce")
    ap.add_argument("--late-allreduce", action="store_true",
                    help="multi-GPU: one dense all-reduce after the whole backward pass instead of starting the top MLP's share early")
    ap.add_argument("--barrier", default="flags", choices=["flags", "nccl"],
                    help="multi-GPU ordering of the fused exchanges: flag barrier kernel over IPC memory, or a one-element NCCL all-reduce")
    ap.add_argument("--e2e-sync", action="store_true",
                    help="e2e leg without the input-prefetch / deferred-loss pipeline (copy, run, read, every step)")
    ap.add_argument("--unfused-mlp", action="store_true",
                    help="plain nn.Linear / ReLU autograd for the MLPs instead of dlrm_jl_b200.dense.FusedMLP")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of as one CUDA graph")
    ap.add_argument("--sweep-quick", action="store_true", help="--workload sweep on a 2 x 2 x 2 x 2 corner of the grid")
    ap.add_argument("--no-host-leg", action="store_true", help="skip the e2e_host leg (hot path through the *_host entry points)")
    ap.add_argument("--opt", action="append", default=[],
                    help="library switch name=value (dlrmb_set_option) for A/B runs; recorded in config.library_options")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, MLP parameters and gradients, the embedding rows "
                         "it looked up after the update) to DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "sweep"):
        ap.error("--dump-outputs applies to the GPU training step (--impl ours, terabyte or kaggle workload)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "sweep":
        run_sweep(args)
    else:
        if args.opt:
            from dlrm_jl_b200 import _lib
            for kv in args.opt:
                name, value = kv.split("=")
                _lib.set_option(name, int(value))
        run_ours(args)


if __name__ == "__main__":
    main()
