"""Host-side logic of bench.py and the step glue that needs no GPU: flat parameter / gradient buckets,
the clock sampler's timed windows, and the shape of the roofline report."""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from dlrm_jl_b200.sharded import FlatGrads  # noqa: E402


def test_flat_grads_and_flat_params_alias_the_parameters():
    torch.manual_seed(0)
    mlp = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 1))
    params = list(mlp.parameters())
    before = [p.detach().clone() for p in params]
    flat = FlatGrads(params, world=1)
    pflat = flat.flatten_params()
    assert pflat.numel() == sum(p.numel() for p in params) == flat.flat.numel()
    off = 0
    for p, b, v in zip(params, before, flat.views):
        assert torch.equal(p.detach(), b)                                   # values survive the re-homing
        assert p.data_ptr() == pflat.data_ptr() + 4 * off                   # and live inside the flat buffer
        assert v.data_ptr() == flat.flat.data_ptr() + 4 * off and v.shape == p.shape
        off += p.numel()
    # one axpy over the flat buffers == per-parameter SGD (Flux.update!: x .-= eta * grad)
    flat.zero()
    mlp(torch.randn(11, 5)).sum().backward()                                # autograd accumulates into the views
    assert all(p.grad is v for p, v in zip(params, flat.views))
    ref = [b - 0.1 * v for b, v in zip(before, flat.views)]
    with torch.no_grad():
        pflat.add_(flat.flat, alpha=-0.1)
    for p, r in zip(params, ref):
        assert torch.allclose(p.detach(), r)
    # the module still computes with the updated parameters
    y = mlp(torch.ones(1, 5))
    assert torch.isfinite(y).all()


def test_clock_sampler_keeps_only_samples_inside_the_timed_windows():
    s = bench.ClockSampler(0)
    s.thread = object()            # pretend a poller ran
    s.source = "synthetic"
    s.samples = [(1.0, 1000.0, 1965.0, set()), (2.0, 1965.0, 1965.0, set()), (2.5, 1950.0, 1965.0, {"sw_power_cap"}),
                 (4.0, 500.0, 1965.0, {"hw_slowdown"})]
    s.windows = [(1.5, 3.0)]
    r = s.stop()
    assert r["samples"] == 2 and r["sm_mhz"] == np.median([1965.0, 1950.0]) and r["reasons"] == ["sw_power_cap"]
    assert r["window"].startswith("inside")
    s2 = bench.ClockSampler(0)
    s2.thread = object()
    s2.samples = [(1.0, 1234.0, 1965.0, set())]
    s2.windows = [(5.0, 6.0)]
    r2 = s2.stop()
    assert r2["samples"] == 1 and r2["window"].startswith("whole run")


def test_hot_path_report_has_the_contract_keys():
    wl = bench.workload("terabyte", 2048)
    se = types.SimpleNamespace(local_ids=list(range(26)))
    prof = {n: {"count": 30, "total_ms": 30 * ms, "avg_ms": ms} for n, ms in
            {"lookup": 0.018, "interaction_fwd": 0.016, "bce": 0.008, "interaction_bwd": 0.022, "update": 0.024}.items()}
    replay = {"lookup": 11.0, "lookup_without_sort": 9.1, "sort_alone": 5.0, "embedding_chain": 25.0, "update": 14.0,
              "interaction_fwd": 13.9, "interaction_bwd": 17.0, "bce": 3.3}
    rep = bench.hot_path_report(wl, 1, 0, se, prof, 0.9, replay)
    roof = rep["roofline"]
    for key in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in roof
    # the dominant kernel and its fraction come from the in-step clock, the conservative one
    assert roof["kernel"] == "update" and roof["bound"] == "hbm" and roof["unit"] == "GB/s"
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12
    k = rep["kernels"]["update"]
    assert abs(roof["achieved"] - k["algorithmic_bytes"] / (24.0e-6) / 1e9) < 1e-3     # bytes are rounded to an int
    assert roof["achieved_back_to_back"] > roof["achieved"]
    # algorithmic bytes per SURVEY 8(d): B * ((d + pairs) + 2 F d + d) * 4 for the backward
    assert rep["kernels"]["interaction_bwd"]["algorithmic_bytes"] == 2048 * ((128 + 351) + 2 * 27 * 128 + 128) * 4
    assert rep["kernels"]["interaction_bwd"]["back_to_back_us"] == 17.0 and rep["kernels"]["interaction_bwd"]["in_step_us"] == 22.0
    assert rep["kernels"]["lookup"]["algorithmic_bytes"] == 26 * (2048 * 128 * 4 + 2048 * 128 * 4 + 2048 * 4)
    emb = rep["embedding"]
    assert abs(emb["us"] - (18.0 + 24.0)) < 1e-9 and emb["back_to_back_us"] == 25.0
    assert emb["frac_hbm_back_to_back"] > emb["frac_hbm"]
    # without replays (multi-GPU lines) only the in-step figure exists
    rep2 = bench.hot_path_report(wl, 1, 0, se, prof, 0.9, None)
    assert "back_to_back_us" not in rep2["kernels"]["update"] and rep2["kernels"]["update"]["in_step_us"] == 24.0


def test_dump_outputs_writes_the_last_step_as_float32(tmp_path):
    """--dump-outputs: loss, MLP parameters, gradients and the looked-up rows of this rank's tables, float32;
    a batch larger than DUMP_SAMPLES is sampled the same way every run."""
    gen = torch.Generator().manual_seed(0)
    tables = [torch.randn(50, 8, generator=gen), torch.randn(70, 8, generator=gen)]
    se = types.SimpleNamespace(local_ids=[1], tables=types.SimpleNamespace(table=lambda j: tables[1 + j]))
    B = bench.DUMP_SAMPLES + 100
    idx = torch.stack([torch.randint(0, 50, (B, 1), generator=gen), torch.randint(0, 70, (B, 1), generator=gen)]).int()
    params, grads = torch.randn(33, generator=gen), torch.randn(33, generator=gen)
    bench.dump_outputs(str(tmp_path / "a"), torch.tensor(0.5), params, grads, se, idx)
    out = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("loss", "dense_params", "dense_grads", "embedding_rows")}
    assert all(a.dtype == np.float32 for a in out.values())
    assert out["loss"].tolist() == [0.5] and np.array_equal(out["dense_params"], params.numpy())
    assert np.array_equal(out["dense_grads"], grads.numpy())
    rows = out["embedding_rows"]
    assert rows.shape == (1, bench.DUMP_SAMPLES, 8)
    pick = np.sort(np.random.default_rng(0).choice(B, size=bench.DUMP_SAMPLES, replace=False))
    assert np.array_equal(rows[0], tables[1][idx[1, pick, 0].long()].numpy())
    bench.dump_outputs(str(tmp_path / "b"), torch.tensor(0.5), params, grads, se, idx)
    assert np.array_equal(np.load(tmp_path / "b" / "embedding_rows.npy"), rows)


def test_cpu_arm_thread_count_ignores_the_launcher_omp_setting(monkeypatch):
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm must still use the host's cores."""
    import os
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    monkeypatch.delenv("DLRMB_CPU_THREADS", raising=False)
    assert bench.host_threads() == len(os.sched_getaffinity(0))
    monkeypatch.setenv("DLRMB_CPU_THREADS", "3")
    assert bench.host_threads() == 3


def test_cpu_arm_row_cap_follows_the_ram_budget():
    wl = bench.workload("terabyte", 2048)
    full = sum(wl["rows"]) * wl["D"] * 4
    assert bench.auto_rows_cap(wl, full) == max(wl["rows"]) == 40_000_000       # everything fits: no cap
    cap = bench.auto_rows_cap(wl, 8 << 30)
    assert cap & (cap - 1) == 0 and sum(min(r, cap) for r in wl["rows"]) * 512 <= 8 << 30
    assert sum(min(r, 2 * cap) for r in wl["rows"]) * 512 > 8 << 30
    total, avail = bench.host_ram_bytes()
    assert total >= avail > 0
