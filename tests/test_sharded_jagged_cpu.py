"""Table-sharded jagged bags (variable length, sum / mean / weighted pooling) without a GPU: the owner-layout reference
on hand-built cases, gloo runs at 2, 3 and 4 ranks of the index exchange and of whole ShardedEmbedding steps with the
NumPy jagged references as the injected compute, the per-step count exchange's refusal of ranks that disagree, the
handles' refusals, and the new C entry points' refusal of bad arguments before any CUDA call."""
import os
import socket
import subprocess

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dlrm_jl_b200.embedding import JaggedIndices
from dlrm_jl_b200.sharded import ShardedEmbedding, TableSharding
from tests import sharded_jagged_oracle as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _jag(values, offsets, weights, lengths, pooling="sum"):
    return JaggedIndices.from_lengths(torch.from_numpy(np.asarray(values)), lengths, pooling,
                                      None if weights is None else torch.from_numpy(weights))


# ---- the owner-layout reference on hand-built cases ----------------------------------------------------
def test_owner_layout_hand_built():
    """Two ranks, three tables, B_local = 2.  Rank 0: table 0 bags [1, 2], []; table 1 bags [], []; table 2 bags [7],
    [8, 9].  Rank 1: table 0 bags [], [3]; table 1 bags [], []; table 2 bags [], [6].  Table 1 has no lookup on any
    rank, and on rank 1 table 0's first bag is empty."""
    r0 = (np.array([1, 2, 7, 8, 9]), np.array([0, 2, 2, 2, 2, 3, 5]), np.array([.5, .25, 2, 3, 4], np.float32))
    r1 = (np.array([3, 6]), np.array([0, 0, 1, 1, 1, 1, 2]), np.array([-1, 6], np.float32))
    v, o, L, w = S.owner_layout([r0, r1], [0, 2], 2)
    assert v.tolist() == [1, 2, 3, 7, 8, 9, 6]
    # bags: table 0 = r0 [1,2], r0 [], r1 [], r1 [3]; table 2 = r0 [7], r0 [8,9], r1 [], r1 [6]
    assert o.tolist() == [0, 2, 2, 2, 3, 4, 6, 6, 7]
    assert L == [3, 4]
    assert w.tolist() == [.5, .25, -1, 2, 3, 4, 6]
    v, o, L, w = S.owner_layout([r0, r1], [1], 2)                       # a table with no lookup anywhere
    assert v.tolist() == [] and o.tolist() == [0, 0, 0, 0, 0] and L == [0] and w.tolist() == []
    v, o, L, w = S.owner_layout([(r0[0], r0[1], None)], [0, 1, 2], 2)   # W = 1: the batch itself
    assert v.tolist() == r0[0].tolist() and o.tolist() == r0[1].tolist() and L == [2, 0, 3] and w is None
    v, o, L, w = S.owner_layout([r0, r1], [], 2)                        # an owner without tables
    assert len(v) == 0 and o.tolist() == [0] and L == []


# ---- gloo runs ----------------------------------------------------------------------------------------
ROWS = [50, 7, 400, 3, 120, 33, 9, 61]
MAXLEN = [3, 1, 7, 0, 2, 12, 1, 5]          # table 3 has no lookup on any rank
HOT = [2, 1, 4, 1, 1, 6, 1, 3]              # plan weights: expected bag lengths
D, BL = 8, 6


def _worker(rank, world, port, q, pooling):
    from oracle import oracle as O
    from dlrm_jl_b200.sharded import exchange_indices_jagged, exchange_jagged_counts
    from tests import jagged_oracle as J
    from tests import jagged_weighted_oracle as JW
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        weighted = pooling == "weighted"
        pool = "mean" if pooling == "mean" else "sum"
        rng = np.random.default_rng(29)                      # same tables / batches on every rank
        tables = [rng.standard_normal((r, D)).astype(np.float32) for r in ROWS]
        sh = TableSharding.build(ROWS, world, HOT)
        mine = sh.local[rank]

        # the index exchange alone, int32 and int64, against the owner-layout reference
        ok_x = True
        for dt in (np.int32, np.int64):
            batches = [S.random_batch(rng, ROWS, BL, MAXLEN, dt, weighted) for _ in range(world)]
            jl = _jag(*batches[rank], pooling=pool)
            counts = exchange_jagged_counts(jl)
            ok_x = ok_x and counts.tolist() == [b[3].sum(axis=1).tolist() for b in batches]
            owned = exchange_indices_jagged(jl, counts, sh, rank)
            v, o, L, w = S.owner_layout([b[:3] for b in batches], mine, BL)
            ok_x = ok_x and owned.B == BL * world and list(owned.L) == L and owned.pooling == pool
            ok_x = ok_x and owned.values.dtype == jl.values.dtype and np.array_equal(owned.values.numpy(), v)
            ok_x = ok_x and np.array_equal(owned.offsets.numpy(), o)
            ok_x = ok_x and (w is None) == (owned.weights is None)
            ok_x = ok_x and (w is None or np.array_equal(owned.weights.numpy(), w))

        # two steps of a whole ShardedEmbedding with the references as the injected compute
        local_tables = [tables[k].copy() for k in mine]

        def lookup_fn(idx, out, slot0):
            if weighted:
                ref = JW.lookup_jagged_weighted(local_tables, idx.values.numpy(), idx.offsets.numpy(),
                                                idx.weights.numpy(), idx.B, slot0)
            else:
                ref = J.lookup_jagged(local_tables, idx.values.numpy(), idx.offsets.numpy(), idx.B, pool, slot0)
            out.copy_(torch.from_numpy(ref))

        def update_fn(idx, g, lr, slot0, presorted=False):
            for j in range(len(mine)):
                part = idx[j]
                delta = np.ascontiguousarray(g[:, slot0 + j].numpy())
                if weighted:
                    JW.sparse_sgd_update_jagged_weighted(local_tables[j], part[0].numpy(), part[1].numpy(),
                                                         part[2].numpy(), delta, lr)
                else:
                    J.sparse_sgd_update_jagged(local_tables[j], part[0].numpy(), part[1].numpy(), delta, lr, pool)

        se = ShardedEmbedding(ROWS, D, rank, world, lookup_fn, update_fn, P=HOT, jagged_cap=[m * BL for m in MAXLEN])
        ref = [t.copy() for t in tables]
        ok_fwd = ok_upd = True
        F = 1 + len(ROWS)
        for step in range(2):
            batches = [S.random_batch(rng, ROWS, BL, MAXLEN, np.int64, weighted) for _ in range(world)]
            x_all = [rng.standard_normal((BL, D)).astype(np.float32) for _ in range(world)]
            gz_all = [rng.standard_normal((BL, D + F * (F - 1) // 2)).astype(np.float32) for _ in range(world)]
            anchor = torch.zeros(1, requires_grad=True)
            T = se.lookup(_jag(*batches[rank], pooling=pool), anchor)

            def ref_lookup(b):
                if weighted:
                    return JW.lookup_jagged_weighted(ref, b[0], b[1], b[2], BL, slot0=1)
                return J.lookup_jagged(ref, b[0], b[1], BL, pool, slot0=1)
            ok_fwd = ok_fwd and np.array_equal(T.detach().numpy()[:, 1:], ref_lookup(batches[rank])[:, 1:])
            Tn = T.detach().numpy().copy()
            Tn[:, 0] = x_all[rank]
            T.backward(torch.from_numpy(O.interaction_bwd(gz_all[rank], Tn)[1]))
            se.update(0.5)
            dT_glob = []
            for r in range(world):
                Tr = ref_lookup(batches[r])
                Tr[:, 0] = x_all[r]
                dT_glob.append(O.interaction_bwd(gz_all[r], Tr)[1])
            dT_glob = np.concatenate(dT_glob, axis=0)
            for k in range(len(ROWS)):                    # the unsharded update over the concatenated global batch
                v, o, _L, w = S.owner_layout([b[:3] for b in batches], [k], BL)
                delta = np.ascontiguousarray(dT_glob[:, 1 + k])
                if weighted:
                    JW.sparse_sgd_update_jagged_weighted(ref[k], v, o, w, delta, 0.5)
                else:
                    J.sparse_sgd_update_jagged(ref[k], v, o, delta, 0.5, pool)
            ok_upd = ok_upd and all(np.array_equal(local_tables[j], ref[k]) for j, k in enumerate(mine))
        q.put((rank, bool(ok_x), bool(ok_fwd), bool(ok_upd), ""))
    except Exception as exc:  # noqa: BLE001
        import traceback
        q.put((rank, False, False, False, repr(exc) + traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _run(target, world, *args):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=target, args=(r, world, port, q) + args) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("pooling", ["sum", "mean", "weighted"])
def test_sharded_jagged_matches_unsharded_oracle(world, pooling):
    """exchange_jagged_counts gathers every rank's counts; exchange_indices_jagged equals the owner-layout reference
    (int32 and int64); two steps of a jagged ShardedEmbedding give the unsharded reference's pooled rows and tables
    bit for bit."""
    for rank, ok_x, ok_fwd, ok_upd, err in _run(_worker, world, pooling):
        assert not err, f"rank {rank}: {err}"
        assert ok_x, f"rank {rank}: the index exchange differs from the owner layout"
        assert ok_fwd, f"rank {rank}: pooled rows differ from the unsharded reference"
        assert ok_upd, f"rank {rank}: tables differ from the unsharded reference"


def _disagree_worker(rank, world, port, q, what):
    from dlrm_jl_b200.sharded import exchange_jagged_counts
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        B = 3 + (rank if what == "B_local" else 0)
        pooling = "mean" if (what == "pooling" and rank == 1) else "sum"
        w = torch.ones(2 * B) if (what == "weighting" and rank == 0) else None
        jag = JaggedIndices.from_lengths(torch.zeros(2 * B, dtype=torch.int64), [[1] * B, [1] * B], pooling, w)
        try:
            exchange_jagged_counts(jag)
            q.put((rank, False, "no error"))
        except ValueError as e:
            q.put((rank, "disagree" in str(e), str(e)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("what", ["pooling", "weighting", "B_local"])
def test_count_exchange_refuses_disagreeing_ranks_on_every_rank(what):
    for rank, ok, msg in _run(_disagree_worker, 2, what):
        assert ok, f"rank {rank}: {msg}"


# ---- refusals -----------------------------------------------------------------------------------------
def _nop(*a, **k):
    return None


def test_fixed_width_handle_refuses_jagged_batches():
    jag = JaggedIndices.from_bags([[[1], [2, 3]], [[], [4]]])
    for P in (None, [1, 2]):
        se = ShardedEmbedding([5, 6], 4, 0, 2, _nop, _nop, P=P)
        with pytest.raises(ValueError, match="jagged_cap"):
            se.lookup(jag, torch.zeros(1, requires_grad=True))


def test_column_wise_plan_refuses_jagged_cap():
    # P = [10, 1] at 2 ranks: table 0 holds 10 of 11 lookups and is split in two by columns
    assert TableSharding.build([100, 100], 2, [10, 1], D=8, max_col_shards=2).split
    with pytest.raises(ValueError, match="jagged_cap"):
        ShardedEmbedding([100, 100], 8, 0, 2, _nop, _nop, P=[10, 1], max_col_shards=2, jagged_cap=[40, 4])
    with pytest.raises(ValueError, match="jagged_cap"):
        ShardedEmbedding.create([100, 100], 8, 4, [10, 1], 0, 2, "cpu", max_col_shards=2, jagged_cap=[40, 4])


def test_jagged_handle_checks_its_batches():
    se = ShardedEmbedding([5, 6], 4, 0, 1, _nop, _nop, jagged_cap=[3, 2])
    with pytest.raises(ValueError, match="takes JaggedIndices"):
        se.lookup(np.zeros((2, 3, 1), np.int64), torch.zeros(1, requires_grad=True))
    with pytest.raises(ValueError, match="jagged_cap\\[1\\] = 2"):
        se.lookup(JaggedIndices.from_bags([[[1], [2]], [[1, 2], [3]]]), torch.zeros(1, requires_grad=True))
    with pytest.raises(ValueError, match="one lookup count per table"):
        ShardedEmbedding([5, 6], 4, 0, 1, _nop, _nop, jagged_cap=[3])


def test_count_group_of_a_non_gloo_subgroup_is_refused(monkeypatch):
    """dist.new_group needs every rank of the job, so a non-gloo proper subgroup cannot make its own gloo group: it is
    refused with a ValueError naming count_group, and the whole-job case makes one gloo group over every rank."""
    from dlrm_jl_b200 import sharded
    sub = object()
    made = []
    monkeypatch.setattr(sharded.dist, "get_backend", lambda g=None: "nccl")
    monkeypatch.setattr(sharded.dist, "get_world_size", lambda g=None: 2 if g is sub else 4)
    monkeypatch.setattr(sharded.dist, "new_group", lambda **kw: made.append(kw) or "gloo group")
    with pytest.raises(ValueError, match="count_group"):
        sharded.gloo_group(sub)
    assert made == []
    assert sharded.gloo_group(None) == "gloo group" and made == [{"backend": "gloo"}]


# ---- the C entry points refuse bad arguments before any CUDA call -------------------------------------
_ARGS_PROGRAM = r"""
#include <stdio.h>
#include "common.cuh"
// Handles built on the host only: every check below runs before the entry point touches the device.
int main() {
    dlrmb_tables t;
    t.ntab = 2;
    t.max_lookups = 100;
    t.D = 8;
    int64_t L[2] = {1, 1};
    int64_t off[5] = {0, 1, 1, 2, 2};
    int32_t v[2] = {0, 0};
    float w[2] = {1.f, 1.f};
    float buf[64];
    float* peers[2] = {buf, buf};
    auto show = [](const char* what, int rc) { printf("%s %d %s\n", what, rc, dlrmb_last_error()); };
    // the fused lookup (B_global = 4 = 2 ranks * 2)
    show("fwd_handle", dlrmb_embedding_fwd_p2p_jagged(nullptr, v, off, nullptr, 8, 0, 4, L, 0, peers, 2, 2, 3, nullptr));
    show("fwd_peers", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, nullptr, 8, 0, 4, L, 0, nullptr, 2, 2, 3, nullptr));
    show("fwd_offsets", dlrmb_embedding_fwd_p2p_sort_jagged(&t, v, nullptr, nullptr, 8, 0, 4, L, 0, peers, 2, 2, 3, nullptr));
    show("fwd_idx_bytes", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, nullptr, 2, 0, 4, L, 0, peers, 2, 2, 3, nullptr));
    show("fwd_weights_mean", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, w, 8, 0, 4, L, 1, peers, 2, 2, 3, nullptr));
    show("fwd_world", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, nullptr, 8, 0, 4, L, 0, peers, 0, 2, 3, nullptr));
    show("fwd_B", dlrmb_embedding_fwd_p2p_sort_jagged(&t, v, off, w, 8, 0, 4, L, 0, peers, 2, 3, 3, nullptr));
    L[1] = 101;
    show("fwd_max_lookups", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, nullptr, 8, 0, 4, L, 0, peers, 2, 2, 3, nullptr));
    L[1] = 1;
    show("fwd_slot_map", dlrmb_embedding_fwd_p2p_jagged(&t, v, off, nullptr, 8, 0, 4, L, 0, peers, 2, 2, 3, nullptr));
    // the index scatter: 2 tables, both on rank 1, B_local = 2, rank 0 sends
    int32_t owner[2] = {1, 1};
    int64_t L_all[4] = {1, 1, 2, 0};                // rank 0: 1, 1; rank 1: 2, 0 -> owner 1 receives 4 entries
    int64_t cap[2] = {0, 4}, small_cap[2] = {0, 3};
    void* pv[2] = {buf, buf};
    void* po[2] = {buf, buf};
    float* pw[2] = {buf, buf};
    auto sc = [&](const void* values, const void* offsets, const float* weights, int ib, int ntab, int world, int rank,
                  void* const* vals, float* const* wts, const int32_t* own, const int64_t* caps) {
        return dlrmb_indices_scatter_p2p_jagged(0, values, offsets, weights, ib, ntab, 2, own, L_all, world, rank, vals,
                                                po, wts, caps, nullptr);
    };
    show("sc_offsets", sc(v, nullptr, nullptr, 8, 2, 2, 0, pv, nullptr, owner, cap));
    show("sc_peer_values", sc(v, off, nullptr, 8, 2, 2, 0, nullptr, nullptr, owner, cap));
    show("sc_idx_bytes", sc(v, off, nullptr, 3, 2, 2, 0, pv, nullptr, owner, cap));
    show("sc_world", sc(v, off, nullptr, 8, 2, 17, 0, pv, nullptr, owner, cap));
    show("sc_rank", sc(v, off, nullptr, 8, 2, 2, 2, pv, nullptr, owner, cap));
    show("sc_ntab", sc(v, off, nullptr, 8, 0, 2, 0, pv, nullptr, owner, cap));
    show("sc_weights_only", sc(v, off, w, 8, 2, 2, 0, pv, nullptr, owner, cap));
    show("sc_peer_weights_only", sc(v, off, nullptr, 8, 2, 2, 0, pv, pw, owner, cap));
    show("sc_cap", sc(v, off, nullptr, 8, 2, 2, 0, pv, nullptr, owner, small_cap));
    int32_t bad_owner[2] = {1, 2};
    show("sc_owner", sc(v, off, nullptr, 8, 2, 2, 0, pv, nullptr, bad_owner, cap));
    L_all[3] = -1;
    show("sc_negative", sc(v, off, nullptr, 8, 2, 2, 0, pv, nullptr, owner, cap));
    L_all[3] = (1ll << 31) - 3;                      // owner 1 would receive 2^31 entries
    int64_t big_cap[2] = {0, 1ll << 40};
    show("sc_int32", sc(v, off, nullptr, 4, 2, 2, 0, pv, nullptr, owner, big_cap));
    return 0;
}
"""


def test_c_entry_points_refuse_bad_arguments(tmp_path):
    from dlrm_jl_b200.csrc import build
    lib = build.build()
    src = tmp_path / "sharded_jagged_args.cu"
    src.write_text(_ARGS_PROGRAM)
    exe = tmp_path / "sharded_jagged_args"
    subprocess.run([build._nvcc(), "-std=c++17", "-I", os.path.join(ROOT, "include"), "-I", build.HERE, str(src),
                    "-o", str(exe), "-L", os.path.dirname(lib), "-ldlrm_b200", "-Xlinker", "-rpath=" + os.path.dirname(lib)],
                   check=True, capture_output=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    got = {line.split(" ", 1)[0]: line.split(" ", 2)[1:] for line in out.splitlines()}
    want = {"fwd_handle": "null argument", "fwd_peers": "null argument", "fwd_offsets": "offsets is null",
            "fwd_idx_bytes": "idx_bytes must be 4 or 8", "fwd_weights_mean": "pooling = 0 (sum) only",
            "fwd_world": "world must be in 1..16", "fwd_B": "B_global (4) must equal B_local (3) * world (2)",
            "fwd_max_lookups": "L[1] = 101 exceeds max_lookups = 100", "fwd_slot_map": "needs dlrmb_tables_set_slot_map",
            "sc_offsets": "null argument", "sc_peer_values": "null argument", "sc_idx_bytes": "idx_bytes must be 4 or 8",
            "sc_world": "bad world / rank (17, 0)", "sc_rank": "bad world / rank (2, 2)", "sc_ntab": "ntab must be in 1..256",
            "sc_weights_only": "both null or both set", "sc_peer_weights_only": "both null or both set",
            "sc_cap": "owner 1 receives 4 entries, its buffer holds cap_values[1] = 3",
            "sc_owner": "owner[1] = 2 is not a rank", "sc_negative": "L_all[1][1] = -1",
            "sc_int32": "4-byte offsets reach 2^31"}
    assert set(got) == set(want)
    for what, msg in want.items():
        rc, text = got[what]
        want_rc = 5 if what == "fwd_slot_map" else 1           # DLRMB_ESTATE without a slot map, else DLRMB_EINVAL
        assert int(rc) == want_rc, (what, rc, text)
        assert msg in text, (what, text)
