"""Shared loaders for the golden fixtures (tests only)."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def reference_parameters():
    """The golden model's parameters before the step, as the PyTorch reference drew them: numpy's
    legacy generator seeded 123, first the 7 tables [1000][16] from U(-sqrt(1/1000), sqrt(1/1000)),
    then for every Linear of the bottom MLP (13-512-256-64-16) and of the top MLP (44-512-256-1)
    a weight [out][in] from N(0, sqrt(2 / (in + out))) and a bias from N(0, sqrt(1 / out)), each
    cast to float32.  RandomState's streams never change, so these are the HDF5 files' values."""
    rng = np.random.RandomState(123)
    p = {}
    for k in range(7):
        p[f"emb_{k}"] = rng.uniform(-np.sqrt(1 / 1000), np.sqrt(1 / 1000), size=(1000, 16)).astype(np.float32)
    for prefix, sizes in (("bot_l", [13, 512, 256, 64, 16]), ("top_l", [44, 512, 256, 1])):
        for i, (n, m) in enumerate(zip(sizes[:-1], sizes[1:])):
            p[f"{prefix}.{i}.weight"] = rng.normal(0.0, np.sqrt(2 / (m + n)), size=(m, n)).astype(np.float32)
            p[f"{prefix}.{i}.bias"] = rng.normal(0.0, np.sqrt(1 / m), size=m).astype(np.float32)
    return p


def params_sha256(params) -> str:
    h = hashlib.sha256()
    for k in sorted(params):
        h.update(k.encode() + str(params[k].shape).encode() + params[k].tobytes())
    return h.hexdigest()


def hdf5_sample_arrays():
    """The datasets of tests/golden/hdf5_sample.h5 (tests/golden/make_hdf5_sample.py): names, dtypes and
    ranks as in the reference's golden files, including a scalar, enough of them for two symbol-table nodes."""
    rng = np.random.default_rng(5)
    f = lambda *shape: rng.standard_normal(shape).astype(np.float32)  # noqa: E731
    return {"bot_l.0.bias": f(4), "bot_l.0.weight": f(4, 3), "emb_0": f(6, 2), "input_bot": f(5, 3),
            "input_emb_0": rng.integers(0, 6, size=5), "input_emb_1": rng.integers(0, 6, size=5),
            "labels": f(5, 1), "loss": np.float32(0.8544201).reshape(()), "update_bot_0.weight": f(4, 3),
            "zpre": f(2, 2, 2)}


def load_golden(name: str):
    """name in {"single", "multi"} -> the 58 datasets of ref/pytorch_reference_<name>.hdf5 as a dict of
    arrays, rebuilt from the compact layout described in tests/golden/make_golden.py."""
    g = {}
    for part in ("", "_update_bot", "_update_top"):
        with np.load(os.path.join(GOLDEN, f"pytorch_reference_{name}{part}.npz")) as z:
            g.update((k, z[k]) for k in z.files)
    params = reference_parameters()
    assert str(g.pop("params_sha256")) == params_sha256(params), "regenerated initial parameters differ from the golden's"
    g.update(params)
    for k in range(7):
        upd = params[f"emb_{k}"].copy()
        upd[np.unique(g[f"input_emb_{k}"])] = g.pop(f"update_emb_{k}_rows")
        g[f"update_emb_{k}"] = upd
    return g


def golden_model(g):
    """Split a golden dict into (bot, top, tables, dense, idx, labels) in oracle layout."""
    bot = [(g[f"bot_l.{i}.weight"], g[f"bot_l.{i}.bias"]) for i in range(4)]
    top = [(g[f"top_l.{i}.weight"], g[f"top_l.{i}.bias"]) for i in range(3)]
    tables = [g[f"emb_{k}"].copy() for k in range(7)]
    B = g["labels"].shape[0]
    idx = [g[f"input_emb_{k}"].reshape(B, -1) for k in range(7)]
    return bot, top, tables, g["input_bot"], idx, g["labels"].reshape(-1)


def golden_updates(g):
    ubot = [(g[f"update_bot_{2 * i}.weight"], g[f"update_bot_{2 * i}.bias"]) for i in range(4)]
    utop = [(g[f"update_top_{2 * i}.weight"], g[f"update_top_{2 * i}.bias"]) for i in range(3)]
    uemb = [g[f"update_emb_{k}"] for k in range(7)]
    return ubot, utop, uemb


def load_known_answer():
    with open(os.path.join(GOLDEN, "known_answer_small.json")) as fh:
        d = json.load(fh)
    return {k: (np.asarray(v, dtype=np.float32) if k != "py_sparse_input" and k != "py_embedding_outputs" else v)
            for k, v in d.items()}
