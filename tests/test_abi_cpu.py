"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol the
header declares, the ctypes binding covers all of them, and the host-side helpers behave.
No compute call is made (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "dlrm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dlrmb_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def built_lib():
    from dlrm_jl_b200.csrc import build
    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    lib = ctypes.CDLL(built_lib)
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/dlrm_b200.h but not exported"


def test_binding_covers_header_exactly(built_lib):
    from dlrm_jl_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_symbols()
    lib = _lib.load()
    assert lib.dlrmb_abi_version() == 1
    assert isinstance(lib.dlrmb_launch_count(), int)


def test_julia_glue_and_integration_guide_only_name_exported_symbols(built_lib):
    """julia/DLRMB200.jl (the ccall side a DLRM.jl maintainer loads) and INTEGRATION.md may only bind
    symbols the header declares and the library exports; every pure query is callable without a GPU."""
    declared = set(_declared_symbols())
    lib = ctypes.CDLL(built_lib)
    for rel in ("julia/DLRMB200.jl", "INTEGRATION.md"):
        text = open(os.path.join(ROOT, rel)).read()
        used = set(re.findall(r"\b(dlrmb_[a-z0-9_]+)\b", text))
        # prose may abbreviate families: dlrmb_xbuf_*, dlrmb_embedding_fwd[_host], dlrmb_tables_create / _upload
        used = {u for u in used if not u.endswith("_")}
        unknown = sorted(u for u in used if u not in declared and not any(d.startswith(u) for d in declared))
        assert not unknown, f"{rel} names symbols the header does not declare: {unknown}"
    jl = open(os.path.join(ROOT, "julia/DLRMB200.jl")).read()
    for n in re.findall(r"ccall\(\(:(dlrmb_[a-z0-9_]+),", jl):
        assert hasattr(lib, n), n
    # every ccall passes as many argument types as the C prototype (= the ctypes binding) has parameters
    from dlrm_jl_b200 import _lib as _binding
    calls = re.findall(r"ccall\(\(:(dlrmb_[a-z0-9_]+), libdlrm_b200\), (\w+),\s*\(([^()]*)\)", jl)
    assert len(calls) >= 12
    for name, ret, types in calls:
        n_types = len([t for t in types.split(",") if t.strip()])
        assert n_types == len(_binding.SIGNATURES[name][1]), (name, n_types)
        assert ret in ("Int32", "Cstring"), (name, ret)
    # the glue extends the reference's own functions for the B200 table type (not private look-alikes)
    for needle in ("function EmbeddingTables.maplookup(strategy::PreallocationStrategy, tables::AbstractVector{<:B200Embedding}",
                   "function EmbeddingTables.update!(opt::Flux.Descent, tables::AbstractVector{<:B200Embedding}",
                   "struct B200Embedding{S,T} <: AbstractEmbeddingTable{S,T}",
                   "ChainRulesCore.rrule(::typeof(EmbeddingTables.maplookup)",
                   "SparseEmbeddingUpdate{Static{D}}(", "Base.isapprox(a::AbstractMatrix, t::B200Embedding"):
        assert needle in jl, needle
    from dlrm_jl_b200 import _lib
    L = _lib.load()
    assert L.dlrmb_interaction_has_warp_path(27, 128) == 1 and L.dlrmb_interaction_has_warp_path(5, 12) == 0
    assert L.dlrmb_dense_bwd_scratch_floats(1024) >= 16 * 1024 + 32


def test_argument_validation_needs_no_gpu(built_lib):
    from dlrm_jl_b200 import _lib
    lib = _lib.load()
    out = ctypes.c_void_p()
    rows = (ctypes.c_int64 * 1)(10)
    rc = lib.dlrmb_tables_create(0, 0, rows, 16, 128, ctypes.byref(out))   # ntab = 0
    assert rc == _lib.EINVAL and b"ntab" in lib.dlrmb_last_error()
    rc = lib.dlrmb_tables_create(0, 1, rows, 3000, 128, ctypes.byref(out))  # bad D
    assert rc == _lib.EINVAL and b"D must be" in lib.dlrmb_last_error()
    rc = lib.dlrmb_interaction_fwd(0, None, None, 4, 8, 16, 1, None, None)
    assert rc == _lib.EINVAL
    with pytest.raises(_lib.DLRMB200Error, match="DLRMB_EINVAL"):
        _lib.check(rc)


def test_library_switches_match_the_header(built_lib):
    """dlrmb_set_option / dlrmb_get_option (host-side state, no GPU): every switch the header documents exists and
    round-trips, defaults are what the header says, unknown names are refused, and bench.py records real names."""
    import re
    from dlrm_jl_b200 import _lib
    header = open(os.path.join(ROOT, "include", "dlrm_b200.h")).read()
    block = header[header.index("Process-wide tuning / test switches"):header.index("int32_t dlrmb_set_option")]
    names = re.findall(r'^ \*   "([a-z_0-9]+)"', block, flags=re.M)
    names += re.findall(r', "([a-z_0-9]+)" [0-9]', block)          # second switch documented on the same line
    assert {"interact_general", "update_two_launches", "update_tile", "bwd_variant", "fwd_tb", "fwd_ks", "fwd_ksplit"} <= set(names)
    defaults = {"fwd_ksplit": 1}
    for n in names:
        before = _lib.get_option(n)
        assert before == defaults.get(n, 0), (n, before)
        _lib.set_option(n, 3)
        assert _lib.get_option(n) == 3
        _lib.set_option(n, before)
    for bad in ("update_prefetch", "lookup_flat", "fwd_rows_per_copy", "no_such_switch"):   # measured and removed / never existed
        with pytest.raises(_lib.DLRMB200Error, match="unknown option"):
            _lib.set_option(bad, 1)
    bench = open(os.path.join(ROOT, "bench.py")).read()
    recorded = re.search(r'for k in \(([^)]*)\)\}', bench[bench.index("def library_options"):]).group(1)
    for n in re.findall(r'"([a-z_0-9]+)"', recorded):
        assert n in names, n


def test_product_path_has_no_cpu_fallback(built_lib):
    from dlrm_jl_b200 import DLRMB200Error
    from dlrm_jl_b200.embedding import EmbeddingTables
    from dlrm_jl_b200.interact import interaction_fwd
    with pytest.raises(DLRMB200Error):
        EmbeddingTables([10], 16, 8, torch.device("cpu"))
    with pytest.raises(DLRMB200Error):
        interaction_fwd(torch.zeros(2, 3, 4))
    # and nothing in the package imports the oracle
    pkg = os.path.join(ROOT, "dlrm_jl_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.lower(), f


def test_index_normalisation_and_widths():
    from dlrm_jl_b200.embedding import _as_index_tensor
    from dlrm_jl_b200.interact import interaction_width
    cpu = torch.device("cpu")
    a = _as_index_tensor([np.arange(4), np.arange(4)], 2, cpu)
    assert a.shape == (2, 4, 1) and a.dtype == torch.int64
    b = _as_index_tensor(np.zeros((3, 5, 2), dtype=np.int32), 3, cpu)
    assert b.shape == (3, 5, 2) and b.dtype == torch.int32
    c = _as_index_tensor([np.zeros((6, 10), dtype=np.int64)] * 7, 7, cpu)   # multi golden: P = 10
    assert c.shape == (7, 6, 10)
    with pytest.raises(ValueError):
        _as_index_tensor(np.zeros((2, 4), dtype=np.int64), 3, cpu)
    assert interaction_width(27, 64) == 415 and interaction_width(8, 16) == 44
    assert interaction_width(27, 128) == 479 and interaction_width(27, 64, 8) == 416


def test_model_constants_match_reference():
    from dlrm_jl_b200.model import KAGGLE_EMBEDDING_SIZES, TERABYTE_EMBEDDING_SIZES
    assert len(KAGGLE_EMBEDDING_SIZES) == 26 and sum(KAGGLE_EMBEDDING_SIZES) == 33762577
    assert len(TERABYTE_EMBEDDING_SIZES) == 26
    assert sum(min(r, 40_000_000) for r in TERABYTE_EMBEDDING_SIZES) == 204184588


def test_hdf5_reader_and_natural_sort():
    """The pure-Python HDF5 reader reads every dataset of a file with the goldens' container shape
    (tests/golden/hdf5_sample.h5), and layer names sort as the reference's NaturalSort does."""
    from dlrm_jl_b200.hdf5_min import read_hdf5
    from dlrm_jl_b200.validation import _natural
    from tests.helpers import hdf5_sample_arrays
    names = ["update_bot_10.weight", "update_bot_2.weight", "update_bot_0.weight"]
    assert sorted(names, key=_natural) == ["update_bot_0.weight", "update_bot_2.weight", "update_bot_10.weight"]
    d = read_hdf5(os.path.join(ROOT, "tests", "golden", "hdf5_sample.h5"))
    want = hdf5_sample_arrays()
    assert sorted(d) == sorted(want)
    for k in d:
        assert d[k].dtype == want[k].dtype and np.array_equal(d[k], want[k]), k
