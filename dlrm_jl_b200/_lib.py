"""ctypes binding of libdlrm_b200.so (the C ABI declared in include/dlrm_b200.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libdlrm_b200.so")

OK, EINVAL, ECUDA, ENOMEM, EOOB, ESTATE, ENCCL = 0, 1, 2, 3, 4, 5, 6
_STATUS_NAMES = {EINVAL: "DLRMB_EINVAL", ECUDA: "DLRMB_ECUDA", ENOMEM: "DLRMB_ENOMEM",
                 EOOB: "DLRMB_EOOB", ESTATE: "DLRMB_ESTATE", ENCCL: "DLRMB_ENCCL"}


class DLRMB200Error(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{_STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


_i32, _i64, _f32, _vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p
_idx_args = [_vp, _i32, _i32, _i32, _i32]  # idx, idx_bytes, idx_base, B, P
_idx_mp_args = [_vp, _i32, _i32, _i32, C.POINTER(_i32)]  # idx, idx_bytes, idx_base, B, P[ntab]
_idx_jagged_args = [_vp, _vp, _i32, _i32, _i32, C.POINTER(_i64)]  # values, offsets, idx_bytes, idx_base, B, L[ntab]

# name -> (restype, argtypes); every symbol include/dlrm_b200.h declares
SIGNATURES = {
    "dlrmb_abi_version": (_i32, []),
    "dlrmb_last_error": (C.c_char_p, []),
    "dlrmb_launch_count": (_i64, []),
    "dlrmb_set_option": (_i32, [C.c_char_p, _i64]),
    "dlrmb_get_option": (_i32, [C.c_char_p, C.POINTER(_i64)]),
    "dlrmb_clock_buffer_bytes": (_i64, []),
    "dlrmb_clock_kernels": (_i32, []),
    "dlrmb_clock_enable": (_i32, [_vp]),
    "dlrmb_tables_create": (_i32, [_i32, _i32, C.POINTER(_i64), _i32, _i64, C.POINTER(_vp)]),
    "dlrmb_tables_create_ex": (_i32, [_i32, _i32, C.POINTER(_i64), _i32, _i64, _i32, C.POINTER(_vp)]),
    "dlrmb_tables_elem_bytes": (_i32, [_vp]),
    "dlrmb_tables_reserve": (_i32, [_vp, _i64]),
    "dlrmb_tables_destroy": (_i32, [_vp]),
    "dlrmb_tables_info": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i64), C.POINTER(_i64)]),
    "dlrmb_tables_upload": (_i32, [_vp, _i32, _vp]),
    "dlrmb_tables_download": (_i32, [_vp, _i32, _vp]),
    "dlrmb_tables_device_ptr": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "dlrmb_tables_init_uniform": (_i32, [_vp, C.c_uint64, _vp]),
    "dlrmb_tables_sync": (_i32, [_vp]),
    "dlrmb_embedding_fwd": (_i32, [_vp, *_idx_args, _vp, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_sort": (_i32, [_vp, *_idx_args, _vp, _i32, _i32, _vp]),
    "dlrmb_interaction_fwd": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "dlrmb_interaction_bwd": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "dlrmb_embedding_sort": (_i32, [_vp, *_idx_args, _vp]),
    "dlrmb_embedding_update_sorted": (_i32, [_vp, _vp, _i32, _i32, _f32, _vp]),
    "dlrmb_embedding_bwd_sgd": (_i32, [_vp, *_idx_args, _vp, _i32, _i32, _f32, _vp]),
    "dlrmb_sort_dedup_export": (_i32, [_vp, _i32, _vp, _vp, _vp, C.POINTER(_i32)]),
    "dlrmb_check_indices": (_i32, [_vp, *_idx_args, _i32]),
    "dlrmb_bce_sigmoid_fwd_bwd": (_i32, [_i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "dlrmb_xbuf_create": (_i32, [_i32, _i64, C.POINTER(_vp)]),
    "dlrmb_xbuf_destroy": (_i32, [_vp]),
    "dlrmb_xbuf_ptr": (_i32, [_vp, C.POINTER(_vp)]),
    "dlrmb_xbuf_ipc_handle": (_i32, [_vp, _vp]),
    "dlrmb_xbuf_open": (_i32, [_i32, _vp, C.POINTER(_vp)]),
    "dlrmb_xbuf_close": (_i32, [_i32, _vp]),
    "dlrmb_tables_set_slot_map": (_i32, [_vp, C.POINTER(_i32)]),
    "dlrmb_tables_set_dest_map": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i32), _i32]),
    "dlrmb_embedding_fwd_p2p": (_i32, [_vp, *_idx_args, C.POINTER(_vp), _i32, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_p2p_sort": (_i32, [_vp, *_idx_args, C.POINTER(_vp), _i32, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_p2p_mp": (_i32, [_vp, *_idx_mp_args, C.POINTER(_vp), _i32, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_p2p_sort_mp": (_i32, [_vp, *_idx_mp_args, C.POINTER(_vp), _i32, _i32, _i32, _vp]),
    "dlrmb_peer_barrier": (_i32, [_i32, C.POINTER(_vp), _i32, _i32, _i32, _vp, _vp]),
    "dlrmb_peer_barrier_flag_bytes": (_i64, []),
    "dlrmb_peer_barrier_state_bytes": (_i64, []),
    "dlrmb_peer_allreduce_f32": (_i32, [_i32, C.POINTER(_vp), C.POINTER(_vp), _i32, _i32, _i32, _vp, _vp, _i64, _vp]),
    "dlrmb_indices_scatter_p2p": (_i32, [_i32, _vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "dlrmb_indices_scatter_p2p_mp": (_i32, [_i32, _vp, _i32, _i32, _i32, C.POINTER(_i32), _vp, _i32, _vp]),
    "dlrmb_indices_scatter_p2p_mp_list": (_i32, [_i32, _vp, _i32, _i32, _i32, C.POINTER(_i32), _i32, C.POINTER(_i32),
                                                 _vp, _i32, _vp]),
    # values, offsets, weights, idx_bytes, ntab, B_local, owner[ntab], L_all[world][ntab], world, rank, peer_values,
    # peer_offsets, peer_weights, cap_values[world], stream
    "dlrmb_indices_scatter_p2p_jagged": (_i32, [_i32, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i32), C.POINTER(_i64),
                                                _i32, _i32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                                C.POINTER(_i64), _vp]),
    # values, offsets, weights, idx_bytes, idx_base, B_global, L[ntab], pooling, peer_T, world, B_local, slots, stream
    "dlrmb_embedding_fwd_p2p_jagged": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i64), _i32, C.POINTER(_vp),
                                              _i32, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_p2p_sort_jagged": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i64), _i32,
                                                   C.POINTER(_vp), _i32, _i32, _i32, _vp]),
    "dlrmb_interaction_has_warp_path": (_i32, [_i32, _i32]),
    "dlrmb_dense_fwd_bias_act": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _vp]),
    "dlrmb_dense_bwd_scratch_floats": (_i64, [_i32]),
    "dlrmb_dense_bwd_act_bias": (_i32, [_i32, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "dlrmb_interaction_bwd_scatter": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _vp]),
    "dlrmb_interaction_bwd_scatter_cols": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _i32, _i64, _vp, _vp]),
    "dlrmb_interaction_bwd_dx": (_i32, [_i32, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "dlrmb_dac_unpack": (_i32, [_i32, _vp, _i32, _vp, _vp, _vp, _vp]),
    "dlrmb_shard_plan": (_i32, [_i32, C.POINTER(_i64), _i32, C.POINTER(_i32)]),
    "dlrmb_shard_plan_mp": (_i32, [_i32, C.POINTER(_i64), C.POINTER(_i32), _i32, C.POINTER(_i32)]),
    "dlrmb_shard_plan_cw": (_i32, [_i32, C.POINTER(_i64), C.POINTER(_i32), _i32, _i32, _i32, C.POINTER(_i32),
                                   C.POINTER(_i32)]),
    "dlrmb_comm_unique_id": (_i32, [_vp]),
    "dlrmb_comm_create": (_i32, [_i32, _vp, _i32, _i32, C.POINTER(_vp)]),
    "dlrmb_comm_destroy": (_i32, [_vp]),
    "dlrmb_comm_info": (_i32, [_vp, C.POINTER(_i32), C.POINTER(_i32)]),
    "dlrmb_comm_a2a_indices": (_i32, [_vp, C.POINTER(_i32), _i32, _vp, _i32, _i32, _i32, _vp, _vp]),
    "dlrmb_comm_a2a_indices_mp": (_i32, [_vp, C.POINTER(_i32), _i32, _vp, _i32, _i32, C.POINTER(_i32), _vp, _vp]),
    "dlrmb_comm_a2a_fwd": (_i32, [_vp, C.POINTER(_i32), _i32, _vp, _i32, _i32, _vp, _vp]),
    "dlrmb_comm_a2a_bwd": (_i32, [_vp, C.POINTER(_i32), _i32, _vp, _i32, _i32, _vp, _vp]),
    "dlrmb_comm_allreduce_f32": (_i32, [_vp, _vp, _i64, _vp]),
    "dlrmb_comm_allgather": (_i32, [_vp, _vp, _vp, _i64, _vp]),
    "dlrmb_embedding_fwd_host": (_i32, [_vp, *_idx_args, _vp, _i32, _i32]),
    "dlrmb_interaction_fwd_host": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "dlrmb_interaction_bwd_host": (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "dlrmb_embedding_bwd_sgd_host": (_i32, [_vp, *_idx_args, _vp, _i32, _i32, _f32]),
    "dlrmb_mp_max_tables": (_i32, []),
    "dlrmb_embedding_fwd_mp": (_i32, [_vp, *_idx_mp_args, _vp, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_sort_mp": (_i32, [_vp, *_idx_mp_args, _vp, _i32, _i32, _vp]),
    "dlrmb_embedding_sort_mp": (_i32, [_vp, *_idx_mp_args, _vp]),
    "dlrmb_embedding_bwd_sgd_mp": (_i32, [_vp, *_idx_mp_args, _vp, _i32, _i32, _f32, _vp]),
    "dlrmb_check_indices_mp": (_i32, [_vp, *_idx_mp_args, _i32]),
    "dlrmb_embedding_fwd_mp_host": (_i32, [_vp, *_idx_mp_args, _vp, _i32, _i32]),
    "dlrmb_embedding_bwd_sgd_mp_host": (_i32, [_vp, *_idx_mp_args, _vp, _i32, _i32, _f32]),
    "dlrmb_embedding_fwd_jagged": (_i32, [_vp, *_idx_jagged_args, _i32, _vp, _i32, _i32, _vp]),
    "dlrmb_embedding_fwd_sort_jagged": (_i32, [_vp, *_idx_jagged_args, _i32, _vp, _i32, _i32, _vp]),
    "dlrmb_embedding_sort_jagged": (_i32, [_vp, *_idx_jagged_args, _i32, _vp]),
    "dlrmb_check_indices_jagged": (_i32, [_vp, *_idx_jagged_args, _i32]),
    # values, offsets, weights, idx_bytes, idx_base, B, L[ntab], out, slots, slot0, stream
    "dlrmb_embedding_fwd_jagged_weighted": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i64), _vp, _i32,
                                                   _i32, _vp]),
    "dlrmb_embedding_fwd_sort_jagged_weighted": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i64), _vp,
                                                        _i32, _i32, _vp]),
    "dlrmb_embedding_sort_jagged_weighted": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, C.POINTER(_i64), _vp]),
    "dlrmb_embedding_weight_grad_jagged": (_i32, [_vp, *_idx_jagged_args, _vp, _i32, _i32, _vp, _vp]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load the shared library and bind every declared symbol (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DLRMB200Error(
            ESTATE,
            f"{LIB_PATH} not found: build it with `python -m dlrm_jl_b200.csrc.build` "
            "(there is no CPU or PyTorch fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.dlrmb_abi_version() != 1:
        raise DLRMB200Error(ESTATE, f"ABI version mismatch: library has {lib.dlrmb_abi_version()}, binding expects 1")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != OK:
        msg = load().dlrmb_last_error()
        raise DLRMB200Error(status, msg.decode("utf-8", "replace") if msg else "")


def launch_count() -> int:
    return int(load().dlrmb_launch_count())


def set_option(name: str, value: int) -> None:
    """Process-wide tuning / test switch of the library (include/dlrm_b200.h: dlrmb_set_option)."""
    check(load().dlrmb_set_option(name.encode(), int(value)))


def get_option(name: str) -> int:
    v = _i64()
    check(load().dlrmb_get_option(name.encode(), C.byref(v)))
    return int(v.value)
