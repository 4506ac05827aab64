"""ctypes binding of libskm_b200.so (the C-ABI declared in include/skm_b200.h).

There is deliberately no CPU fallback: if the shared library is missing or no
CUDA device is present, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libskm_b200.so")

SKM_OK = 0
SKM_DENSE_MAX_SPACE = 1 << 27


class SkmError(RuntimeError):
    """A libskm_b200 call failed (the message carries skm_last_error())."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libskm_b200 error {code}: {message}")
        self.code = code


_lib = None
_lock = threading.Lock()

_p = C.c_void_p
_i64 = C.c_int64
_u64 = C.c_uint64
_int = C.c_int
_sz = C.c_size_t

# name -> (restype, argtypes); mirrors include/skm_b200.h one to one
SIGNATURES = {
    "skm_version": (_int, []),
    "skm_last_error": (C.c_char_p, []),
    "skm_device_info": (_int, [C.POINTER(_int), C.POINTER(_int), C.POINTER(_int)]),
    "skm_lut_build": (_int, [C.c_char_p, C.c_char_p, _int, C.c_char_p, _int, C.POINTER(C.c_uint8)]),
    "skm_reduce_bytes": (_int, [_p, _i64, _p, _p, _p]),
    "skm_encode_windows": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _int, _p, _p]),
    "skm_basis_accumulate": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _u64, _p, _p, _p]),
    "skm_basis_order_max_space": (_int, []),
    "skm_basis_first_progressive": (_int, [_p, _i64, _p, _p, _i64, _p, _int, _int, _u64, _p, _p, _i64, _int, _p]),
    "skm_basis_finalize_workspace": (_sz, [_i64]),
    "skm_basis_finalize": (_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_basis_colmap": (_int, [_p, _i64, _i64, _p, _p]),
    "skm_count_dense": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _i64, _int, _p, _i64, _p]),
    "skm_count_csr_workspace": (_sz, [_i64, _i64]),
    "skm_count_csr": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_learn_dense": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _i64, _p, _p, _i64, _p, _p, _p]),
    "skm_apply_dense_workspace": (_sz, [_i64, _i64, _i64]),
    "skm_apply_dense": (_int, [_p, _i64, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_learn_sparse_workspace": (_sz, [_i64]),
    "skm_learn_sparse": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_learn_wide_workspace": (_sz, [_i64]),
    "skm_learn_wide": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_basis_sorted_local_workspace": (_sz, [_i64]),
    "skm_basis_sorted_local": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_basis_sorted_finalize_workspace": (_sz, [_i64]),
    "skm_basis_sorted_finalize": (_int, [_p, _p, _p, _i64, _int, _i64, _i64, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_codes_to_columns": (_int, [_p, _i64, _p, _p, _i64, _p, _p]),
    "skm_count_csr_wide_workspace": (_sz, [_i64, _i64]),
    "skm_count_csr_wide": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _p, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_count_csr_sorted_workspace": (_sz, [_i64, _i64, _i64, _int]),
    "skm_count_csr_sorted": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _int, _p, _i64, _p, _p, _i64, _i64, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_learn_sparse_group_workspace": (_sz, [_i64]),
    "skm_learn_sparse_group": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _i64, _p, _p, _i64, _p, _p, _sz, _p]),
    "skm_learn_sparse_group_place": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _i64, _p, _p, _i64, _p, _p, _p, _i64, _p, _p, _p, _sz, _p]),
    "skm_gather_sequences": (_int, [_p, _p, _p, _i64, _p, _p, _p]),
    "skm_coo_merge_workspace": (_sz, [_i64]),
    "skm_coo_merge": (_int, [_p, _p, _i64, _u64, _p, _p, _p, _p, _sz, _p]),
    "skm_coo_colsum": (_int, [_p, _p, _i64, _i64, _p, _p]),
    "skm_coo_merge_runs_workspace": (_sz, [_i64, _int]),
    "skm_coo_merge_runs": (_int, [_p, _p, _p, _int, _p, _p, _p, _p, _sz, _p]),
    "skm_csc_build_workspace": (_sz, [_i64, _i64]),
    "skm_csc_build_workspace_cols": (_sz, [_i64, _i64, _i64]),
    "skm_csc_build": (_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_csc_pack": (_int, [_p, _p, _i64, _p, _p]),
    "skm_apply_sparse": (_int, [_p, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _int, _p, _p, _p, _p, _p, _p]),
    "skm_apply_sparse_rows": (_int, [_p, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _int, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "skm_apply_tc_planes_bytes": (_sz, [_i64, _i64]),
    "skm_apply_tc_prepare": (_int, [_p, _i64, _i64, _p, _sz, C.POINTER(_int), _p]),
    "skm_apply_tc_workspace": (_sz, [_i64, _i64, _i64]),
    "skm_apply_tc": (_int, [_p, _i64, _i64, _p, _int, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "skm_top2_merge": (_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _p]),
    "skm_top2_rows_f64": (_int, [_p, _i64, _i64, _p, _p, _p, _p, _p]),
    "skm_confidence_hist": (_int, [_p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p]),
    "skm_confidence_classify": (_int, [_p, _p, _i64, _i64, _p, _p, _i64, _p, _p]),
    "skm_fasta_scan": (_int, [_p, _i64, _int, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "skm_fasta_pack": (_int, [_p, _i64, _int, _p, _p, _p, _p]),
    "skm_row_norm2_i32": (_int, [_p, _i64, _i64, _p, _p]),
    "skm_row_norm2_i64": (_int, [_p, _i64, _i64, _p, _p]),
    "skm_gather_columns": (_int, [_p, _i64, _i64, _int, _p, _i64, _p, _p]),
    "skm_pack_counts_u8": (_int, [_p, _i64, _i64, _int, _p, _p, _p, _p, _i64, _p, _p]),
    "skm_pack_presence_bits": (_int, [_p, _i64, _i64, _int, _p, _p]),
    "skm_rows_out_of_range_i32": (_int, [_p, _i64, _i64, C.c_int32, C.c_int32, _p, _i64, _p, _p]),
    "skm_bench_fma_f32": (_int, [_i64, _int, _p, C.POINTER(C.c_double), _p]),
    "skm_coo_pack": (_int, [_p, _p, _i64, _int, _p, _p, _p]),
    "skm_coo_merge_runs_packed_workspace": (_sz, [_i64, _int]),
    "skm_coo_merge_runs_packed": (_int, [_p, _p, _int, _int, _p, _p, _p, _p, _sz, _p]),
    "skm_peer_alloc": (_int, [_sz, C.POINTER(C.c_void_p), _p]),
    "skm_peer_open": (_int, [_p, C.POINTER(C.c_void_p)]),
    "skm_peer_close": (_int, [_p]),
    "skm_peer_free": (_int, [_p]),
    "skm_coo_pack_push": (_int, [_p, _p, _p, _int, _int, _p, _p, _p, _p]),
    "skm_rows_accumulate": (_int, [_p, _i64, _p, _i64, _p, _int, _int, _p, _i64, _p, _p]),
    "skm_rows_block": (_int, []),
    "skm_rows_block_counts": (_int, [_p, _i64, _i64, _p, _p]),
    "skm_rows_emit": (_int, [_p, _i64, _i64, _p, _p, _p, _p, _p, _i64, _p]),
    "skm_rows_colsum": (_int, [_p, _i64, _i64, _p, _p]),
    "skm_scatter_add_i64": (_int, [_p, _i64, _i64, _p, _p, _p, _i64, _i64, _p]),
    "skm_csv_f64_host": (_int, [C.c_double, C.c_char_p]),
    "skm_csv_rows_workspace": (_sz, [_i64]),
    "skm_csv_assoc_measure": (_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_csv_assoc_write": (_int, [_p, _i64, _i64, _i64, _p, _p, _p, _p, _p]),
    "skm_csv_top2_measure": (_int, [_p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_csv_top2_write": (_int, [_p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _p]),
    "skm_csv_counts_measure": (_int, [_p, _p, _i64, _i64, _p, _p, _p, _p, _int, _p, _p, _sz, _p]),
    "skm_csv_counts_write": (_int, [_p, _p, _p, _i64, _i64, _p, _p, _p, _p, _int, _p, _p, _p]),
    "skm_csv_parse_workspace": (_sz, [_i64]),
    "skm_csv_parse_rows": (_int, [_p, _i64, _p, _p, _p, _p, _sz, _p]),
    "skm_csv_parse_cells": (_int, [_p, _p, _p, _p, _i64, _p, _int, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
}


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise SkmError(-100, f"{LIB_PATH} is not built; run `python -m snekmer_b200.build` "
                                 "(nvcc, sm_100a). There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != SKM_OK:
        raise SkmError(rc, lib().skm_last_error().decode("utf-8", "replace"))


def lut_build(map_from: str, map_to: str, symbols: str):
    """Host-side 256-entry residue→symbol LUT (bytes object of length 256)."""
    buf = (C.c_uint8 * 256)()
    check(lib().skm_lut_build(map_from.encode("latin-1"), map_to.encode("latin-1"), len(map_from),
                              symbols.encode("latin-1"), len(symbols), buf))
    return bytes(buf)
