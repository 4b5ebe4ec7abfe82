"""ctypes binding of libswb200.so -- the same C ABI (include/swb200.h) a Java host binds
through Panama FFM / JNI (INTEGRATION.md).  Loading never falls back to anything else:
a missing library or a missing CUDA device is an error."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libswb200.so")

SWB_OK = 0
SWB_F_SCORES_ONLY = 1
SWB_F_NO_FETCH = 2
SWB_F_TIE_GT = 4
SWB_F_BOTH_STRANDS = 8

# every symbol include/swb200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I64P = C.POINTER(C.c_int64)
_I32P = C.POINTER(C.c_int32)
SIGNATURES = {
    "swb_abi_version": (C.c_int, []),
    "swb_last_error": (C.c_char_p, []),
    "swb_device_count": (C.c_int, []),
    "swb_create": (C.c_int, [C.c_int, C.c_int64, C.POINTER(_P)]),
    "swb_destroy": (None, [_P]),
    "swb_refset_load": (C.c_int, [_P, C.c_int64, C.c_char_p, _I64P, C.POINTER(_P)]),
    "swb_refset_free": (None, [_P]),
    "swb_refset_count": (C.c_int64, [_P]),
    "swb_refset_total_bases": (C.c_int64, [_P]),
    "swb_reads_upload": (C.c_int, [_P, _P, C.c_int64, C.c_char_p, _I64P, C.POINTER(_P)]),
    "swb_reads_free": (None, [_P]),
    "swb_reads_count": (C.c_int64, [_P]),
    "swb_align": (C.c_int, [_P, _P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32,
                            C.c_uint32, C.POINTER(_P)]),
    "swb_align_resident": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.POINTER(_P)]),
    "swb_align_pair": (C.c_int, [_P, C.c_char_p, C.c_int64, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_uint32, C.POINTER(_P)]),
    "swb_queue_stats": (C.c_int, [_P, _I64P, C.c_int]),
    "swb_align_hits": (C.c_int, [_P, _P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_uint32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "swb_align_resident_hits": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_int32, C.c_int32,
                                          C.POINTER(_P)]),
    "swb_result_hits": (_I32P, [_P, _I32P]),
    "swb_align_all_hits": (C.c_int, [_P, _P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_uint32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "swb_align_resident_all_hits": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32, C.c_int32, C.c_int32,
                                              C.POINTER(_P)]),
    "swb_result_hit_offsets": (_I64P, [_P, _I64P]),
    "swb_result_hit_list": (_I32P, [_P]),
    "swb_result_fetch": (C.c_int, [_P]),
    "swb_result_free": (None, [_P]),
    "swb_result_n_refs": (C.c_int64, [_P]),
    "swb_result_n_reads": (C.c_int64, [_P]),
    "swb_result_scores": (_I32P, [_P]),
    "swb_result_ref_totals": (_I32P, [_P]),
    "swb_result_best_hits": (_I32P, [_P]),
    "swb_result_cell_offsets": (_I64P, [_P]),
    "swb_result_total_cells": (C.c_int64, [_P]),
    "swb_result_cells": (_I32P, [_P]),
    "swb_result_beginnings": (_I32P, [_P]),
    "swb_result_op_lens": (_I32P, [_P]),
    "swb_result_pair_cell_count": (C.c_int64, [_P, C.c_int64]),
    "swb_result_pair_cell": (C.c_int, [_P, C.c_int64, C.c_int64, _I32P, _I32P, _I32P, _I32P]),
    "swb_result_ops": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_uint8), C.c_int64]),
    "swb_result_materialize": (C.c_int, [_P, C.c_int64, C.c_char_p, C.c_int64, C.c_char_p, C.c_int64,
                                         C.c_char_p, C.c_char_p, C.c_int64]),
    "swb_result_stats": (C.c_int, [_P, C.POINTER(C.c_double), C.c_int]),
    "swb_result_device_ptr": (C.c_int, [_P, C.c_int, C.POINTER(_P), _I64P]),
    "swb_get_stream": (C.c_int, [_P, C.POINTER(_P)]),
    "swb_microbench_json": (C.c_int, [C.c_int, C.c_int, C.c_char_p, C.c_int]),
    # multi-GPU (single process, n devices)
    "swb_multi_create": (C.c_int, [_I32P, C.c_int32, C.c_int64, C.POINTER(_P)]),
    "swb_multi_destroy": (None, [_P]),
    "swb_multi_device_count": (C.c_int32, [_P]),
    "swb_multi_ctx": (_P, [_P, C.c_int32]),
    "swb_multi_refset_load": (C.c_int, [_P, C.c_int64, C.c_char_p, _I64P]),
    "swb_multi_ref_count": (C.c_int64, [_P]),
    "swb_multi_ref_location": (C.c_int, [_P, C.c_int64, _I32P, _I64P]),
    "swb_multi_shard_refs": (_I64P, [_P, C.c_int32, _I64P]),
    "swb_multi_align": (C.c_int, [_P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                  C.POINTER(_P)]),
    "swb_multi_result_free": (None, [_P]),
    "swb_multi_result_shard": (_P, [_P, C.c_int32]),
    "swb_multi_result_best_hits": (_I32P, [_P]),
    "swb_multi_align_hits": (C.c_int, [_P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                       C.c_int32, C.c_int32, C.POINTER(_P)]),
    "swb_multi_result_hits": (_I32P, [_P, _I32P]),
    "swb_multi_align_all_hits": (C.c_int, [_P, C.c_int64, C.c_char_p, _I64P, C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                           C.c_int32, C.c_int32, C.POINTER(_P)]),
    "swb_multi_result_hit_offsets": (_I64P, [_P, _I64P]),
    "swb_multi_result_hit_list": (_I32P, [_P]),
    "swb_multi_result_stats": (C.c_int, [_P, C.POINTER(C.c_double), C.c_int]),
    # multi-GPU (one process per device)
    "swb_comm_unique_id": (C.c_int, [C.c_char_p]),
    "swb_comm_create": (C.c_int, [_P, C.c_char_p, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "swb_comm_destroy": (None, [_P]),
    "swb_comm_allgather_best": (C.c_int, [_P, _P, _I64P, C.c_int64, _I32P]),
    "swb_comm_merged_device_ptr": (C.c_int, [_P, C.POINTER(_P), _I64P]),
    "swb_comm_allgather_hits": (C.c_int, [_P, _P, _I64P, C.c_int64, _I32P]),
    "swb_comm_allgather_all_hits": (C.c_int, [_P, _P, _I64P, C.c_int64, C.POINTER(_I64P), C.POINTER(_I32P), _I64P]),
}

_lib = None


class SwbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libswb200 error {code}: {msg}")
        self.code = code


def load():
    """Load the in-tree library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} is missing: run `python -m sparksmithwaterman_b200.build` "
                "(there is no CPU fallback for the CUDA path)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the ABI is incomplete
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != SWB_OK:
        raise SwbError(rc, (load().swb_last_error() or b"").decode("utf-8", "replace"))
