"""ctypes binding of libvet_b200.so (the C ABI declared in include/vet_b200.h).

There is no CPU fallback: if the shared library is missing or a symbol is
absent, loading raises, and every compute entry point needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

LIB_PATH = Path(__file__).resolve().parent / "_lib" / "libvet_b200.so"

VET_OK = 0
VET_ERR_INVALID_ARG = -1
VET_ERR_CUDA = -2
VET_ERR_UNSUPPORTED = -3
VET_ERR_NOMEM = -4

VET_F32, VET_F64 = 0, 1
VET_TRANSITION_LITERAL, VET_TRANSITION_TEXTBOOK = 0, 1
VET_MISSING = 0xFFFF
VET_FLAG_OUT_OF_RANGE, VET_FLAG_EMPTY_FRAME, VET_FLAG_NO_COMMON_USER = 1, 2, 4
VET_REGIME_AUTO, VET_REGIME_DIRECT = 0, 1
# vet_set_option: name -> (option id, {value name -> value})
# include/vet_b200.h VET_I8_MIN_FRAMES: frames per call from which the automatic dispatch of the weighted histogram
# takes the tensor-core kernel (tests/test_host_logic.py checks the two against each other)
I8_MIN_FRAMES = 384
# include/vet_b200.h VET_UT_SMEM_RECORDS: pair records of one user that vet_user_transitions sorts in shared memory;
# more go through global scratch (the tests cover both sides)
UT_SMEM_RECORDS = 3712

OPTIONS = {
    "weighted_kernel": (0, {"auto": 0, "fp64": 1, "i8": 2}),
    "stream_kernel": (1, {"auto": 0, "simple": 1, "cells": 2, "global": 3}),
    "transition_kernel": (2, {"auto": 0, "v1": 1, "v2": 2, "v3": 3}),
    "cluster_tail": (3, {"off": 0, "auto": 1, "force": 2}),
    "t3_pair_scratch": (4, {"off": 0, "on": 1}),
    "t3_assume_missing": (5, {"off": 0, "on": 1}),
    "analyze_overlap": (6, {"off": 0, "on": 1}),
    "host_batch_frames": (7, {"auto": 0}),
    "t4_list_cap": (8, {"auto": 0}),
    "cuda_graph": (9, {"off": 0, "on": 1}),
    "host_layout": (10, {"tuv": 0, "uv": 1}),
}


class VetConfig(C.Structure):
    """struct vet_config (include/vet_b200.h)."""
    _fields_ = [
        ("device", C.c_int32),
        ("video_width", C.c_int32),
        ("video_height", C.c_int32),
        ("num_tile_counts", C.c_int32),
        ("tile_counts", C.POINTER(C.c_int32)),
        ("fov_angle", C.c_double),
        ("power_factor", C.c_double),
        ("use_weight_distribution", C.c_int32),
        ("centres", C.POINTER(C.POINTER(C.c_double))),
        ("lon_by_px", C.POINTER(C.c_double)),
        ("lat_by_py", C.POINTER(C.c_double)),
        ("num_tiles", C.POINTER(C.c_int32)),
        ("naive_tile_width", C.c_int32),
        ("naive_tile_height", C.c_int32),
        ("regime", C.c_int32),
    ]


_P = C.c_void_p
_I64 = C.c_int64
# name -> (restype, argtypes); must list every symbol include/vet_b200.h declares
SYMBOLS = {
    "vet_last_error": (C.c_char_p, []),
    "vet_version": (C.c_char_p, []),
    "vet_set_option": (C.c_int, [_P, C.c_int, C.c_int]),
    "vet_get_option": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int)]),
    "vet_create": (C.c_int, [C.POINTER(_P), C.POINTER(VetConfig)]),
    "vet_destroy": (C.c_int, [_P]),
    "vet_num_tiles": (C.c_int, [_P, C.c_int]),
    "vet_num_cells": (_I64, [_P]),
    "vet_lattice": (C.c_int, [_P, C.c_int, _P]),
    "vet_cell_lut": (C.c_int, [_P, C.c_int, _P]),
    "vet_decode": (C.c_int, [_P, _P, C.c_int, _I64, _P, _P, _P]),
    "vet_nearest_tile": (C.c_int, [_P, C.c_int, _P, _I64, _P, _P]),
    "vet_tile_weights": (C.c_int, [_P, C.c_int, _P, _I64, _P, _P]),
    "vet_angular_distances": (C.c_int, [_P, C.c_int, _P, _I64, _P, _P]),
    "vet_vector_angles": (C.c_int, [_P, _P, _P, _I64, _P, _P]),
    "vet_spatial_vectors": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _P, _P]),
    "vet_transition_vectors": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _P, C.c_int, _P]),
    "vet_spatial": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P, _P]),
    "vet_transition": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P, C.c_int, _P]),
    "vet_analyze": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "vet_spatial_host": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P]),
    "vet_transition_host": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P, C.c_int]),
    "vet_analyze_host": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int]),
    "vet_users_accumulate": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _I64, _P, _P]),
    "vet_users_finish": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P, _P]),
    "vet_transition_counts_accumulate": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P]),
    "vet_transition_counts_finish": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "vet_user_transitions": (C.c_int, [_P, _P, C.c_int, _I64, _I64, _P, _P, _P, _P]),
    "vet_naive_points": (C.c_int, [_P, _P, _I64, _I64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "vet_poll_flags": (C.c_int, [_P, _P, C.POINTER(C.c_uint32)]),
    "vet_launch_count": (_I64, [_P]),
    "vet_graph_replays": (_I64, [_P]),
    "vet_profile_enable": (C.c_int, [_P, C.c_int]),
    "vet_profile_read": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
}
KERNEL_NAMES = ("stream", "epilogue", "transition", "transition_tail", "user_rows", "user_entropy")  # VET_KERNEL_* of vet_b200.h

_lib: Optional[C.CDLL] = None


class NativeLibraryError(RuntimeError):
    """The CUDA library is missing or incomplete (build it with
    `python __graft_entry__.py`)."""


def load_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("VET_B200_LIB", LIB_PATH))
    if not path.exists():
        raise NativeLibraryError(
            f"{path} not found: the CUDA extension is not built (run `python __graft_entry__.py`); "
            "there is no CPU fallback")
    lib = C.CDLL(str(path))
    for name, (restype, argtypes) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{path} does not export {name}") from e
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def last_error() -> str:
    return load_library().vet_last_error().decode("utf-8", "replace")
