"""ctypes binding of include/lanpaint_b200.h.

There is deliberately no fallback: if the library is missing or a call fails
the caller gets an exception.  (The product never routes through `oracle/`.)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_LIB_PATH = os.environ.get("LANPAINT_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib",
                                                               "liblanpaint_b200.so")

ABI_VERSION = 6
TABLE_STRIDE = 32

RNG_TAPE, RNG_PHILOX, RNG_TORCH = 0, 1, 2
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
T_INVS = 2  # LP_T_INVS
SUBSTEP_FIRST, SUBSTEP_FUSE_NEXT, SUBSTEP_STORE_C, SUBSTEP_MERGE_NOISE = 1, 2, 4, 8

# every symbol include/lanpaint_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = (
    "lp_abi_version", "lp_status_string", "lp_last_cuda_error", "lp_set_option", "lp_selftest_index_math", "lp_selftest_box_muller", "lp_build_coef_table", "lp_build_coef_table_dt",
    "lp_torch_randn_geometry", "lp_pack_mask_f32", "lp_prologue_f32", "lp_substep", "lp_substep_f32", "lp_substep_cfg_f32", "lp_advance_f32",
    "lp_boundary", "lp_synth_denoiser",
    "lp_epilogue_f32", "lp_epilogue_euler_f32", "lp_step_boundary_f32", "lp_epilogue_cfg_f32", "lp_stop_stats_f32", "lp_fill_normal_f32", "lp_synth_denoiser_f32", "lp_torch_cpu_randn_f32",
)


class NativeError(RuntimeError):
    pass


class Hyper(C.Structure):
    _fields_ = [("step_size", C.c_double), ("lam", C.c_double), ("beta", C.c_double),
                ("min_step_frac", C.c_double), ("flow", C.c_int32), ("reserved", C.c_int32)]


class Heads(C.Structure):
    """lp_heads: the model's prediction(s) of one call (x0 / x0_BIG, or raw cond / uncond with combine=1)."""
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("dtype", C.c_int32), ("combine", C.c_int32),
                ("cfg", C.c_float), ("cfg_big", C.c_float)]


class Dims(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("per_row", C.c_int64), ("spatial", C.c_int64),
                ("mask_row_stride", C.c_int64), ("mask_channel_stride", C.c_int64), ("row_split", C.c_int64)]


class Rng(C.Structure):
    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("tape0", C.c_void_p), ("tape1", C.c_void_p),
                ("seed", C.c_uint64), ("draw0", C.c_uint64), ("draw1", C.c_uint64), ("state", C.c_void_p)]


_lib: Optional[C.CDLL] = None


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load (once) and type the library.  Raises NativeError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise NativeError(
            f"{_LIB_PATH} is missing: build it with `python -m lanpaint_b200.build` "
            "(nvcc, sm_100a).  lanpaint_b200 has no CPU or eager-PyTorch fallback.")
    lib = C.CDLL(_LIB_PATH)
    p, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int
    lib.lp_abi_version.restype = i32
    lib.lp_abi_version.argtypes = []
    lib.lp_status_string.restype = C.c_char_p
    lib.lp_status_string.argtypes = [i32]
    lib.lp_last_cuda_error.restype = i32
    lib.lp_last_cuda_error.argtypes = []
    lib.lp_set_option.restype = i32
    lib.lp_set_option.argtypes = [C.c_char_p, i32]
    lib.lp_selftest_index_math.restype = i64
    lib.lp_selftest_index_math.argtypes = [i64]
    lib.lp_selftest_box_muller.restype = i32
    lib.lp_selftest_box_muller.argtypes = [i64, u64, p, p]
    lib.lp_build_coef_table.restype = i32
    lib.lp_build_coef_table.argtypes = [p, p, p, p, p, i64, C.POINTER(Hyper), p]
    lib.lp_build_coef_table_dt.restype = i32
    lib.lp_build_coef_table_dt.argtypes = [p, p, p, p, C.c_double, C.c_int32, i64, p]
    lib.lp_torch_randn_geometry.restype = i32
    lib.lp_torch_randn_geometry.argtypes = [i64, i32, C.POINTER(i64), C.POINTER(u64)]
    lib.lp_pack_mask_f32.restype = i32
    lib.lp_pack_mask_f32.argtypes = [p, p, i64, i32, p]
    lib.lp_prologue_f32.restype = i32
    lib.lp_prologue_f32.argtypes = [p, p, p, p, p, p, p, C.POINTER(Dims), p]
    lib.lp_substep.restype = i32
    lib.lp_substep.argtypes = [p, C.POINTER(Heads), p, p, p, p, p, p, C.POINTER(Dims), C.POINTER(Rng), i32, p]
    lib.lp_boundary.restype = i32
    lib.lp_boundary.argtypes = [C.POINTER(Heads), p, p, p, p, p, C.c_float, p, C.POINTER(Dims), p]
    lib.lp_synth_denoiser.restype = i32
    lib.lp_synth_denoiser.argtypes = [p, p, p, i32, i64, p, p]
    lib.lp_substep_f32.restype = i32
    lib.lp_substep_f32.argtypes = [p, p, p, p, p, p, p, p, p, C.POINTER(Dims), C.POINTER(Rng), i32, p]
    lib.lp_substep_cfg_f32.restype = i32
    lib.lp_substep_cfg_f32.argtypes = [p, p, p, C.c_float, C.c_float, p, p, p, p, p, p, C.POINTER(Dims), C.POINTER(Rng),
                                       i32, p]
    lib.lp_epilogue_cfg_f32.restype = i32
    lib.lp_epilogue_cfg_f32.argtypes = [p, p, C.c_float, p, p, p, p, C.c_float, C.POINTER(Dims), p]
    lib.lp_advance_f32.restype = i32
    lib.lp_advance_f32.argtypes = [p, p, p, p, C.POINTER(Dims), C.POINTER(Rng), i32, p]
    lib.lp_epilogue_f32.restype = i32
    lib.lp_epilogue_f32.argtypes = [p, p, p, p, C.POINTER(Dims), p]
    lib.lp_epilogue_euler_f32.restype = i32
    lib.lp_epilogue_euler_f32.argtypes = [p, p, p, p, p, C.c_float, C.POINTER(Dims), p]
    lib.lp_step_boundary_f32.restype = i32
    lib.lp_step_boundary_f32.argtypes = [p, p, p, p, p, p, C.c_float, p, C.POINTER(Dims), p]
    lib.lp_stop_stats_f32.restype = i32
    lib.lp_stop_stats_f32.argtypes = [p, p, p, p, p, C.POINTER(Dims), p, p]
    lib.lp_fill_normal_f32.restype = i32
    lib.lp_fill_normal_f32.argtypes = [p, i64, C.POINTER(Rng), p]
    lib.lp_synth_denoiser_f32.restype = i32
    lib.lp_synth_denoiser_f32.argtypes = [p, p, p, i64, p, p]
    lib.lp_torch_cpu_randn_f32.restype = i32
    lib.lp_torch_cpu_randn_f32.argtypes = [p, i64, u64, p, C.POINTER(i64), p]
    v = lib.lp_abi_version()
    if v != ABI_VERSION:
        raise NativeError(f"ABI mismatch: library {v}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        lib = load()
        msg = lib.lp_status_string(rc).decode()
        raise NativeError(f"{what}: {msg} (status {rc}, cudaError {lib.lp_last_cuda_error()})")
