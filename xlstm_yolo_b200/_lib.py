"""ctypes binding of ``lib/libmlstm_b200.so`` (C ABI: include/mlstm_b200.h).

There is no fallback: if the library is missing or does not export the expected symbols,
importing a CUDA op raises.  ``build.build()`` compiles it in-tree.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# MLSTM_B200_LIB: developer override for A/B builds (build.build_variant); the product path is the in-tree library
LIB_PATH = os.environ.get("MLSTM_B200_LIB") or os.path.join(_PKG, "lib", "libmlstm_b200.so")

ABI_VERSION = 6
MLSTM_F32, MLSTM_BF16 = 0, 1

STATUS = {0: "OK", -1: "INVALID_ARG", -2: "UNSUPPORTED", -3: "WORKSPACE", -4: "CUDA", -5: "NO_DEVICE"}

EXPORTS = (
    "mlstm_b200_abi_version",
    "mlstm_b200_workspace_bytes",
    "mlstm_b200_state_bytes",
    "mlstm_b200_fwd",
    "mlstm_b200_bwd",
    "mlstm_b200_bwd_part",
    "mlstm_b200_kernel_name",
    "mlstm_b200_kernel_variant",
    "mlstm_b200_qkv_supported",
    "mlstm_b200_qkv_fwd",
    "mlstm_b200_qkv_bwd_workspace_bytes",
    "mlstm_b200_qkv_bwd",
    "mlstm_b200_conv_bwd_workspace_bytes",
    "mlstm_b200_conv_bwd",
    "mlstm_b200_colsum_workspace_bytes",
    "mlstm_b200_colsum",
    "mlstm_b200_gates_supported",
    "mlstm_b200_gates_workspace_bytes",
    "mlstm_b200_gates_fwd_workspace_bytes",
    "mlstm_b200_gates_fwd",
    "mlstm_b200_gates_bwd",
    "mlstm_b200_glue_supported",
    "mlstm_b200_glue_workspace_bytes",
    "mlstm_b200_glue_fwd",
    "mlstm_b200_glue_bwd",
    "mlstm_b200_launch_count",
    "mlstm_b200_last_error",
)


class Act(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride_b", C.c_int64), ("stride_h", C.c_int64), ("stride_s", C.c_int64)]


class Gate(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride_b", C.c_int64), ("stride_h", C.c_int64), ("stride_s", C.c_int64)]


class Params(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("B", C.c_int32), ("NH", C.c_int32), ("S", C.c_int32),
        ("DHQK", C.c_int32), ("DHV", C.c_int32),
        ("dtype", C.c_int32), ("reverse", C.c_int32), ("chunk_size", C.c_int32),
        ("eps", C.c_float), ("qk_scale", C.c_float),
        ("q", Act), ("k", Act), ("v", Act),
        ("i", Gate), ("f", Gate),
        ("c_initial", C.c_void_p), ("n_initial", C.c_void_p), ("m_initial", C.c_void_p),
        ("h", Act),
        ("n_row", C.c_void_p), ("m_row", C.c_void_p),
        ("c_last", C.c_void_p), ("n_last", C.c_void_p), ("m_last", C.c_void_p),
        ("dh", Act),
        ("dq", Act), ("dk", Act), ("dv", Act),
        ("di", Gate), ("df", Gate),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("states", C.c_void_p), ("states_bytes", C.c_size_t),
        ("gate_mode", C.c_int32), ("reserved_", C.c_int32),
    ]


class GateProjParams(C.Structure):
    """ctypes mirror of ``mlstm_gate_proj_params`` (include/mlstm_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("T", C.c_int32), ("D", C.c_int32), ("NH", C.c_int32), ("dtype", C.c_int32),
        ("ld", C.c_int64),
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p),
        ("w_i", C.c_void_p), ("w_f", C.c_void_p), ("b_i", C.c_void_p), ("b_f", C.c_void_p),
        ("i", C.c_void_p), ("f", C.c_void_p),
        ("di", C.c_void_p), ("df", C.c_void_p),
        ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("ld_d", C.c_int64),
        ("dw_i", C.c_void_p), ("dw_f", C.c_void_p), ("db_i", C.c_void_p), ("db_f", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class GlueParams(C.Structure):
    """ctypes mirror of ``mlstm_glue_params`` (include/mlstm_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("T", C.c_int32), ("D", C.c_int32), ("NH", C.c_int32), ("dtype", C.c_int32),
        ("eps", C.c_float),
        ("h", C.c_void_p), ("ld_h", C.c_int64), ("c", C.c_void_p), ("ld_c", C.c_int64), ("z", C.c_void_p), ("ld_z", C.c_int64),
        ("w", C.c_void_p), ("b", C.c_void_p), ("skip", C.c_void_p),
        ("y", C.c_void_p), ("ld_y", C.c_int64), ("dy", C.c_void_p), ("ld_dy", C.c_int64),
        ("dh", C.c_void_p), ("ld_dh", C.c_int64), ("dc", C.c_void_p), ("ld_dc", C.c_int64), ("dz", C.c_void_p), ("ld_dz", C.c_int64),
        ("dw", C.c_void_p), ("db", C.c_void_p), ("dskip", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class QkvParams(C.Structure):
    """ctypes mirror of ``mlstm_qkv_params`` (include/mlstm_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("B", C.c_int32), ("GH", C.c_int32), ("GW", C.c_int32), ("D", C.c_int32), ("NH", C.c_int32),
        ("rotate", C.c_int32), ("x_dtype", C.c_int32),
        ("x", C.c_void_p), ("ld_x", C.c_int64),
        ("conv_w", C.c_void_p), ("conv_b", C.c_void_p),
        ("wq", C.c_void_p), ("wk", C.c_void_p), ("wv", C.c_void_p),
        ("bq", C.c_void_p), ("bk", C.c_void_p), ("bv", C.c_void_p),
        ("c", C.c_void_p), ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("sp", C.c_void_p),
    ]


class ConvBwdParams(C.Structure):
    """ctypes mirror of ``mlstm_conv_bwd_params`` (include/mlstm_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("B", C.c_int32), ("GH", C.c_int32), ("GW", C.c_int32), ("D", C.c_int32), ("NH", C.c_int32),
        ("rotate", C.c_int32), ("x_dtype", C.c_int32),
        ("x", C.c_void_p), ("ld_x", C.c_int64),
        ("dxc", C.c_void_p), ("dxv", C.c_void_p), ("sp", C.c_void_p),
        ("conv_w", C.c_void_p), ("dx", C.c_void_p), ("dwc", C.c_void_p), ("dbc", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


class QkvBwdParams(C.Structure):
    """ctypes mirror of ``mlstm_qkv_bwd_params`` (include/mlstm_b200.h)."""
    _fields_ = [
        ("abi_version", C.c_int32), ("T", C.c_int32), ("D", C.c_int32), ("NH", C.c_int32), ("x_dtype", C.c_int32),
        ("reserved_", C.c_int32),
        ("x", C.c_void_p), ("ld_x", C.c_int64),
        ("c", C.c_void_p), ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p), ("dc", C.c_void_p),
        ("wq", C.c_void_p), ("wk", C.c_void_p), ("wv", C.c_void_p),
        ("dxc", C.c_void_p), ("dxv", C.c_void_p),
        ("dwq", C.c_void_p), ("dwk", C.c_void_p), ("dwv", C.c_void_p), ("db", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


_lock = threading.Lock()
_lib = None


class LibraryMissing(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once). Raises LibraryMissing if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                f"{LIB_PATH} not found: build it with `python -m xlstm_yolo_b200.build` "
                "(there is no CPU or PyTorch fallback for CUDA tensors)")
        lib = C.CDLL(LIB_PATH)
        for name in EXPORTS:
            if not hasattr(lib, name):
                raise LibraryMissing(f"{LIB_PATH} does not export {name}")
        lib.mlstm_b200_abi_version.restype = C.c_int
        lib.mlstm_b200_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_workspace_bytes.argtypes = [C.POINTER(Params), C.c_int]
        lib.mlstm_b200_state_bytes.restype = C.c_size_t
        lib.mlstm_b200_state_bytes.argtypes = [C.POINTER(Params)]
        lib.mlstm_b200_fwd.restype = C.c_int
        lib.mlstm_b200_fwd.argtypes = [C.POINTER(Params), C.c_void_p]
        lib.mlstm_b200_bwd.restype = C.c_int
        lib.mlstm_b200_bwd.argtypes = [C.POINTER(Params), C.c_void_p]
        lib.mlstm_b200_bwd_part.restype = C.c_int
        lib.mlstm_b200_bwd_part.argtypes = [C.POINTER(Params), C.c_int, C.c_void_p]
        lib.mlstm_b200_kernel_name.restype = C.c_char_p
        lib.mlstm_b200_kernel_variant.restype = C.c_char_p
        lib.mlstm_b200_kernel_variant.argtypes = [C.POINTER(Params), C.c_int]
        lib.mlstm_b200_kernel_name.argtypes = [C.POINTER(Params), C.c_int]
        lib.mlstm_b200_gates_supported.restype = C.c_int
        lib.mlstm_b200_gates_supported.argtypes = [C.c_int, C.c_int64]
        lib.mlstm_b200_qkv_supported.restype = C.c_int
        lib.mlstm_b200_qkv_supported.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64]
        lib.mlstm_b200_qkv_bwd_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_qkv_bwd_workspace_bytes.argtypes = [C.POINTER(QkvBwdParams)]
        lib.mlstm_b200_qkv_bwd.restype = C.c_int
        lib.mlstm_b200_qkv_bwd.argtypes = [C.POINTER(QkvBwdParams), C.c_void_p]
        lib.mlstm_b200_conv_bwd_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_conv_bwd_workspace_bytes.argtypes = [C.POINTER(ConvBwdParams)]
        lib.mlstm_b200_conv_bwd.restype = C.c_int
        lib.mlstm_b200_conv_bwd.argtypes = [C.POINTER(ConvBwdParams), C.c_void_p]
        lib.mlstm_b200_colsum_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_colsum_workspace_bytes.argtypes = [C.c_int, C.c_int]
        lib.mlstm_b200_colsum.restype = C.c_int
        lib.mlstm_b200_colsum.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_size_t, C.c_void_p]
        lib.mlstm_b200_qkv_fwd.restype = C.c_int
        lib.mlstm_b200_qkv_fwd.argtypes = [C.POINTER(QkvParams), C.c_void_p]
        lib.mlstm_b200_glue_supported.restype = C.c_int
        lib.mlstm_b200_glue_supported.argtypes = [C.c_int, C.c_int]
        lib.mlstm_b200_gates_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_gates_workspace_bytes.argtypes = [C.POINTER(GateProjParams)]
        lib.mlstm_b200_gates_fwd_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_gates_fwd_workspace_bytes.argtypes = [C.POINTER(GateProjParams)]
        lib.mlstm_b200_gates_fwd.restype = C.c_int
        lib.mlstm_b200_gates_fwd.argtypes = [C.POINTER(GateProjParams), C.c_void_p]
        lib.mlstm_b200_gates_bwd.restype = C.c_int
        lib.mlstm_b200_gates_bwd.argtypes = [C.POINTER(GateProjParams), C.c_void_p]
        lib.mlstm_b200_glue_workspace_bytes.restype = C.c_size_t
        lib.mlstm_b200_glue_workspace_bytes.argtypes = [C.POINTER(GlueParams)]
        lib.mlstm_b200_glue_fwd.restype = C.c_int
        lib.mlstm_b200_glue_fwd.argtypes = [C.POINTER(GlueParams), C.c_void_p]
        lib.mlstm_b200_glue_bwd.restype = C.c_int
        lib.mlstm_b200_glue_bwd.argtypes = [C.POINTER(GlueParams), C.c_void_p]
        lib.mlstm_b200_launch_count.restype = C.c_uint64
        lib.mlstm_b200_last_error.restype = C.c_char_p
        if lib.mlstm_b200_abi_version() != ABI_VERSION:
            raise LibraryMissing(f"ABI mismatch: library {lib.mlstm_b200_abi_version()} vs binding {ABI_VERSION}")
        _lib = lib
    return _lib


def last_error() -> str:
    return load().mlstm_b200_last_error().decode("utf-8", "replace")


def launch_count() -> int:
    return int(load().mlstm_b200_launch_count())
