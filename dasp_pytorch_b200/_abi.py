"""ctypes binding of libdasp_b200.so (the C ABI declared in include/dasp_b200.h).

There is no fallback: if the shared library is missing or fails to load, importing the
ops raises -- the product path never silently degrades to PyTorch/CPU code.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdasp_b200.so")

ABI_VERSION = 2


class DaspError(RuntimeError):
    """A C-ABI call returned a negative status."""


_lib = None


class ReverbGeom(ctypes.Structure):
    """mirror of ``dasp_reverb_geom`` (include/dasp_b200.h)"""

    _fields_ = [(name, c_int64) for name in (
        "nb", "hop", "nbk", "leff", "rpp", "conv_block", "x_blocks", "ir_partitions", "chunk_items",
        "f_floats", "xspec_c64", "irspec_c64", "wet_floats", "fwd_workspace_bytes", "bwd_workspace_bytes")]

P = c_void_p       # device pointer
I64 = c_int64

# name -> (restype, argtypes); mirrors include/dasp_b200.h one to one
_SIGNATURES = {
    "dasp_abi_version": (c_int, []),
    "dasp_last_error": (c_char_p, []),
    "dasp_compiled_arch": (c_int, []),
    "dasp_shutdown": (None, []),
    "dasp_debug_force_warps": (None, [c_int]),
    "dasp_debug_reverb_last_path": (c_int, []),
    "dasp_debug_reverb_flat_filterbank": (None, [c_int]),
    "dasp_denormalize": (c_int, [P, P, P, P, P, I64, I64, P]),
    "dasp_gain_fwd": (c_int, [P, P, P, I64, I64, I64, P]),
    "dasp_gain_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, I64, P]),
    "dasp_distortion_fwd": (c_int, [P, P, P, I64, I64, P]),
    "dasp_distortion_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, P]),
    "dasp_pointwise_bwd_workspace_floats": (I64, [I64, I64]),
    "dasp_stereo_bwd_workspace_floats": (I64, [I64, I64]),
    "dasp_widener_fwd": (c_int, [P, P, P, I64, I64, P]),
    "dasp_widener_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, P]),
    "dasp_panner_fwd": (c_int, [P, P, P, I64, I64, I64, P]),
    "dasp_panner_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, I64, P]),
    "dasp_bus_fwd": (c_int, [P, P, P, I64, I64, I64, P]),
    "dasp_bus_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, I64, P]),
    "dasp_eq_tile_len": (I64, [I64]),
    "dasp_eq_ckpt_floats": (I64, [I64, I64, I64]),
    "dasp_eq_bwd_workspace_floats": (I64, [I64, I64]),
    "dasp_eq_fwd": (c_int, [P, P, P, P, I64, I64, I64, c_float, P]),
    "dasp_eq_bwd": (c_int, [P, P, P, P, P, P, P, I64, I64, I64, I64, c_float, P]),
    "dasp_reverb_geometry": (c_int, [I64, I64, I64, I64, I64, ctypes.POINTER(ReverbGeom)]),
    "dasp_reverb_fwd": (c_int, [P, I64, P, P, P, P, P, P, P, P, P, I64, I64, I64, I64, I64, I64, c_float, P]),
    "dasp_reverb_bwd": (c_int, [P, P, I64, P, P, P, P, P, P, P, P, I64, I64, I64, I64, I64, I64, I64, P]),
    "dasp_reverb_filterbank": (c_int, [I64, c_double, ctypes.POINTER(c_float)]),
    "dasp_dynamics_tile_len": (I64, [I64, I64]),
    "dasp_dynamics_fwd": (c_int, [c_int, P, P, P, P, P, P, P, P, I64, I64, I64, c_float, c_float, I64, P]),
    "dasp_dynamics_bwd": (c_int, [c_int, P, P, P, P, P, P, P, P, P, P, P, I64, I64, I64, c_float, c_float, I64, P]),
}


def exported_symbols():
    """Names every build of the library must export (checked by the CPU test-suite)."""
    return sorted(_SIGNATURES)


def lib():
    """Load (once) and return the ctypes handle.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m dasp_pytorch_b200.build` "
            "(nvcc, sm_100a).  dasp_pytorch_b200 has no CPU / PyTorch fallback."
        )
    handle = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(handle, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    got = handle.dasp_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libdasp_b200.so ABI version {got}, python side expects {ABI_VERSION}")
    _lib = handle
    return _lib


def check(status: int, what: str):
    if status != 0:
        msg = lib().dasp_last_error()
        raise DaspError(f"{what} failed with status {status}: {msg.decode() if msg else '?'}")


def ptr(t: torch.Tensor | None):
    return None if t is None else t.data_ptr()


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    """The kernels take contiguous fp32 CUDA tensors; anything else is an explicit error
    (no silent host fallback)."""
    if not t.is_cuda:
        raise DaspError(
            f"{name}: dasp_pytorch_b200 runs on CUDA (B200) tensors only, got device {t.device}; "
            "there is no CPU path"
        )
    if t.dtype != torch.float32:
        raise DaspError(f"{name}: expected float32, got {t.dtype}")
    return t.contiguous()
