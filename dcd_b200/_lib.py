"""ctypes binding of libdcd_b200.so (the C ABI declared in include/dcd_b200.h and include/dcd_b200_grad.h).

There is no CPU fallback: if the library is missing or a tensor is not on a CUDA device the
call raises.  The library is built in-tree by `python -m dcd_b200.build` (or
`__graft_entry__.build()`); it has no torch dependency, tensors cross the boundary as raw
device pointers and the current CUDA stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

# DCD_B200_LIB selects a debug variant of the library built by `python -m dcd_b200.build --trace` (profiling aids only)
LIB_PATH = os.environ.get("DCD_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libdcd_b200.so")

# name -> (restype, argtypes); mirrors include/dcd_b200.h line by line
SIGNATURES = {
    "dcd_version": (c_int, []),
    "dcd_strerror": (c_char_p, [c_int]),
    "dcd_edge_solve_fwd": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_float, c_float, c_int, c_void_p, c_void_p, c_void_p]),
    "dcd_edge_select_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "dcd_edge_select_fwd": (c_int, [c_void_p] * 5 + [c_int64, c_int, c_int, c_float, c_float, c_int] + [c_void_p] * 5),
    "dcd_edge_solve_bwd": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_float, c_float, c_int, c_void_p, c_int] + [c_void_p] * 5),
    "dcd_dgde_locate_fwd": (c_int, [c_void_p] * 9 + [c_int64, c_int, c_float, c_float, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "dcd_dgde_frame_fwd": (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 6 + [c_void_p] * 4 + [c_int64, c_int, c_float, c_float, c_int, c_float]
                           + [c_void_p] * 5),
    "dcd_dgde_depth_ensemble_fwd": (c_int, [c_void_p] * 7 + [c_int64, c_float, c_float, c_float, c_float] + [c_void_p] * 6),
    "dcd_poi_gather_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    "dcd_poi_gather_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    "dcd_dgde_locate_bwd": (c_int, [c_void_p] * 6 + [c_int64, c_float] + [c_void_p] * 4),
    "dcd_dgde_depth_ensemble_bwd": (c_int, [c_void_p] * 7 + [c_int64, c_float, c_float, c_float, c_float] + [c_void_p] * 11),
    "dcd_gmw_ray_rescale_fwd": (c_int, [c_void_p] * 3 + [c_int64, c_void_p, c_void_p]),
    "dcd_gmw_param_count": (c_size_t, [c_int, c_int]),
    "dcd_gmw_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "dcd_gmw_weights_fwd": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int] + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "dcd_gmw_transport_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "dcd_gmw_transport_fwd": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_float, c_float, c_int] + [c_void_p] * 5 + [c_size_t, c_void_p]),
    "dcd_gmw_bwd_scratch_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "dcd_gmw_transport_bwd_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "dcd_gmw_transport_bwd": (c_int, [c_void_p] * 6 + [c_int64, c_int, c_float, c_int, c_float] + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "dcd_gmw_transport_terms_bwd": (c_int, [c_void_p] * 3 + [c_size_t] + [c_void_p] * 3 + [c_int64, c_int, c_float, c_int, c_float]
                                    + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "dcd_gmw_weights_bwd": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int] + [c_void_p] * 6 + [c_size_t, c_void_p, c_size_t, c_void_p]),
    "dcd_gmw_kpts_bwd": (c_int, [c_void_p] * 2 + [c_int64, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "dcd_gmw_aggregate_fwd": (c_int, [c_void_p] * 3 + [c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dcd_gmw_aggregate_bwd": (c_int, [c_void_p] * 3 + [c_int64, c_int64, c_int, c_int] + [c_void_p] * 4),
    "dcd_gmw_depth_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int64]),
    "dcd_gmw_depth_fwd": (c_int, [c_void_p] * 5 + [c_int64, c_int, c_int, c_int, c_float, c_float, c_int64]
                          + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "dcd_dgde_gmw_refine_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int64]),
    "dcd_dgde_gmw_refine_fwd": (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 6 + [c_void_p] * 6 + [c_int64, c_int, c_int, c_int, c_int64]
                                + [c_void_p] * 8 + [c_size_t, c_void_p]),
}

# name -> (restype, argtypes); mirrors include/dcd_b200_grad.h (backward of the fused frame-epilogue entry points)
GRAD_SIGNATURES = {
    "dcd_dgde_frame_bwd": (c_int, [c_void_p] * 3 + [c_int64] + [c_int] * 6 + [c_void_p] * 4 + [c_int64, c_int, c_float, c_float, c_int, c_float]
                           + [c_void_p] * 7),
    "dcd_dgde_locate_solve_bwd": (c_int, [c_void_p] * 8 + [c_int64, c_int, c_float, c_float, c_int, c_float] + [c_void_p] * 8),
    "dcd_gmw_ray_rescale_bwd": (c_int, [c_void_p] * 4 + [c_int64] + [c_void_p] * 4),
}

_lib = None


def load_library(path: str = LIB_PATH) -> ctypes.CDLL:
    """dlopen the library and attach the prototypes.  Works without a GPU (symbol checks only)."""
    if not os.path.exists(path):
        raise RuntimeError(
            "libdcd_b200.so is not built (%s missing): run `python -m dcd_b200.build`; "
            "dcd_b200 has no CPU or PyTorch fallback" % path)
    lib = ctypes.CDLL(path)
    for name, (res, args) in list(SIGNATURES.items()) + list(GRAD_SIGNATURES.items()):
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dcd_version() != 2:
        raise RuntimeError("libdcd_b200.so ABI version mismatch")
    return lib


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = load_library()
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError("%s failed: %s (rc=%d)" % (what, lib().dcd_strerror(rc).decode(), rc))


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("dcd_b200 ops need CUDA tensors (sm_100a kernels only, no CPU fallback); got %s" % t.device)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("dcd_b200 ops need all tensors on one device")
    if dev is None:
        raise RuntimeError("dcd_b200 ops need at least one CUDA tensor")
    if dev.index is not None and dev.index != torch.cuda.current_device():
        # the library launches on the CURRENT device and stream (include/dcd_b200.h)
        raise RuntimeError("dcd_b200 ops run on the current CUDA device (cuda:%d) but the tensors live on %s; "
                           "wrap the call in `with torch.cuda.device(t.device):`" % (torch.cuda.current_device(), dev))
    return dev


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def f32c(t: torch.Tensor) -> torch.Tensor:
    """FP32 contiguous view/copy (materialises stride-0 expands, casts float64 calibration)."""
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t.contiguous()
