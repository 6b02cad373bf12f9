"""ctypes binding of ``libtgp_b200.so`` (the C ABI declared in ``include/tgp_b200.h``).

There is NO fallback: if the shared library is missing, or a tensor is not a
contiguous CUDA tensor, the call raises.  Signatures carry plain pointers and sizes
only; torch is used for device memory and the current stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_size_t, c_uint32, c_void_p
from typing import Optional

import torch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libtgp_b200.so")
_lib = None

F32, BF16 = 0, 1
SUM, MEAN, MAX, MIN, MUL = 0, 1, 2, 3, 4
OPS = {"sum": SUM, "add": SUM, "mean": MEAN, "max": MAX, "min": MIN, "mul": MUL}
REMOVE_SELF_LOOPS, DEGREE_NORM, ADJ_TRANSPOSE, EDGE_WEIGHT_NORM, HAS_WEIGHT = 1, 2, 4, 8, 16

_ERR = {-1: "invalid argument", -2: "workspace too small", -3: "CUDA launch failed", -4: "unsupported shape/dtype"}

# name -> (restype, argtypes); mirrors include/tgp_b200.h one to one
_P, _I64, _SZ, _INT, _U32, _F = c_void_p, c_int64, c_size_t, c_int, c_uint32, c_float
SIGNATURES = {
    "tgpb200_abi_version": (_INT, []),
    "tgpb200_debug_launch_count": (ctypes.c_longlong, []),
    "tgpb200_debug_time_kernel": (None, [ctypes.c_char_p]),
    "tgpb200_debug_kernel_time_ms": (ctypes.c_double, [ctypes.POINTER(ctypes.c_int)]),
    "tgpb200_debug_kernel_times": (_SZ, [ctypes.c_char_p, _SZ]),
    "tgpb200_build_csr_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_build_csr": (_INT, [_P, _I64, _I64, _P, _P, _P, _SZ, _P]),
    "tgpb200_segment_reduce_fwd": (_INT, [_P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _INT, _INT, _P, _P]),
    "tgpb200_segment_reduce_bwd_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I64, _INT]),
    "tgpb200_segment_reduce_bwd": (
        _INT,
        [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _INT, _INT, _P, _P, _P, _SZ, _P],
    ),
    "tgpb200_reduce_batch": (_INT, [_P, _P, _P, _P, _I64, _P, _P]),
    "tgpb200_filter_relabel_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_filter_relabel_count": (_INT, [_P, _P, _P, _I64, _P, _I64, _I64, _U32, _F, _P, _P, _SZ, _P]),
    "tgpb200_filter_relabel_emit": (_INT, [_P, _P, _P, _I64, _I64, _U32, _F, _P, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_filter_relabel_onepass_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_filter_relabel_onepass": (_INT, [_P, _P, _P, _I64, _P, _I64, _I64, _U32, _F, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_filter_relabel_bwd": (_INT, [_P, _P, _I64, _P, _I64, _P, _P]),
    "tgpb200_remap_coalesce_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_remap_coalesce_count": (_INT, [_P, _P, _P, _I64, _P, _I64, _I64, _INT, _U32, _F, _P, _P, _SZ, _P]),
    "tgpb200_remap_coalesce_emit": (_INT, [_I64, _I64, _INT, _U32, _F, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_coalesce_bwd_workspace_bytes": (_SZ, [_I64, _I64, _INT]),
    "tgpb200_coalesce_bwd": (_INT, [_P, _P, _P, _P, _P, _P, _I64, _I64, _INT, _P, _P, _SZ, _P]),
    "tgpb200_bucket_coalesce_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "tgpb200_bucket_coalesce_plan": (_INT, [_P, _I64, _P, _P, _P, _I64, _I64, _P, _P, _SZ, _P]),
    "tgpb200_bucket_coalesce_count": (
        _INT, [_P, _P, _P, _I64, _P, _P, _P, _I64, _I64, _INT, _U32, _F, _I64, _I64, _INT, _P, _P, _SZ, _P]),
    "tgpb200_bucket_coalesce_emit": (_INT, [_I64, _I64, _I64, _INT, _I64, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_edge_norm_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_rows_sorted": (_INT, [_P, _I64, _P, _P]),
    "tgpb200_degree_norm_fwd": (_INT, [_P, _P, _P, _I64, _P, _I64, _F, _INT, _P, _P, _P, _SZ, _P]),
    "tgpb200_degree_norm_bwd": (_INT, [_P, _P, _P, _P, _P, _I64, _P, _I64, _F, _INT, _P, _P, _P, _SZ, _P]),
    "tgpb200_degree_accumulate": (_INT, [_P, _P, _I64, _P, _I64, _INT, _P, _P, _SZ, _P]),
    "tgpb200_degree_apply": (_INT, [_P, _P, _P, _P, _I64, _P, _I64, _F, _P, _P]),
    "tgpb200_degree_bwd_accumulate": (_INT, [_P, _P, _P, _P, _P, _I64, _P, _I64, _F, _INT, _P, _P, _SZ, _P]),
    "tgpb200_degree_bwd_apply": (_INT, [_P, _P, _P, _P, _P, _I64, _P, _I64, _F, _P, _P]),
    "tgpb200_weight_max_accumulate": (_INT, [_P, _P, _P, _I64, _P, _I64, _P, _P]),
    "tgpb200_weight_max_apply": (_INT, [_P, _P, _P, _P, _I64, _P, _I64, _P, _P]),
    "tgpb200_weight_norm_fwd": (_INT, [_P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P]),
    "tgpb200_weight_norm_bwd": (_INT, [_P, _P, _P, _P, _P, _P, _I64, _P, _I64, _I64, _INT, _P, _P, _P, _SZ, _P]),
    "tgpb200_tc_gemm": (
        _INT,
        [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _INT, _I64, _I64, _INT, _I64, _I64, _I64, _INT, _INT, _F, _INT, _P],
    ),
    "tgpb200_bmm": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _I64, _I64, _INT, _I64, _I64, _INT, _INT, _P]),
    "tgpb200_topk_select_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_topk_select": (_INT, [_P, _P, _I64, _I64, _F, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_block_diag_workspace_bytes": (_SZ, [_I64, _I64]),
    "tgpb200_block_diag_count": (_INT, [_P, _P, _I64, _I64, _INT, _F, _P, _P, _P, _SZ, _P]),
    "tgpb200_block_diag_emit": (_INT, [_P, _P, _I64, _I64, _INT, _F, _P, _P, _P, _P, _P, _SZ, _P]),
    "tgpb200_block_diag_bwd": (_INT, [_P, _P, _I64, _I64, _INT, _P, _P]),
    "tgpb200_graph_ptr": (_INT, [_P, _I64, _I64, _P, _P, _SZ, _P]),
    "tgpb200_to_dense_batch": (_INT, [_P, _P, _P, _I64, _I64, _I64, _I64, _INT, _P, _P, _P]),
    "tgpb200_to_dense_adj": (_INT, [_P, _P, _P, _P, _P, _I64, _I64, _I64, _INT, _P, _P]),
    "tgpb200_dense_pool_saved_bytes": (_SZ, [_I64, _I64, _I64]),
    "tgpb200_dense_pool_bwd_workspace_bytes": (_SZ, [_I64, _I64, _I64, _INT]),
    "tgpb200_dense_pool_fwd": (
        _INT,
        [_P, _P, _P, _I64, _I64, _I64, _I64, _INT, _U32, _INT, _F, _F, _F, _P, _P, _P, _P, _SZ, _P],
    ),
    "tgpb200_dense_pool_bwd": (
        _INT,
        [_P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _U32, _INT, _F, _F, _F, _P, _P, _P, _P, _SZ, _P, _SZ, _P],
    ),
    "tgpb200_dense_pool_fwd_v2": (
        _INT,
        [_P, _P, _P, _I64, _I64, _I64, _I64, _INT, _U32, _INT, _F, _F, _F, _P, _P, _P, _P, _SZ, _P, _P],
    ),
    "tgpb200_dense_pool_bwd_v2": (
        _INT,
        [_P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I64, _INT, _U32, _INT, _F, _F, _F, _P, _P, _P, _P, _SZ, _P, _SZ, _P,
         _P],
    ),
}


def lib_path() -> str:
    return _LIB_PATH


def load() -> ctypes.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(_LIB_PATH):
            raise RuntimeError(
                f"tgp_b200: {_LIB_PATH} not found. Build it with "
                "`bash torch-geometric-pool_b200/csrc/build.sh` (or __graft_entry__.build()). "
                "There is no CPU / eager fallback."
            )
        lib = ctypes.CDLL(_LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a contiguous CUDA tensor (None stays NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("tgp_b200 kernels need CUDA tensors (there is no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("tgp_b200: tensor must be contiguous")
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise RuntimeError(f"tgp_b200: unsupported dtype {dt} (float32 and bfloat16 only)")


def workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"tgp_b200.{what} failed: {_ERR.get(rc, rc)}")


def kernel_launches() -> int:
    """Kernels launched by libtgp_b200.so in this process so far."""
    return int(load().tgpb200_debug_launch_count())


def time_kernel(name_filter: Optional[str]) -> None:
    """Bracket every kernel whose name contains ``name_filter`` with CUDA events (None stops)."""
    load().tgpb200_debug_time_kernel(None if name_filter is None else name_filter.encode())


def kernel_time_ms():
    """(mean ms, launches) of the kernels recorded since ``time_kernel``."""
    n = ctypes.c_int(0)
    ms = load().tgpb200_debug_kernel_time_ms(ctypes.byref(n))
    return float(ms), int(n.value)


def kernel_trace() -> list:
    """[(kernel name, ms)] in launch order for the launches recorded since ``time_kernel("*")``."""
    buf = ctypes.create_string_buffer(1 << 20)
    load().tgpb200_debug_kernel_times(buf, len(buf))
    out = []
    for line in buf.value.decode().splitlines():
        name, ms = line.split("\t")
        out.append((name, float(ms)))
    return out


_NVTX = os.environ.get("TGPB200_NVTX", "0") == "1"


def call(name: str, *args) -> None:
    """One C-ABI entry point.  ``TGPB200_NVTX=1`` brackets every call with an NVTX range named after the entry point
    (the dispatcher ops of ``libtgp_b200_ops.so`` are visible to ``torch.autograd.profiler.emit_nvtx`` as usual)."""
    if _NVTX:
        torch.cuda.nvtx.range_push(name)
        try:
            check(getattr(load(), name)(*args), name)
        finally:
            torch.cuda.nvtx.range_pop()
        return
    check(getattr(load(), name)(*args), name)
