"""ctypes binding of libspotv2_gat.so (declared in include/spotv2_gat.h).

There is no fallback: if the library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libspotv2_gat.so"

_i32, _i64, _f32, _vp, _sz = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t


class GatDesc(C.Structure):
    """struct spotv2_gat_desc (include/spotv2_gat.h)."""
    _fields_ = [("B", _i32), ("N", _i32), ("F", _i32), ("Fe", _i32), ("H", _i32), ("C", _i32),
                ("R", _i32), ("concat", _i32), ("negative_slope", _f32), ("ldp", _i32),
                ("gemm_algo", _i32), ("attn_bwd_algo", _i32),
                ("dropout_p", _f32), ("edge_mode", _i32), ("dropout_seed_lo", C.c_uint32), ("dropout_seed_hi", C.c_uint32),
                ("p_format", _i32)]


class SpotV2Error(RuntimeError):
    pass


_DP = C.POINTER(GatDesc)
# name -> (restype, argtypes); every symbol include/spotv2_gat.h declares
SIGNATURES = {
    "spotv2_last_error": (C.c_char_p, []),
    "spotv2_abi_version": (_i32, []),
    "spotv2_gat_ldp": (_i32, [_i32, _i32]),
    "spotv2_gat_n_aug": (_i32, [_DP]),
    "spotv2_gat_pair_format_supported": (C.c_int, [_DP]),
    "spotv2_gat_head_pitch": (_i32, [_DP]),
    "spotv2_gat_workspace_bytes": (C.c_int, [_DP, C.POINTER(_sz), C.POINTER(_sz), C.POINTER(_sz)]),
    "spotv2_proj_fwd_pair": (C.c_int, [_DP] + [_vp] * 9 + [_sz, _vp]),
    "spotv2_gat_attn_fwd_pair": (C.c_int, [_DP] + [_vp] * 12),
    "spotv2_gat_attn_bwd_pair": (C.c_int, [_DP] + [_vp] * 16 + [_sz, _vp]),
    "spotv2_gat_attn_bwd_pair_dalpha": (C.c_int, [_DP] + [_vp] * 16 + [_sz, _vp, _vp]),
    "spotv2_edge_table_build": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp]),
    "spotv2_edge_table_dense": (C.c_int, [_i32, _vp, _vp]),
    "spotv2_gat_fold": (C.c_int, [_DP] + [_vp] * 8),
    "spotv2_gat_uses_tensor_cores": (C.c_int, [_DP]),
    "spotv2_gat_ld16": (_i32, [_i32]),
    "spotv2_split_f16": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp]),
    "spotv2_proj_fwd": (C.c_int, [_DP] + [_vp] * 8 + [_sz, _vp]),
    "spotv2_gat_attn_fwd_workspace_bytes": (C.c_int, [_DP, C.POINTER(_sz)]),
    "spotv2_gat_edge_terms_bytes": (C.c_int, [_DP, C.POINTER(_sz)]),
    "spotv2_gat_attn_fwd": (C.c_int, [_DP] + [_vp] * 9 + [_sz, _vp]),
    "spotv2_gat_attn_bwd": (C.c_int, [_DP] + [_vp] * 15 + [_sz, _vp]),
    "spotv2_gat_attn_bwd_dalpha": (C.c_int, [_DP] + [_vp] * 15 + [_sz, _vp, _vp]),
    "spotv2_gat_edge_rows_grad": (C.c_int, [_DP] + [_vp] * 5),
    "spotv2_edge_terms_from_windows_workspace_bytes": (C.c_int, [_DP, C.POINTER(_sz)]),
    "spotv2_edge_terms_from_windows": (C.c_int, [_DP, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "spotv2_windows_dv_workspace_bytes": (C.c_int, [_DP, C.POINTER(_sz)]),
    "spotv2_windows_dv": (C.c_int, [_DP, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "spotv2_proj_bwd_weight": (C.c_int, [_DP] + [_vp] * 10 + [_sz, _vp]),
    "spotv2_proj_bwd_input": (C.c_int, [_DP] + [_vp] * 7 + [_sz, _vp]),
    "spotv2_gat_unfold": (C.c_int, [_DP] + [_vp] * 13),
    "spotv2_alpha_to_pyg": (C.c_int, [_DP, _vp, _vp, _vp, _vp]),
    "spotv2_alpha_to_pyg_grad": (C.c_int, [_DP, _vp, _vp, _vp, _vp]),
    "spotv2_collate_windows": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp]),
    "spotv2_stack_scale": (C.c_int, [_vp, _i64, _vp, _vp]),
    "spotv2_collate_windows_pair": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "spotv2_diag_dout_pair_ws_bytes": (_sz, [_i32, _i32, _i32]),
    "spotv2_diag_dout_pair": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "spotv2_diag_counters": (C.c_int, [_vp, C.c_int]),
    "spotv2_diag_weight_grad_splits": (_i32, [_i32, _i32, _i32]),
    "spotv2_diag_gemm": (C.c_int, [C.c_int] * 5 + [_vp, C.c_int, _vp, C.c_int, _vp, C.c_int] + [C.c_int] * 4 + [_vp, _sz, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("SPOTV2_GAT_LIB", LIB_PATH))
    if not path.exists():
        raise SpotV2Error(
            f"{path} not found: build it with `python -m spotv2net_b200.build` "
            "(or __graft_entry__.build()).  spotv2net_b200 has no CPU or eager fallback.")
    lib = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.spotv2_abi_version() != 5:
        raise SpotV2Error(f"ABI version mismatch: library reports {lib.spotv2_abi_version()}, binding expects 5")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().spotv2_last_error()
        raise SpotV2Error(f"{what} failed (status {rc}): {msg.decode() if msg else '?'}")


def ptr(t: torch.Tensor | None):
    """Device pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "spotv2 kernels take contiguous tensors"
    return t.data_ptr()


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise SpotV2Error(
            f"{name} is on {t.device}: spotv2net_b200 runs on sm_100a CUDA devices only "
            "(no CPU fallback by design).")
    if t.dtype != torch.float32 and t.is_floating_point():
        raise SpotV2Error(f"{name} has dtype {t.dtype}; this build computes in float32")
