"""ctypes binding of the C-ABI library declared in ``include/veomni_b200.h``.

The product path has no CPU fallback: if the CUDA library is missing or a call fails,
:class:`VB200Error` is raised.  ``torch`` must be imported first so that the same
``libcudart.so.12`` is shared with PyTorch's streams and allocations.
"""

from __future__ import annotations

import ctypes
import re
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_void_p
from pathlib import Path

import torch  # noqa: F401  (loads libcudart before our library)

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libveomni_b200.so"
HEADER = PKG.parent / "include" / "veomni_b200.h"


class VB200Error(RuntimeError):
    pass


_lib = None

_F = c_float
_P = c_void_p
_I32 = c_int32
_I64 = c_int64

# name -> (restype, argtypes).  Kept next to the header; tests/test_abi.py checks that every
# symbol declared in include/veomni_b200.h is listed here and exported by the library.
SIGNATURES = {
    "vb200_abi_version": (c_int, []),
    "vb200_last_error": (c_char_p, []),
    "vb200_launch_count": (_I64, []),
    "vb200_reset_launch_count": (None, []),
    "vb200_rmsnorm_fwd": (c_int, [_P, _P, _P, _P, _I64, _I64, _F, _P]),
    "vb200_rmsnorm_bwd_partials": (_I64, [_I64, _I64]),
    "vb200_rmsnorm_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _P]),
    "vb200_rope": (c_int, [_P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _I32] + [_I64] * 8 + [_I32, _P]),
    "vb200_qknorm_rope_fwd": (c_int, [_P] * 10 + [_I64, _I32, _I32, _I32, _F, _P]),
    "vb200_qknorm_rope_bwd": (c_int, [_P] * 15 + [_I64, _I32, _I32, _I32, _P]),
    "vb200_qknorm_rope_bwd_partials": (_I64, [_I64]),
    "vb200_multi_sumsq_partials": (c_int64, [_I32]),
    "vb200_multi_sumsq": (c_int, [_P, _P, _I32, _I32, _P, _P, _P, _P]),
    "vb200_multi_scale": (c_int, [_P, _P, _I32, _I32, _P, _P]),
    "vb200_add_rmsnorm_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _I64, _I64, _F, _P]),
    "vb200_rmsnorm_bwd_add": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _P]),
    "vb200_multi_adamw": (c_int, [_P, _P, _P, _P, _P, _P, _I32, _I32, _F, _F, _F, _F, _F, _F, _F, _P, _P]),
    "vb200_cross_entropy": (c_int, [_P, _I32, _I64, _I64, _I64, _P, _I64, _P, _P, _I32, _P, _I64, _F, _P, _P, _P]),
    "vb200_count_valid_labels": (c_int, [_P, _I64, _I64, _P, _P]),
    "vb200_token_logprobs": (c_int, [_P, _I32, _I64, _I64, _I64, _P, _I64, _F, _P, _P, _P, _I32, _P, _P, _I32, _I32, _F,
                                     _P, _P, _P, _P]),
    "vb200_token_logprobs_bwd": (c_int, [_P, _I32, _I64, _I64, _I64, _P, _I64, _F, _P, _P, _P, _P, _P, _I32, _P, _P,
                                         _I32, _I32, _F, _P, _I64, _P]),
    "vb200_swiglu_fwd": (c_int, [_P, _P, _P, _I64, _I64, _I64, _I64, _P]),
    "vb200_swiglu_bwd": (c_int, [_P] * 5 + [_I64] * 5 + [_P]),
    "vb200_attn_varlen_fwd": (c_int, [_P] * 6 + [_I32] * 6 + [_P, _F, _I32, _P]),
    "vb200_attn_varlen_fwd_tc": (c_int, [_P] * 6 + [_I32] * 6 + [_P, _F, _I32, _P]),
    "vb200_attn_bwd_delta": (c_int, [_P, _P, _P, _I32, _I32, _I32, _I64, _I64, _I64, _I64, _P]),
    "vb200_attn_varlen_bwd_tc": (c_int, [_P] * 10 + [_I32] * 6 + [_P, _F, _I32, _P]),
    "vb200_attn_debug_trace": (c_int, [_P]),
    "vb200_attn_varlen_bwd": (c_int, [_P] * 11 + [_I32] * 6 + [_P, _F, _I32, _P]),
    "vb200_moe_route_workspace": (_I64, [_I64, _I32]),
    "vb200_moe_route": (c_int, [_P, _I32, _I64, _I32, _P, _P, _P, _P, _P]),
    "vb200_moe_scatter": (c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I64, _P]),
    "vb200_moe_gather": (c_int, [_P, _P, _P, _P, _I64, _I32, _I64, _P]),
    "vb200_moe_weight_grad": (c_int, [_P, _P, _P, _P, _I64, _I32, _I64, _P]),
    "vb200_group_gemm": (c_int, [_I32, _P, _P, _P, _P, _I32, _I64, _I32, _I32, _I32, _P]),
    "vb200_symm_alloc": (c_int, [ctypes.POINTER(_P), _I64]),
    "vb200_symm_free": (c_int, [_P]),
    "vb200_ipc_get_handle": (c_int, [_P, _P]),
    "vb200_ipc_open_handle": (c_int, [_P, ctypes.POINTER(_P)]),
    "vb200_ipc_close_handle": (c_int, [_P]),
    "vb200_comm_signal_bytes": (_I64, []),
    "vb200_comm_create": (c_int, [ctypes.POINTER(_P), _I32, _I32, ctypes.POINTER(_P), ctypes.POINTER(_P), _I64]),
    "vb200_comm_destroy": (c_int, [_P]),
    "vb200_comm_check": (c_int, [_P]),
    "vb200_comm_barrier": (c_int, [_P, _I32, _P]),
    "vb200_allgather": (c_int, [_P, _I32, _I64, _I64, _I32, _P]),
    "vb200_reduce_scatter_f32": (c_int, [_P, _I32, _I64, _I64, _F, _P, _I32, _P]),
    "vb200_reduce_scatter_bf16": (c_int, [_P, _I32, _I64, _I64, _F, _P, _I32, _P]),
    "vb200_allgather_scatter": (c_int, [_P, _I32, _I64, _I64, _P, _I32, _I32, _P]),
    "vb200_reduce_scatter_push_bf16": (c_int, [_P, _I32, _I64, _P, _I32, _I64, _F, _P, _I32, _P]),
    "vb200_fsdp_pack_bf16": (c_int, [_P, _I32, _I32, _I64, _P, _I32, _P]),
    "vb200_all_to_all": (c_int, [_P, _I32, _I64, _I32, _P, _I32, _P]),
    "vb200_chunk_pull": (c_int, [_P, _I32, _I64, _P, _I32, _P, _I32, _P]),
}


def declared_symbols() -> list[str]:
    """Function names declared in the public header (used by the ABI test)."""
    text = HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vb200_[a-z0-9_]+)\s*\(", text)))


def load() -> ctypes.CDLL:
    """Load (once) and return the library; raise loudly when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VB200Error(
            f"{LIB_PATH} is missing: build it with `python -m veomni_b200.build` "
            "(there is no CPU / PyTorch fallback for the veomni_b200 hot path)"
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    got = lib.vb200_abi_version()
    if got != 1:
        raise VB200Error(f"ABI version mismatch: library {got}, binding 1")
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = load().vb200_last_error().decode(errors="replace")
        raise VB200Error(f"{what} failed with code {code}: {msg}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
    return int(load().vb200_launch_count())


def reset_launch_count() -> None:
    load().vb200_reset_launch_count()
