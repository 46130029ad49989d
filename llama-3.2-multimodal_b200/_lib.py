"""ctypes binding of the C-ABI library libl32ffn.so (include/l32_ffn.h).

There is deliberately NO fallback here: if the library is missing or a call fails, the caller gets an
exception.  (The PyTorch expressions in `modules.py` that serve fp32 / CPU tensors are the reference's own
semantics for those inputs, Model/model.py:165-171 and Tools/swiglu/FusedSwiglu.py:17-20 -- they are not a
fallback for the CUDA path.)
"""
from __future__ import annotations

import ctypes
import os
import re
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# L32_LIB_PATH: A/B experiments against another build of the same ABI (never set in production)
LIB_PATH = os.environ.get("L32_LIB_PATH") or os.path.join(_HERE, "libl32ffn.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "l32_ffn.h")

_lock = threading.Lock()
_lib = None

c_void_p, c_int, c_int64, c_size_t, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float

# name -> (restype, argtypes); mirrors include/l32_ffn.h one to one (tests/test_abi.py checks the header).
SIGNATURES = {
    "l32_abi_version": (c_int, []),
    "l32_kernel_launch_count": (ctypes.c_ulonglong, []),
    "l32_error_string": (ctypes.c_char_p, [c_int]),
    "l32_add_rmsnorm_forward": (c_int, [c_void_p] * 6 + [c_int64, c_int, c_float, c_int, c_void_p]),
    "l32_rmsnorm_backward_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "l32_rmsnorm_backward": (c_int, [c_void_p] * 7 + [c_size_t, c_int64, c_int, c_int, c_void_p]),
    "l32_rmsnorm_backward_add": (c_int, [c_void_p] * 9 + [c_size_t, c_int64, c_int, c_int, c_void_p]),
    "l32_swiglu_forward": (c_int, [c_void_p] * 8 + [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_swiglu_backward_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "l32_swiglu_backward": (c_int, [c_void_p] * 10 + [c_size_t, c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_linear_forward": (c_int, [c_void_p] * 4 + [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_linear_group_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p]),
    "l32_ffn_forward": (c_int, [c_void_p] * 11 + [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_block_tail_forward": (c_int, [c_void_p] * 3 + [c_float] + [c_void_p] * 6 + [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_block_tail_forward_ex": (c_int, [c_void_p] * 3 + [c_float] + [c_void_p] * 11 + [c_float] + [c_void_p] * 2 +
                                  [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_linear_lora_forward": (c_int, [c_void_p] * 8 + [c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_linear_lora_backward": (c_int, [c_void_p] * 11 + [c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_lm_head_ce_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "l32_lm_head_ce_forward": (c_int, [c_void_p] * 3 + [ctypes.c_longlong] + [c_void_p] * 5 + [c_size_t, c_int64, c_int, c_int, c_int,
                                                                                             c_void_p]),
    "l32_lm_head_ce_backward": (c_int, [c_void_p] * 3 + [ctypes.c_longlong, c_void_p, c_void_p] + [c_void_p] * 5 +
                                [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_rope_kv_append": (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_float, c_int, c_void_p]),
    "l32_gqa_attention_workspace_bytes": (c_size_t, [c_int] * 6),
    "l32_gqa_attention_forward": (c_int, [c_void_p] * 6 + [c_size_t] + [c_int] * 10 + [c_void_p]),
    "l32_gqa_attention_forward_train": (c_int, [c_void_p] * 6 + [c_int] * 8 + [c_void_p]),
    "l32_gqa_attention_backward_workspace_bytes": (c_size_t, [c_int] * 3),
    "l32_gqa_attention_backward": (c_int, [c_void_p] * 12 + [c_size_t] + [c_int] * 7 + [c_float, c_int, c_void_p]),
    "l32_rope_kv_append_paged": (c_int, [c_void_p] * 9 + [c_int] * 7 + [c_float, c_int, c_void_p]),
    "l32_gqa_attention_forward_paged": (c_int, [c_void_p] * 8 + [c_size_t] + [c_int] * 9 + [c_void_p]),
    "l32_ffn_backward_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "l32_ffn_backward": (c_int, [c_void_p] * 12 + [c_size_t, c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_ffn_lora_forward": (c_int, [c_void_p] * 11 + [c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_ffn_lora_backward_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "l32_ffn_lora_backward": (c_int, [c_void_p] * 16 + [c_size_t, c_int64, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_gemm": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_int64, c_void_p, c_int64,
                         c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_debug_tile_order": (c_int, [c_int, c_int, c_void_p, c_void_p]),
    "l32_debug_gemm_plan": (c_int, [c_int] * 6 + [c_void_p]),
    "l32_swiglu_act": (c_int, [c_void_p] * 3 + [c_int64, c_int, c_void_p]),
    "l32_tp_peer_copy": (c_int, [c_void_p, c_void_p, c_size_t, c_int, c_int, c_int, c_int, c_void_p]),
    "l32_tp_signal": (c_int, [c_void_p, c_int, c_int, ctypes.c_uint32, c_void_p, c_void_p]),
    "l32_tp_swiglu_forward_allgather": (c_int, [c_void_p] * 4 + [ctypes.c_uint32, c_int, c_int, c_int64] + [c_void_p] * 7 +
                                        [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_tp_linear_forward_reduce_scatter": (c_int, [c_void_p] * 3 + [c_int, c_int, c_int64, c_int64, c_int, c_int, c_int,
                                                                      c_void_p]),
    "l32_tp_ffn_backward_dact_allgather": (c_int, [c_void_p] * 4 + [ctypes.c_uint32, c_int, c_int, c_int64] + [c_void_p] * 6 +
                                           [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_tp_ffn_backward_dx_reduce_scatter": (c_int, [c_void_p] * 5 + [c_int, c_int, c_int64, c_int64, c_int, c_int, c_int,
                                                                       c_void_p]),
    "l32_tp_linear_group_forward_allgather": (c_int, [c_void_p] * 4 + [ctypes.c_uint32, c_int, c_int, c_int64] + [c_void_p] * 3 +
                                              [c_int, c_int64, c_int, c_int, c_void_p]),
    "l32_tp_linear_forward_allgather": (c_int, [c_void_p] * 4 + [ctypes.c_uint32, c_int, c_int, c_int64, c_void_p, c_int, c_void_p,
                                                                 c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_tp_linear_group_backward_dx_reduce_scatter": (c_int, [c_void_p] * 3 + [c_int, c_void_p, c_int, c_int, c_int64, c_int64,
                                                                                c_int, c_int, c_void_p]),
    "l32_tp_ffn_forward_fused": (c_int, [c_void_p] * 4 + [ctypes.c_uint32, c_int, c_int, c_int64] + [c_void_p] * 6 +
                                 [c_int64, c_int, c_int, c_int, c_void_p]),
    "l32_tp_reduce_partials": (c_int, [c_void_p, c_void_p, ctypes.c_uint32, c_int, c_int, c_void_p, c_void_p, c_int64,
                                       c_int64, c_int, c_int, c_void_p]),
}


class L32Error(RuntimeError):
    """Raised when a C-ABI call returns a non-zero code."""


def header_symbols() -> list[str]:
    """Every function name declared in include/l32_ffn.h."""
    with open(HEADER_PATH) as f:
        text = f.read()
    return sorted(set(re.findall(r"L32_API\s+[\w\s\*]+?\b(l32_\w+)\s*\(", text)))


def lib() -> ctypes.CDLL:
    """Load (once) and return the C-ABI library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise L32Error(
                    f"{LIB_PATH} not found: build it with `python setup.py build_ext --inplace` "
                    "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback "
                    "for the CUDA path.")
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            got = handle.l32_abi_version()
            if got != ABI_VERSION:
                raise L32Error(f"{LIB_PATH} has ABI version {got}, this package needs {ABI_VERSION}: rebuild the library "
                               "(python -c 'import __graft_entry__ as g; g.build()')")
            _lib = handle
    return _lib


ABI_VERSION = 3   # must match l32_abi_version() of the loaded library (include/l32_ffn.h)


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().l32_error_string(code)
        raise L32Error(f"{what} failed with code {code}: {msg.decode() if msg else '?'}")
