"""ctypes binding of the C-ABI declared in ``include/b200_attn_mlp.h``.

There is no CPU or PyTorch fallback: if the shared library is missing this module raises on first use, and
every compute entry point fails with ``B200Error`` when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes
import os
import threading
from pathlib import Path
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_uint32, c_void_p, POINTER

from .build import LIB_PATH

c_int64_p = POINTER(c_int64)

B200_OK = 0
DTYPE_BF16, DTYPE_FP16 = 0, 1
ACT_NONE, ACT_GELU_TANH, ACT_GELU_ERF, ACT_RELU, ACT_SWIGLU = 0, 1, 2, 3, 4
KV_CONTIGUOUS, KV_PAGED = 0, 1

#: every symbol include/b200_attn_mlp.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "b200_version": (c_char_p, []),
    "b200_last_error": (c_char_p, []),
    "b200_arch_ok": (c_int, []),
    "b200_set_sm_limit": (c_int, [c_int]),
    "b200_set_gemm_group_rows": (c_int, [c_int]),
    "b200_launch_count": (c_int64, []),
    "b200_last_gemm_kernel": (c_char_p, []),
    "b200_last_kernel": (c_char_p, []),
    "b200_fa_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                            c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_float, c_int, c_int64, c_void_p, c_int,
                            c_void_p]),
    "b200_fa_fwd_accum": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_float, c_int, c_int64, c_void_p,
                                  c_int, c_int, c_void_p]),
    "b200_fa_fwd_paged": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int64_p,
                                  c_int64_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_float, c_int, c_int, c_void_p]),
    "b200_lse_merge": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int64_p, c_int,
                               c_void_p]),
    "b200_cast_out": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int64_p, c_int, c_void_p]),
    "b200_fa_decode_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "b200_fa_decode_num_splits": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "b200_fa_decode": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                               c_int, c_float, c_int, c_int64, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_int,
                               c_void_p, c_int64, c_int, c_void_p]),
    "b200_kv_append": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int64,
                               c_int64, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "b200_fa_decode_fp8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                   c_int, c_float, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int64,
                                   c_float, c_float, c_int, c_void_p]),
    "b200_kv_append_fp8": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                   c_int, c_int, c_int, c_int, c_float, c_float, c_int, c_void_p]),
    "b200_fused_mlp_workspace_bytes": (c_int64, [c_int64, c_int, c_int]),
    "b200_fused_mlp": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_int64, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_int64, c_int, c_void_p]),
    "b200_layernorm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_int64,
                               c_float, c_float, c_int, c_void_p]),
    "b200_tp_allreduce_flag_bytes": (c_int64, []),
    "b200_tp_allreduce": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_int, c_int64, c_int64, c_int64, c_uint32, c_void_p,
                                  c_int, c_int, c_int, c_void_p, c_void_p]),
    "b200_linear_act_workspace_bytes": (c_int64, [c_int64, c_int, c_int, c_int]),
    "b200_linear_act": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                c_int, c_int, c_int, c_void_p, c_int64, c_int, c_void_p]),
}


class B200Error(RuntimeError):
    """A C-ABI call returned a negative status."""

    def __init__(self, fn: str, code: int, message: str):
        super().__init__(f"{fn} failed ({code}): {message}")
        self.fn, self.code, self.message = fn, code, message


_lock = threading.Lock()
_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library (once). Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = LIB_PATH
        if os.environ.get("B200_LIB_PATH"):  # developer A/B runs only: another build of the SAME library (tests/*_probe.py)
            path = Path(os.environ["B200_LIB_PATH"]).resolve()
        if not path.exists():
            raise RuntimeError(
                f"{path} is missing: the sm_100a extension has not been built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` (or `python -m ml_inference_optimizer_b200.build`). "
                "There is deliberately no CPU / PyTorch fallback for the attention + FusedMLP hot path.")
        lib = ctypes.CDLL(str(path))
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the header and the library disagree
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def last_error() -> str:
    return (load().b200_last_error() or b"").decode("utf-8", "replace")


def check(fn_name: str, rc: int) -> None:
    if rc != B200_OK:
        raise B200Error(fn_name, rc, last_error())


def strides3(values) -> ctypes.Array:
    return (c_int64 * 3)(*[int(v) for v in values])
