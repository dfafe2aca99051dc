"""ctypes binding of libvitb200.so (the C ABI in include/vitb200.h).

There is no fallback: if the library is missing, or a call is made without a CUDA device, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VITB_LIB_PATH") or os.path.join(HERE, "libvitb200.so")  # (override: A/B builds of experiments)

F32 = 0
BF16 = 1

GEMM_GELU = 1
GEMM_OUT_F32 = 2
GEMM_DY_F32 = 4

ABI_VERSION = 1

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_f = C.c_float
_sz = C.c_size_t

class DropoutDesc(C.Structure):
    """vitb_dropout_t (include/vitb200.h): one nn.Dropout site for the fused kernels."""
    _fields_ = [("p", C.c_float), ("seed", C.c_uint64), ("site", C.c_uint32), ("step", C.c_uint32), ("step_dev", C.c_void_p)]


_dp = C.POINTER(DropoutDesc)

# name -> (restype, argtypes); mirrors include/vitb200.h exactly (checked by tests/test_abi.py)
SIGNATURES = {
    "vitb_version": (_i, []),
    "vitb_last_error": (C.c_char_p, []),
    "vitb_device_supported": (_i, []),
    "vitb_launch_count": (C.c_ulonglong, []),
    "vitb_set_l2_persisting_window": (_i, [_p, _sz, _sz]),
    "vitb_cast_f32_to_bf16": (_i, [_p, _p, _i64, _p]),
    "vitb_patch_embed_fwd_ws_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "vitb_patch_embed_fwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, _sz, _i, _i, _i, _i, _i, _i, _p]),
    "vitb_patch_embed_bwd_ws_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "vitb_patch_embed_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _sz, _i, _i, _i, _i, _i, _i, _p]),
    "vitb_layernorm_fwd": (_i, [_p, _i64, _p, _p, _p, _p, _p, _i, _i, _f, _i, _p]),
    "vitb_layernorm_bwd_ws_bytes": (_sz, [_i, _i]),
    "vitb_layernorm_bwd": (_i, [_p, _p, _i64, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _i, _i, _i, _p]),
    "vitb_gemm_bias_act_fwd": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vitb_gemm_dgrad": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "vitb_gemm_wgrad_ws_bytes": (_sz, [_i, _i, _i, _i]),
    "vitb_gemm_wgrad_dbias": (_i, [_p, _p, _p, _p, _p, _sz, _i, _i, _i, _i, _i, _p]),
    "vitb_attn_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _f, _i, _p]),
    "vitb_attn_bwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _i, _p]),
    "vitb_colsum_ws_bytes": (_sz, [_i, _i]),
    "vitb_gelu_bwd_colsum": (_i, [_p, _p, _p, _p, _p, _sz, _i, _i, _i, _p]),
    "vitb_colsum": (_i, [_p, _p, _p, _sz, _i, _i, _i, _p]),
    "vitb_pool_fwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "vitb_pool_bwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "vitb_augment_crop_flip_normalize": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vitb_augment_autoaugment": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _i, _i, _i, _p]),
    "vitb_augment_crop_flip_normalize_gather": (_i, [_p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vitb_augment_autoaugment_gather": (_i, [_p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p, _i, _i, _i, _p]),
    "vitb_random_crop_paste": (_i, [_p, _p, _p, _i, _i, _p]),
    "vitb_batch_mix": (_i, [_p, _p, _p, _i, _i, _i, _i, C.c_double, _i, _i, _i, _i, _p]),
    "vitb_dropout_threshold": (C.c_uint32, [_f]),
    "vitb_dropout": (_i, [_p, _p, _p, _i64, _f, C.c_uint64, C.c_uint32, C.c_uint32, _p, _i, _p]),
    "vitb_ls_ce_fwd_bwd": (_i, [_p, _p, _p, _p, _i, _i, _f, _f, _p]),
    "vitb_ls_ce_mix_fwd_bwd": (_i, [_p, _p, _p, _f, _p, _p, _p, _i, _i, _f, _f, _p]),
    "vitb_ls_ce_batch_fwd_bwd": (_i, [_p, _p, _p, _f, _p, _p, _p, _p, _i, _i, _f, _f, _p]),
    "vitb_ls_ce_ws_bytes": (_sz, []),
    "vitb_ls_ce_blocks_fwd_bwd": (_i, [_p, _p, _p, _f, _p, _p, _p, _p, _i, _i, _f, _f, _p, _sz, _p]),
    "vitb_eval_metrics_ws_bytes": (_sz, []),
    "vitb_eval_metrics": (_i, [_p, _p, _p, _i, _i, _f, _p, _p, _sz, _p]),
    "vitb_train_loss_accumulate": (_i, [_p, _p, _i, _p, _p]),
    "vitb_gemm_bias_act_fwd_drop": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _dp, _p]),
    "vitb_gemm_dgrad_drop": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _dp, _p]),
    "vitb_gelu_bwd_colsum_drop": (_i, [_p, _p, _p, _p, _p, _sz, _i, _i, _i, _dp, _p]),
    "vitb_layernorm_bwd_fused": (_i, [_p, _p, _i64, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _dp, _p, _sz, _i, _i, _i, _p]),
    "vitb_gemm_bwd_fused_ws_bytes": (_sz, [_i, _i, _i, _i]),
    "vitb_gemm_bwd_fused": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _sz, _i, _i, _i, _i, _p]),
    "vitb_defer_begin": (_i, [_p, _sz]),
    "vitb_defer_flush": (_i, [_p]),
    "vitb_defer_flush_partial": (_i, [_p]),
    "vitb_defer_used": (_sz, []),
    "vitb_adam_multi": (_i, [_p, _p, _p, _p, _p, _i64, _p, _p, _p]),
    "vitb_sgd_multi": (_i, [_p, _p, _p, _p, _i64, _p, _p, _p]),
    "vitb_dp_reduce_adam": (_i, [_p, _p, _p, _p, _p, _p, _p, _i64, _i, _i, _i, _p, _p, _p]),
    "vitb_dp_set_timeout": (_i, [C.c_double]),
    "vitb_ipc_export": (_i, [_p, _p, _p]),
    "vitb_ipc_open": (_i, [_p, _i64, _p]),
}

_lock = threading.Lock()
_lib = None


class VitbError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise VitbError(
                f"{LIB_PATH} not found: build it with `python vit-cifar_b200/build.py` "
                "(or __graft_entry__.build()); there is no CPU or PyTorch fallback for this path")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        v = lib.vitb_version()
        if v != ABI_VERSION:
            raise VitbError(f"libvitb200 ABI version {v} != expected {ABI_VERSION}; rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().vitb_last_error().decode(errors="replace")
        kind = "bad argument" if rc < 0 else f"cudaError {rc}"
        raise VitbError(f"libvitb200 {what} failed ({kind}): {msg}")
