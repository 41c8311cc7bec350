"""ctypes binding of libphotoverse_b200.so (the C ABI declared in include/photoverse_b200.h).

There is deliberately no fallback: if the shared object is missing or a call fails, we raise.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_ulonglong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PV_LIB_PATH") or os.path.join(_HERE, "libphotoverse_b200.so")   # PV_LIB_PATH: debug (trace) builds

PV_F32 = 0
PV_BF16 = 1
PV_F16 = 2          # inference only (include/photoverse_b200.h)
PV_KEYS_PAD = 96


class PhotoverseB200Error(RuntimeError):
    pass


_lib = None

_SIGNATURES = {
    "pv_version": (c_int, []),
    "pv_last_error": (c_char_p, []),
    "pv_launch_count": (c_ulonglong, []),
    "pv_set_option": (c_int, [c_char_p, c_int]),
    "pv_debug_trace": (c_int, [c_void_p, c_int]),
    "pv_pack_weight": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pv_linear_fwd": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int64] * 11 + [c_void_p]),
    "pv_kv_tile_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "pv_kv_pack_fwd": (c_int, [c_int] + [c_void_p] * 9 + [c_int] * 6 + [c_void_p]),
    "pv_dual_attn_sync_words": (c_int64, [c_int, c_int]),
    "pv_dual_attn_fwd": (c_int, [c_int] + [c_void_p] * 11 + [c_int] * 6 + [c_float, c_float, c_void_p]),
    "pv_dual_attn_core_fwd": (c_int, [c_int] + [c_void_p] * 6 + [c_int] * 6 + [c_float, c_float, c_void_p]),
    "pv_ip_mask_downsample": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "pv_dual_attn_masked_fwd": (c_int, [c_int] + [c_void_p] * 11 + [c_int] * 6 + [c_float, c_float, c_void_p, c_void_p]),
    "pv_dual_attn_masked_core_fwd": (c_int, [c_int] + [c_void_p] * 6 + [c_int] * 6 + [c_float, c_float, c_void_p, c_void_p]),
    "pv_ln_lrelu_fwd": (c_int, [c_int] + [c_void_p] * 6 + [c_int64, c_int, c_int64, c_int64, c_int64, c_float, c_float, c_void_p]),
    "pv_group_mean_fwd": (c_int, [c_int, c_int, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64, c_void_p]),
    "pv_inject_concept_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pv_inject_concept_bwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pv_train_loss_ws_bytes": (c_int64, []),
    "pv_train_loss_fwd": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_float, c_float, c_void_p,
                                  c_void_p, c_void_p]),
    "pv_train_loss_bwd": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_float, c_float, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p]),
    "pv_self_attn_ws_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "pv_self_attn_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "pv_dropout_bwd_acc": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_float, c_int64, c_void_p]),
    "pv_pack_weight_t": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_int, c_int, c_int, c_void_p]),
    "pv_transpose_2d": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p]),
    "pv_linear_bwd_weight_ws_bytes": (c_int64, [c_int, c_int64, c_int64, c_int64]),
    "pv_linear_bwd_weight": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int64] * 5 + [c_float, c_float, c_void_p]),
    "pv_lora_bwd_ws_bytes": (c_int64, [c_int64, c_int, c_int, c_int]),
    "pv_lora_bwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                            c_int64, c_int64, c_void_p]),
    "pv_col_sum_ws_bytes": (c_int64, [c_int64, c_int64]),
    "pv_col_sum": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "pv_ln_lrelu_bwd_ws_bytes": (c_int64, [c_int64, c_int64, c_int]),
    "pv_ln_lrelu_bwd": (c_int, [c_int] + [c_void_p] * 10 + [c_int64, c_int64, c_int, c_float, c_void_p]),
    "pv_group_mean_bwd": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int, c_int, c_int64, c_void_p]),
    "pv_dual_attn_bwd_ws_bytes": (c_int64, [c_int] * 6),
    "pv_dual_attn_bwd": (c_int, [c_int] + [c_void_p] * 7 + [c_int] * 6 + [c_float, c_float, c_void_p]),
    "pv_dual_attn_masked_bwd": (c_int, [c_int] + [c_void_p] * 7 + [c_int] * 6 + [c_float, c_float, c_void_p, c_void_p]),
    "pv_kv_pack_bwd": (c_int, [c_int] + [c_void_p] * 6 + [c_int] * 6 + [c_void_p]),
    "pv_group_norm_nhwc_ws_bytes": (c_int64, [c_int64, c_int64, c_int, c_int]),
    "pv_group_norm_nhwc_fwd": (c_int, [c_int] + [c_void_p] * 7 + [c_int64, c_int64, c_int, c_int, c_float, c_int, c_void_p]),
    "pv_group_norm_nhwc_bwd": (c_int, [c_int] + [c_void_p] * 8 + [c_int64, c_int64, c_int, c_int, c_int, c_void_p]),
    "pv_add_bias_nhwc_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "pv_layer_norm_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_float, c_void_p]),
    "pv_layer_norm_bwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_float, c_void_p]),
    "pv_geglu_fwd": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p]),
    "pv_geglu_bwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p]),
    "pv_linear_geglu_fwd": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int64] * 5 + [c_void_p]),
    "pv_convert_fwd": (c_int, [c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
}

# every declared symbol must be exported by the build
REQUIRED_SYMBOLS = list(_SIGNATURES)


def lib() -> ctypes.CDLL:
    """Load (once) and return the native library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PhotoverseB200Error(
                f"{LIB_PATH} is missing: build it with `python -m photoverse_b200.build` "
                "(photoverse_b200 has no CPU / PyTorch fallback)")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            try:
                fn = getattr(l, name)
            except AttributeError:
                if name in REQUIRED_SYMBOLS:
                    raise PhotoverseB200Error(f"{LIB_PATH} does not export {name}")
                continue
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pv_last_error()
        raise PhotoverseB200Error(f"{what or 'photoverse_b200 call'} failed (code {rc}): "
                                  f"{msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(lib().pv_launch_count())


def set_option(name: str, value: int) -> None:
    check(lib().pv_set_option(name.encode(), int(value)), f"pv_set_option({name})")
