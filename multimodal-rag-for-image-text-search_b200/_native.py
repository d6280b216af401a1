"""ctypes binding of libmmr_b200.so (include/mmr_b200.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MMR_LIB_PATH") or os.path.join(HERE, "libmmr_b200.so")  # override: experiments only

MMR_OK = 0
MMR_BF16, MMR_F32, MMR_F16 = 0, 1, 2
MMR_MAX_K = 64
ABI_VERSION = 2
MMR_QP_AUTO, MMR_QP_F32, MMR_QP_RESCORE = 0, 1, 2

# every symbol include/mmr_b200.h declares: (name, restype, argtypes)
_i32, _i64, _sz, _p, _f64 = C.c_int32, C.c_int64, C.c_size_t, C.c_void_p, C.c_double
SYMBOLS = [
    ("mmr_abi_version", C.c_int, []),
    ("mmr_last_error", C.c_char_p, []),
    ("mmr_set_option", C.c_int, [C.c_char_p, C.c_char_p]),
    ("mmr_get_option", C.c_int, [C.c_char_p]),
    ("mmr_index_set_query_precision", C.c_int, [_p, C.c_int]),
    ("mmr_search_ranges_workspace_bytes", _sz, [_p, _i32, _i32, _i64]),
    ("mmr_search_exchange_host", C.c_int, [_p, _p, _p, _i32, _i32, _p, _i32, _i32, C.c_uint32, _p, _p, _p]),
    ("mmr_index_create", C.c_int, [C.c_int, C.c_int, C.c_int, _i64, _p, _p, _i32, _i64, C.POINTER(_p)]),
    ("mmr_index_destroy", C.c_int, [_p]),
    ("mmr_index_update", C.c_int, [_p, _i64, _p, _p, _i32]),
    ("mmr_convert_rows_f32", C.c_int, [_p, _p, C.c_int, _i64, C.c_int, C.c_int, _p]),
    ("mmr_load_rows_f32_host", C.c_int, [C.c_int, _p, _p, C.c_int, _i64, C.c_int, C.c_int, _p]),
    ("mmr_load_rows_f32_host_scatter", C.c_int, [C.c_int, _p, _p, C.c_int, _i64, C.c_int, C.c_int, _p, _p]),
    ("mmr_hash_strings", C.c_int, [_p, _p, _i64, _p]),
    ("mmr_search_workspace_bytes", _sz, [_p, _i32, _i32]),
    ("mmr_search", C.c_int, [_p, _p, _p, _i32, _i32, _p, _p, _p, _sz, _p]),
    ("mmr_search_ranges", C.c_int, [_p, _p, _i32, _i32, _p, _p, _p, _p, _p, _sz, _p]),
    ("mmr_search_host", C.c_int, [_p, _p, _p, _i32, _i32, _p, _p, _p]),
    ("mmr_merge_topk", C.c_int, [_p, _p, _i32, _i32, _i32, _p, _p, _p]),
    ("mmr_merge_topk_strided", C.c_int, [_p, _p, _i64, _i64, _i32, _i32, _i32, _p, _p, _p]),
    ("mmr_exchange_buffer_bytes", _sz, [_i32, _i32, _i32]),
    ("mmr_search_exchange_workspace_bytes", _sz, [_p, _i32, _i32]),
    ("mmr_search_exchange", C.c_int, [_p, _p, _p, _i32, _i32, _p, _i32, _i32, C.c_uint32, _p, _p, _p, _sz, _p]),
    ("mmr_multi_create", C.c_int, [_p, _i32, C.POINTER(_p)]),
    ("mmr_multi_destroy", C.c_int, [_p]),
    ("mmr_multi_search_host", C.c_int, [_p, _p, _i32, _i32, _p, _p, _p, _p]),
    ("mmr_encoder_create", C.c_int, [C.c_int, _p, C.POINTER(_p)]),
    ("mmr_encoder_destroy", C.c_int, [_p]),
    ("mmr_encoder_out_dim", C.c_int, [_p]),
    ("mmr_encoder_set_weight", C.c_int, [_p, C.c_char_p, _p, _i64, _p]),
    ("mmr_encoder_forward", C.c_int, [_p, _p, _p, _p, _i32, _i32, _p, _p]),
    ("mmr_encoder_create_vision", C.c_int, [C.c_int, _p, C.POINTER(_p)]),
    ("mmr_encoder_forward_pixels", C.c_int, [_p, _p, _i32, _p, _p]),
    ("mmr_image_preprocess", C.c_int, [C.c_int, _p, _p, _i64, _p, _i32, _p, _p]),
    ("mmr_fuse", C.c_int, [_p, _p, _i32, _p, _p, _i32, _i32, _i32, _f64, _p, _p, _p, _p, _p, _p]),
    ("mmr_fuse_f64", C.c_int, [_p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _f64, _p, _p, _p, _p]),
    ("mmr_debug_umma_scores", C.c_int, [_p, _p, _i32, _i64, _i64, _p, _i64, _p, _sz, _p]),
    ("mmr_debug_enc_gemm", C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, C.c_float, _p, _p, _p, _p, _p, _p, _p]),
    ("mmr_debug_enc_attention", C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p]),
    ("mmr_debug_enc_layernorm", C.c_int, [_i32, _i32, _p, _p, _p, C.c_float, _p, _p, _p]),
    ("mmr_debug_enc_patch_embed", C.c_int, [_i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, C.c_float, _p, _p, _p, _p]),
    ("mmr_launch_count", _i64, []),
    ("mmr_device_sm_count", C.c_int, [C.c_int, C.POINTER(C.c_int)]),
    ("mmr_last_kernel", C.c_int, []),
    ("mmr_rescore_reruns", _i64, []),
]


MMR_ENC_MINILM, MMR_ENC_CLIP_TEXT, MMR_ENC_CROSS, MMR_ENC_CLIP_VISION = 0, 1, 2, 3


class EncoderConfig(C.Structure):
    """mmr_encoder_config (include/mmr_b200.h)."""
    _fields_ = [("kind", _i32), ("vocab_size", _i32), ("hidden", _i32), ("layers", _i32), ("heads", _i32),
                ("intermediate", _i32), ("max_positions", _i32), ("type_vocab", _i32), ("proj_dim", _i32),
                ("eos_token_id", _i32), ("ln_eps", C.c_float)]


class VisionConfig(C.Structure):
    """mmr_vision_config (include/mmr_b200.h)."""
    _fields_ = [("hidden", _i32), ("layers", _i32), ("heads", _i32), ("intermediate", _i32), ("image_size", _i32),
                ("patch_size", _i32), ("channels", _i32), ("proj_dim", _i32), ("ln_eps", C.c_float)]


class ImagePrep(C.Structure):
    """mmr_image_prep (include/mmr_b200.h)."""
    _fields_ = [("crop_h", _i32), ("crop_w", _i32), ("table", (C.c_float * 256) * 3)]


class NativeError(RuntimeError):
    """Raised for every non-zero status from the C ABI (propagates like the reference's search errors,
    app/storage/lancedb_store.py:103-123 has no try/except)."""


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). This package has no CPU or eager fallback."
            )
        handle = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(handle, name)  # AttributeError = ABI mismatch, surface it
            fn.restype = res
            fn.argtypes = args
        if handle.mmr_abi_version() != ABI_VERSION:
            raise NativeError(f"ABI version mismatch: library {handle.mmr_abi_version()} != binding {ABI_VERSION}")
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != MMR_OK:
        msg = lib().mmr_last_error()
        raise NativeError(f"mmr status {status}: {msg.decode() if msg else '?'}")


def set_option(name: str, value) -> None:
    """Change a library switch (MMR_PDL, MMR_ENC_ATT_MMA, ...) after load; None restores the default."""
    check(lib().mmr_set_option(name.encode(), None if value is None else str(value).encode()))


def get_option(name: str) -> int:
    return int(lib().mmr_get_option(name.encode()))
