"""ctypes binding of ``libhmocr.so`` (the C ABI declared in ``include/hmocr.h``).

There is no fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libhmocr.so")


class HmocrConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("vocab_size", "d_model", "nhead", "dim_feedforward", "num_layers",
                                         "max_seq_len", "sos_id", "eos_id", "pad_id", "encoder_arch",
                                         "enc_num_layers")]


_p, _i, _i64p, _fp = C.c_void_p, C.c_int, C.POINTER(C.c_int64), C.c_void_p

# name -> (restype, argtypes); must list every symbol include/hmocr.h declares
SIGNATURES = {
    "hmocr_last_error": (C.c_char_p, []),
    "hmocr_version": (C.c_char_p, []),
    "hmocr_launch_count": (C.c_int64, []),
    "hmocr_create": (_i, [C.POINTER(HmocrConfig), C.POINTER(_p)]),
    "hmocr_destroy": (None, [_p]),
    "hmocr_load_weight": (_i, [_p, C.c_char_p, _p, _i64p, _i, _i]),
    "hmocr_finalize_weights": (_i, [_p]),
    "hmocr_set_option": (_i, [_p, C.c_char_p, _i]),
    "hmocr_decode_max_clusters": (_i, [C.POINTER(C.c_int)]),
    "hmocr_set_pos_table": (_i, [_p, _p, _i, _i, _p]),
    "hmocr_workspace_bytes": (_i, [_p, _i, _i, _i, C.POINTER(C.c_size_t)]),
    "hmocr_set_workspace": (_i, [_p, _p, C.c_size_t, _p]),
    "hmocr_read_trace": (_i, [_p, _i64p, _i]),
    "hmocr_encode": (_i, [_p, _p, _i, _p, _p]),
    "hmocr_decoder_forward": (_i, [_p, _p, _p, _i, _i, _p, _p]),
    "hmocr_generate": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_generate_from_memory": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_generate_nbest": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_score": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_score_workspace_bytes": (_i, [_p, _i, _i, C.POINTER(C.c_size_t)]),
    "hmocr_generate_host": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_preprocess_u8": (_i, [_p, _p, _i, _p, _p]),
    "hmocr_pack_tokens": (_i, [_p, _p, _i, _i, _p, _p, _p]),
    "hmocr_preprocess_image_u8": (_i, [_p, _p, _i, _i, _i, _p, _p]),
    "hmocr_preprocess_cv2_u8": (_i, [_p, _p, _i, _i, _p, _p]),
    "hmocr_generate_host_u8": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_last_decode_steps": (_i, [_p, C.POINTER(C.c_int32)]),
    "hmocr_last_timings": (_i, [_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "hmocr_gemm_f16": (_i, [_p, _i, _i, _i, _p, _i, _p, _i, _p, _i, _p, _i, _p, _i, _p, _p, _i, _p]),
    "hmocr_swin_mlp": (_i, [_p, _i, _i, _p, _p, _p, _p, _p, _p]),
    "hmocr_layernorm": (_i, [_p, _i, _i, _p, _p, _p, _p, _p]),
    "hmocr_patch_embed": (_i, [_p, _i, _p, _p, _p, _p, _p, _p]),
    "hmocr_patch_merge_ln": (_i, [_p, _i, _i, _i, _i, _p, _p, _p, _p]),
    "hmocr_window_attention": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "hmocr_self_attention": (_i, [_p, _i, _i, _i, _i, _p, _p]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m handwritten_math_ocr_api_b200.build` "
                "(there is no CPU or PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().hmocr_last_error()
        raise RuntimeError(f"{what} failed ({rc}): {msg.decode() if msg else 'unknown error'}")
