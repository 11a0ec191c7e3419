"""ctypes binding of libplangen_b200.so (the C-ABI in include/plangen_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails,
an exception is raised."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_LIB = None


class PgDims(C.Structure):
    _fields_ = [
        ("D", C.c_int32), ("L", C.c_int32), ("H", C.c_int32), ("head_dim", C.c_int32), ("F", C.c_int32),
        ("vocab", C.c_int32), ("img_vocab", C.c_int32), ("code_dim", C.c_int32), ("img_embed", C.c_int32),
        ("grid", C.c_int32), ("rms_eps", C.c_float), ("rope_theta", C.c_float),
        ("vq_ch", C.c_int32), ("vq_nres", C.c_int32), ("vq_ch_mult", C.c_int32 * 8), ("vq_z", C.c_int32),
        ("vq_res_blocks", C.c_int32), ("mode", C.c_int32), ("max_rows", C.c_int32), ("max_prompt", C.c_int32),
        ("max_steps", C.c_int32),
        ("sig_width", C.c_int32), ("sig_layers", C.c_int32), ("sig_heads", C.c_int32), ("sig_patch", C.c_int32),
        ("sig_image", C.c_int32), ("sig_mlp", C.c_int32), ("max_images", C.c_int32),
    ]


class PgError(RuntimeError):
    pass


EXPORTS = {
    "pg_last_error": (C.c_char_p, []),
    "pg_abi_version": (C.c_int, []),
    "pg_engine_create": (C.c_int, [C.POINTER(PgDims), C.c_int, C.POINTER(C.c_void_p)]),
    "pg_engine_destroy": (C.c_int, [C.c_void_p]),
    "pg_engine_query_bytes": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "pg_engine_bind_buffers": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]),
    "pg_engine_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t]),
    "pg_engine_finalize": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pg_embed_tokens": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_prefill": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "pg_decode_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_gen_head": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_cfg_sample_embed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_uint64, C.c_uint64,
                                      C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "pg_prepare_gen_img_embeds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_sample_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                  C.c_uint64, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pg_generate_greedy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.POINTER(C.c_int), C.c_void_p]),
    "pg_vq_decode_code": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_vq_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_prepare_inputs_embeds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                           C.c_void_p, C.c_void_p]),
    "pg_vision_features": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_images_to_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "pg_engine_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "pg_engine_get_counter": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64)]),
    "pg_debug_copy": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "pg_test_attn_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "pg_debug_zero_part": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "pg_host_group_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pg_test_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_void_p, C.c_void_p]),
}


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Load the shared library (building it in-tree first if it is missing or stale)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get("PG_LIB_PATH")          # A/B testing of kernel variants
    if not path:
        if build_if_missing:
            _build.build()
        path = _build.LIB
    if not os.path.exists(path):
        raise PgError(f"{path} is missing: build it with `python -m plangen_b200.build`; there is no fallback path")
    lib = C.CDLL(path)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.pg_abi_version() != 3:
        raise PgError("ABI version mismatch")
    _LIB = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise PgError(load().pg_last_error().decode("utf-8", "replace"))
