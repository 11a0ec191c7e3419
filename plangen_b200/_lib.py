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


class PgImageSampling(C.Structure):
    """pg_image_sampling: one image's sampling settings (include/plangen_b200.h)."""
    _fields_ = [("seed", C.c_uint64), ("offset", C.c_uint64), ("cfg_weight", C.c_float), ("temperature", C.c_float),
                ("top_k", C.c_int32), ("top_p", C.c_double)]


class PgTestContraction(C.Structure):
    """pg_test_contraction: one contraction of pg_test_contraction_run (include/plangen_b200.h)."""
    _fields_ = [
        ("mode", C.c_int32), ("weights", C.c_int32), ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("splits", C.c_int32),
        ("X", C.c_void_p), ("W", C.c_void_p), ("w_tiled", C.c_void_p), ("w_tiled_bytes", C.c_size_t),
        ("C", C.c_void_p), ("c_bytes", C.c_size_t), ("out", C.c_void_p), ("bias", C.c_void_p), ("gelu", C.c_int32),
        ("add16", C.c_void_p), ("resid", C.c_void_p), ("q_out", C.c_void_p), ("kcache", C.c_void_p), ("vcache", C.c_void_p),
        ("row_off", C.c_void_p), ("kv_start", C.c_void_p), ("rope_start", C.c_void_p),
        ("R", C.c_int32), ("P", C.c_int32), ("H", C.c_int32), ("Tmax", C.c_int32), ("ctas", C.c_int32),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t), ("counters", C.c_void_p), ("n_counters", C.c_int32),
        ("img_b", C.c_int32), ("img_h", C.c_int32), ("img_w", C.c_int32), ("path", C.c_int32), ("path_nt", C.c_int32),
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
    "pg_cfg_sample_embed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(PgImageSampling), C.c_int, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pg_prepare_gen_img_embeds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_sample_image": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(PgImageSampling),
                                  C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pg_score_image_tokens": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.POINTER(PgImageSampling), C.c_void_p, C.c_void_p, C.c_void_p]),
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
    "pg_test_attn_decode_io": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                         C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pg_test_attn_prefill_io": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "pg_test_vit_attn_io": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p]),
    "pg_host_group_rows":(C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pg_test_gemm": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_void_p, C.c_void_p]),
    "pg_test_contraction_run": (C.c_int, [C.c_void_p, C.POINTER(PgTestContraction), C.c_void_p]),
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
    if lib.pg_abi_version() != 10:
        raise PgError("ABI version mismatch")
    _LIB = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise PgError(load().pg_last_error().decode("utf-8", "replace"))
