"""torch custom-op layer over the C-ABI (north_star: "a thin C-ABI torch custom-op layer").

Every hot-path entry point of include/plangen_b200.h is registered with `torch.library` under the namespace
`plangen_b200`, so the calls are visible to the dispatcher (`torch.ops.plangen_b200.sample_image(...)`), carry a schema
with their mutated arguments, run on torch's CURRENT CUDA stream and can be traced / profiled like any other operator.
The ops take the engine as an integer handle (`FastJanus.handle`); all tensors are CUDA tensors owned by the caller.
There is no CPU implementation: a CPU tensor fails in the dispatcher, a missing shared library fails at import of
`_lib` - nothing falls back.

    op                          C-ABI                         reference call (plangen_base.py)
    embed_tokens                pg_embed_tokens               language_model.get_input_embeddings()(ids)      :548
    prefill                     pg_prefill                    language_model.model(inputs_embeds, mask)       :571-576 (i = 0)
    decode_step                 pg_decode_step                language_model.model(..., past_key_values)      :571-576 (i >= 1)
    gen_head                    pg_gen_head                   gen_head(h)                                     :579
    prepare_gen_img_embeds      pg_prepare_gen_img_embeds     prepare_gen_img_embeds(ids)                     :603
    cfg_sample_embed            pg_cfg_sample_embed           CFG + softmax + multinomial + embed             :580-604
    sample_image                pg_sample_image               System.sample_image                             :567-607
    vq_decode_code              pg_vq_decode_code             gen_vision_model.decode_code                    :555
    vq_encode                   pg_vq_encode                  gen_vision_model.encode(img)[-1][-1]            :532
    prepare_inputs_embeds       pg_prepare_inputs_embeds      prepare_inputs_embeds                           :289,366,855
    images_to_u8                pg_images_to_u8               denorm_pt + uint8                               funcs.py:511,497
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Optional

import torch

from . import _lib

_ENGINES: "weakref.WeakValueDictionary[int, object]" = weakref.WeakValueDictionary()
NS = "plangen_b200"


def register_engine(eng) -> int:
    h = int(eng._h.value)
    _ENGINES[h] = eng
    return h


def _eng(handle: int):
    e = _ENGINES.get(int(handle))
    if e is None:
        raise RuntimeError(f"plangen_b200: no live engine with handle {handle}")
    return e


def _p(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _st(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("plangen_b200 ops take CUDA tensors only (there is no CPU path)")


def _top_p(top_p: float):
    if not 0.0 <= float(top_p) <= 1.0:          # NaN fails too
        raise ValueError(f"`top_p` has to be a float in [0, 1], but is {top_p}")


@torch.library.custom_op(f"{NS}::embed_tokens", mutates_args=("out",), device_types="cuda")
def embed_tokens(handle: int, ids: torch.Tensor, out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(ids, out)
    _lib.check(e._lib.pg_embed_tokens(e._h, _p(ids), ids.numel(), _p(out), _st(out)))


@torch.library.custom_op(f"{NS}::prefill", mutates_args=("x", "hidden_out"), device_types="cuda")
def prefill(handle: int, x: torch.Tensor, kv_start: torch.Tensor, hidden_out: torch.Tensor, all_positions: bool) -> None:
    e = _eng(handle); _cuda(x, kv_start, hidden_out)
    R, P = x.shape[0], x.shape[1]
    _lib.check(e._lib.pg_prefill(e._h, _p(x), _p(kv_start), R, P, _p(hidden_out), int(all_positions), _st(x)))


@torch.library.custom_op(f"{NS}::decode_step", mutates_args=("hidden_out",), device_types="cuda")
def decode_step(handle: int, x: torch.Tensor, kv_start: torch.Tensor, pos: int, hidden_out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(x, kv_start, hidden_out)
    _lib.check(e._lib.pg_decode_step(e._h, _p(x), _p(kv_start), x.shape[0], int(pos), _p(hidden_out), _st(x)))


@torch.library.custom_op(f"{NS}::gen_head", mutates_args=("logits_out",), device_types="cuda")
def gen_head(handle: int, hidden: torch.Tensor, logits_out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(hidden, logits_out)
    _lib.check(e._lib.pg_gen_head(e._h, _p(hidden), hidden.shape[0], _p(logits_out), _st(hidden)))


@torch.library.custom_op(f"{NS}::prepare_gen_img_embeds", mutates_args=("out",), device_types="cuda")
def prepare_gen_img_embeds(handle: int, ids: torch.Tensor, out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(ids, out)
    _lib.check(e._lib.pg_prepare_gen_img_embeds(e._h, _p(ids), ids.numel(), _p(out), _st(out)))


@torch.library.custom_op(f"{NS}::cfg_sample_embed", mutates_args=("tokens_out", "x_next"), device_types="cuda")
def cfg_sample_embed(handle: int, logits: torch.Tensor, cfg_weight: float, temperature: float, seed: int, philox_offset: int,
                     greedy: bool, top_k: int, edit_region: Optional[torch.Tensor], gt_labels: Optional[torch.Tensor], step: int,
                     n_steps: int, tokens_out: torch.Tensor, x_next: torch.Tensor, top_p: float = 1.0) -> None:
    e = _eng(handle); _cuda(logits, edit_region, gt_labels, tokens_out, x_next); _top_p(top_p)
    _lib.check(e._lib.pg_cfg_sample_embed(e._h, _p(logits), logits.shape[0] // 2, float(cfg_weight), float(temperature), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                          int(philox_offset), int(greedy), int(top_k), float(top_p), _p(edit_region), _p(gt_labels), int(step),
                                          int(n_steps), _p(tokens_out), _p(x_next), _st(logits)))


@torch.library.custom_op(f"{NS}::sample_image", mutates_args=("x_prompt", "tokens_out"), device_types="cuda")
def sample_image(handle: int, x_prompt: torch.Tensor, kv_start: torch.Tensor, n_steps: int, cfg_weight: float, temperature: float,
                 seed: int, greedy: bool, top_k: int, edit_region: Optional[torch.Tensor], gt_labels: Optional[torch.Tensor],
                 tokens_out: torch.Tensor, top_p: float = 1.0) -> None:
    e = _eng(handle); _cuda(x_prompt, kv_start, edit_region, gt_labels, tokens_out); _top_p(top_p)
    R, P = x_prompt.shape[0], x_prompt.shape[1]
    _lib.check(e._lib.pg_sample_image(e._h, _p(x_prompt), _p(kv_start), R, P, int(n_steps), float(cfg_weight), float(temperature),
                                      int(seed) & 0xFFFFFFFFFFFFFFFF, int(greedy), int(top_k), float(top_p), _p(edit_region), _p(gt_labels), _p(tokens_out), _st(x_prompt)))


@torch.library.custom_op(f"{NS}::vq_decode_code", mutates_args=("image_out",), device_types="cuda")
def vq_decode_code(handle: int, codes: torch.Tensor, gh: int, gw: int, image_out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(codes, image_out)
    _lib.check(e._lib.pg_vq_decode_code(e._h, _p(codes), codes.shape[0], int(gh), int(gw), _p(image_out), _st(codes)))


@torch.library.custom_op(f"{NS}::vq_encode", mutates_args=("codes_out",), device_types="cuda")
def vq_encode(handle: int, image: torch.Tensor, codes_out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(image, codes_out)
    B, _, H, W = image.shape
    _lib.check(e._lib.pg_vq_encode(e._h, _p(image), B, H, W, _p(codes_out), _st(image)))


@torch.library.custom_op(f"{NS}::prepare_inputs_embeds", mutates_args=("embeds_out",), device_types="cuda")
def prepare_inputs_embeds(handle: int, pixel_values: torch.Tensor, input_ids: torch.Tensor, images_seq_mask: torch.Tensor,
                          images_emb_mask: torch.Tensor, embeds_out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(pixel_values, input_ids, images_seq_mask, images_emb_mask, embeds_out)
    b, T = input_ids.shape
    _lib.check(e._lib.pg_prepare_inputs_embeds(e._h, _p(pixel_values), pixel_values.shape[0], _p(input_ids), _p(images_seq_mask),
                                               _p(images_emb_mask), b, T, _p(embeds_out), _st(input_ids)))


@torch.library.custom_op(f"{NS}::images_to_u8", mutates_args=("out",), device_types="cuda")
def images_to_u8(handle: int, image: torch.Tensor, out: torch.Tensor) -> None:
    e = _eng(handle); _cuda(image, out)
    _lib.check(e._lib.pg_images_to_u8(e._h, _p(image), image.numel(), _p(out), _st(image)))


OP_NAMES = ("embed_tokens", "prefill", "decode_step", "gen_head", "prepare_gen_img_embeds", "cfg_sample_embed", "sample_image",
            "vq_decode_code", "vq_encode", "prepare_inputs_embeds", "images_to_u8")
