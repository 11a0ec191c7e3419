"""torch custom-op layer over the C-ABI (north_star: "a thin C-ABI torch custom-op layer").

Every hot-path entry point of include/plangen_b200.h is registered with `torch.library` under the namespace
`plangen_b200`, so the calls are visible to the dispatcher (`torch.ops.plangen_b200.sample_image(...)`), carry a schema
with their mutated arguments, run on torch's CURRENT CUDA stream and can be traced / profiled like any other operator.
The ops take the engine as an integer handle (`FastJanus.handle`); all tensors are CUDA tensors owned by the caller.
There is no CPU implementation: a CPU tensor fails in the dispatcher, a missing shared library fails at import of
`_lib` - nothing falls back.  The sampling ops take one value per image as list arguments (seeds as two's-complement
int64; a batch-wide setting is the same value repeated) and pass them to the C-ABI as a host array of pg_image_sampling.
sample_image and score_image_tokens take an optional guidance schedule as a CPU fp32 (B, n) tensor, passed as the
C-ABI's host array; it replaces the per-image cfg_weight, which is then ignored.  A weight of 1 there is u + 1 * (c - u)
rounded per op (not the conditional logits alone), and the unconditional rows are computed on every step whatever the
schedule.  logprobs_out (None: none, for the step and the loop) receives log p(token) per image and step.  These
optional arguments have no default: torch.library's version bookkeeping indexes every mutated argument positionally.

    op                          C-ABI                         reference call (plangen_base.py)
    embed_tokens                pg_embed_tokens               language_model.get_input_embeddings()(ids)      :548
    prefill                     pg_prefill                    language_model.model(inputs_embeds, mask)       :571-576 (i = 0)
    decode_step                 pg_decode_step                language_model.model(..., past_key_values)      :571-576 (i >= 1)
    gen_head                    pg_gen_head                   gen_head(h)                                     :579
    prepare_gen_img_embeds      pg_prepare_gen_img_embeds     prepare_gen_img_embeds(ids)                     :603
    cfg_sample_embed            pg_cfg_sample_embed           CFG + softmax + multinomial + embed             :580-604
    sample_image                pg_sample_image               System.sample_image                             :567-607
    score_image_tokens          pg_score_image_tokens         log p(given tokens): one teacher-forced prefill + gen_head
    vq_decode_code              pg_vq_decode_code             gen_vision_model.decode_code                    :555
    vq_encode                   pg_vq_encode                  gen_vision_model.encode(img)[-1][-1]            :532
    prepare_inputs_embeds       pg_prepare_inputs_embeds      prepare_inputs_embeds                           :289,366,855
    images_to_u8                pg_images_to_u8               denorm_pt + uint8                               funcs.py:511,497
"""
from __future__ import annotations

import ctypes as C
import weakref
from typing import List, Optional

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


def _per_image(B: int, cfg_weight, temperature, top_k, top_p, seed, offset):
    """pg_image_sampling[B] (a host array) from the per-image lists; seeds arrive as two's-complement int64."""
    if any(len(v) != B for v in (cfg_weight, temperature, top_k, top_p, seed, offset)):
        raise ValueError(f"per-image settings need {B} entries each")
    arr = (_lib.PgImageSampling * B)()
    for i in range(B):
        if not 0.0 <= float(top_p[i]) <= 1.0:          # NaN fails too
            raise ValueError(f"image {i}: `top_p` has to be a float in [0, 1], but is {top_p[i]}")
        if int(top_k[i]) < 0:
            raise ValueError(f"image {i}: `top_k` has to be >= 0, but is {top_k[i]}")
        arr[i] = _lib.PgImageSampling(int(seed[i]) & 0xFFFFFFFFFFFFFFFF, int(offset[i]), float(cfg_weight[i]),
                                      float(temperature[i]), int(top_k[i]), float(top_p[i]))
    return arr


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


def _schedule(cfg_schedule: Optional[torch.Tensor], B: int, n: int):
    """The host pointer of a guidance schedule: a CPU fp32 contiguous (B, n) tensor (the C-ABI checks the values)."""
    if cfg_schedule is None:
        return None
    if cfg_schedule.device.type != "cpu" or cfg_schedule.dtype != torch.float32 or not cfg_schedule.is_contiguous():
        raise ValueError("`cfg_schedule` must be a contiguous CPU float32 tensor (it is read on the host)")
    if tuple(cfg_schedule.shape) != (B, n):
        raise ValueError(f"`cfg_schedule` must be (images, steps) = {(B, n)}, got {tuple(cfg_schedule.shape)}")
    return C.c_void_p(cfg_schedule.data_ptr())


@torch.library.custom_op(f"{NS}::cfg_sample_embed", mutates_args=("tokens_out", "x_next", "logprobs_out"), device_types="cuda")
def cfg_sample_embed(handle: int, logits: torch.Tensor, cfg_weight: List[float], temperature: List[float], top_k: List[int],
                     top_p: List[float], seed: List[int], philox_offset: List[int], rng_per_image: bool, greedy: bool,
                     edit_region: Optional[torch.Tensor], gt_labels: Optional[torch.Tensor], step: int, n_steps: int,
                     tokens_out: torch.Tensor, x_next: torch.Tensor, logprobs_out: Optional[torch.Tensor]) -> None:
    e = _eng(handle); _cuda(logits, edit_region, gt_labels, tokens_out, x_next, logprobs_out)
    B = logits.shape[0] // 2
    pi = _per_image(B, cfg_weight, temperature, top_k, top_p, seed, philox_offset)
    _lib.check(e._lib.pg_cfg_sample_embed(e._h, _p(logits), B, pi, int(rng_per_image), int(greedy), _p(edit_region),
                                          _p(gt_labels), int(step), int(n_steps), _p(tokens_out), _p(x_next),
                                          _p(logprobs_out), _st(logits)))


@torch.library.custom_op(f"{NS}::sample_image", mutates_args=("x_prompt", "tokens_out", "logprobs_out"), device_types="cuda")
def sample_image(handle: int, x_prompt: torch.Tensor, kv_start: torch.Tensor, n_steps: int, cfg_weight: List[float],
                 temperature: List[float], top_k: List[int], top_p: List[float], seed: List[int], philox_offset: List[int],
                 rng_per_image: bool, greedy: bool, edit_region: Optional[torch.Tensor], gt_labels: Optional[torch.Tensor],
                 tokens_out: torch.Tensor, cfg_schedule: Optional[torch.Tensor], logprobs_out: Optional[torch.Tensor]) -> None:
    e = _eng(handle); _cuda(x_prompt, kv_start, edit_region, gt_labels, tokens_out, logprobs_out)
    R, P = x_prompt.shape[0], x_prompt.shape[1]
    sched = _schedule(cfg_schedule, R // 2, int(n_steps))
    pi = _per_image(R // 2, cfg_weight, temperature, top_k, top_p, seed, philox_offset)
    _lib.check(e._lib.pg_sample_image(e._h, _p(x_prompt), _p(kv_start), R, P, int(n_steps), pi, int(rng_per_image), int(greedy),
                                      _p(edit_region), _p(gt_labels), sched, _p(tokens_out), _p(logprobs_out), _st(x_prompt)))


@torch.library.custom_op(f"{NS}::score_image_tokens", mutates_args=("x_seq", "logprobs_out"), device_types="cuda")
def score_image_tokens(handle: int, x_seq: torch.Tensor, kv_start: torch.Tensor, P: int, image_tokens: torch.Tensor,
                       cfg_weight: List[float], temperature: List[float], top_k: List[int], top_p: List[float],
                       logprobs_out: torch.Tensor, cfg_schedule: Optional[torch.Tensor]) -> None:
    e = _eng(handle); _cuda(x_seq, kv_start, image_tokens, logprobs_out)
    R, n = x_seq.shape[0], image_tokens.shape[1]
    B = R // 2
    sched = _schedule(cfg_schedule, B, n)
    pi = _per_image(B, cfg_weight, temperature, top_k, top_p, [0] * B, [0] * B)
    _lib.check(e._lib.pg_score_image_tokens(e._h, _p(x_seq), _p(kv_start), R, int(P), n, _p(image_tokens), pi, sched,
                                            _p(logprobs_out), _st(x_seq)))


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
            "score_image_tokens", "vq_decode_code", "vq_encode", "prepare_inputs_embeds", "images_to_u8")
