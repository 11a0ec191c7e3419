"""Host-side mirror of the reference interface for the CFG image-token decode path.

`FastJanus` exposes the attribute surface PlanGen's `System` touches on `self.vl_gpt`
(SURVEY.md §8b; project/plangen/plangen_base.py:525-607):

    vl_gpt.language_model.get_input_embeddings()(ids)
    vl_gpt.language_model.model(inputs_embeds=, attention_mask=, use_cache=True, past_key_values=)
    vl_gpt.gen_head(h)
    vl_gpt.prepare_gen_img_embeds(ids)
    vl_gpt.gen_vision_model.decode_code(code_b, shape=[B, 8, h, w], channel_first=True)

plus the fused fast path with the reference's own signatures, `sample_image(...)` / `t2i(...)`,
which runs the whole 576-step loop on the device (CUDA graph, no host sync, no logits round trip).
PyTorch is used only for device memory, streams and host<->device copies; all arithmetic happens in
the sm_100a kernels behind the C-ABI (include/plangen_b200.h), reached through the torch custom-op layer
`torch.ops.plangen_b200.*` (plangen_b200/ops.py).  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional, Sequence

import torch

from . import _lib
from . import ops as _ops          # registers torch.ops.plangen_b200.* (the custom-op layer over the C-ABI)
from .config import Dims
from .weights import pack_state_dict

MODE_IDS = {"bf16": 0, "fp32": 1}


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


OPS = torch.ops.plangen_b200


def _i64(v: int) -> int:
    """uint64 seeds through an int64 schema slot (two's complement)."""
    v = int(v) & 0xFFFFFFFFFFFFFFFF
    return v - (1 << 64) if v >= (1 << 63) else v


def kv_start_from_mask(mask: torch.Tensor, P: int) -> torch.Tensor:
    """Lossless encoding of the reference's 0/1 mask (LEFT padding only, image part all ones;
    plangen_base.py:708-712,668,686): number of leading pad columns per row.  Any other mask shape is
    rejected - the reference never produces one on this path."""
    m = (mask[:, :P] != 0)
    first = torch.where(m.any(1), m.int().argmax(1), torch.full((m.shape[0],), P, device=m.device))
    ar = torch.arange(P, device=m.device)[None, :]
    tail_ok = (mask[:, P:] != 0).all() if mask.shape[1] > P else torch.ones((), dtype=torch.bool, device=m.device)
    left_ok = (m == (ar >= first[:, None])).all()
    ok = int(tail_ok) + 2 * int(left_ok) if mask.device.type == "cpu" else int((tail_ok.int() + 2 * left_ok.int()).item())  # one sync
    if not ok & 1:
        raise ValueError("attention_mask must be all ones on the image-token part")
    if not ok & 2:
        raise ValueError("attention_mask must be LEFT padded (zeros then ones)")
    return first.to(torch.int32).contiguous()


@dataclass
class ModelOutput:
    """BaseModelOutputWithPast stand-in (`.last_hidden_state`, `.past_key_values`)."""
    last_hidden_state: torch.Tensor
    past_key_values: "KVHandle"


class KVHandle:
    """Opaque `past_key_values` the caller threads back (the cache itself lives in the engine)."""

    def __init__(self, rows: int, length: int, kv_start: torch.Tensor, serial: int):
        self.rows, self.length, self.kv_start, self.serial = rows, length, kv_start, serial

    def get_seq_length(self) -> int:
        return self.length


class _Embedding:
    def __init__(self, eng: "FastJanus"):
        self._e = eng

    def __call__(self, ids: torch.Tensor) -> torch.Tensor:
        e = self._e
        ids32 = ids.to(device=e.device, dtype=torch.int32).contiguous()
        out = torch.empty(*ids32.shape, e.dims.D, device=e.device, dtype=torch.float32)
        OPS.embed_tokens(e.handle, ids32, out)
        return out


class _LlamaModel:
    def __init__(self, eng: "FastJanus"):
        self._e = eng

    def __call__(self, inputs_embeds=None, attention_mask=None, use_cache=True, past_key_values=None, **kw):
        e = self._e
        if inputs_embeds is None:
            raise ValueError("inputs_embeds is required (the reference never passes input_ids here)")
        R, q, D = inputs_embeds.shape
        st = _stream_ptr(e.device)
        if past_key_values is None:
            P = q
            if attention_mask is None:
                kv_start = torch.zeros(R, dtype=torch.int32, device=e.device)
            else:
                kv_start = kv_start_from_mask(attention_mask.to(e.device), P)
            x = inputs_embeds.to(device=e.device, dtype=torch.float32).contiguous().clone()
            hidden = torch.empty(R, P, D, device=e.device, dtype=torch.float32)
            OPS.prefill(e.handle, x, kv_start, hidden, True)
            e._serial += 1
            return ModelOutput(hidden, KVHandle(R, P, kv_start, e._serial))
        h = past_key_values
        if not isinstance(h, KVHandle) or h.serial != e._serial or h.rows != R or q != 1:
            raise ValueError("past_key_values does not belong to the engine's live cache")
        x = inputs_embeds.to(device=e.device, dtype=torch.float32).contiguous().view(R, D)
        hidden = torch.empty(R, 1, D, device=e.device, dtype=torch.float32)
        OPS.decode_step(e.handle, x, h.kv_start, h.length, hidden.view(R, D))
        h.length += 1
        return ModelOutput(hidden, h)


class _LanguageModel:
    def __init__(self, eng: "FastJanus"):
        self.model = _LlamaModel(eng)
        self._emb = _Embedding(eng)

    def get_input_embeddings(self):
        return self._emb

    @torch.inference_mode()
    def generate(self, inputs_embeds=None, attention_mask=None, pad_token_id=None, bos_token_id=None, eos_token_id=None,
                 max_new_tokens=512, do_sample=False, use_cache=True, **kw):
        """`LlamaForCausalLM.generate` as System.x2t calls it (plangen_base.py:513-523): greedy search from
        `inputs_embeds` with a LEFT-padded `attention_mask`; returns the NEW token ids only, int64
        (R, n) with n <= max_new_tokens (HF stops once every row has emitted eos; finished rows are filled
        with pad_token_id).  The whole loop runs on the device (pg_generate_greedy)."""
        e = self.model._e
        if inputs_embeds is None:
            raise ValueError("inputs_embeds is required (the reference never passes input_ids here)")
        if do_sample or kw.get("num_beams", 1) != 1:
            raise NotImplementedError("only greedy search (do_sample=False, num_beams=1) is implemented; x2t uses nothing else")
        if not use_cache:
            raise NotImplementedError("use_cache=False is not supported")
        if eos_token_id is None:
            raise ValueError("eos_token_id is required")
        if isinstance(eos_token_id, (list, tuple)):
            if len(eos_token_id) != 1:
                raise NotImplementedError("a single eos_token_id is supported")
            eos_token_id = eos_token_id[0]
        pad = eos_token_id if pad_token_id is None else pad_token_id
        R, P, D = inputs_embeds.shape
        if attention_mask is None:
            kv_start = torch.zeros(R, dtype=torch.int32, device=e.device)
        else:
            kv_start = kv_start_from_mask(attention_mask.to(e.device), P)
        x = inputs_embeds.to(device=e.device, dtype=torch.float32).contiguous().clone()
        tokens = torch.zeros(R, int(max_new_tokens), dtype=torch.int32, device=e.device)
        n = C.c_int(0)
        e._keep = (kv_start, x)
        _lib.check(e._lib.pg_generate_greedy(e._h, _ptr(x), _ptr(kv_start), R, P, int(max_new_tokens), int(eos_token_id),
                                             int(pad), _ptr(tokens), C.byref(n), _stream_ptr(e.device)))
        e._serial += 1
        return tokens[:, :n.value].to(torch.int64)


class _GenVisionModel:
    def __init__(self, eng: "FastJanus"):
        self._e = eng

    def decode_code(self, code_b: torch.Tensor, shape: Optional[Sequence[int]] = None, channel_first: bool = True):
        e = self._e
        if not channel_first:
            raise NotImplementedError("the reference only calls decode_code(channel_first=True)")
        codes = code_b.to(device=e.device, dtype=torch.int32).contiguous()
        if shape is None:
            B, g = codes.shape[0], int(round(codes.shape[1] ** 0.5))
            gh = gw = g
        else:
            B, _, gh, gw = [int(s) for s in shape]
        codes = codes.reshape(B, gh * gw)
        up = 2 ** (len(e.dims.vq_ch_mult) - 1)
        out = torch.empty(B, 3, gh * up, gw * up, device=e.device, dtype=torch.float32)
        OPS.vq_decode_code(e.handle, codes, gh, gw, out)
        return out.to(e.out_dtype)


    def encode(self, img: torch.Tensor):
        """`VQModel.encode` as the editing path uses it (plangen_base.py:532: `encode(img)[-1][-1]`): returns
        `(None, None, (None, None, indices))` with the flat int64 nearest-code indices (B * H/16 * W/16,);
        the quantised tensor and the losses of the training branch are not produced."""
        e = self._e
        x = img.to(device=e.device, dtype=torch.float32).contiguous()
        B, C, H, W = x.shape
        if C != 3:
            raise ValueError("encode expects (B, 3, H, W) images")
        down = 2 ** (len(e.dims.vq_ch_mult) - 1)
        codes = torch.empty(B, (H // down) * (W // down), dtype=torch.int32, device=e.device)
        OPS.vq_encode(e.handle, x, codes)
        return None, None, (None, None, codes.reshape(-1).to(torch.int64))


class FastJanus:
    """B200 engine behind the `MultiModalityCausalLM` attribute surface."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], dims: Dims, mode: str = "bf16",
                 max_batch: int = 16, max_prompt: int = 512, max_steps: Optional[int] = None,
                 device: str = "cuda:0", seed: int = 0, with_vq: bool = True, options: Optional[dict] = None,
                 use_teacher_forcing: bool = False, top_k: int = 0, max_images: int = 0, top_p: float = 1.0):
        if not torch.cuda.is_available():
            raise RuntimeError("plangen_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if mode not in MODE_IDS:
            raise ValueError(mode)
        self.dims, self.mode, self.seed = dims, mode, seed
        self.use_teacher_forcing = bool(use_teacher_forcing)      # args.use_teacher_forcing (plangen_base.py:528,556,593)
        self.top_k = int(top_k)                                   # 0 = off (the reference has no top-k)
        self.top_p = float(top_p)                                 # 1 = off (nor top-p)
        _ops._top_p(self.top_p)
        self.device = torch.device(device)
        self.out_dtype = torch.bfloat16 if mode == "bf16" else torch.float32
        self.max_rows = 2 * max_batch
        self.max_prompt = max_prompt
        self.max_steps = max_steps or dims.n_img_tokens
        self._lib = _lib.load()
        self._serial = 0
        pd = _lib.PgDims()
        for k in ("D", "L", "H", "head_dim", "F", "vocab", "img_vocab", "code_dim", "img_embed", "grid", "vq_ch",
                  "vq_z", "vq_res_blocks"):
            setattr(pd, k, getattr(dims, k))
        pd.rms_eps, pd.rope_theta = dims.rms_eps, dims.rope_theta
        pd.vq_nres = len(dims.vq_ch_mult)
        for i, m in enumerate(dims.vq_ch_mult):
            pd.vq_ch_mult[i] = m
        pd.mode, pd.max_rows, pd.max_prompt, pd.max_steps = MODE_IDS[mode], self.max_rows, max_prompt, self.max_steps
        # mmu front-end: built when the state dict carries the vision tower and max_images > 0
        self.with_vision = max_images > 0 and "vision_model.vision_tower.pos_embed" in state_dict
        self.max_images = int(max_images) if self.with_vision else 0
        if self.with_vision:
            for k in ("sig_width", "sig_layers", "sig_heads", "sig_patch", "sig_image", "sig_mlp"):
                setattr(pd, k, getattr(dims, k))
            pd.max_images = self.max_images
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pg_engine_create(C.byref(pd), self.device.index or 0, C.byref(h)))
            self._h = h
            for k, v in (options or {}).items():
                self.set_option(k, v)
            kvb, wsb = C.c_size_t(), C.c_size_t()
            _lib.check(self._lib.pg_engine_query_bytes(h, C.byref(kvb), C.byref(wsb)))
            self._kv = torch.zeros(kvb.value, dtype=torch.uint8, device=self.device)   # TMA tiles read past `pos`: keep it finite
            self._ws = torch.empty(wsb.value, dtype=torch.uint8, device=self.device)
            _lib.check(self._lib.pg_engine_bind_buffers(h, _ptr(self._kv), kvb.value, _ptr(self._ws), wsb.value))
            tmax = self.counter("tmax")
            self._weights = pack_state_dict(state_dict, dims, mode, self.device, tmax, with_vq=with_vq,
                                            with_vision=self.with_vision)
            for name, t in self._weights.items():
                _lib.check(self._lib.pg_engine_set_tensor(h, name.encode(), _ptr(t), t.numel() * t.element_size()))
            _lib.check(self._lib.pg_engine_finalize(h, _stream_ptr(self.device)))
        self.handle = _ops.register_engine(self)      # the integer the torch.ops.plangen_b200.* operators take
        self.language_model = _LanguageModel(self)
        self.gen_vision_model = _GenVisionModel(self)
        self.weight_bytes_per_step = self._weight_bytes_per_step()

    # ------------------------------------------------------------------ plumbing
    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.pg_engine_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def set_option(self, key: str, value: int):
        _lib.check(self._lib.pg_engine_set_option(self._h, key.encode(), int(value)))

    def counter(self, key: str) -> int:
        v = C.c_int64()
        _lib.check(self._lib.pg_engine_get_counter(self._h, key.encode(), C.byref(v)))
        return v.value

    def eval(self):
        return self

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("plangen_b200 is an inference engine")
        return self

    def parameters(self):
        return iter(self._weights.values())

    def _weight_bytes_per_step(self) -> int:
        """Algorithmic weight bytes one decode step must stream (BASELINE.md §4; the gen_aligner
        MLP is replaced by a table gather so its weights are not counted)."""
        d = self.dims
        es = 2 if self.mode == "bf16" else 4
        HD = d.H * d.head_dim
        per_layer = (3 * HD * d.D + d.D * HD + 2 * d.F * d.D + d.D * d.F) * es + 2 * d.D * 4
        head = (d.img_embed * d.D + d.img_vocab * d.img_embed) * es + (d.img_embed + d.img_vocab) * 4
        return d.L * per_layer + d.D * 4 + head

    # ------------------------------------------------------------------ duck-typed pieces
    @torch.inference_mode()
    def prepare_inputs_embeds(self, input_ids, pixel_values, images_seq_mask, images_emb_mask, **kwargs):
        """`MultiModalityCausalLM.prepare_inputs_embeds` (modeling_vlm.py:221-268; called at plangen_base.py:289,366,855):
        input_ids (b, T), pixel_values (b, n, 3, h, w), images_seq_mask (b, T), images_emb_mask (b, n, n_image_tokens)
        -> inputs_embeds (b, T, D) fp32 (the text embedding's dtype).  SigLIP tower + aligner + scatter on the device
        (pg_prepare_inputs_embeds); raises if the two masks select different counts, as the reference asserts."""
        if not self.with_vision:
            raise RuntimeError("this engine was built without the vision tower: pass a state_dict with "
                               "vision_model.vision_tower.* / aligner.* and max_images > 0")
        ids = input_ids.to(device=self.device, dtype=torch.int32).contiguous()
        b, T = ids.shape
        pv = pixel_values.to(device=self.device)
        if pv.dim() != 5 or pv.shape[0] != b or pv.shape[2] != 3:
            raise ValueError("pixel_values must be (b, n_images, 3, h, w)")
        n_img = pv.shape[0] * pv.shape[1]
        S = self.dims.sig_image
        if pv.shape[3] != S or pv.shape[4] != S:
            raise ValueError(f"the vision tower takes {S}x{S} images")
        if self.mode == "bf16":
            pv = pv.to(torch.bfloat16)                    # `images.bfloat16()` (:249) - also when the caller passes fp32
        pv = pv.to(torch.float32).reshape(n_img, 3, S, S).contiguous()
        seq = images_seq_mask.to(self.device).reshape(b, T).ne(0).to(torch.uint8).contiguous()
        emb = images_emb_mask.to(self.device).reshape(n_img, -1).ne(0).to(torch.uint8).contiguous()
        if emb.shape[1] != self.dims.sig_patches:
            raise ValueError(f"images_emb_mask must have {self.dims.sig_patches} entries per image")
        out = torch.empty(b, T, self.dims.D, device=self.device, dtype=torch.float32)
        OPS.prepare_inputs_embeds(self.handle, pv, ids, seq, emb, out)
        return out

    @torch.inference_mode()
    def vision_features(self, images: torch.Tensor) -> torch.Tensor:
        """`aligner(vision_model(images))` (modeling_vlm.py:250): (n, 3, S, S) -> (n, n_patches, D) in the engine's dtype."""
        if not self.with_vision:
            raise RuntimeError("this engine was built without the vision tower")
        pv = images.to(device=self.device)
        if self.mode == "bf16":
            pv = pv.to(torch.bfloat16)
        pv = pv.to(torch.float32).contiguous()
        n = pv.shape[0]
        out = torch.empty(n, self.dims.sig_patches, self.dims.D, device=self.device, dtype=torch.float32)
        _lib.check(self._lib.pg_vision_features(self._h, _ptr(pv), n, _ptr(out), _stream_ptr(self.device)))
        return out.to(self.out_dtype)

    def gen_head(self, h: torch.Tensor) -> torch.Tensor:
        R = h.shape[0]
        x = h.to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty(R, self.dims.img_vocab, device=self.device, dtype=torch.float32)
        OPS.gen_head(self.handle, x, out)
        return out.to(self.out_dtype)

    def prepare_gen_img_embeds(self, image_ids: torch.Tensor) -> torch.Tensor:
        ids = image_ids.to(device=self.device, dtype=torch.int32).contiguous()
        out = torch.empty(*ids.shape, self.dims.D, device=self.device, dtype=torch.float32)
        OPS.prepare_gen_img_embeds(self.handle, ids, out)
        return out.to(self.out_dtype)

    def cfg_sample_embed(self, logits: torch.Tensor, cfg_weight: float, temperature: float, seed: int, offset: int,
                         step: int, n_steps: int, tokens_out: torch.Tensor, greedy: bool = False,
                         edit_region: Optional[torch.Tensor] = None, gt_labels: Optional[torch.Tensor] = None,
                         top_k: int = 0, top_p: float = 1.0):
        """plangen_base.py:580-604 in one launch; returns the next inputs_embeds (2B, D) fp32.  `top_k` / `top_p` filter the
        CFG logits as HF's TopKLogitsWarper then TopPLogitsWarper do (0 / 1 = off)."""
        B = logits.shape[0] // 2
        lg = logits.to(device=self.device, dtype=torch.float32).contiguous()
        x_next = torch.empty(2 * B, self.dims.D, device=self.device, dtype=torch.float32)
        OPS.cfg_sample_embed(self.handle, lg, float(cfg_weight), float(temperature), _i64(seed), int(offset), bool(greedy), int(top_k),
                             edit_region, gt_labels, int(step), int(n_steps), tokens_out, x_next, float(top_p))
        return x_next

    def philox_offset_per_step(self, B: int) -> int:
        numel = B * self.dims.img_vocab
        grid = min((numel + 255) // 256, self.counter("num_sms") * (self.counter("max_threads_per_sm") // 256))
        return ((numel - 1) // (256 * grid * 4) + 1) * 4

    # ------------------------------------------------------------------ fused fast path
    def _teacher_inputs(self, batch, gt_labels, num_gen: int, n: int):
        """`edit_region` / `gt_labels` of the reference's override loop (plangen_base.py:593-598) as (num_gen, n) int32.
        The reference overrides rows `bid in range(len(edit_region))` only: with parallel_size > 1 the extra copies are
        sampled freely, so rows >= bs get edit_region = 1 (no override)."""
        if batch is None or batch.get("edit_region") is None:
            raise ValueError("use_teacher_forcing needs batch['edit_region'] (plangen_base.py:594)")
        if gt_labels is None:
            raise ValueError("use_teacher_forcing needs gt_labels (or gt_image for t2i to encode, plangen_base.py:528-532)")
        er = batch["edit_region"].to(device=self.device, dtype=torch.int32)
        bs = er.shape[0]
        er = er.reshape(bs, -1)
        gl = gt_labels.to(device=self.device, dtype=torch.int32).reshape(gt_labels.shape[0], -1)
        if gl.shape[0] != bs:
            raise ValueError(f"gt_labels has {gl.shape[0]} rows, edit_region {bs}")
        if bs > num_gen:
            raise ValueError(f"edit_region has {bs} rows but only {num_gen} images are generated")
        if er.shape[1] < n or gl.shape[1] < n:
            raise ValueError(f"edit_region / gt_labels need at least {n} columns (got {er.shape[1]}, {gl.shape[1]})")
        er, gl = er[:, :n], gl[:, :n]
        if bs < num_gen:
            er = torch.cat([er, torch.ones(num_gen - bs, n, dtype=torch.int32, device=self.device)])
            gl = torch.cat([gl, torch.zeros(num_gen - bs, n, dtype=torch.int32, device=self.device)])
        return er.contiguous(), gl.contiguous()

    @torch.inference_mode()
    def sample_image(self, inputs_embeds, num_gen, image_token_num_per_image, mask, cfg_weight, temperature,
                     generator=None, batch=None, gt_labels=None, greedy: bool = False,
                     use_teacher_forcing: Optional[bool] = None, top_k: Optional[int] = None,
                     top_p: Optional[float] = None):
        """System.sample_image (plangen_base.py:567-607).  `generator`: torch CUDA generator (its seed and
        philox offset are honoured and advanced) or an int seed.  Teacher forcing (:593-598) is gated on
        `use_teacher_forcing` (default: the engine's flag = `args.use_teacher_forcing`), never on the mere presence
        of batch['edit_region'] - the reference's datasets emit an all-zero edit_region for non-edit samples.
        `top_k` > 0 keeps the k largest CFG logits before the softmax (north_star (4); 0 = off = the reference).
        `top_p` < 1 then keeps the nucleus, as HF's TopPLogitsWarper after TopKLogitsWarper (1 = off = the reference).
        None: the engine's defaults."""
        R, P, D = inputs_embeds.shape
        if R != 2 * num_gen:
            raise ValueError("inputs_embeds rows must be 2 * num_gen (interleaved cond/uncond)")
        n = int(image_token_num_per_image)
        if isinstance(generator, torch.Generator):
            seed, off = generator.initial_seed(), generator.get_offset()
        else:
            seed, off = int(self.seed if generator is None else generator), 0
        if off != 0:
            raise ValueError("generator must be freshly seeded (the reference reseeds per t2i call, :526)")
        kv_start = (kv_start_from_mask(mask.to(self.device), P) if mask is not None
                    else torch.zeros(R, dtype=torch.int32, device=self.device))
        x = inputs_embeds.to(device=self.device, dtype=torch.float32).contiguous().clone()
        tokens = torch.zeros(num_gen, n, dtype=torch.int32, device=self.device)
        teacher = self.use_teacher_forcing if use_teacher_forcing is None else bool(use_teacher_forcing)
        er = gl = None
        if teacher:
            er, gl = self._teacher_inputs(batch, gt_labels, num_gen, n)
        k = int(self.top_k if top_k is None else top_k)
        p = float(self.top_p if top_p is None else top_p)
        self._keep = (kv_start, x, er, gl)        # keep alive until the stream has consumed them
        OPS.sample_image(self.handle, x, kv_start, n, float(cfg_weight), float(temperature), _i64(seed), bool(greedy), k, er, gl, tokens, p)
        self._serial += 1
        if isinstance(generator, torch.Generator):
            generator.set_offset(off + n * self.philox_offset_per_step(num_gen))
        return tokens

    @torch.inference_mode()
    def t2i(self, inputs_ids=None, parallel_size=1, image_token_num_per_image=None, cfg_weight=5.0, temperature=1.0,
            img_size=None, patch_size=None, gt_image=None, batch=None, mask=None, tokens=None, emb=None,
            gt_labels=None, greedy: bool = False, use_teacher_forcing: Optional[bool] = None, top_k: Optional[int] = None,
            top_p: Optional[float] = None):
        """System.t2i (plangen_base.py:525-565), `tokens`/`emb` branches.  Returns (dec, mask_image).
        Teacher forcing (layout-guided editing, :528-532, :593-598, :557-562) follows `use_teacher_forcing` (default: the
        engine's flag, the counterpart of `args.use_teacher_forcing`): `gt_image` is encoded with the VQ encoder as the
        reference does (or ready-made `gt_labels` are used), and `mask_image` is returned.  With the flag off `gt_image` and
        batch['edit_region'] are ignored, exactly as in the reference."""
        n = image_token_num_per_image or self.dims.n_img_tokens
        img_size = img_size or self.dims.img_size
        patch_size = patch_size or 2 ** (len(self.dims.vq_ch_mult) - 1)      # 16 for VQ-16
        if tokens is None and emb is None:
            raise NotImplementedError("pass `tokens` (2B, P) or `emb`; the un-batched branch is unused by PlanGen")
        teacher = self.use_teacher_forcing if use_teacher_forcing is None else bool(use_teacher_forcing)
        if teacher and gt_labels is None and gt_image is not None:
            gt_images = gt_image.to(device=self.device, dtype=self.out_dtype)          # `gt_image.bfloat16()` (:530)
            gt_labels = self.gen_vision_model.encode(gt_images)[-1][-1].reshape(gt_images.shape[0], -1)
        if tokens is not None:
            tokens = torch.cat([tokens.to(self.device)] * parallel_size)
            inputs_embeds = self.language_model.get_input_embeddings()(tokens)
        else:
            inputs_embeds = emb
        mask = torch.cat([mask.to(self.device)] * parallel_size)
        num_gen = inputs_embeds.shape[0] // 2
        gen = self.sample_image(inputs_embeds, num_gen, n, mask, cfg_weight, temperature, None, batch, gt_labels, greedy,
                                use_teacher_forcing=teacher, top_k=top_k, top_p=top_p)
        g = img_size // patch_size
        dec = self.gen_vision_model.decode_code(gen.to(dtype=torch.int), shape=[num_gen, self.dims.code_dim, g, g])
        self.last_tokens = gen
        mask_image = None
        if teacher:
            # resize_pt(edit_region.reshape(bs,1,g,g).repeat(1,3,1,1), janus_hw).to(dec)   (:559-560).  resize_pt is a
            # torchvision Resize on the LONG tensor: bilinear interpolation in float, then round and cast back to int64,
            # so the reference's mask is binary before `.to(dec)`
            er = batch["edit_region"].to(self.device).reshape(-1, 1, g, g).repeat(1, 3, 1, 1).float()
            mask_image = torch.nn.functional.interpolate(er, size=(img_size, img_size), mode="bilinear",
                                                         align_corners=False).round().to(dec)
        return dec, mask_image

    def images_to_uint8(self, dec: torch.Tensor) -> torch.Tensor:
        """denorm_pt (src/utils/funcs.py:511-512) then `(x*255).astype(np.uint8)` (funcs.py:497-498, truncation) on the
        device: (B,3,H,W) float -> uint8, one kernel (pg_images_to_u8)."""
        x = dec.to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty(x.shape, dtype=torch.uint8, device=self.device)
        OPS.images_to_u8(self.handle, x, out)
        return out

    # ------------------------------------------------------------------ host-buffer entry (end to end)
    @torch.inference_mode()
    def generate_from_host(self, ids_host: torch.Tensor, mask_host: torch.Tensor, cfg_weight=5.0, temperature=1.0,
                           out_host: Optional[torch.Tensor] = None):
        """ids/mask in (pinned) host memory -> uint8 images in host memory; H2D / D2H inside."""
        ids = ids_host.to(self.device, non_blocking=True)
        mask = mask_host.to(self.device, non_blocking=True)
        dec, _ = self.t2i(tokens=ids, mask=mask, cfg_weight=cfg_weight, temperature=temperature)
        img = self.images_to_uint8(dec)
        if out_host is None:
            out_host = torch.empty(img.shape, dtype=torch.uint8, pin_memory=True)
        out_host.copy_(img, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return out_host
