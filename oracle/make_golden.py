"""ORACLE tooling: regenerate tests/golden/*.npz in the AUTHORING container.

Golden vectors come from the real pieces, not from the restatement:
  * LM arithmetic: the installed HF `LlamaModel` (transformers, third-party
    dependency of the reference) driven through the reference's loop shape
    (plangen_base.py:567-607) with the reference's mask / no-position_ids call
    pattern (:571-576);
  * VQ decode: the reference's own `three_party/Janus/janus/models/vq_model.py`
    imported by file path from /root/reference (read-only), both the real
    `VQ_models['VQ-16']()` class on a 4x4 token grid and a tiny-channel Decoder.

Run:  python oracle/make_golden.py          (needs /root/reference; CPU only)
The GPU box never runs this; it only reads the committed .npz files.
"""
from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import janus_oracle as O            # noqa: E402
from oracle.philox import PhiloxSampler         # noqa: E402

REF_VQ = "/root/reference/three_party/Janus/janus/models/vq_model.py"
OUT = os.path.join(ROOT, "tests", "golden")


def load_ref_vq():
    spec = importlib.util.spec_from_file_location("ref_vq_model", REF_VQ)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["ref_vq_model"] = mod
    spec.loader.exec_module(mod)
    return mod


def hf_llama(d: O.JanusDims, sd):
    from transformers import LlamaConfig, LlamaModel
    cfg = LlamaConfig(hidden_size=d.D, intermediate_size=d.F, num_hidden_layers=d.L,
                      num_attention_heads=d.H, num_key_value_heads=d.H, head_dim=d.head_dim,
                      vocab_size=d.vocab, rms_norm_eps=d.rms_eps, rope_theta=d.rope_theta,
                      max_position_embeddings=4096, attn_implementation="eager")
    m = LlamaModel(cfg).eval()
    pre = "language_model.model."
    missing, unexpected = m.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)},
                                            strict=True)
    assert not missing and not unexpected
    return m


def versions():
    import transformers
    return np.array([torch.__version__, transformers.__version__])


def logit_columns(vocab: int, keep: int) -> np.ndarray:
    """The image-vocab columns whose CFG logits a golden stores: all of them, or a fixed seeded sorted sample of `keep`
    (a golden file stays under 1 MB; random fp32 logits do not compress)."""
    if keep >= vocab:
        return np.arange(vocab, dtype=np.int64)
    return np.sort(np.random.default_rng(0).choice(vocab, keep, replace=False)).astype(np.int64)


def golden_lm(name: str, d: O.JanusDims, batch: int, steps: int, lo: int, hi: int, neg_len: int, logit_cols: int):
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    hf = hf_llama(d, sd)
    cond, neg = O.synthetic_prompts(d, batch, seed=1234, lo=lo, hi=hi, neg_len=neg_len)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    trace: dict = {}
    with torch.inference_mode():
        emb = O.embed_tokens(sd, ids)
        toks = O.sample_image(sd, d, emb, batch, steps, mask, 5.0, 1.0, PhiloxSampler(0, 148),
                              mode="fp32", trace=trace,
                              lm_forward=lambda **kw: hf(**kw))
    cols = logit_columns(d.img_vocab, logit_cols)
    np.savez_compressed(
        os.path.join(OUT, name), dims=np.array(d.name), ids=ids.numpy(), mask=mask.numpy(),
        hidden=torch.stack(trace["hidden"]).numpy(), logits=torch.stack(trace["logits"]).numpy()[..., cols],
        logit_cols=cols, tokens=toks.numpy(), cfg_weight=5.0, temperature=1.0, seed=0, num_sms=148,
        versions=versions())
    print(name, "tokens", toks.tolist())


def golden_vq_ref_class(name: str):
    """The reference's real VQ-16 (ch=128, 71.9M params) on a 4x4 token grid."""
    ref = load_ref_vq()
    d = O.JANUS_1P3B
    sd = O.init_state_dict(d, seed=0, only="gen_vision_model.")
    m = ref.VQ_models["VQ-16"]().eval()
    pre = "gen_vision_model."
    res = m.load_state_dict({k[len(pre):]: v for k, v in sd.items()}, strict=False)
    assert not res.unexpected_keys
    assert all(k.startswith(("encoder.", "quant_conv.", "quantize.codebook_used")) for k in res.missing_keys), res.missing_keys
    g = torch.Generator().manual_seed(7)
    codes = torch.randint(0, d.img_vocab, (1, 16), generator=g, dtype=torch.int32)
    with torch.inference_mode():
        out = m.decode_code(codes, shape=[1, 8, 4, 4])
    np.savez_compressed(os.path.join(OUT, name), codes=codes.numpy(), out=out.numpy(), versions=versions())
    print(name, tuple(out.shape), float(out.abs().mean()))


def golden_vq_tiny(name: str, d: O.JanusDims, batch: int):
    """Reference Decoder / VectorQuantizer classes at test-sized channel counts."""
    ref = load_ref_vq()
    sd = O.init_state_dict(d, seed=0, only="gen_vision_model.")
    dec = ref.Decoder(z_channels=d.vq_z, ch=d.vq_ch, ch_mult=d.vq_ch_mult,
                      num_res_blocks=d.vq_res_blocks).eval()
    quant = ref.VectorQuantizer(d.img_vocab, d.code_dim, 0.25, 0.0, True, False).eval()
    pqc = torch.nn.Conv2d(d.code_dim, d.vq_z, 1)
    pre = "gen_vision_model."
    dec.load_state_dict({k[len(pre + "decoder."):]: v for k, v in sd.items() if k.startswith(pre + "decoder.")})
    quant.load_state_dict({"embedding.weight": sd[pre + "quantize.embedding.weight"]})
    pqc.load_state_dict({"weight": sd[pre + "post_quant_conv.weight"], "bias": sd[pre + "post_quant_conv.bias"]})
    g = torch.Generator().manual_seed(11)
    codes = torch.randint(0, d.img_vocab, (batch, d.n_img_tokens), generator=g, dtype=torch.int32)
    with torch.inference_mode():
        zq = quant.get_codebook_entry(codes, [batch, d.code_dim, d.grid, d.grid], True)
        out = dec(pqc(zq))
    np.savez_compressed(os.path.join(OUT, name), dims=np.array(d.name), codes=codes.numpy(),
                        out=out.numpy(), versions=versions())
    print(name, tuple(out.shape), float(out.abs().mean()))


def hf_llama_causal(d: O.JanusDims, sd):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(hidden_size=d.D, intermediate_size=d.F, num_hidden_layers=d.L,
                      num_attention_heads=d.H, num_key_value_heads=d.H, head_dim=d.head_dim,
                      vocab_size=d.vocab, rms_norm_eps=d.rms_eps, rope_theta=d.rope_theta, tie_word_embeddings=False,
                      max_position_embeddings=4096, attn_implementation="eager")
    m = LlamaForCausalLM(cfg).eval()
    pre = "language_model."
    missing, unexpected = m.load_state_dict({k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}, strict=True)
    assert not missing and not unexpected
    return m


def golden_x2t(name: str, d: O.JanusDims, batch: int, max_new: int, lo: int, hi: int, eos_from=(0, 3)):
    """Stage-1 layout-text decode (System.x2t, plangen_base.py:513-523): the REAL HF `generate` on left-padded
    prompts.  eos_token_id is chosen as the token row eos_from[0] emits at step eos_from[1] in a free run, so
    that row finishes early and the pad-fill / early-stop bookkeeping is exercised."""
    sd = O.init_state_dict(d, seed=0, with_vq=False, with_lm_head=True)
    hf = hf_llama_causal(d, sd)
    cond, _ = O.synthetic_prompts(d, batch, seed=4321, lo=lo, hi=hi, neg_len=4)
    ids, mask = O.pad_input_ids(cond, d.pad_id)
    kw = dict(bos_token_id=1, max_new_tokens=max_new, do_sample=False, use_cache=True, output_logits=True,
              return_dict_in_generate=True)
    with torch.inference_mode():
        emb = hf.get_input_embeddings()(ids.long())
        free = hf.generate(inputs_embeds=emb, attention_mask=mask.long(), pad_token_id=d.vocab - 1,
                           eos_token_id=d.vocab - 1, **kw)
        row = free.sequences[eos_from[0]].tolist()
        # first step >= eos_from[1] whose token did not occur earlier in that row: the row then finishes exactly there
        k = next((j for j in range(eos_from[1], len(row)) if row[j] not in row[:j]), eos_from[1])
        eos = int(row[k])
        out = hf.generate(inputs_embeds=emb, attention_mask=mask.long(), pad_token_id=eos, eos_token_id=eos, **kw)
        # second case: every row finishes early (eos = most frequent first token is not guaranteed; use per-run stop)
    np.savez_compressed(os.path.join(OUT, name), dims=np.array(d.name), ids=ids.numpy(), mask=mask.numpy(), eos=eos,
                        max_new=max_new, tokens=out.sequences.numpy(), free_tokens=free.sequences.numpy(),
                        logits=torch.stack(out.logits, 0)[:4].numpy(), versions=versions())
    print(name, "eos", eos, "tokens", out.sequences.tolist())


def golden_vq_encode(name: str, d: O.JanusDims, batch: int, size: int):
    """VQ encode side (editing path, plangen_base.py:528-532): the reference's own Encoder / quant_conv /
    VectorQuantizer classes (imported by file path) at test-sized channel counts with the oracle's weights."""
    ref = load_ref_vq()
    sd = O.init_state_dict(d, seed=0, with_vq=True, with_vq_encoder=True, only="gen_vision_model.")
    enc = ref.Encoder(ch=d.vq_ch, ch_mult=tuple(d.vq_ch_mult), num_res_blocks=d.vq_res_blocks, z_channels=d.vq_z).eval()
    qc = torch.nn.Conv2d(d.vq_z, d.code_dim, 1).eval()
    vq = ref.VectorQuantizer(d.img_vocab, d.code_dim, 0.25, 0.0, True, False).eval()
    pre = "gen_vision_model."
    missing, unexpected = enc.load_state_dict({k[len(pre + "encoder."):]: v for k, v in sd.items() if k.startswith(pre + "encoder.")}, strict=True)
    assert not missing and not unexpected
    qc.load_state_dict({"weight": sd[pre + "quant_conv.weight"], "bias": sd[pre + "quant_conv.bias"]})
    vq.embedding.weight.data.copy_(sd[pre + "quantize.embedding.weight"])
    g = torch.Generator().manual_seed(5)
    img = torch.rand(batch, 3, size, size, generator=g) * 2 - 1
    with torch.inference_mode():
        z = qc(enc(img))
        _, _, info = vq(z)
    idx = info[-1]
    mine = O.vq_encode(sd, d, img)
    assert torch.equal(mine, idx), "oracle restatement disagrees with the reference classes"
    np.savez_compressed(os.path.join(OUT, name), dims=np.array(d.name), img=img.numpy(), z=z.numpy(), indices=idx.numpy(),
                        versions=versions())
    print(name, "indices", idx.tolist()[:12], "...")


REF_SIGLIP = "/root/reference/three_party/Janus/janus/models/siglip_vit.py"


def load_ref_siglip():
    """The reference's own siglip_vit.py (its Attention / Block / VisionTransformer), executed with oracle/timm_stub.py
    standing in for the few timm layers it imports when timm is not installed."""
    from oracle import timm_stub
    timm_stub.install()
    spec = importlib.util.spec_from_file_location("ref_siglip_vit", REF_SIGLIP)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["ref_siglip_vit"] = mod
    spec.loader.exec_module(mod)
    return mod


def golden_siglip(name: str, v: O.SigLIPDims, d: O.JanusDims, batch: int):
    """mmu front-end (oracle only this round): the reference VisionTransformer (ignore_head) with the oracle's weights."""
    ref = load_ref_siglip()
    sd = O.init_siglip_state_dict(v, d, seed=0)
    m = ref.VisionTransformer(img_size=v.image, patch_size=v.patch, embed_dim=v.width, depth=v.layers, num_heads=v.heads,
                              mlp_ratio=v.mlp_ratio, class_token=False, global_pool="map", ignore_head=True,
                              weight_init="skip", num_classes=0).eval()
    pre = "vision_model.vision_tower."
    missing, unexpected = m.load_state_dict({k[len(pre):]: t for k, t in sd.items() if k.startswith(pre)}, strict=False)
    assert not unexpected and all(k.startswith("attn_pool") for k in missing), (missing, unexpected)
    g = torch.Generator().manual_seed(8)
    img = torch.rand(batch, 3, v.image, v.image, generator=g) * 2 - 1
    with torch.inference_mode():
        want = m(img)
        mine = O.siglip_forward(sd, v, img)
    err = (mine - want).abs().max().item()
    assert err <= 1e-5 * max(1.0, want.abs().max().item()), err
    np.savez_compressed(os.path.join(OUT, name), dims=np.array(v.name), img=img.numpy(), features=want.numpy(), versions=versions())
    print(name, "features", tuple(want.shape), "max|restatement - reference| =", err)


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    if len(sys.argv) > 1 and sys.argv[1] == "siglip":  # only the mmu front-end vectors
        golden_siglip("siglip_tiny.npz", O.SIGLIP_TINY, O.TINY, batch=2)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "vqenc":   # only the VQ encode-side vectors
        golden_vq_encode("vqenc_tiny.npz", O.TINY, batch=3, size=8)
        golden_vq_encode("vqenc_small.npz", O.SMALL, batch=2, size=24)
        return
    if len(sys.argv) > 1 and sys.argv[1] == "x2t":     # only the stage-1 text-decode vectors
        golden_x2t("x2t_tiny_fp32.npz", O.TINY, batch=3, max_new=24, lo=5, hi=14)
        golden_x2t("x2t_small_fp32.npz", O.SMALL, batch=4, max_new=20, lo=9, hi=40, eos_from=(1, 5))
        golden_x2t("x2t_tiny_stop_fp32.npz", O.TINY, batch=1, max_new=24, lo=11, hi=11, eos_from=(0, 6))   # all rows finish early
        return
    golden_lm("lm_tiny_fp32.npz", O.TINY, batch=2, steps=8, lo=5, hi=12, neg_len=7, logit_cols=O.TINY.img_vocab)
    golden_lm("lm_small_fp32.npz", O.SMALL, batch=3, steps=6, lo=9, hi=40, neg_len=13, logit_cols=8192)
    golden_vq_tiny("vq_tiny.npz", O.TINY, batch=2)
    golden_vq_tiny("vq_small.npz", O.SMALL, batch=1)
    golden_vq_ref_class("vq16_grid4.npz")
    golden_x2t("x2t_tiny_fp32.npz", O.TINY, batch=3, max_new=24, lo=5, hi=14)
    golden_x2t("x2t_small_fp32.npz", O.SMALL, batch=4, max_new=20, lo=9, hi=40, eos_from=(1, 5))
    golden_x2t("x2t_tiny_stop_fp32.npz", O.TINY, batch=1, max_new=24, lo=11, hi=11, eos_from=(0, 6))
    golden_vq_encode("vqenc_tiny.npz", O.TINY, batch=3, size=8)
    golden_vq_encode("vqenc_small.npz", O.SMALL, batch=2, size=24)
    golden_siglip("siglip_tiny.npz", O.SIGLIP_TINY, O.TINY, batch=2)


if __name__ == "__main__":
    main()
