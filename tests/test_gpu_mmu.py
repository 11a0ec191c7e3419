"""-m gpu: mmu front-end (SURVEY §8f rank 2) - `vl_gpt.prepare_inputs_embeds` (plangen_base.py:289,366,855 ->
modeling_vlm.py:221-268): SigLIP vision tower + aligner + embedding scatter through the C-ABI
(pg_prepare_inputs_embeds / pg_vision_features), against the golden made with the reference's own VisionTransformer class
(tests/golden/siglip_tiny.npz, oracle/make_golden.py::golden_siglip) and the oracle restatement."""
import os

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from tests.gpu_util import assert_close

pytestmark = pytest.mark.gpu

_ENG = {}


def _dims(d, v):
    from plangen_b200.config import Dims
    return Dims.from_any(d, vision=v)


def _engine(d, v, mode, max_images=4, with_lm_head=False):
    from plangen_b200.engine import FastJanus
    key = (d.name, v.name, mode, max_images, with_lm_head)
    if key not in _ENG:
        sd = {**O.init_state_dict(d, seed=0, with_vq=False, with_lm_head=with_lm_head), **O.init_siglip_state_dict(v, d, seed=0)}
        _ENG[key] = (FastJanus(sd, _dims(d, v), mode=mode, max_batch=4, max_prompt=64, with_vq=False, max_images=max_images), sd)
    return _ENG[key]


def test_fp32_vision_features_match_reference_class_golden(golden_dir):
    """fp32 check mode: tower + aligner on the golden images = aligner(features the reference's own VisionTransformer
    produced) to 1e-4; and equal to the oracle restatement."""
    g = np.load(os.path.join(golden_dir, "siglip_tiny.npz"))
    v, d = O.SIGLIP_TINY, O.TINY
    eng, sd = _engine(d, v, "fp32")
    img = torch.from_numpy(g["img"])
    with torch.inference_mode():
        want = O.understanding_aligner(sd, torch.from_numpy(g["features"]))
        want2 = O.understanding_aligner(sd, O.siglip_forward(sd, v, img))
    got = eng.vision_features(img.cuda()).float().cpu()
    assert got.shape == want.shape == (2, v.n_patches, d.D)
    assert_close(got.numpy(), want.numpy(), 1e-4, 1e-5, "aligner(SigLIP features) vs reference-class golden")
    assert_close(got.numpy(), want2.numpy(), 1e-4, 1e-5, "aligner(SigLIP features) vs oracle")


def _mmu_batch(v, d, b, n_img, seed, drop=0):
    """ids / pixel_values / masks shaped like mmu_collate's: `n_img` images per row, each image's placeholder run in the
    sequence, `drop` image tokens of the last image of every row left unused (emb mask False)."""
    g = torch.Generator().manual_seed(seed)
    n = v.n_patches
    pix = torch.rand(b, n_img, 3, v.image, v.image, generator=g) * 2 - 1
    T = n_img * n + 7
    ids = torch.randint(1, d.vocab - 2, (b, T), generator=g)
    seq = torch.zeros(b, T, dtype=torch.bool)
    emb = torch.ones(b, n_img, n, dtype=torch.bool)
    for r in range(b):
        start = 1 + r                                           # ragged placement
        seq[r, start:start + n_img * n - drop] = True
        if drop:
            emb[r, -1, n - drop:] = False
    ids[seq] = -1
    return ids, pix, seq, emb


@pytest.mark.parametrize("n_img,drop", [(1, 0), (2, 3)])
def test_fp32_prepare_inputs_embeds_matches_oracle_and_scatter_is_exact(n_img, drop):
    v, d = O.SIGLIP_TINY, O.TINY
    eng, sd = _engine(d, v, "fp32")
    ids, pix, seq, emb = _mmu_batch(v, d, 2, n_img, seed=11 + n_img, drop=drop)
    with torch.inference_mode():
        want = O.prepare_inputs_embeds(sd, v, ids.clone(), pix, seq, emb)
    got = eng.prepare_inputs_embeds(ids.cuda(), pix.cuda(), seq.cuda(), emb.cuda()).cpu()
    assert got.shape == want.shape and got.dtype == torch.float32
    keep = ~seq
    assert torch.equal(got[keep], want[keep])                  # text slots: embed_tokens rows, bit for bit
    assert_close(got[seq].numpy(), want[seq].numpy(), 1e-4, 1e-5, "image slots")
    # scatter order: slot k of the sequence mask holds selected image token k (row-major), checked against the
    # engine's own tower output
    feats = eng.vision_features(pix.reshape(-1, 3, v.image, v.image).cuda()).float().cpu().reshape(2, n_img * v.n_patches, d.D)
    assert torch.equal(got[seq], feats[emb.reshape(2, -1)])


def test_prepare_inputs_embeds_rejects_mismatched_masks():
    from plangen_b200._lib import PgError
    v, d = O.SIGLIP_TINY, O.TINY
    eng, _ = _engine(d, v, "fp32")
    ids, pix, seq, emb = _mmu_batch(v, d, 2, 1, seed=3)
    emb[0, 0, 0] = False
    with pytest.raises(PgError):
        eng.prepare_inputs_embeds(ids.cuda(), pix.cuda(), seq.cuda(), emb.cuda())
    from plangen_b200.engine import FastJanus
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    plain = FastJanus(sd, _dims(d, v), mode="fp32", max_batch=2, max_prompt=64, with_vq=False)
    with pytest.raises(RuntimeError):
        plain.prepare_inputs_embeds(ids.cuda(), pix.cuda(), seq.cuda(), emb.cuda())


SIGLIP_SMALL64 = O.SigLIPDims(name="siglip-small-hd64", width=128, layers=3, heads=2, patch=16, image=96)     # 36 patches, head_dim 64


@pytest.mark.parametrize("tc", [1, 0])
def test_bf16_small_tower_vs_autocast_reference(tc):
    """bf16 regime at a small width with head_dim 64 (the tcgen05 attention's shape; tc = 0: CUDA-core attention):
    features vs the oracle under autocast on the same GPU, rtol 2e-2."""
    v, d = SIGLIP_SMALL64, O.TINY
    eng, sd = _engine(d, v, "bf16")
    sdc = {k: t.cuda() for k, t in sd.items()}
    g = torch.Generator().manual_seed(8)
    img = (torch.rand(3, 3, v.image, v.image, generator=g) * 2 - 1).cuda()
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        want = O.understanding_aligner(sdc, O.siglip_forward(sdc, v, img.bfloat16())).float().cpu()
    eng.set_option("sig_attn_tc", tc)
    try:
        got = eng.vision_features(img).float().cpu()
    finally:
        eng.set_option("sig_attn_tc", 1)
    assert_close(got.numpy(), want.numpy(), 2e-2, 2e-2, f"bf16 SigLIP features (tc attention = {tc})")


def test_fullsize_siglip_l_bf16_vs_autocast_reference():
    """The real tower size (SigLIP-L/16-384: width 1024, 24 layers, 16 heads, 576 patches) + aligner to D = 2048, B = 2,
    through prepare_inputs_embeds: vs the oracle under autocast on the same GPU.  Criteria as in test_gpu_fullsize:
    >= 99.9 % of the feature values within rtol 2e-2 + max(2e-2 max|ref|, 2 x q99.9 of the reference's own bf16 noise),
    and the engine's error against the fp32 reference no larger than 1.25x the reference bf16 path's own."""
    from plangen_b200 import synthetic
    from plangen_b200.config import Dims
    from plangen_b200.engine import FastJanus
    v, od = O.SIGLIP_L16_384, O.JANUS_1P3B
    d = Dims.from_any(od, vision=v)
    dev = torch.device("cuda", 0)
    # LM layers are irrelevant here: a 2-layer LM keeps the engine small, the tower / aligner / embedding are full size
    d2 = Dims(**{**d.__dict__, "L": 2, "name": "janus-1.3b-2layer"})
    sd = synthetic.random_state_dict(d2, dev, seed=0, with_vq=False, with_vision=True)
    eng = FastJanus(sd, d2, mode="bf16", max_batch=2, max_prompt=1024, with_vq=False, max_images=2)
    try:
        b, n = 2, v.n_patches
        g = torch.Generator().manual_seed(21)
        pix = (torch.rand(b, 1, 3, v.image, v.image, generator=g) * 2 - 1).to(dev)
        T = n + 44
        ids = torch.randint(1, 100000, (b, T), generator=g).to(dev)
        seq = torch.zeros(b, T, dtype=torch.bool, device=dev)
        seq[0, 20:20 + n] = True
        seq[1, 31:31 + n] = True
        ids[seq] = -1
        emb = torch.ones(b, 1, n, dtype=torch.bool, device=dev)
        with torch.inference_mode():
            want16 = O.prepare_inputs_embeds(sd, v, ids.clone(), pix, seq, emb, mode="autocast").float().cpu().numpy()
            want32 = O.prepare_inputs_embeds(sd, v, ids.clone(), pix, seq, emb, mode="fp32").float().cpu().numpy()
        got = eng.prepare_inputs_embeds(ids, pix, seq, emb).float().cpu().numpy()
        m = seq.cpu().numpy()
        assert np.array_equal(got[~m], want32[~m])                                   # text slots exact
        a, r16, r32 = got[m], want16[m], want32[m]
        e_mine, e_ref = np.abs(a - r32), np.abs(r16 - r32)
        add = max(2e-2 * np.abs(r16).max(), 2.0 * np.quantile(e_ref, 0.999))
        frac_ok = float((np.abs(a - r16) <= 2e-2 * np.abs(r16) + add).mean())
        assert frac_ok >= 0.999, f"only {frac_ok:.5f} of the image features within rtol 2e-2 + {add:.3e}"
        assert e_mine.mean() <= 1.25 * e_ref.mean(), (e_mine.mean(), e_ref.mean())
        assert np.quantile(e_mine, 0.999) <= 1.25 * np.quantile(e_ref, 0.999), (np.quantile(e_mine, 0.999), np.quantile(e_ref, 0.999))
        # batch independence: image 1 alone gives the same features
        solo = eng.vision_features(pix[1]).float().cpu().numpy()
        assert np.array_equal(solo[0], got[1][m[1]])
    finally:
        del eng, sd
        torch.cuda.empty_cache()


def test_mmu_flow_prepare_inputs_embeds_then_generate_fp32_tokens_match_oracle():
    """The mmu call stack (plangen_base.py:855-881 shape): prepare_inputs_embeds -> language_model.generate, fp32 check
    mode: greedy token ids identical to the oracle's restatement of the same two calls."""
    v, d = O.SIGLIP_TINY, O.TINY
    eng, sd = _engine(d, v, "fp32", with_lm_head=True)
    ids, pix, seq, emb = _mmu_batch(v, d, 2, 2, seed=5)
    # three more columns on the left: text for row 0, padding for row 1 (LEFT padded, as mmu_collate / pad_input_ids do)
    head = torch.tensor([[11, 12, 13], [d.pad_id] * 3])
    ids = torch.cat([head, ids], 1)
    seq = torch.cat([torch.zeros(2, 3, dtype=torch.bool), seq], 1)
    mask = torch.ones(2, ids.shape[1], dtype=torch.int32)
    mask[1, :3] = 0
    eos = 7
    with torch.inference_mode():
        x = O.prepare_inputs_embeds(sd, v, ids.clone(), pix, seq, emb)
        want = O.generate_greedy(sd, d, x, mask, max_new_tokens=12, eos_token_id=eos, pad_token_id=eos)
    xe = eng.prepare_inputs_embeds(ids.cuda(), pix.cuda(), seq.cuda(), emb.cuda())
    got = eng.language_model.generate(inputs_embeds=xe, attention_mask=mask.cuda(), pad_token_id=eos, bos_token_id=1,
                                      eos_token_id=eos, max_new_tokens=12, do_sample=False, use_cache=True)
    assert got.cpu().tolist() == want.tolist()


def test_describe_then_ground_host_flow_runs_the_mmu_stack():
    """prompts.PromptPipeline.describe_then_ground (the `mmu` mode, plangen_base.py:851-881): mmu_collate-shaped batch ->
    prepare_inputs_embeds -> generate; same token ids as the two engine calls made by hand."""
    from plangen_b200.prompts import PromptPipeline, IMAGE_PLACEHOLDER
    v, d = O.SIGLIP_TINY, O.TINY

    class Tok:
        def encode(self, s):
            out = []
            for part in s.split(IMAGE_PLACEHOLDER):
                out += [ord(c) % 800 + 10 for c in part] + [900]
            return out[:-1]

        def decode(self, ids):
            return " ".join(str(int(t)) for t in ids)

    eng, _ = _engine(d, v, "fp32", with_lm_head=True)
    pp = PromptPipeline(Tok(), pad_id=d.pad_id, image_token_num=v.n_patches, image_id=900, image_start_id=901, image_end_id=902)
    g = torch.Generator().manual_seed(2)
    images = torch.rand(2, 3, v.image, v.image, generator=g) * 2 - 1
    b = pp.mmu_batchify([pp.mmu_process_one(images[i:i + 1], "", question=q) for i, q in enumerate(["hi", "what is it?"])])   # short: T <= 64
    assert int(b["images_seq_mask"].sum()) == 2 * v.n_patches and b["input_ids"].shape[1] <= 64
    x = eng.prepare_inputs_embeds(b["input_ids"], b["pixel_values"], b["images_seq_mask"], b["images_emb_mask"])
    want = eng.language_model.generate(inputs_embeds=x, attention_mask=b["attention_mask"].cuda(), pad_token_id=7, eos_token_id=7,
                                       max_new_tokens=6)
    pp.mmu_infer_batch = lambda images, answers=None: b              # same batch through the one-call flow
    texts = pp.describe_then_ground(eng, images, eos_token_id=7, max_new_tokens=6)
    assert texts == [" ".join(str(int(t)) for t in row if int(t) != 7) for row in want.cpu().tolist()]
