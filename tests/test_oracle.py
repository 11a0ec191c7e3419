"""CPU tests pinning the oracle (oracle/) against the committed golden vectors
(produced by the installed HF LlamaModel and the reference's own vq_model.py, see
oracle/make_golden.py) and against the live pieces when they are importable."""
import os

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from oracle import philox as PX


# ------------------------------------------------------------------ Philox / sampler
def test_philox_known_answers():
    # Random123 kat_vectors for philox4x32-10
    kats = [
        ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
        ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
        ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
         (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ]
    for c, k, want in kats:
        got = PX.philox4x32_10(*[np.uint32(x) for x in c], *[np.uint32(x) for x in k])
        assert tuple(int(x) for x in got) == want


def test_execution_policy_matches_torch_formula():
    # B*16384 elements on a 148-SM part with 2048 threads/SM
    assert PX.execution_policy(16 * 16384, 148, 2048) == (4, 1024, 256)
    off, grid, _ = PX.execution_policy(32 * 16384, 148, 2048)
    assert grid == 1184 and off == 4
    off, grid, _ = PX.execution_policy(128 * 16384, 148, 2048)
    assert grid == 1184 and off == 8


def test_exponential_clamp_and_sign():
    u = np.array([1.0, np.float32(1.0) - np.float32(2.0 ** -24), 0.5, 2.0 ** -33], dtype=np.float32)
    q = PX.exponential_from_uniform(u)
    assert q[0] == np.float32(2.0 ** -24) and q[1] == np.float32(2.0 ** -24)
    assert np.isclose(q[2], np.log(2.0)) and np.all(q > 0)


def test_multinomial_statistics():
    # argmax(p / Exp(1)) is an exact categorical sampler: check frequencies
    p = np.array([[0.5, 0.25, 0.125, 0.125]], dtype=np.float32).repeat(4096, 0)
    tok, off = PX.cuda_multinomial1(p, seed=3, offset=0, num_sms=148)
    freq = np.bincount(tok, minlength=4) / tok.size
    assert np.allclose(freq, p[0], atol=0.03) and off == 4


# ------------------------------------------------------------------------ host layout
def test_collate_layout():
    d = O.TINY
    cond = [[1, 2, 3, 4, 5], [6, 7, 8]]
    neg = [[9, 10], [9, 10]]
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    assert ids.dtype == torch.int32 and mask.dtype == torch.int32
    assert ids.shape == (4, 5) and mask.shape == (4, 5 + d.n_img_tokens)
    assert ids[0].tolist() == [1, 2, 3, 4, 5]                       # cond0
    assert ids[1].tolist() == [d.pad_id] * 3 + [9, 10]             # neg0, LEFT padded
    assert ids[2].tolist() == [d.pad_id] * 2 + [6, 7, 8]           # cond1
    assert mask[1, :5].tolist() == [0, 0, 0, 1, 1] and bool(mask[:, 5:].all())


def test_empty_and_ragged_prompts():
    d = O.TINY
    ids, mask = O.pad_input_ids([[], [1], [1, 2, 3]], d.pad_id)
    assert ids.shape == (3, 3) and mask.sum(1).tolist() == [0, 1, 3]


# ------------------------------------------------------------------- LM vs golden / HF
@pytest.mark.parametrize("name,dims,steps", [("lm_tiny_fp32.npz", O.TINY, 8), ("lm_small_fp32.npz", O.SMALL, 6)])
def test_lm_oracle_matches_hf_golden(golden_dir, name, dims, steps):
    g = np.load(os.path.join(golden_dir, name))
    sd = O.init_state_dict(dims, seed=0, with_vq=False)
    ids, mask = torch.from_numpy(g["ids"]), torch.from_numpy(g["mask"])
    trace = {}
    toks, _ = O.t2i(sd, dims, ids, mask, sampler=PX.PhiloxSampler(int(g["seed"]), int(g["num_sms"])),
                    mode="fp32", image_token_num_per_image=steps, decode=False, trace=trace)
    assert np.array_equal(toks.numpy(), g["tokens"])                 # index work: bit-exact
    logits = torch.stack(trace["logits"]).numpy()[..., g["logit_cols"]]
    # fp32, same library GEMMs on both sides: tolerance 1e-4 relative (north_star)
    np.testing.assert_allclose(logits, g["logits"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(torch.stack(trace["hidden"]).numpy(), g["hidden"], rtol=1e-4, atol=1e-5)


def test_lm_oracle_matches_live_hf_with_padding_and_cache():
    transformers = pytest.importorskip("transformers")
    from oracle.make_golden import hf_llama
    d = O.TINY
    sd = O.init_state_dict(d, seed=5, with_vq=False)
    hf = hf_llama(d, sd)
    torch.manual_seed(0)
    R, P = 4, 9
    ids = torch.randint(0, d.vocab - 1, (R, P))
    mask = torch.ones(R, P + 3, dtype=torch.int32)
    mask[1, :4] = 0
    mask[3, :7] = 0
    emb = O.embed_tokens(sd, ids)
    with torch.inference_mode():
        a = O.llama_model_forward(sd, d, emb, mask)
        b = hf(inputs_embeds=emb, attention_mask=mask, use_cache=True)
        np.testing.assert_allclose(a.last_hidden_state[:, -1].numpy(), b.last_hidden_state[:, -1].numpy(),
                                   rtol=1e-4, atol=1e-5)
        nxt = torch.randn(R, 1, d.D)
        a2 = O.llama_model_forward(sd, d, nxt, mask, past_key_values=a.past_key_values)
        b2 = hf(inputs_embeds=nxt, attention_mask=mask, use_cache=True, past_key_values=b.past_key_values)
        np.testing.assert_allclose(a2.last_hidden_state.numpy(), b2.last_hidden_state.numpy(), rtol=1e-4, atol=1e-5)


def test_autocast_mode_runs_and_is_close_to_fp32():
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    cond, neg = O.synthetic_prompts(d, 1, lo=5, hi=8, neg_len=4)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    tr32, tr16 = {}, {}
    forced = torch.zeros(1, 3, dtype=torch.long)
    gt = torch.tensor([[5, 6, 7]])
    for mode, tr in (("fp32", tr32), ("autocast", tr16)):
        O.t2i(sd, d, ids, mask, sampler=O.greedy_sampler, mode=mode, image_token_num_per_image=3,
              decode=False, trace=tr, edit_region=forced, gt_labels=gt)
    a, b = torch.stack(tr32["logits"]), torch.stack(tr16["logits"])
    assert (a - b).abs().max() < 2e-2 * a.abs().max() + 2e-2


def test_teacher_forcing_overrides_tokens():
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    cond, neg = O.synthetic_prompts(d, 2, lo=5, hi=8, neg_len=4)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    edit = torch.tensor([[0, 1, 0, 1], [1, 1, 0, 0]])
    gt = torch.tensor([[11, 12, 13, 14], [21, 22, 23, 24]])
    toks, _ = O.t2i(sd, d, ids, mask, sampler=PX.PhiloxSampler(0, 148), image_token_num_per_image=4,
                    decode=False, edit_region=edit, gt_labels=gt)
    assert toks[0, 0] == 11 and toks[0, 2] == 13 and toks[1, 2] == 23 and toks[1, 3] == 24


# ------------------------------------------------------------------- VQ vs golden / ref
@pytest.mark.parametrize("name,dims", [("vq_tiny.npz", O.TINY), ("vq_small.npz", O.SMALL)])
def test_vq_oracle_matches_reference_golden(golden_dir, name, dims):
    g = np.load(os.path.join(golden_dir, name))
    sd = O.init_state_dict(dims, seed=0, only="gen_vision_model.")
    codes = torch.from_numpy(g["codes"])
    with torch.inference_mode():
        out = O.decode_code(sd, dims, codes, [codes.shape[0], dims.code_dim, dims.grid, dims.grid])
    np.testing.assert_allclose(out.numpy(), g["out"], rtol=1e-4, atol=1e-5)


def test_vq16_oracle_matches_reference_class_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "vq16_grid4.npz"))
    d = O.JANUS_1P3B
    sd = O.init_state_dict(d, seed=0, only="gen_vision_model.")
    with torch.inference_mode():
        out = O.decode_code(sd, d, torch.from_numpy(g["codes"]), [1, 8, 4, 4])
    np.testing.assert_allclose(out.numpy(), g["out"], rtol=1e-4, atol=2e-5)


@pytest.mark.parametrize("name,dims", [("vq_tiny.npz", O.TINY), ("vq_small.npz", O.SMALL)])
def test_vq_oracle_bf16_autocast_matches_reference_golden(golden_dir, name, dims):
    """The VQ decoder restatement under bf16 autocast (the reference's regime) yields bf16 images of the reference's
    shape, within bf16 rounding of the reference's own fp32 Decoder output (oracle/make_golden.py::golden_vq_tiny)."""
    g = np.load(os.path.join(golden_dir, name))
    sd = O.init_state_dict(dims, seed=0, only="gen_vision_model.")
    codes = torch.from_numpy(g["codes"])
    with torch.inference_mode(), torch.autocast("cpu", dtype=torch.bfloat16):
        out = O.decode_code(sd, dims, codes, [codes.shape[0], dims.code_dim, dims.grid, dims.grid])
    assert out.dtype == torch.bfloat16 and out.shape == g["out"].shape
    err = np.abs(out.float().numpy() - g["out"])
    scale = np.abs(g["out"]).max()
    assert err.max() <= 5e-2 * scale and err.mean() <= 1e-2 * scale, (err.max(), err.mean(), scale)


# ------------------------------------------------------- stage-1 layout-text decode (x2t)
X2T_GOLDENS = [("x2t_tiny_fp32.npz", O.TINY), ("x2t_small_fp32.npz", O.SMALL), ("x2t_tiny_stop_fp32.npz", O.TINY)]


@pytest.mark.parametrize("name,dims", X2T_GOLDENS)
def test_generate_greedy_matches_hf_generate_golden(golden_dir, name, dims):
    """The restated greedy search (System.x2t, plangen_base.py:513-523) against the committed output of the
    real HF `LlamaForCausalLM.generate` (oracle/make_golden.py::golden_x2t): identical token ids incl. the
    pad fill of finished rows and the early stop, logits within 1e-5."""
    g = np.load(os.path.join(golden_dir, name))
    sd = O.init_state_dict(dims, seed=0, with_vq=False, with_lm_head=True)
    ids, mask = torch.from_numpy(g["ids"]), torch.from_numpy(g["mask"])
    eos = int(g["eos"])
    seq, logits = O.generate_greedy(sd, dims, O.embed_tokens(sd, ids), mask, int(g["max_new"]), eos, eos, return_logits=True)
    assert seq.tolist() == g["tokens"].tolist()
    n = min(len(logits), g["logits"].shape[0])
    got = torch.stack(logits[:n]).numpy()
    assert np.abs(got - g["logits"][:n]).max() <= 1e-5 * np.abs(g["logits"]).max()


def test_generate_greedy_positions_are_mask_aware():
    """generate() derives position_ids from the attention mask: a row's result must not depend on how many pad
    columns sit in front of it (the image loop's absolute positions would change the rotary phases)."""
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False, with_lm_head=True)
    prompt = [11, 12, 13, 14, 15, 16, 17]
    ids1, mask1 = O.pad_input_ids([prompt], d.pad_id)
    ids2, mask2 = O.pad_input_ids([prompt, list(range(20, 40))], d.pad_id)
    a = O.generate_greedy(sd, d, O.embed_tokens(sd, ids1), mask1, 6, d.vocab - 1, d.vocab - 1, return_logits=True)[1]
    b = O.generate_greedy(sd, d, O.embed_tokens(sd, ids2), mask2, 6, d.vocab - 1, d.vocab - 1, return_logits=True)[1]
    for x, y in zip(a, b):
        assert torch.allclose(x[0], y[0], atol=2e-6)


# ------------------------------------------------------------------ VQ encode side (editing path)
@pytest.mark.parametrize("name,dims", [("vqenc_tiny.npz", O.TINY), ("vqenc_small.npz", O.SMALL)])
def test_vq_encode_matches_reference_classes_golden(golden_dir, name, dims):
    """`gen_vision_model.encode(img)[-1][-1]` (plangen_base.py:532): the restated Encoder / quant_conv / nearest-code
    search against the committed output of the reference's own classes (oracle/make_golden.py::golden_vq_encode)."""
    g = np.load(os.path.join(golden_dir, name))
    sd = O.init_state_dict(dims, seed=0, with_vq=True, with_vq_encoder=True, only="gen_vision_model.")
    img = torch.from_numpy(g["img"])
    with torch.inference_mode():
        z = O.vq_encoder_forward(sd, dims, img)
    assert np.abs(z.numpy() - g["z"]).max() <= 1e-5 * max(1.0, np.abs(g["z"]).max())
    assert O.vq_encode(sd, dims, img).tolist() == g["indices"].tolist()


def test_vq_encode_decode_round_trip_codes():
    """decode_code(encode(x)) re-encoded lands on codes whose embeddings are the nearest ones (idempotence of the
    quantiser on its own code vectors): quantising the exact code embeddings returns the codes themselves."""
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=True, with_vq_encoder=True, only="gen_vision_model.")
    codes = torch.arange(0, d.img_vocab, 97)[:16].reshape(1, 16)
    zq = O.get_codebook_entry(sd, codes, [1, d.code_dim, 4, 4])
    assert O.vq_quantize_indices(sd, zq).tolist() == codes.reshape(-1).tolist()


@pytest.mark.parametrize("seed,batch,eos_step", [(11, 2, 2), (12, 4, 5), (13, 1, 9)])
def test_generate_greedy_matches_live_hf_generate(seed, batch, eos_step):
    """Beyond the committed goldens: the restated greedy search against the INSTALLED HF `generate` on fresh ragged
    batches (left padding, eos chosen from a free run so rows stop at different steps / all rows stop early)."""
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_llama_causal
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False, with_lm_head=True)
    hf = hf_llama_causal(d, sd)
    cond, _ = O.synthetic_prompts(d, batch, seed=seed, lo=4, hi=19, neg_len=3)
    ids, mask = O.pad_input_ids(cond, d.pad_id)
    kw = dict(bos_token_id=1, max_new_tokens=14, do_sample=False, use_cache=True)
    with torch.inference_mode():
        emb = hf.get_input_embeddings()(ids.long())
        free = hf.generate(inputs_embeds=emb, attention_mask=mask.long(), pad_token_id=d.vocab - 1, eos_token_id=d.vocab - 1, **kw)
        eos = int(free[0, eos_step])
        want = hf.generate(inputs_embeds=emb, attention_mask=mask.long(), pad_token_id=eos, eos_token_id=eos, **kw)
    got = O.generate_greedy(sd, d, O.embed_tokens(sd, ids), mask, 14, eos, eos)
    assert got.tolist() == want.tolist()


# ---------------------------------------------------------- mmu front-end (oracle only; CUDA path not built yet)
def test_siglip_restatement_matches_reference_class_golden(golden_dir):
    """SigLIP vision tower (SURVEY §8f rank 2): the restated forward against the committed output of the reference's own
    VisionTransformer (oracle/make_golden.py::golden_siglip; timm's PatchEmbed / Mlp come from oracle/timm_stub.py)."""
    g = np.load(os.path.join(golden_dir, "siglip_tiny.npz"))
    v, d = O.SIGLIP_TINY, O.TINY
    sd = O.init_siglip_state_dict(v, d, seed=0)
    with torch.inference_mode():
        out = O.siglip_forward(sd, v, torch.from_numpy(g["img"]))
    assert out.shape == (2, v.n_patches, v.width)
    assert np.abs(out.numpy() - g["features"]).max() <= 1e-5 * max(1.0, np.abs(g["features"]).max())


def test_prepare_inputs_embeds_scatters_image_features():
    """modeling_vlm.py:221-268: aligned image features land exactly on the masked sequence slots, in order; text slots
    keep their embed_tokens rows; negative (image) ids are embedded as id 0 before being overwritten."""
    v, d = O.SIGLIP_TINY, O.TINY
    sd = {**O.init_state_dict(d, seed=0, with_vq=False), **O.init_siglip_state_dict(v, d, seed=0)}
    n = v.n_patches
    g = torch.Generator().manual_seed(4)
    pix = torch.rand(2, 1, 3, v.image, v.image, generator=g) * 2 - 1
    T = n + 5
    ids = torch.randint(1, 900, (2, T), generator=g)
    seq_mask = torch.zeros(2, T, dtype=torch.bool)
    seq_mask[0, 2:2 + n] = True
    seq_mask[1, 4:4 + n] = True
    ids[seq_mask] = -1
    emb_mask = torch.ones(2, 1, n, dtype=torch.bool)
    with torch.inference_mode():
        out = O.prepare_inputs_embeds(sd, v, ids, pix, seq_mask, emb_mask)
        feats = O.understanding_aligner(sd, O.siglip_forward(sd, v, pix.reshape(2, 3, v.image, v.image)))
    assert out.shape == (2, T, d.D)
    assert torch.allclose(out[0, 2:2 + n], feats[0]) and torch.allclose(out[1, 4:4 + n], feats[1])
    keep = ~seq_mask
    assert torch.equal(out[keep], O.embed_tokens(sd, ids.clamp_min(0))[keep])
