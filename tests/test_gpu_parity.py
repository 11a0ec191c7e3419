"""-m gpu: parity of the CUDA path (through the C-ABI) against the oracle and the golden vectors."""
import os

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from oracle import philox as PX
from tests.gpu_util import get_engine, assert_close

pytestmark = pytest.mark.gpu


def _num_sms():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.max_threads_per_multi_processor


# ------------------------------------------------------------------------------- fp32 check mode
@pytest.mark.parametrize("name,dims,steps", [("lm_tiny_fp32.npz", O.TINY, 8), ("lm_small_fp32.npz", O.SMALL, 6)])
def test_fp32_dropin_api_matches_golden(golden_dir, name, dims, steps):
    """Drive the engine exactly the way System.sample_image drives vl_gpt (plangen_base.py:567-607),
    teacher-forced on the golden tokens, and compare hidden states / CFG logits (rtol 1e-4)."""
    g = np.load(os.path.join(golden_dir, name))
    eng = get_engine(dims, "fp32", with_vq=False)
    ids = torch.from_numpy(g["ids"]).cuda()
    mask = torch.from_numpy(g["mask"]).cuda()
    emb = eng.language_model.get_input_embeddings()(ids)
    sd_emb = O.init_state_dict(dims, seed=0, with_vq=False)["language_model.model.embed_tokens.weight"]
    assert torch.equal(emb.cpu(), sd_emb[ids.cpu().long()])
    outputs = None
    for i in range(steps):
        outputs = eng.language_model.model(inputs_embeds=emb, attention_mask=mask, use_cache=True,
                                           past_key_values=outputs.past_key_values if i != 0 else None)
        h = outputs.last_hidden_state[:, -1, :]
        assert_close(h.cpu().numpy(), g["hidden"][i], 1e-4, 1e-5, f"hidden step {i}")
        logits = eng.gen_head(h)
        cfg = logits[1::2] + 5.0 * (logits[0::2] - logits[1::2])
        assert_close(cfg.cpu().numpy()[:, g["logit_cols"]], g["logits"][i], 1e-4, 2e-5, f"cfg logits step {i}")
        tok = torch.from_numpy(g["tokens"][:, i]).cuda().long()
        nxt = torch.stack([tok, tok], 1).view(-1)
        emb = eng.prepare_gen_img_embeds(nxt).unsqueeze(1)


@pytest.mark.parametrize("name,dims,steps", [("lm_tiny_fp32.npz", O.TINY, 8), ("lm_small_fp32.npz", O.SMALL, 6)])
@pytest.mark.parametrize("graph", [0, 1])
def test_fp32_fused_loop_reproduces_golden_tokens(golden_dir, name, dims, steps, graph):
    """The fused device loop with the torch-compatible Philox sampler must emit the golden token ids
    when the box has the SM count the golden was made for; otherwise compare with the oracle re-run."""
    g = np.load(os.path.join(golden_dir, name))
    eng = get_engine(dims, "fp32", with_vq=False)
    eng.set_option("use_graph", graph)
    ids = torch.from_numpy(g["ids"]).cuda()
    mask = torch.from_numpy(g["mask"]).cuda()
    emb = eng.language_model.get_input_embeddings()(ids)
    dbg = torch.zeros(steps, ids.shape[0] // 2, dims.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())
    try:
        toks = eng.sample_image(emb, ids.shape[0] // 2, steps, mask, 5.0, 1.0, generator=0)
        torch.cuda.synchronize()
    finally:
        eng.set_option("dbg_logits_ptr", 0)
        eng.set_option("use_graph", 1)
    sms, mt = _num_sms()
    if sms == int(g["num_sms"]):
        want = g["tokens"]
    else:
        sd = O.init_state_dict(dims, seed=0, with_vq=False)
        want, _ = O.t2i(sd, dims, ids.cpu(), mask.cpu(), sampler=PX.PhiloxSampler(0, sms, mt),
                        image_token_num_per_image=steps, decode=False)
        want = want.numpy()
    assert toks.cpu().numpy().tolist() == want.tolist()
    if sms == int(g["num_sms"]):
        assert_close(dbg.cpu().numpy()[..., g["logit_cols"]], g["logits"], 1e-4, 2e-5, "fused-loop CFG logits")


def test_fp32_greedy_sequence_identical_and_ragged_batch():
    """fp32 greedy tokens identical to the oracle on a ragged batch (rows with 0..many pad columns)."""
    d = O.SMALL
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    eng = get_engine(d, "fp32", with_vq=False)
    cond = [[5, 6, 7], list(range(10, 45)), [9] * 17, [3]]
    neg = [[1, 2]] * 4
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    steps = 12
    want, _ = O.t2i(sd, d, ids, mask, sampler=O.greedy_sampler, image_token_num_per_image=steps, decode=False)
    emb = eng.language_model.get_input_embeddings()(ids.cuda())
    got = eng.sample_image(emb, 4, steps, mask.cuda(), 5.0, 1.0, generator=0, greedy=True)
    assert got.cpu().tolist() == want.tolist()


# --------------------------------------------------------------------------- bf16 (autocast) regime
@pytest.mark.parametrize("dims,steps", [(O.TINY, 6), (O.SMALL, 6)])
@pytest.mark.parametrize("use_tc", [1, 0])
def test_bf16_logits_match_autocast_reference(dims, steps, use_tc):
    """Reference regime: fp32 master weights under torch.autocast(bf16) on the SAME GPU (the reference
    PyTorch path).  Teacher-forced on the reference's tokens; CFG logits within rtol 2e-2 (north_star)."""
    sd = O.init_state_dict(dims, seed=0, with_vq=False)
    sdc = {k: v.cuda() for k, v in sd.items()}
    cond, neg = O.synthetic_prompts(dims, 3, seed=77, lo=9, hi=40, neg_len=13)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    trace = {}
    ref_tok, _ = O.t2i(sdc, dims, ids.cuda(), mask.cuda(), sampler=O.greedy_sampler, mode="autocast",
                       image_token_num_per_image=steps, decode=False, trace=trace)
    ref_logits = torch.stack(trace["logits"]).numpy()
    eng = get_engine(dims, "bf16", with_vq=False)
    eng.set_option("use_tc", use_tc)
    dbg = torch.zeros(steps, 3, dims.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())
    try:
        emb = eng.language_model.get_input_embeddings()(ids.cuda())
        forced = {"edit_region": torch.zeros(3, steps, dtype=torch.int32)}
        got = eng.sample_image(emb, 3, steps, mask.cuda(), 5.0, 1.0, generator=0, batch=forced,
                               gt_labels=ref_tok, greedy=True, use_teacher_forcing=True)
        torch.cuda.synchronize()
    finally:
        eng.set_option("dbg_logits_ptr", 0)
        eng.set_option("use_tc", 1)
    assert got.cpu().tolist() == ref_tok.cpu().tolist()            # forced
    assert_close(dbg.cpu().numpy(), ref_logits, 2e-2, 2e-2, f"bf16 CFG logits (tc={use_tc})")


# ----------------------------------------------------------------------------------------- VQ decode
@pytest.mark.parametrize("name,dims", [("vq_tiny.npz", O.TINY), ("vq_small.npz", O.SMALL)])
def test_vq_fp32_matches_reference_golden(golden_dir, name, dims):
    g = np.load(os.path.join(golden_dir, name))
    eng = get_engine(dims, "fp32", with_vq=True)
    codes = torch.from_numpy(g["codes"]).cuda()
    out = eng.gen_vision_model.decode_code(codes, shape=[codes.shape[0], dims.code_dim, dims.grid, dims.grid])
    assert_close(out.cpu().numpy(), g["out"], 1e-4, 2e-5, "vq fp32")


def test_vq16_fp32_matches_reference_class_golden(golden_dir):
    """The real VQ-16 architecture (ch 128, 5 levels) on a 4x4 token grid vs the reference class output."""
    g = np.load(os.path.join(golden_dir, "vq16_grid4.npz"))
    d = O.JanusDims(**{**O.TINY.__dict__, "name": "tiny-vq16", "img_vocab": 16384, "vq_ch": 128,
                       "vq_ch_mult": (1, 1, 2, 2, 4), "vq_z": 256})
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    sd.update(O.init_state_dict(O.JANUS_1P3B, seed=0, only="gen_vision_model."))
    eng = get_engine(d, "fp32", sd=sd, cache=False)
    out = eng.gen_vision_model.decode_code(torch.from_numpy(g["codes"]).cuda(), shape=[1, 8, 4, 4])
    assert_close(out.cpu().numpy(), g["out"], 1e-4, 5e-5, "vq16 fp32")


@pytest.mark.parametrize("dims", [O.TINY, O.SMALL])
def test_vq_bf16_matches_autocast_reference(dims):
    sd = O.init_state_dict(dims, seed=0, only="gen_vision_model.")
    sdc = {k: v.cuda() for k, v in sd.items()}
    g = torch.Generator().manual_seed(5)
    codes = torch.randint(0, dims.img_vocab, (3, dims.n_img_tokens), generator=g, dtype=torch.int32)
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        want = O.decode_code(sdc, dims, codes.cuda(), [3, dims.code_dim, dims.grid, dims.grid]).float()
    eng = get_engine(dims, "bf16", with_vq=True)
    out = eng.gen_vision_model.decode_code(codes.cuda(), shape=[3, dims.code_dim, dims.grid, dims.grid]).float()
    # Two bf16 evaluations of this ~30-conv GroupNorm decoder differ by accumulated rounding noise: the
    # reference under autocast vs the reference in fp32 differ by max 6.5e-2 / mean 8e-3 on SMALL
    # (measured with the oracle on CPU), max|out| ~ 1.9.  Tolerance: rtol 2e-2 plus 5% of max|ref|
    # per element, and a mean error below 1% of max|ref|.
    a, b = out.cpu().numpy(), want.cpu().numpy()
    assert_close(a, b, 2e-2, 5e-2, "vq bf16")
    assert np.abs(a - b).mean() < 1e-2 * np.abs(b).max()
    # the convolution epilogue fused into the contraction (bias + skip + bf16 store) rounds at the same points as the
    # separate epilogue kernel it replaced: identical images with the switch off
    eng.set_option("fuse_conv_epilogue", 0)
    try:
        out2 = eng.gen_vision_model.decode_code(codes.cuda(), shape=[3, dims.code_dim, dims.grid, dims.grid]).float()
    finally:
        eng.set_option("fuse_conv_epilogue", 1)
    assert torch.equal(out, out2)


def test_t2i_end_to_end_small():
    """System.t2i shape/dtype contract + host-buffer entry."""
    d = O.SMALL
    eng = get_engine(d, "bf16", with_vq=True)
    cond, neg = O.synthetic_prompts(d, 2, seed=3, lo=9, hi=30, neg_len=11)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    dec, _ = eng.t2i(tokens=ids.cuda(), mask=mask.cuda(), cfg_weight=5.0, temperature=1.0)
    assert dec.shape == (2, 3, d.img_size, d.img_size) and dec.dtype == torch.bfloat16
    assert torch.isfinite(dec.float()).all()
    img = eng.generate_from_host(ids.pin_memory(), mask.pin_memory())
    assert img.dtype == torch.uint8 and img.shape == (2, 3, d.img_size, d.img_size) and not img.is_cuda
    # pg_images_to_u8 = denorm_pt + `(x*255).astype(np.uint8)` (src/utils/funcs.py:511-512, :497-498)
    want = (((dec.float().clamp(-1, 1) + 1) / 2) * 255).to(torch.uint8)
    assert torch.equal(eng.images_to_uint8(dec), want)
    edge = torch.tensor([-3.0, -1.0, -0.999, 0.0, 0.5, 0.9999, 1.0, 7.0, 0.25, -0.25, 0.1, 0.7], device="cuda").reshape(1, 3, 2, 2)
    assert torch.equal(eng.images_to_uint8(edge), (((edge.clamp(-1, 1) + 1) / 2) * 255).to(torch.uint8))


def test_save_images_writes_the_decoded_pixels(tmp_path):
    """PNG side of the result writers (plangen_base.py:1174-1177): files hold exactly denorm_pt(dec) * 255 truncated."""
    from plangen_b200.prompts import save_images
    d = O.SMALL
    eng = get_engine(d, "bf16", with_vq=True)
    codes = torch.randint(0, d.img_vocab, (2, d.n_img_tokens), dtype=torch.int32, device="cuda")
    dec = eng.gen_vision_model.decode_code(codes, shape=[2, d.code_dim, d.grid, d.grid])
    paths = save_images(eng, dec, str(tmp_path / "pr_{}.png"), start_index=5)
    assert [os.path.basename(p) for p in paths] == ["pr_5.png", "pr_6.png"]
    try:
        from PIL import Image
    except ImportError:
        pytest.skip("PIL not installed")
    want = eng.images_to_uint8(dec).permute(0, 2, 3, 1).cpu().numpy()
    for i, p in enumerate(paths):
        assert np.array_equal(np.asarray(Image.open(p)), want[i])


@pytest.mark.parametrize("path", ["perop_v5", "perop_plain"])
def test_bf16_long_ragged_context(path):
    """Long, ragged prompts (many 32-token KV tiles per row, cond/uncond lengths very different) through the
    TMA-staged decode attention and through the plain attention kernel: CFG logits vs the autocast reference on
    the same GPU, teacher-forced."""
    attn_impl = {"perop_v5": 3, "perop_plain": 0}[path]
    dims = O.SMALL
    steps = 10
    sd = O.init_state_dict(dims, seed=0, with_vq=False)
    sdc = {k: v.cuda() for k, v in sd.items()}
    g = torch.Generator().manual_seed(3)
    lens = [211, 37, 160, 1, 97]
    cond = [torch.randint(0, dims.vocab - 2, (n,), generator=g).tolist() for n in lens]
    neg = [torch.randint(0, dims.vocab - 2, (29,), generator=g).tolist()] * len(lens)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    trace = {}
    ref_tok, _ = O.t2i(sdc, dims, ids.cuda(), mask.cuda(), sampler=O.greedy_sampler, mode="autocast",
                       image_token_num_per_image=steps, decode=False, trace=trace)
    ref_logits = torch.stack(trace["logits"]).numpy()
    eng = get_engine(dims, "bf16", with_vq=False, max_batch=8, max_prompt=256)
    eng.set_option("attn_impl", attn_impl)
    dbg = torch.zeros(steps, len(lens), dims.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())
    try:
        emb = eng.language_model.get_input_embeddings()(ids.cuda())
        forced = {"edit_region": torch.zeros(len(lens), steps, dtype=torch.int32)}
        eng.sample_image(emb, len(lens), steps, mask.cuda(), 5.0, 1.0, generator=0, batch=forced, gt_labels=ref_tok,
                         greedy=True, use_teacher_forcing=True)
        torch.cuda.synchronize()
    finally:
        eng.set_option("dbg_logits_ptr", 0)
        eng.set_option("attn_impl", 3)
    assert_close(dbg.cpu().numpy(), ref_logits, 2e-2, 2e-2, f"bf16 long-context CFG logits ({path})")


def test_packed_prefill_is_bit_identical_to_padded_prefill():
    """The fused loops prefill the real tokens only (packed row after row, lm_kernels.cuh packed_row_of); the reference runs
    the LEFT-padded (R, P) block.  Pad positions never reach a real position, and every real position goes through the same
    arithmetic in the same order, so the CFG logits of the following steps are bit-identical with packing on and off (rows
    with 1 token, rows without padding, tiles straddling the first real column)."""
    dims = O.SMALL
    steps = 4
    g = torch.Generator().manual_seed(12)
    lens = [200, 1, 129, 128, 77, 255, 256, 3]
    cond = [torch.randint(0, dims.vocab - 2, (n,), generator=g).tolist() for n in lens]
    neg = [torch.randint(0, dims.vocab - 2, (31,), generator=g).tolist()] * len(lens)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    eng = get_engine(dims, "bf16", with_vq=False, max_batch=8, max_prompt=256)
    outs, toks = [], []
    # third pass: V from the key-contiguous copy instead of the cache rows read in place (MN-major operand, the default);
    # fourth: SwiGLU as its own kernel instead of in the gate|up contraction's epilogue
    # fifth: RoPE + q / cache stores as their own kernel instead of in the QKV contraction's epilogue (also with the padded block)
    for pack, v_direct, swiglu_fuse, qkv_fuse in ((1, 1, 1, 1), (0, 1, 1, 1), (1, 0, 1, 1), (1, 1, 0, 1), (1, 1, 1, 0), (0, 1, 1, 0)):
        eng.set_option("prefill_pack", pack)
        eng.set_option("prefill_v_direct", v_direct)
        eng.set_option("prefill_swiglu_fuse", swiglu_fuse)
        eng.set_option("prefill_qkv_fuse", qkv_fuse)
        dbg = torch.zeros(steps, len(lens), dims.img_vocab, device="cuda")
        eng.set_option("dbg_logits_ptr", dbg.data_ptr())
        try:
            emb = eng.language_model.get_input_embeddings()(ids.cuda())
            toks.append(eng.sample_image(emb, len(lens), steps, mask.cuda(), 5.0, 1.0, generator=0).cpu())
            torch.cuda.synchronize()
        finally:
            eng.set_option("dbg_logits_ptr", 0)
            eng.set_option("prefill_pack", 1)
            eng.set_option("prefill_v_direct", 1)
            eng.set_option("prefill_swiglu_fuse", 1)
            eng.set_option("prefill_qkv_fuse", 1)
        outs.append(dbg.cpu())
    for k in (1, 2, 3, 4, 5):
        assert torch.equal(outs[0], outs[k]) and torch.equal(toks[0], toks[k]), k
    # and for the text prefill of language_model.generate (mask-aware RoPE positions)
    sd = O.init_state_dict(dims, seed=0, with_vq=False, with_lm_head=True)
    from plangen_b200.engine import FastJanus
    from tests.gpu_util import product_dims
    te = FastJanus(sd, product_dims(dims), mode="bf16", max_batch=4, max_prompt=256, max_steps=32, with_vq=False)
    tid, tmask = O.pad_input_ids([c[:n] for c, n in zip(cond, (200, 1, 64, 130, 9, 255, 256, 3))], dims.pad_id)
    got = []
    for pack, qkv_fuse in ((1, 1), (0, 1), (1, 0)):
        te.set_option("prefill_pack", pack)
        te.set_option("prefill_qkv_fuse", qkv_fuse)
        emb = te.language_model.get_input_embeddings()(tid.cuda())
        got.append(te.language_model.generate(inputs_embeds=emb, attention_mask=tmask.cuda(), pad_token_id=7, eos_token_id=7,
                                              max_new_tokens=8).cpu())
    te.set_option("prefill_qkv_fuse", 1)
    assert torch.equal(got[0], got[1]) and torch.equal(got[0], got[2])


def test_prefill_row_dedup_is_bit_identical():
    """Rows that repeat an earlier row (PlanGen's unconditional rows all carry the same negative prompt, cfg/base.py:129;
    `parallel_size` > 1 repeats whole batches) are prefilled once and their K / V strips copied (lm_kernels.cuh
    kv_broadcast_rows_kernel).  Mixed batch: six prompts share a negative prompt (rows 1, 3, 5, 7, 11, 15), two carry their
    own (one of the same length), one conditional prompt appears three times (rows 0, 2, 10); the CFG logits of the following
    steps and the sampled tokens are bit-identical with `prefill_dedup` / `attn_alias` on and off."""
    dims = O.SMALL
    steps = 5
    g = torch.Generator().manual_seed(77)
    rnd = lambda n: torch.randint(0, dims.vocab - 2, (n,), generator=g).tolist()
    a, shared = rnd(60), rnd(23)
    # prompts 0 and 1 are the same text (rows 0 / 2 repeat); prompt 3 has the same length as 2 but other tokens; prompt 7
    # shares only a suffix with prompt 6
    cond = [a, list(a), rnd(200), rnd(200), rnd(5), list(a), rnd(256), None]
    cond[7] = rnd(196) + cond[6][-60:]
    neg = [shared, shared, shared, shared, rnd(23), shared, rnd(9), shared]
    lens = [len(c) for c in cond]
    ids, mask = O.t2i_infer_collate_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    eng = get_engine(dims, "bf16", with_vq=False, max_batch=8, max_prompt=256)
    outs, toks = [], []
    for dedup, alias in ((1, 1), (0, 1), (1, 0)):
        eng.set_option("prefill_dedup", dedup)
        eng.set_option("attn_alias", alias)           # decode attention reads a duplicate row's prompt K / V from its source row
        dbg = torch.zeros(steps, len(lens), dims.img_vocab, device="cuda")
        eng.set_option("dbg_logits_ptr", dbg.data_ptr())
        try:
            emb = eng.language_model.get_input_embeddings()(ids.cuda())
            toks.append(eng.sample_image(emb, len(lens), steps, mask.cuda(), 5.0, 1.0, generator=3).cpu())
            torch.cuda.synchronize()
        finally:
            eng.set_option("dbg_logits_ptr", 0)
            eng.set_option("prefill_dedup", 1)
            eng.set_option("attn_alias", 1)
        outs.append(dbg.cpu())
    assert torch.equal(outs[0], outs[1]) and torch.equal(toks[0], toks[1])
    assert torch.equal(outs[0], outs[2]) and torch.equal(toks[0], toks[2])
    assert float(outs[0].abs().max()) > 0
    # identical adjacent-pair rows in a text prefill (rows r and r - 2 the same prompt)
    sd = O.init_state_dict(dims, seed=0, with_vq=False, with_lm_head=True)
    from plangen_b200.engine import FastJanus
    from tests.gpu_util import product_dims
    te = FastJanus(sd, product_dims(dims), mode="bf16", max_batch=6, max_prompt=256, max_steps=32, with_vq=False)
    tid, tmask = O.pad_input_ids([cond[0], cond[2], cond[0], cond[2][:150], cond[0], cond[4]], dims.pad_id)
    got = []
    for dedup in (1, 0):
        te.set_option("prefill_dedup", dedup)
        emb = te.language_model.get_input_embeddings()(tid.cuda())
        got.append(te.language_model.generate(inputs_embeds=emb, attention_mask=tmask.cuda(), pad_token_id=7, eos_token_id=7,
                                              max_new_tokens=8).cpu())
    assert torch.equal(got[0], got[1])
    assert torch.equal(got[0][0], got[0][2]) and torch.equal(got[0][0], got[0][4])
    # parallel_size = 2 (plangen_base.py:547-549: the whole (2B, P) block repeated): every row of the second copy repeats a
    # row 2B earlier; same images with the shortcut on and off, and the two copies differ (independent sampling)
    ve = get_engine(dims, "bf16", with_vq=True, max_batch=8, max_prompt=256)
    ids4, mask4 = O.t2i_infer_collate_batch(cond[2:5], neg[2:5], dims.pad_id, dims.n_img_tokens)
    imgs = []
    for dedup in (1, 0):
        ve.set_option("prefill_dedup", dedup)
        try:
            dec, _ = ve.t2i(tokens=ids4.cuda(), mask=mask4.cuda(), parallel_size=2, image_token_num_per_image=dims.n_img_tokens)
        finally:
            ve.set_option("prefill_dedup", 1)
        imgs.append(dec.float().cpu())
    assert imgs[0].shape[0] == 6 and torch.equal(imgs[0], imgs[1])
    assert not torch.equal(imgs[0][:3], imgs[0][3:])


@pytest.mark.parametrize("B", [5, 16, 32])
def test_bf16_streamk_gate_up_matches_reference(B):
    """Stream-K gate|up + SwiGLU (gemm_sk.cuh; the default for Janus-Pro-7B, forced here): token tiles of 16 / 32 / 64
    rows, unit ranges of one or two k-blocks (176 units over 148 CTAs: up to eight partial contributors per tile,
    fragments whose only k-block falls to one MMA issuer): CFG logits vs the autocast reference on the same GPU,
    teacher-forced, and deterministic across runs."""
    dims = O.SMALL
    steps = 6
    sd = O.init_state_dict(dims, seed=0, with_vq=False)
    sdc = {k: v.cuda() for k, v in sd.items()}
    g = torch.Generator().manual_seed(40 + B)
    lens = torch.randint(5, 120, (B,), generator=g).tolist()
    cond = [torch.randint(0, dims.vocab - 2, (n,), generator=g).tolist() for n in lens]
    neg = [torch.randint(0, dims.vocab - 2, (17,), generator=g).tolist()] * B
    ids, mask = O.t2i_infer_collate_batch(cond, neg, dims.pad_id, dims.n_img_tokens)
    trace = {}
    ref_tok, _ = O.t2i(sdc, dims, ids.cuda(), mask.cuda(), sampler=O.greedy_sampler, mode="autocast",
                       image_token_num_per_image=steps, decode=False, trace=trace)
    ref_logits = torch.stack(trace["logits"]).numpy()
    eng = get_engine(dims, "bf16", with_vq=False, max_batch=32, max_prompt=128)
    eng.set_option("gu_streamk", 2)
    try:
        outs = []
        for _ in range(2):
            dbg = torch.zeros(steps, B, dims.img_vocab, device="cuda")
            eng.set_option("dbg_logits_ptr", dbg.data_ptr())
            emb = eng.language_model.get_input_embeddings()(ids.cuda())
            forced = {"edit_region": torch.zeros(B, steps, dtype=torch.int32)}
            eng.sample_image(emb, B, steps, mask.cuda(), 5.0, 1.0, generator=0, batch=forced, gt_labels=ref_tok, greedy=True,
                             use_teacher_forcing=True)
            torch.cuda.synchronize()
            outs.append(dbg.cpu().numpy())
    finally:
        eng.set_option("dbg_logits_ptr", 0)
        eng.set_option("gu_streamk", 1)
    assert np.array_equal(outs[0], outs[1]), "stream-K gate|up is not deterministic"
    assert_close(outs[0], ref_logits, 2e-2, 2e-2, f"bf16 CFG logits, stream-K gate|up, B={B}")


def test_fp32_t2i_parallel_size_two_matches_oracle():
    """System.t2i with parallel_size = 2 (plangen_base.py:547-549: ids and mask tiled, num_gen = B * parallel_size
    images sampled in one batch from one Philox stream): token ids identical to the oracle, images within fp32 noise."""
    d = O.SMALL
    sd = O.init_state_dict(d, seed=0, with_vq=True)
    eng = get_engine(d, "fp32", with_vq=True)
    cond, neg = O.synthetic_prompts(d, 2, seed=31, lo=9, hi=33, neg_len=11)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    sms, mt = _num_sms()
    want_tok, want_img = O.t2i(sd, d, ids, mask, parallel_size=2, sampler=PX.PhiloxSampler(0, sms, mt), mode="fp32")
    dec, _ = eng.t2i(tokens=ids.cuda(), mask=mask.cuda(), parallel_size=2, cfg_weight=5.0, temperature=1.0)
    assert eng.last_tokens.shape == (4, d.n_img_tokens)
    assert eng.last_tokens.cpu().tolist() == want_tok.tolist()
    assert not torch.equal(eng.last_tokens[:2], eng.last_tokens[2:])          # the two copies are different samples
    err = (dec.float().cpu() - want_img).abs().max().item()
    assert err < 1e-3 * want_img.abs().max().item() + 1e-4, err
