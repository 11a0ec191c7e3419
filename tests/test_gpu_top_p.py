"""-m gpu: top-p (nucleus) filtering in the fused CFG sampler, HF TopPLogitsWarper after TopKLogitsWarper.

The reference for every check is the torch idiom (tests/top_p_ref.py) on the same scaled CFG logits,
followed by softmax and torch.multinomial with the same generator.  Where the boundary of the nucleus sits within 1e-6
(fp64 cumulative mass) of the threshold, torch's fp32 cumsum order legitimately decides which tokens stay: a mismatch in
such a row is excused and counted, and more than 1 % excused rows fail the test."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200 import _lib
from tests import top_p_ref as R
from tests.gpu_util import get_engine, product_dims

pytestmark = pytest.mark.gpu

CFG_W = 5.0


def _scaled_cfg(logits, mode, temperature):
    """The kernel's t: CFG combine rounded per op in the engine's dtype, then a correctly rounded division by the
    temperature (a tensor divisor: torch divides by a Python scalar through its reciprocal)."""
    lg = logits.bfloat16() if mode == "bf16" else logits
    c, u = lg[0::2], lg[1::2]
    t = (u + CFG_W * (c - u)).float() / torch.tensor(temperature, device=logits.device)
    return t.bfloat16().float() if mode == "bf16" else t


def _ambiguous(t, top_k, top_p, tol=1e-6):
    """Rows whose fp64 cumulative mass, in the ascending order, comes within tol of fp32(1 - top_p) before the last."""
    t = R.top_k_top_p_filter(t, top_k, 1.0).double()
    s = torch.sort(t, dim=-1).values.softmax(-1).cumsum(-1)[:, :-1]
    thr = float(np.float32(1.0 - top_p))
    return ((s - thr).abs() < tol).any(-1)


class _Tally:
    def __init__(self):
        self.rows = self.excused = 0

    def check(self, got, want, kept, amb, what):
        inside = kept.gather(1, got[:, None].long()).squeeze(1)
        bad = (got != want) | ~inside
        assert not bool((bad & ~amb).any()), f"{what}: rows {torch.nonzero(bad & ~amb).flatten().tolist()}"
        self.rows += got.numel()
        self.excused += int((bad & amb).sum())

    def done(self, what):
        print(f"{what}: {self.excused} of {self.rows} rows excused (boundary within 1e-6 of the threshold)")
        assert self.excused <= 0.01 * self.rows


def test_torch_sort_orders_ties_by_index():
    """HF's order among equal logits is whatever torch.sort yields on the device; the kernel removes the lowest indices
    of the boundary tie group first, so torch.sort must keep index order within ties on (B, 16384) fp32 rows."""
    g = torch.Generator(device="cuda").manual_seed(3)
    for B in (3, 16, 20):
        x = (torch.randn(B, 16384, device="cuda", generator=g) * 2).bfloat16().float()
        x[:, 7::1000] = x.max()
        vals, idx = torch.sort(x, dim=-1, descending=False)
        same = vals[:, 1:] == vals[:, :-1]
        assert int(same.sum()) > 1000
        assert bool((idx[:, 1:][same] > idx[:, :-1][same]).all())


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,V", [(3, 16384), (16, 16384), (20, 16384), (4, 2048)])
def test_sampler_top_p_matches_torch_idiom_multinomial(mode, B, V):
    d = O.JanusDims(**{**O.TINY.__dict__, "name": f"tiny-v{V}", "img_vocab": V})
    eng = get_engine(d, mode, max_batch=max(B, 4), with_vq=False)
    tg = torch.Generator(device="cuda").manual_seed(100 + B)
    tally = _Tally()
    cases = [(p, k, temp) for p in (0.0, 0.3, 0.9, 0.999) for k in (0, 50) for temp in (1.0, 0.7)]
    n_steps = 4
    for p, k, temp in cases:
        gen = torch.Generator(device="cuda").manual_seed(77)
        toks = torch.zeros(B, n_steps, dtype=torch.int32, device="cuda")
        off = 0
        for step in range(n_steps):
            logits = torch.randn(2 * B, V, device="cuda", generator=tg) * 0.5
            if step == 1:                                   # every logit tied with another one: ties at the boundary
                logits[:, : V // 2] = logits[:, V // 2: 2 * (V // 2)]
            if step == 2:                                   # tied maxima
                m = _scaled_cfg(logits, mode, temp).argmax(-1)
                for b in range(B):
                    for j in (3, V // 3, V - 2):
                        logits[2 * b: 2 * b + 2, j] = logits[2 * b: 2 * b + 2, m[b]]
            t = _scaled_cfg(logits, mode, temp)
            filt = R.top_k_top_p_filter(t, k, p)
            want = torch.multinomial(torch.softmax(filt, -1), 1, generator=gen).squeeze(-1)
            eng.cfg_sample_embed(logits, CFG_W, temp, 77, off, step, n_steps, toks, top_k=k, top_p=p)
            torch.cuda.synchronize()
            tally.check(toks[:, step], want.int(), ~torch.isinf(filt), _ambiguous(t, k, p),
                        f"{mode} B={B} V={V} top_p={p} top_k={k} T={temp} step {step}")
            off = gen.get_offset()
    tally.done(f"{mode} B={B} V={V}")


def test_sampler_top_p_one_is_the_unfiltered_path_and_bad_values_fail():
    d = O.JanusDims(**{**O.TINY.__dict__, "name": "tiny-v16384", "img_vocab": 16384})
    eng = get_engine(d, "fp32", max_batch=4, with_vq=False)
    logits = torch.randn(8, 16384, device="cuda")
    outs, launches = [], []
    for kw in ({}, {"top_p": 1.0}):
        t = torch.zeros(4, 1, dtype=torch.int32, device="cuda")
        before = eng.counter("launches")
        eng.cfg_sample_embed(logits, CFG_W, 1.0, 5, 0, 0, 1, t, **kw)
        launches.append(eng.counter("launches") - before)
        outs.append(t.cpu())
    assert torch.equal(outs[0], outs[1]) and launches[0] == launches[1] == 1
    # greedy: top-p is skipped, the arg-max is always inside the nucleus
    g = [torch.zeros(4, 1, dtype=torch.int32, device="cuda") for _ in range(2)]
    eng.cfg_sample_embed(logits, CFG_W, 1.0, 5, 0, 0, 1, g[0], greedy=True)
    eng.cfg_sample_embed(logits, CFG_W, 1.0, 5, 0, 0, 1, g[1], greedy=True, top_p=0.3)
    assert torch.equal(g[0], g[1])
    t = torch.zeros(4, 1, dtype=torch.int32, device="cuda")
    for bad in (-0.1, 1.5, math.nan):
        with pytest.raises(ValueError):
            eng.cfg_sample_embed(logits, CFG_W, 1.0, 5, 0, 0, 1, t, top_p=bad)
        x = torch.empty(8, d.D, device="cuda")
        arr = (_lib.PgImageSampling * 4)(*[_lib.PgImageSampling(5, 0, CFG_W, 1.0, 0, bad)] * 4)
        rc = eng._lib.pg_cfg_sample_embed(eng._h, C.c_void_p(logits.data_ptr()), 4, arr, 0, 0, None, None, 0, 1,
                                          C.c_void_p(t.data_ptr()), C.c_void_p(x.data_ptr()), None, None)
        assert rc != 0 and b"top_p" in eng._lib.pg_last_error()


def _small_batch(d, B):
    cond, neg = O.synthetic_prompts(d, B, lo=20, hi=60, neg_len=12)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    return ids.cuda(), mask.cuda()


def test_fp32_loop_top_p_matches_oracle_graph_plain_and_editing():
    d, steps, B = O.SMALL, 8, 2
    eng = get_engine(d, "fp32", with_vq=False)
    sd = {k: v.cuda() for k, v in O.init_state_dict(d, seed=0, with_vq=False).items()}
    ids, mask = _small_batch(d, B)
    want = R.t2i_tokens(sd, d, ids, mask, steps, top_k=100, top_p=0.8, seed=0)
    runs = []
    for graph in (1, 0, 1):
        eng.set_option("use_graph", graph)
        try:
            emb = eng.language_model.get_input_embeddings()(ids)
            runs.append(eng.sample_image(emb, B, steps, mask, 5.0, 1.0, generator=0, top_k=100, top_p=0.8).cpu())
        finally:
            eng.set_option("use_graph", 1)
    assert runs[0].tolist() == want.cpu().tolist()
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])      # plain launches, replay determinism
    # editing: teacher forcing composes with top-p (forced columns take the ground truth, the others match the oracle)
    er = torch.ones(B, steps, dtype=torch.int32)
    er[:, ::3] = 0
    gt = torch.randint(0, d.img_vocab, (B, steps), dtype=torch.int32)
    want_e = R.t2i_tokens(sd, d, ids, mask, steps, top_k=100, top_p=0.8, seed=0, edit_region=er, gt_labels=gt.cuda())
    emb = eng.language_model.get_input_embeddings()(ids)
    got_e = eng.sample_image(emb, B, steps, mask, 5.0, 1.0, generator=0, batch={"edit_region": er}, gt_labels=gt,
                             use_teacher_forcing=True, top_k=100, top_p=0.8).cpu()
    assert got_e.tolist() == want_e.cpu().tolist()
    assert bool((got_e[er == 0] == gt[er == 0]).all())


def test_fullsize_top_p_tokens_inside_the_nucleus_and_deterministic():
    from plangen_b200 import synthetic
    from plangen_b200.engine import FastJanus
    d = product_dims(O.JANUS_1P3B)
    B, steps, p = 16, 6, 0.9
    sd = synthetic.random_state_dict(d, torch.device("cuda", 0), seed=0, with_vq=False)
    eng = FastJanus(sd, d, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
    del sd
    cond, neg = synthetic.layoutsam_prompts(d, B, seed=1234, lo=150, hi=480)
    ids, mask = synthetic.collate_cfg_batch(cond, neg, d.pad_id, d.n_img_tokens)
    ids, mask = ids.cuda(), mask.cuda()

    def run(**kw):
        emb = eng.language_model.get_input_embeddings()(ids)
        return eng.sample_image(emb, B, steps, mask, 5.0, 1.0, generator=0, **kw).cpu()

    dbg = torch.zeros(steps, B, d.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())
    try:
        got = run(top_p=p)
        torch.cuda.synchronize()
    finally:
        eng.set_option("dbg_logits_ptr", 0)
    tally = _Tally()
    for s in range(steps):
        t = dbg[s]
        kept = ~torch.isinf(R.top_k_top_p_filter(t, 0, p))
        tok = got[:, s].cuda()
        tally.check(tok, tok, kept, _ambiguous(t, 0, p), f"full size step {s}")
        assert int(kept.sum(-1).min()) >= 1
    tally.done("full size")
    assert torch.equal(got, run(top_p=p))
    assert torch.equal(run(), run(top_p=1.0))
