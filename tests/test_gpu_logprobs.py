"""-m gpu: image-token log-probabilities from the fused sampler and the teacher-forced scorer.

The reference is tests/logprob_ref.py: log_softmax of the filtered scaled CFG logits (tests/per_image_ref.py) gathered
at the emitted token.  Rows whose nucleus boundary is ambiguous are excused as in test_gpu_top_p / test_gpu_per_image."""
import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200 import _lib
from tests import logprob_ref as LR
from tests import per_image_ref as PR
from tests.gpu_util import get_engine, product_dims

pytestmark = pytest.mark.gpu


def _mixed(B):
    return dict(cfg_weight=[(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)],
                temperature=[(1.0, 0.7, 1.3)[b % 3] for b in range(B)],
                top_k=[(0, 50, 1000)[(b // 2) % 3] for b in range(B)],
                top_p=[(1.0, 0.9, 0.5)[(b + 1) % 3] for b in range(B)])


def _tiny(V):
    return O.JanusDims(**{**O.TINY.__dict__, "name": f"tiny-v{V}", "img_vocab": V})


def _logits(B, V, step, tg):
    logits = torch.randn(2 * B, V, device="cuda", generator=tg) * 0.5
    if step == 1:                                       # every logit tied with another one: ties at the boundary
        logits[:, : V // 2] = logits[:, V // 2: 2 * (V // 2)]
    return logits


def _check_lp(got, want, excused, what, tol=1e-5):
    keep = ~excused
    g, w = got[keep], want[keep]
    assert torch.equal(torch.isneginf(g), torch.isneginf(w)), what
    fin = torch.isfinite(w)
    assert torch.isfinite(g[fin]).all(), what
    if fin.any():
        err = (g[fin] - w[fin]).abs().max().item()
        assert err <= tol, f"{what}: log-prob error {err:.3e}"


@pytest.mark.parametrize("greedy", [0, 1])
@pytest.mark.parametrize("rng_per_image", [0, 1])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,V", [(1, 16384), (3, 16384), (16, 16384), (20, 16384), (3, 2048), (20, 2048)])
def test_kernel_logprobs_match_torch_and_leave_tokens_alone(greedy, rng_per_image, mode, B, V):
    eng = get_engine(_tiny(V), mode, max_batch=20, with_vq=False)
    s = _mixed(B)
    tg = torch.Generator(device="cuda").manual_seed(300 + B)
    seeds = [1000 + 7 * b for b in range(B)] if rng_per_image else 77
    n_steps = 3
    a = torch.zeros(B, n_steps, dtype=torch.int32, device="cuda")
    b_ = torch.zeros(B, n_steps, dtype=torch.int32, device="cuda")
    lp = torch.full((B, n_steps), 7.0, device="cuda")
    top_p = [1.0] * B if greedy else s["top_p"]          # greedy: top-k only, as the draw
    for step in range(n_steps):
        logits = _logits(B, V, step, tg)
        offs = [4 * step] * B if rng_per_image else 4 * step
        xa = eng.cfg_sample_embed(logits, s["cfg_weight"], s["temperature"], seeds, offs, step, n_steps, a, greedy=bool(greedy),
                                  top_k=s["top_k"], top_p=s["top_p"])
        xb = eng.cfg_sample_embed(logits, s["cfg_weight"], s["temperature"], seeds, offs, step, n_steps, b_, greedy=bool(greedy),
                                  top_k=s["top_k"], top_p=s["top_p"], logprobs_out=lp)
        torch.cuda.synchronize()
        assert torch.equal(a[:, step], b_[:, step]) and torch.equal(xa, xb), (mode, B, V, step)
        t = PR.scaled_cfg(logits, mode, s["cfg_weight"], s["temperature"])
        want = LR.logprobs_of(PR.filter_rows(t, s["top_k"], top_p), b_[:, step])
        _check_lp(lp[:, step], want, PR.ambiguous_rows(t, s["top_k"], top_p), f"{mode} B={B} V={V} step {step}")
        assert torch.isfinite(lp[:, step]).all()         # sampled tokens are never removed


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_kernel_forced_tokens_removed_are_minus_inf_and_far_tail_is_finite(mode):
    B, V = 4, 16384
    eng = get_engine(_tiny(V), mode, max_batch=20, with_vq=False)
    tg = torch.Generator(device="cuda").manual_seed(17)
    s = dict(cfg_weight=[5.0, 5.0, 3.0, 5.0], temperature=[1.0, 0.7, 1.0, 1.3], top_k=[50, 0, 0, 0], top_p=[1.0, 0.5, 1.0, 1.0])
    logits = torch.randn(2 * B, V, device="cuda", generator=tg) * 0.5
    logits[6, 123], logits[7, 123] = -30.0, 0.0         # image 3: t = 5 * -30 = -150 below ~0, still kept
    t = PR.scaled_cfg(logits, mode, s["cfg_weight"], s["temperature"])
    filt = PR.filter_rows(t, s["top_k"], s["top_p"])
    gt = torch.tensor([int(t[0].argmin()), int(t[1].argmin()), int(t[2].argmax()), 123], dtype=torch.int32, device="cuda")
    assert torch.isinf(filt[0, gt[0]]) and torch.isinf(filt[1, gt[1]])
    assert (t[3, 123] - t[3].max()).item() < -100
    er = torch.zeros(B, 1, dtype=torch.int32, device="cuda")
    toks = torch.zeros(B, 1, dtype=torch.int32, device="cuda")
    lp = torch.zeros(B, 1, device="cuda")
    eng.cfg_sample_embed(logits, s["cfg_weight"], s["temperature"], 5, 0, 0, 1, toks, edit_region=er,
                         gt_labels=gt.view(B, 1), top_k=s["top_k"], top_p=s["top_p"], logprobs_out=lp)
    torch.cuda.synchronize()
    assert toks.view(-1).tolist() == gt.tolist()
    want = LR.logprobs_of(filt, gt)
    assert torch.isneginf(lp[0, 0]) and torch.isneginf(lp[1, 0])
    assert torch.isfinite(lp[2:, 0]).all() and lp[3, 0].item() < -100
    assert (lp[2:, 0] - want[2:]).abs().max().item() <= 1e-5


def _small_batch(d, B, n=None):
    cond, neg = O.synthetic_prompts(d, B, lo=20, hi=60, neg_len=12)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, n or d.n_img_tokens)
    return ids.cuda(), mask.cuda()


def _gens(seeds):
    return [torch.Generator(device="cuda").manual_seed(s) for s in seeds]


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_loop_logprobs_leave_tokens_alone_graph_equals_plain(mode):
    d, steps, B = O.SMALL, 7, 3
    eng = get_engine(d, mode, with_vq=False)
    ids, mask = _small_batch(d, B)
    s = _mixed(B)
    er = torch.ones(B, steps, dtype=torch.int32)
    er[:, ::3] = 0
    gt = torch.randint(0, d.img_vocab, (B, steps), dtype=torch.int32)
    cases = [dict(cfg_weight=5.0, temperature=1.0, generator=3, top_k=50, top_p=0.9),
             dict(cfg_weight=s["cfg_weight"], temperature=s["temperature"], generator=[11, 22, 33], top_k=s["top_k"],
                  top_p=s["top_p"]),
             dict(cfg_weight=s["cfg_weight"], temperature=s["temperature"], generator=[11, 22, 33], top_k=s["top_k"],
                  top_p=s["top_p"], batch={"edit_region": er}, gt_labels=gt, use_teacher_forcing=True)]
    for c in cases:
        runs = []
        for graph, lps in ((1, False), (1, True), (0, False), (0, True)):
            eng.set_option("use_graph", graph)
            try:
                c2 = dict(c)
                if isinstance(c2["generator"], list):
                    c2["generator"] = list(c2["generator"])
                emb = eng.language_model.get_input_embeddings()(ids)
                runs.append(eng.sample_image(emb, B, steps, mask, c2.pop("cfg_weight"), c2.pop("temperature"),
                                             return_logprobs=lps, **c2))
            finally:
                eng.set_option("use_graph", 1)
        toks = [r[0] if isinstance(r, tuple) else r for r in runs]
        assert all(torch.equal(toks[0], t) for t in toks), (mode, c.keys())
        assert torch.equal(runs[1][1], runs[3][1])                       # graph replay == plain launches, bit for bit
        assert torch.isfinite(runs[1][1][er.cuda() != 0] if "batch" in c else runs[1][1]).all()


def test_new_settings_with_logprobs_replay_the_same_graph():
    d, steps, B = O.SMALL, 5, 3
    eng = get_engine(d, "bf16", max_batch=3, with_vq=False, cache=False)
    ids, mask = _small_batch(d, B)
    calls = [dict(cfg_weight=[3.0, 5.0, 7.5], temperature=[1.0, 0.7, 1.3], top_k=[0, 50, 100], top_p=[0.9, 1.0, 0.5]),
             dict(cfg_weight=[1.0, 2.0, 4.0], temperature=[1.3, 1.0, 0.8], top_k=[10, 0, 5], top_p=[1.0, 0.6, 0.95])]
    before = eng.counter("graph_captures")
    for i, c in enumerate(calls):
        emb = eng.language_model.get_input_embeddings()(ids)
        eng.sample_image(emb, B, steps, mask, c["cfg_weight"], c["temperature"], generator=[i, i + 1, i + 2], top_k=c["top_k"],
                         top_p=c["top_p"], return_logprobs=True)
    assert eng.counter("graph_captures") - before == 1


def test_fp32_loop_logprobs_match_the_oracle_loop():
    d, steps, B = O.SMALL, 6, 3
    eng = get_engine(d, "fp32", with_vq=False)
    sd = {k: v.cuda() for k, v in O.init_state_dict(d, seed=0, with_vq=False).items()}
    ids, mask = _small_batch(d, B)
    s = {"cfg_weight": [3.0, 5.0, 7.5], "temperature": [1.0, 0.7, 1.3], "top_k": [0, 50, 100], "top_p": [0.9, 1.0, 0.5]}
    seeds = [11, 22, 33]
    want_t, want_lp = LR.loop_ref(sd, d, ids, mask, steps, generator=_gens(seeds), **s)
    emb = eng.language_model.get_input_embeddings()(ids)
    got_t, got_lp = eng.sample_image(emb, B, steps, mask, s["cfg_weight"], s["temperature"], generator=_gens(seeds),
                                     top_k=s["top_k"], top_p=s["top_p"], return_logprobs=True)
    assert got_t.tolist() == want_t.tolist()
    bound = 2e-4 / torch.tensor(s["temperature"], device="cuda")[:, None]
    assert ((got_lp - want_lp).abs() <= bound).all(), (got_lp - want_lp).abs().max()


def _score_setup(d, mode, B, n, max_prompt=128):
    eng = get_engine(d, mode, with_vq=False, max_prompt=max_prompt)
    sd = {k: v.cuda() for k, v in O.init_state_dict(d, seed=0, with_vq=False).items()}
    ids, mask = _small_batch(d, B, n)
    img = torch.randint(0, d.img_vocab, (B, n), generator=torch.Generator().manual_seed(4)).cuda()
    return eng, sd, ids, mask, img


def test_fp32_scorer_matches_full_forward_teacher_forced_loop_and_its_own_samples():
    d, B, n = O.SMALL, 3, 8
    eng, sd, ids, mask, img = _score_setup(d, "fp32", B, n)
    s = {"cfg_weight": [3.0, 5.0, 7.5], "temperature": [1.0, 0.7, 1.3], "top_k": [0, 0, 0], "top_p": [1.0, 1.0, 1.0]}
    bound = 2e-4 / torch.tensor(s["temperature"], device="cuda")[:, None]
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, **s)
    want = LR.score_ref(sd, d, ids, mask, img, **s)
    assert ((got - want).abs() <= bound).all(), (got - want).abs().max()
    # the engine's own teacher-forced loop on the same tokens (edit_region all 0)
    emb = eng.language_model.get_input_embeddings()(ids)
    forced = {"edit_region": torch.zeros(B, n, dtype=torch.int32)}
    t_loop, lp_loop = eng.sample_image(emb, B, n, mask, s["cfg_weight"], s["temperature"], generator=[1, 2, 3], batch=forced,
                                       gt_labels=img, use_teacher_forcing=True, return_logprobs=True)
    assert torch.equal(t_loop, img.int())
    assert ((got - lp_loop).abs() <= bound).all(), (got - lp_loop).abs().max()
    # self-consistency: score the loop's own samples
    emb = eng.language_model.get_input_embeddings()(ids)
    t_s, lp_s = eng.sample_image(emb, B, n, mask, s["cfg_weight"], s["temperature"], generator=[5, 6, 7], return_logprobs=True)
    again = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=t_s, **s)
    assert ((again - lp_s).abs() <= bound).all(), (again - lp_s).abs().max()


def test_scorer_filters_give_minus_inf_exactly_where_the_reference_removes():
    d, B, n = O.SMALL, 3, 8
    eng, sd, ids, mask, img = _score_setup(d, "fp32", B, n)
    s = {"cfg_weight": [3.0, 5.0, 5.0], "temperature": [1.0, 0.7, 1.0], "top_k": [50, 0, 1000], "top_p": [1.0, 0.5, 0.9]}
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, **s)
    want = LR.score_ref(sd, d, ids, mask, img, **s)
    assert torch.isneginf(want).any() and torch.isfinite(want).any()
    assert torch.equal(torch.isneginf(got), torch.isneginf(want))
    fin = torch.isfinite(want)
    bound = (2e-4 / torch.tensor(s["temperature"], device="cuda")[:, None]).expand_as(want)
    assert ((got[fin] - want[fin]).abs() <= bound[fin]).all()


def test_bf16_scorer_small_dims_vs_autocast_oracle():
    d, B, n = O.SMALL, 2, 8
    eng, sd, ids, mask, img = _score_setup(d, "bf16", B, n)
    s = {"cfg_weight": [5.0, 3.0], "temperature": [1.0, 0.7], "top_k": [0, 0], "top_p": [1.0, 1.0]}
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, **s)
    want = LR.score_ref(sd, d, ids, mask, img, mode="autocast", **s)
    want32 = LR.score_ref(sd, d, ids, mask, img, mode="fp32", **s)
    # log p moves by at most twice the largest CFG-logit error; §2's logit bound is 2e-2 of the logit range, divided by T
    rng = 1.0 + (want32.max() - want32.min()).item()
    bound = 2 * 2e-2 * rng / torch.tensor(s["temperature"], device="cuda")[:, None]
    assert ((got - want).abs() <= bound).all(), (got - want).abs().max()
    assert (got - want32).abs().mean() <= 1.25 * (want - want32).abs().mean() + 1e-6


def test_scorer_failures_name_the_limit_and_the_argument():
    d, B, n = O.SMALL, 2, 8
    eng, sd, ids, mask, img = _score_setup(d, "fp32", B, n, max_prompt=64)
    P = ids.shape[1]
    big = 64 - P + 2                                    # P + n - 1 = 65 > max_prompt
    if big <= eng.max_steps:
        ids2, mask2 = _small_batch(d, B, big)
        with pytest.raises(_lib.PgError, match="max_prompt"):
            eng.score_image_tokens(tokens=ids2, mask=mask2[:, : P + big], image_tokens=torch.zeros(B, big, dtype=torch.int64))
    with pytest.raises(ValueError, match="image_tokens"):
        eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img + d.img_vocab)
    with pytest.raises(ValueError, match="image_tokens"):
        eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img[:1])
    with pytest.raises(ValueError, match="mask"):
        eng.score_image_tokens(tokens=ids, mask=mask[:, :-1], image_tokens=img)
    with pytest.raises(ValueError, match="max_steps"):
        eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=torch.zeros(B, eng.max_steps + 1, dtype=torch.int64))


def test_fullsize_scorer_vs_autocast_reference_and_sampled_logprobs_finite():
    from plangen_b200 import synthetic
    from plangen_b200.engine import FastJanus
    d = O.JANUS_1P3B
    pd = product_dims(d)
    B, n = 2, 48
    sd = synthetic.random_state_dict(pd, torch.device("cuda", 0), seed=0, with_vq=False)
    eng = FastJanus(sd, pd, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
    cond, neg = synthetic.layoutsam_prompts(pd, B, seed=1234, lo=150, hi=400)
    ids, mask = synthetic.collate_cfg_batch(cond, neg, pd.pad_id, n)
    ids, mask = ids.cuda(), mask.cuda()
    img = torch.randint(0, pd.img_vocab, (B, n), generator=torch.Generator().manual_seed(9)).cuda()
    s = {"cfg_weight": [5.0, 5.0], "temperature": [1.0, 1.0], "top_k": [0, 0], "top_p": [1.0, 1.0]}
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, **s).cpu().numpy()
    ref16 = LR.score_ref(sd, d, ids, mask, img, mode="autocast", **s).cpu().numpy()
    ref32 = LR.score_ref(sd, d, ids, mask, img, mode="fp32", **s).cpu().numpy()
    e_mine, e_ref = np.abs(got - ref32), np.abs(ref16 - ref32)
    add = max(2e-2 * np.abs(ref16).max(), 2.0 * np.quantile(e_ref, 0.999))
    frac_ok = float((np.abs(got - ref16) <= 2e-2 * np.abs(ref16) + add).mean())
    assert frac_ok >= 0.999, frac_ok
    assert e_mine.mean() <= 1.25 * e_ref.mean(), (e_mine.mean(), e_ref.mean())
    assert np.quantile(e_mine, 0.999) <= 1.25 * np.quantile(e_ref, 0.999), (np.quantile(e_mine, 0.999), np.quantile(e_ref, 0.999))
    emb = eng.language_model.get_input_embeddings()(ids)
    _, lp = eng.sample_image(emb, B, 6, mask, 5.0, 1.0, generator=0, return_logprobs=True)
    assert torch.isfinite(lp).all()
