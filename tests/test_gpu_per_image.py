"""-m gpu: per-image seeds, guidance scale, temperature, top-k and top-p within one image batch.

The reference for every check is tests/per_image_ref.py: each row with its own scalars (the scalar path's rounding), HF's
filter idiom, softmax, then torch.multinomial on the row alone with its own generator (per-image RNG) or on the whole
batch with one generator (batch-wide RNG).  Rows whose nucleus boundary is ambiguous are excused as in test_gpu_top_p."""
import ctypes as C
import math

import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200 import _lib
from tests import per_image_ref as PR
from tests.gpu_util import get_engine, product_dims
from tests.test_gpu_top_p import _Tally

pytestmark = pytest.mark.gpu


def _mixed(B):
    return dict(cfg_weight=[(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)],
                temperature=[(1.0, 0.7, 1.3)[b % 3] for b in range(B)],
                top_k=[(0, 50, 1000)[(b // 2) % 3] for b in range(B)],
                top_p=[(1.0, 0.9, 0.5)[(b + 1) % 3] for b in range(B)])


def _tiny(V):
    return O.JanusDims(**{**O.TINY.__dict__, "name": f"tiny-v{V}", "img_vocab": V})


def _logits(B, V, step, tg, t_of=None):
    logits = torch.randn(2 * B, V, device="cuda", generator=tg) * 0.5
    if step == 1:                                       # every logit tied with another one: ties at the boundary
        logits[:, : V // 2] = logits[:, V // 2: 2 * (V // 2)]
    if step == 2 and t_of is not None:                  # tied maxima
        m = t_of(logits).argmax(-1)
        for b in range(B):
            for j in (3, V // 3, V - 2):
                logits[2 * b: 2 * b + 2, j] = logits[2 * b: 2 * b + 2, m[b]]
    return logits


@pytest.mark.parametrize("rng_per_image", [0, 1])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("B,V", [(1, 16384), (3, 16384), (16, 16384), (20, 16384), (3, 2048), (20, 2048)])
def test_kernel_mixed_settings_match_per_row_torch(rng_per_image, mode, B, V):
    eng = get_engine(_tiny(V), mode, max_batch=20, with_vq=False)
    s = _mixed(B)
    tg = torch.Generator(device="cuda").manual_seed(200 + B)
    if rng_per_image:
        seeds = [1000 + 7 * b for b in range(B)]
        twins = [torch.Generator(device="cuda").manual_seed(x) for x in seeds]
    else:
        seeds, twins = 77, torch.Generator(device="cuda").manual_seed(77)
    n_steps, tally = 4, _Tally()
    toks = torch.zeros(B, n_steps, dtype=torch.int32, device="cuda")
    t_of = lambda lg: PR.scaled_cfg(lg, mode, s["cfg_weight"], s["temperature"])
    for step in range(n_steps):
        logits = _logits(B, V, step, tg, t_of)
        offs = [g.get_offset() for g in twins] if rng_per_image else twins.get_offset()
        t = t_of(logits)
        filt = PR.filter_rows(t, s["top_k"], s["top_p"])
        want = PR.draw(filt, twins)
        eng.cfg_sample_embed(logits, s["cfg_weight"], s["temperature"], seeds, offs, step, n_steps, toks,
                             top_k=s["top_k"], top_p=s["top_p"])
        torch.cuda.synchronize()
        tally.check(toks[:, step], want.int(), ~torch.isinf(filt), PR.ambiguous_rows(t, s["top_k"], s["top_p"]),
                    f"{mode} B={B} V={V} rng_per_image={rng_per_image} step {step}")
    tally.done(f"{mode} B={B} V={V} rng_per_image={rng_per_image}")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_kernel_uniform_lists_are_the_scalar_path(mode):
    B, V = 16, 16384
    eng = get_engine(_tiny(V), mode, max_batch=20, with_vq=False)
    tg = torch.Generator(device="cuda").manual_seed(5)
    for cfg, temp, k, p in ((5.0, 1.0, 0, 1.0), (3.0, 0.7, 50, 0.9), (7.5, 1.3, 1000, 0.5)):
        for step in range(3):
            logits = _logits(B, V, step, tg)
            outs = []
            for per_image in (False, True):
                toks = torch.zeros(B, 3, dtype=torch.int32, device="cuda")
                kw = dict(cfg_weight=[cfg] * B, temperature=[temp] * B, top_k=[k] * B, top_p=[p] * B) if per_image else \
                    dict(cfg_weight=cfg, temperature=temp, top_k=k, top_p=p)
                x = eng.cfg_sample_embed(logits, kw.pop("cfg_weight"), kw.pop("temperature"), 41, 12 * step, step, 3, toks, **kw)
                outs.append((toks.clone(), x))
            assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), (cfg, temp, k, p, step)


def test_kernel_b1_per_image_generator_is_the_scalar_path():
    V = 16384
    eng = get_engine(_tiny(V), "bf16", max_batch=20, with_vq=False)
    tg = torch.Generator(device="cuda").manual_seed(9)
    for step in range(4):
        logits = _logits(1, V, step, tg)
        a = torch.zeros(1, 4, dtype=torch.int32, device="cuda")
        b = torch.zeros(1, 4, dtype=torch.int32, device="cuda")
        xa = eng.cfg_sample_embed(logits, 5.0, 0.7, 123, 4 * step + 8, step, 4, a, top_k=50, top_p=0.9)
        xb = eng.cfg_sample_embed(logits, [5.0], [0.7], [123], [4 * step + 8], step, 4, b, top_k=[50], top_p=[0.9])
        assert torch.equal(a, b) and torch.equal(xa, xb)


def test_kernel_token_does_not_depend_on_position_or_batch_size():
    V = 16384
    eng = get_engine(_tiny(V), "bf16", max_batch=20, with_vq=False)
    tg = torch.Generator(device="cuda").manual_seed(13)
    pair = torch.randn(2, V, device="cuda", generator=tg)
    n_steps = 5
    seen = {}
    for B, pos in ((1, 0), (5, 2), (16, 0), (16, 15), (20, 9)):
        s = _mixed(B)
        s["cfg_weight"][pos], s["temperature"][pos], s["top_k"][pos], s["top_p"][pos] = 3.0, 0.7, 1000, 0.9
        toks = torch.zeros(B, n_steps, dtype=torch.int32, device="cuda")
        for step in range(n_steps):
            logits = torch.randn(2 * B, V, device="cuda", generator=tg)
            logits[2 * pos: 2 * pos + 2] = pair
            seeds = [500 + b for b in range(B)]
            seeds[pos] = 4242
            offs = [40 + 4 * step] * B
            eng.cfg_sample_embed(logits, s["cfg_weight"], s["temperature"], seeds, offs, step, n_steps, toks,
                                 top_k=s["top_k"], top_p=s["top_p"])
        seen[(B, pos)] = toks[pos].tolist()
    assert len({tuple(v) for v in seen.values()}) == 1, seen


def _small_batch(d, B):
    cond, neg = O.synthetic_prompts(d, B, lo=20, hi=60, neg_len=12)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    return ids.cuda(), mask.cuda()


def _gens(seeds, predraw=0):
    out = []
    for i, s in enumerate(seeds):
        g = torch.Generator(device="cuda").manual_seed(s)
        if predraw:                                     # a generator that has already drawn
            torch.rand(predraw + 100 * i, device="cuda", generator=g)
        out.append(g)
    return out


def test_fp32_loop_mixed_settings_generators_graph_plain_and_editing():
    d, steps, B = O.SMALL, 8, 3
    eng = get_engine(d, "fp32", with_vq=False)
    sd = {k: v.cuda() for k, v in O.init_state_dict(d, seed=0, with_vq=False).items()}
    ids, mask = _small_batch(d, B)
    s = {"cfg_weight": [3.0, 5.0, 7.5], "temperature": [1.0, 0.7, 1.3], "top_k": [0, 50, 100], "top_p": [0.9, 1.0, 0.5]}
    seeds = [11, 22, 33]
    twins = _gens(seeds, predraw=1000)
    want = PR.t2i_tokens(sd, d, ids, mask, steps, s["cfg_weight"], s["temperature"], s["top_k"], s["top_p"], twins)
    runs = []
    for graph in (1, 0, 1):
        eng.set_option("use_graph", graph)
        try:
            gens = _gens(seeds, predraw=1000)
            emb = eng.language_model.get_input_embeddings()(ids)
            runs.append(eng.sample_image(emb, B, steps, mask, s["cfg_weight"], s["temperature"], generator=gens,
                                         top_k=s["top_k"], top_p=s["top_p"]).cpu())
            # each generator moved on as by `steps` torch.multinomial draws on a (1, img_vocab) tensor
            assert [g.get_offset() for g in gens] == [g.get_offset() for g in twins]
        finally:
            eng.set_option("use_graph", 1)
    assert runs[0].tolist() == want.cpu().tolist()
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])
    # editing: teacher forcing composes (forced columns take the ground truth, the others match the reference)
    er = torch.ones(B, steps, dtype=torch.int32)
    er[:, ::3] = 0
    gt = torch.randint(0, d.img_vocab, (B, steps), dtype=torch.int32)
    want_e = PR.t2i_tokens(sd, d, ids, mask, steps, s["cfg_weight"], s["temperature"], s["top_k"], s["top_p"],
                           _gens(seeds), edit_region=er, gt_labels=gt.cuda())
    emb = eng.language_model.get_input_embeddings()(ids)
    got_e = eng.sample_image(emb, B, steps, mask, s["cfg_weight"], s["temperature"], generator=_gens(seeds),
                             batch={"edit_region": er}, gt_labels=gt, use_teacher_forcing=True, top_k=s["top_k"],
                             top_p=s["top_p"]).cpu()
    assert got_e.tolist() == want_e.cpu().tolist()
    assert bool((got_e[er == 0] == gt[er == 0]).all())


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_loop_uniform_lists_and_b1_generator_are_the_scalar_path(mode):
    d, steps = O.SMALL, 6
    eng = get_engine(d, mode, with_vq=False)
    for graph in (1, 0):
        eng.set_option("use_graph", graph)
        try:
            B = 2
            ids, mask = _small_batch(d, B)
            emb = eng.language_model.get_input_embeddings()(ids)
            a = eng.sample_image(emb, B, steps, mask, 3.0, 0.7, generator=7, top_k=50, top_p=0.9)
            emb = eng.language_model.get_input_embeddings()(ids)
            b = eng.sample_image(emb, B, steps, mask, [3.0] * B, [0.7] * B, generator=7, top_k=[50] * B, top_p=[0.9] * B)
            assert torch.equal(a, b), (mode, graph)
            # B = 1: one generator per image is the scalar path with that generator
            ids, mask = _small_batch(d, 1)
            ga, gb = _gens([99]), _gens([99])
            emb = eng.language_model.get_input_embeddings()(ids)
            a = eng.sample_image(emb, 1, steps, mask, 5.0, 1.0, generator=ga[0], top_p=0.9)
            emb = eng.language_model.get_input_embeddings()(ids)
            b = eng.sample_image(emb, 1, steps, mask, 5.0, 1.0, generator=gb, top_p=0.9)
            assert torch.equal(a, b) and ga[0].get_offset() == gb[0].get_offset(), (mode, graph)
        finally:
            eng.set_option("use_graph", 1)


def test_new_seeds_and_settings_replay_the_same_graph():
    d, steps, B = O.SMALL, 5, 3
    eng = get_engine(d, "bf16", max_batch=3, with_vq=False, cache=False)
    ids, mask = _small_batch(d, B)
    calls = [dict(cfg_weight=[3.0, 5.0, 7.5], temperature=[1.0, 0.7, 1.3], top_k=[0, 50, 100], top_p=[0.9, 1.0, 0.5],
                  seeds=[1, 2, 3]),
             dict(cfg_weight=[1.0, 2.0, 4.0], temperature=[1.3, 1.0, 0.8], top_k=[10, 0, 5], top_p=[1.0, 0.6, 0.95],
                  seeds=[4, 5, 6])]

    def run(c):
        emb = eng.language_model.get_input_embeddings()(ids)
        return eng.sample_image(emb, B, steps, mask, c["cfg_weight"], c["temperature"], generator=_gens(c["seeds"]),
                                top_k=c["top_k"], top_p=c["top_p"]).cpu()

    before = eng.counter("graph_captures")
    got = [run(c) for c in calls]
    assert eng.counter("graph_captures") - before == 1
    eng.set_option("use_graph", 0)
    try:
        plain = [run(c) for c in calls]
    finally:
        eng.set_option("use_graph", 1)
    assert torch.equal(got[0], plain[0]) and torch.equal(got[1], plain[1])
    assert not torch.equal(got[0], got[1])


def test_fullsize_mixed_settings_per_image_generators_match_torch_and_are_deterministic():
    from plangen_b200 import synthetic
    from plangen_b200.engine import FastJanus
    d = product_dims(O.JANUS_1P3B)
    B, steps = 16, 6
    sd = synthetic.random_state_dict(d, torch.device("cuda", 0), seed=0, with_vq=False)
    eng = FastJanus(sd, d, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
    del sd
    cond, neg = synthetic.layoutsam_prompts(d, B, seed=1234, lo=150, hi=480)
    ids, mask = synthetic.collate_cfg_batch(cond, neg, d.pad_id, d.n_img_tokens)
    ids, mask = ids.cuda(), mask.cuda()
    s = _mixed(B)
    seeds = [300 + 17 * b for b in range(B)]

    def run():
        emb = eng.language_model.get_input_embeddings()(ids)
        return eng.sample_image(emb, B, steps, mask, s["cfg_weight"], s["temperature"], generator=_gens(seeds),
                                top_k=s["top_k"], top_p=s["top_p"]).cpu()

    dbg = torch.zeros(steps, B, d.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())
    try:
        got = run()
        torch.cuda.synchronize()
    finally:
        eng.set_option("dbg_logits_ptr", 0)
    twins = _gens(seeds)
    tally = _Tally()
    for st in range(steps):
        t = dbg[st]
        filt = PR.filter_rows(t, s["top_k"], s["top_p"])
        want = PR.draw(filt, twins)
        tally.check(got[:, st].cuda(), want.int(), ~torch.isinf(filt), PR.ambiguous_rows(t, s["top_k"], s["top_p"]),
                    f"full size step {st}")
    tally.done("full size")
    assert torch.equal(got, run())


def test_bad_sampling_entries_fail_naming_the_image():
    V = 2048
    eng = get_engine(_tiny(V), "fp32", max_batch=20, with_vq=False)
    B = 4
    logits = torch.randn(2 * B, V, device="cuda")
    t = torch.zeros(B, 1, dtype=torch.int32, device="cuda")
    x = torch.empty(2 * B, eng.dims.D, device="cuda")
    for field, bad in (("top_p", 1.5), ("top_p", -0.1), ("top_p", math.nan), ("top_k", -1)):
        arr = (_lib.PgImageSampling * B)()
        for b in range(B):
            arr[b] = _lib.PgImageSampling(b, 0, 5.0, 1.0, 0, 1.0)
        setattr(arr[3], field, bad)
        rc = eng._lib.pg_cfg_sample_embed(eng._h, C.c_void_p(logits.data_ptr()), B, arr, 1, 0, None, None, 0, 1,
                                          C.c_void_p(t.data_ptr()), C.c_void_p(x.data_ptr()), None, None)
        err = eng._lib.pg_last_error()
        assert rc != 0 and b"image 3" in err and field.encode() in err, err
        vals = {"top_k": [0] * B, "top_p": [1.0] * B}
        vals[field][3] = bad
        with pytest.raises(ValueError, match=r"\[3\]"):
            eng.cfg_sample_embed(logits, [5.0] * B, 1.0, 1, 0, 0, 1, t, **vals)
    # wrong length, a CPU generator, the same generator twice
    with pytest.raises(ValueError):
        eng.cfg_sample_embed(logits, [5.0] * (B - 1), 1.0, 1, 0, 0, 1, t)
    d = O.SMALL
    eng2 = get_engine(d, "fp32", with_vq=False)
    ids, mask = _small_batch(d, 2)
    emb = eng2.language_model.get_input_embeddings()(ids)
    g = torch.Generator(device="cuda").manual_seed(1)
    for gens in ([g, g], [torch.Generator().manual_seed(1), g], [g]):
        with pytest.raises(ValueError):
            eng2.sample_image(emb, 2, 3, mask, 5.0, 1.0, generator=gens)
