"""-m gpu: guidance schedules - a CFG weight per image and per step - in the image loop, its log-probs and the scorer.

The reference is tests/cfg_schedule_ref.py: step i of image b sampled and scored exactly as the per-image path does with
cfg_weight[b] = schedule[b][i].  Log-probs are held to the 2e-4 / temperature bound of test_gpu_logprobs."""
import ctypes as C
import math

import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200 import _lib
from plangen_b200.engine import OPS, kv_start_from_mask
from tests import cfg_schedule_ref as SR
from tests import per_image_ref as PR
from tests.gpu_util import get_engine, product_dims
from tests.test_gpu_top_p import _Tally

pytestmark = pytest.mark.gpu

S3 = {"temperature": [1.0, 0.7, 1.3], "top_k": [0, 50, 100], "top_p": [0.9, 1.0, 0.5]}
W3 = [3.0, 5.0, 7.5]
SEEDS = [11, 22, 33]
_SD = {}


def _sd(d):
    if d.name not in _SD:
        _SD[d.name] = {k: v.cuda() for k, v in O.init_state_dict(d, seed=0, with_vq=False).items()}
    return _SD[d.name]


def _small_batch(d, B, n):
    cond, neg = O.synthetic_prompts(d, B, lo=20, hi=60, neg_len=12)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, n)
    return ids.cuda(), mask.cuda()


def _gens(seeds):
    return [torch.Generator(device="cuda").manual_seed(s) for s in seeds]


def _schedules(n, w=W3, seed=0):
    """MAR's linear ramp from 1 to w, LlamaGen's interval (w, then 1 from step n // 2) and a random table."""
    w = torch.tensor(w)[:, None]
    return {"ramp": 1.0 + (w - 1.0) * torch.linspace(0, 1, n),
            "interval": torch.where(torch.arange(n) < n // 2, w, torch.tensor(1.0)),
            "random": torch.rand(len(w), n, generator=torch.Generator().manual_seed(seed)) * 8.0}


def _check_lp(got, want, temperature, what):
    assert torch.equal(torch.isneginf(got), torch.isneginf(want)), what
    fin = torch.isfinite(want)
    assert torch.isfinite(got[fin]).all(), what
    bound = (2e-4 / torch.tensor(temperature, device=got.device)[:, None]).expand_as(want)
    err = (got - want).abs()
    assert (err[fin] <= bound[fin]).all(), f"{what}: log-prob error {err[fin].max().item():.3e}"


def _sample(eng, ids, mask, steps, cfg_weight, s, **kw):
    emb = eng.language_model.get_input_embeddings()(ids)
    return eng.sample_image(emb, ids.shape[0] // 2, steps, mask, cfg_weight, s["temperature"], top_k=s["top_k"],
                            top_p=s["top_p"], **kw)


# ------------------------------------------------------------------------------------------- 1. fp32 loop vs the oracle
@pytest.mark.parametrize("name", ["ramp", "interval", "random"])
def test_fp32_loop_schedules_match_the_oracle_with_graph_and_plain_launches(name):
    d, steps, B = O.SMALL, 8, 3
    eng = get_engine(d, "fp32", with_vq=False)
    ids, mask = _small_batch(d, B, d.n_img_tokens)
    sched = _schedules(steps)[name]
    twins = _gens(SEEDS)
    want_t, want_lp = SR.loop_ref(_sd(d), d, ids, mask, steps, sched, generator=twins, **S3)
    for graph in (1, 0):
        eng.set_option("use_graph", graph)
        try:
            gens = _gens(SEEDS)
            got_t, got_lp = _sample(eng, ids, mask, steps, sched, S3, generator=gens, return_logprobs=True)
        finally:
            eng.set_option("use_graph", 1)
        assert got_t.tolist() == want_t.tolist(), (name, graph)
        # each generator moved on as by `steps` torch.multinomial draws on a (1, img_vocab) tensor
        assert [g.get_offset() for g in gens] == [g.get_offset() for g in twins], (name, graph)
        _check_lp(got_lp, want_lp, S3["temperature"], f"{name} graph={graph}")


def test_fp32_loop_schedule_with_teacher_forcing_and_greedy_matches_the_oracle():
    d, steps, B = O.SMALL, 8, 3
    eng = get_engine(d, "fp32", with_vq=False)
    ids, mask = _small_batch(d, B, d.n_img_tokens)
    sched = _schedules(steps)["random"]
    er = torch.ones(B, steps, dtype=torch.int32)
    er[:, ::3] = 0
    gt = torch.randint(0, d.img_vocab, (B, steps), dtype=torch.int32, generator=torch.Generator().manual_seed(2))
    twins = _gens(SEEDS)
    want_t, want_lp = SR.loop_ref(_sd(d), d, ids, mask, steps, sched, generator=twins, edit_region=er.cuda(),
                                  gt_labels=gt.cuda(), **S3)
    gens = _gens(SEEDS)
    got_t, got_lp = _sample(eng, ids, mask, steps, sched, S3, generator=gens, batch={"edit_region": er}, gt_labels=gt,
                            use_teacher_forcing=True, return_logprobs=True)
    assert got_t.tolist() == want_t.tolist()
    assert bool((got_t.cpu()[er == 0] == gt[er == 0]).all())
    assert [g.get_offset() for g in gens] == [g.get_offset() for g in twins]
    _check_lp(got_lp, want_lp, S3["temperature"], "teacher forcing")
    # greedy: the arg-max of the top-k-filtered scheduled distribution
    want_t, want_lp = SR.loop_ref(_sd(d), d, ids, mask, steps, sched, greedy=True, **S3)
    got_t, got_lp = _sample(eng, ids, mask, steps, sched, S3, generator=SEEDS, greedy=True, return_logprobs=True)
    assert got_t.tolist() == want_t.tolist()
    _check_lp(got_lp, want_lp, S3["temperature"], "greedy")


# ------------------------------------------------------------------------- 2. a constant schedule is the per-image path
def _c_abi_scheduled(eng, ids, mask, steps, sched, arr, rng_per_image=1):
    """pg_sample_image with a schedule, called directly (tokens, log-probs and the return code)."""
    emb = eng.language_model.get_input_embeddings()(ids)
    R, P, _ = emb.shape
    x = emb.contiguous().clone()
    kv = kv_start_from_mask(mask, P)
    toks = torch.zeros(R // 2, steps, dtype=torch.int32, device="cuda")
    lp = torch.zeros(R // 2, steps, device="cuda")
    sched = sched.float().contiguous()
    p = lambda t: C.c_void_p(t.data_ptr())
    rc = eng._lib.pg_sample_image(eng._h, p(x), p(kv), R, P, steps, arr, rng_per_image, 0, None, None, p(sched), p(toks),
                                  p(lp), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, toks, lp


def _arr(s, seeds, cfg_weight):
    arr = (_lib.PgImageSampling * len(seeds))()
    for b, seed in enumerate(seeds):
        arr[b] = _lib.PgImageSampling(seed, 0, cfg_weight, s["temperature"][b], s["top_k"][b], s["top_p"][b])
    return arr


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_constant_schedule_samples_as_per_image_weights_bit_for_bit(mode):
    d, steps, B = O.SMALL, 6, 3
    eng = get_engine(d, mode, with_vq=False)
    ids, mask = _small_batch(d, B, d.n_img_tokens)
    const = torch.tensor(W3)[:, None].expand(B, steps)
    for graph in (1, 0):
        eng.set_option("use_graph", graph)
        try:
            runs = []
            for cw in (W3, const):
                gens = _gens(SEEDS)
                t, lp = _sample(eng, ids, mask, steps, cw, S3, generator=gens, return_logprobs=True)
                t2 = _sample(eng, ids, mask, steps, cw, S3, generator=_gens(SEEDS))          # without log-probs
                runs.append((t, lp, t2, [g.get_offset() for g in gens]))
        finally:
            eng.set_option("use_graph", 1)
        (ta, la, ua, oa), (tb, lb, ub, ob) = runs
        assert torch.equal(ta, tb) and torch.equal(la, lb) and torch.equal(ua, ub) and oa == ob, (mode, graph)
        assert torch.equal(ta, ua)
    # at the C-ABI, with every per-image cfg_weight NaN: no read site falls back to the struct
    rc, toks, lp = _c_abi_scheduled(eng, ids, mask, steps, const, _arr(S3, SEEDS, math.nan))
    assert rc == 0, eng._lib.pg_last_error()
    want_t, want_lp = _sample(eng, ids, mask, steps, W3, S3, generator=SEEDS, return_logprobs=True)
    assert torch.equal(toks, want_t) and torch.equal(lp, want_lp)


# ------------------------------------------------------------------------------------------------------ 3. graph reuse
def test_new_schedules_replay_the_same_graph():
    d, steps, B = O.SMALL, 5, 3
    eng = get_engine(d, "bf16", max_batch=3, with_vq=False, cache=False)
    ids, mask = _small_batch(d, B, d.n_img_tokens)
    sch = _schedules(steps)
    calls = [sch["ramp"], sch["random"]]
    run = lambda s: _sample(eng, ids, mask, steps, s, S3, generator=[1, 2, 3]).cpu()
    before = eng.counter("graph_captures")
    got = [run(s) for s in calls]
    assert eng.counter("graph_captures") - before == 1
    eng.set_option("use_graph", 0)
    try:
        plain = [run(s) for s in calls]
    finally:
        eng.set_option("use_graph", 1)
    assert torch.equal(got[0], plain[0]) and torch.equal(got[1], plain[1])
    assert not torch.equal(got[0], got[1])


# ---------------------------------------------------------------------------------------------------------- 4. scorer
def _score_setup(d, mode, B, n, max_prompt=128, max_batch=4):
    eng = get_engine(d, mode, with_vq=False, max_prompt=max_prompt, max_batch=max_batch)
    ids, mask = _small_batch(d, B, n)
    img = torch.randint(0, d.img_vocab, (B, n), generator=torch.Generator().manual_seed(4)).cuda()
    return eng, ids, mask, img


NOFILTER3 = {"temperature": [1.0, 0.7, 1.3], "top_k": [0, 0, 0], "top_p": [1.0, 1.0, 1.0]}


def test_fp32_scheduled_scorer_matches_full_forward_teacher_forced_loop_and_its_own_samples():
    d, B, n = O.SMALL, 3, 8
    eng, ids, mask, img = _score_setup(d, "fp32", B, n)
    s = NOFILTER3
    sched = _schedules(n)["random"]
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=sched, **s)
    _check_lp(got, SR.score_ref(_sd(d), d, ids, mask, img, sched, **s), s["temperature"], "vs full forward")
    # the engine's own teacher-forced scheduled loop on the same tokens (edit_region all 0)
    forced = {"edit_region": torch.zeros(B, n, dtype=torch.int32)}
    t_loop, lp_loop = _sample(eng, ids, mask, n, sched, s, generator=[1, 2, 3], batch=forced, gt_labels=img,
                              use_teacher_forcing=True, return_logprobs=True)
    assert torch.equal(t_loop, img.int())
    _check_lp(got, lp_loop, s["temperature"], "vs teacher-forced loop")
    # self-consistency: score the loop's own samples
    t_s, lp_s = _sample(eng, ids, mask, n, sched, s, generator=[5, 6, 7], return_logprobs=True)
    again = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=t_s, cfg_weight=sched, **s)
    _check_lp(again, lp_s, s["temperature"], "own samples")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_constant_schedule_scorer_is_the_per_image_scorer(mode):
    d, B, n = O.SMALL, 3, 8
    eng, ids, mask, img = _score_setup(d, mode, B, n)
    a = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=W3, **S3)
    b = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=torch.tensor(W3)[:, None].expand(B, n),
                               **S3)
    assert torch.equal(a, b), mode


def test_scheduled_scorer_over_several_gen_head_chunks():
    # pg_score_image_tokens runs gen_head over at most part_bytes / (img_vocab * 4) rows at a time.  At SMALL dims with
    # max_batch 8 and max_prompt 128 the gen_aligner table's img_vocab * D * 4 bytes set part_bytes: 512 rows, so the
    # 2B * n = 576 rows run in two chunks and the second starts mid-image (pair 256 = image 7, position 4).
    d, B, n = O.SMALL, 8, 36
    eng, ids, mask, img = _score_setup(d, "fp32", B, n, max_batch=8)
    w = [3.0, 5.0, 7.5, 2.0] * 2
    s = {"temperature": [1.0, 0.7, 1.3, 1.0] * 2, "top_k": [0] * B, "top_p": [1.0] * B}
    sched = _schedules(n, w=w)["random"]
    got = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=sched, **s)
    _check_lp(got, SR.score_ref(_sd(d), d, ids, mask, img, sched, **s), s["temperature"], "two chunks")
    const = torch.tensor(w)[:, None].expand(B, n)
    a = eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=w, **s)
    assert torch.equal(a, eng.score_image_tokens(tokens=ids, mask=mask, image_tokens=img, cfg_weight=const, **s))


# ------------------------------------------------------------------------------------------------ 5. full size, bf16
def test_fullsize_bf16_schedule_columns_land_on_their_steps_and_tokens_match_torch():
    from plangen_b200 import synthetic
    from plangen_b200.engine import FastJanus
    d = product_dims(O.JANUS_1P3B)
    B, steps, k = 16, 6, 3
    sd = synthetic.random_state_dict(d, torch.device("cuda", 0), seed=0, with_vq=False)
    eng = FastJanus(sd, d, mode="bf16", max_batch=B, max_prompt=512, with_vq=False)
    del sd
    cond, neg = synthetic.layoutsam_prompts(d, B, seed=1234, lo=150, hi=480)
    ids, mask = synthetic.collate_cfg_batch(cond, neg, d.pad_id, d.n_img_tokens)
    ids, mask = ids.cuda(), mask.cuda()
    s = dict(temperature=[(1.0, 0.7, 1.3)[b % 3] for b in range(B)], top_k=[(0, 50, 1000)[(b // 2) % 3] for b in range(B)],
             top_p=[(1.0, 0.9, 0.5)[(b + 1) % 3] for b in range(B)])
    w = torch.tensor([(1.0, 3.0, 5.0, 7.5)[b % 4] for b in range(B)])[:, None]
    sa = 1.0 + (w - 1.0) * torch.linspace(0, 1, steps)
    sb = sa.clone()
    sb[:, k:] += 0.5                                    # agrees with sa on the columns < k only
    seeds = [300 + 17 * b for b in range(B)]
    dbg = torch.zeros(steps, B, d.img_vocab, device="cuda")
    eng.set_option("dbg_logits_ptr", dbg.data_ptr())

    def run(sched):
        got = _sample(eng, ids, mask, steps, sched, s, generator=_gens(seeds)).cpu()
        torch.cuda.synchronize()
        return got, dbg.clone()

    try:
        (ta, la), (tb, lb) = run(sa), run(sb)
        again, _ = run(sa)
    finally:
        eng.set_option("dbg_logits_ptr", 0)
    assert torch.equal(la[:k], lb[:k]) and torch.equal(ta[:, :k], tb[:, :k])
    assert bool((la[k] != lb[k]).any(dim=-1).all())      # every image's step-k logits moved with its column k
    tally = _Tally()
    for toks, lg in ((ta, la), (tb, lb)):
        twins = _gens(seeds)
        for st in range(steps):
            t = lg[st]
            filt = PR.filter_rows(t, s["top_k"], s["top_p"])
            want = PR.draw(filt, twins)
            tally.check(toks[:, st].cuda(), want.int(), ~torch.isinf(filt), PR.ambiguous_rows(t, s["top_k"], s["top_p"]),
                        f"full size step {st}")
    tally.done("full size schedules")
    assert torch.equal(ta, again)


# ---------------------------------------------------------------------------------------------------------- 6. failures
def test_bad_schedules_fail_naming_the_image_and_step_at_the_single_entry_points():
    d, B, steps = O.SMALL, 3, 4
    eng = get_engine(d, "fp32", with_vq=False)
    ids, mask = _small_batch(d, B, d.n_img_tokens)
    arr = _arr(S3, SEEDS, 5.0)
    P = 8
    x_seq = torch.zeros(2 * B, P + steps - 1, d.D, device="cuda")
    kv0 = torch.zeros(2 * B, dtype=torch.int32, device="cuda")
    img = torch.zeros(B, steps, dtype=torch.int32, device="cuda")
    lp = torch.zeros(B, steps, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    for bad in (math.nan, math.inf, -math.inf):
        sched = torch.full((B, steps), 5.0)
        sched[1, 2] = bad
        rc, _, _ = _c_abi_scheduled(eng, ids, mask, steps, sched, arr)
        err = eng._lib.pg_last_error()
        assert rc != 0 and b"image 1, step 2" in err, err
        rc = eng._lib.pg_score_image_tokens(eng._h, p(x_seq), p(kv0), 2 * B, P, steps, p(img), arr, p(sched), p(lp), None)
        err = eng._lib.pg_last_error()
        assert rc != 0 and b"image 1, step 2" in err, err
        with pytest.raises(ValueError, match=r"cfg_weight\[1, 2\]"):
            _sample(eng, ids, mask, steps, sched, S3)
        with pytest.raises(ValueError, match=r"cfg_weight\[1, 2\]"):
            _sample(eng, ids, mask, steps, sched.tolist(), S3)
    # n past max_steps
    n_big = eng.max_steps + 1
    rc, _, _ = _c_abi_scheduled(eng, ids, mask, n_big, torch.full((B, n_big), 5.0), arr)
    assert rc != 0 and b"n_steps" in eng._lib.pg_last_error()
    with pytest.raises(_lib.PgError, match="n_steps"):
        _sample(eng, ids, mask, n_big, torch.full((B, n_big), 5.0), S3)
    # wrong shapes: in sample_image, and at the op (which passes the table to the C-ABI as a host array)
    for bad in (torch.ones(B, steps + 1), torch.ones(B + 1, steps), torch.ones(B, steps, 1), [[5.0] * steps] * (B - 1)):
        with pytest.raises(ValueError, match="cfg_weight"):
            _sample(eng, ids, mask, steps, bad, S3)
    emb = eng.language_model.get_input_embeddings()(ids)
    kv = kv_start_from_mask(mask, emb.shape[1])
    toks = torch.zeros(B, steps, dtype=torch.int32, device="cuda")
    for bad in (torch.ones(B, steps + 1), torch.ones(B, steps, device="cuda"), torch.ones(B, steps, dtype=torch.float64)):
        with pytest.raises(ValueError, match="cfg_schedule"):
            OPS.sample_image(eng.handle, emb.clone(), kv, steps, [5.0] * B, S3["temperature"], S3["top_k"], S3["top_p"], SEEDS,
                             [0] * B, True, False, None, None, toks, bad, None)
