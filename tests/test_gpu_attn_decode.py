"""-m gpu: the decode-attention kernels against an fp64 reference of their own operation (tests/attn_ref.py).

Each case launches one decode attention exactly as a decode step does (pg_test_attn_decode_io) on operands the test owns:
split-K QKV partials, a KV cache, kv_start, and optionally a source row per row whose prompt columns are read instead of
the row's own (prefill de-duplication).  Compared: attn_decode_v5_kernel (impl 3, bf16) and the plain attn_decode_kernel
(impl 0, bf16 and fp32, with T-splits).

Tolerance, |got - ref| <= 2^-8 |ref| + 1e-4 max|V of the item|:
  * the kernel's output is an fp32 value rounded to bf16 with RNE.  For |x| in [2^e, 2^(e+1)) the rounding moves x by at
    most half an ulp, 2^(e-8) <= 2^-8 |x|;
  * the fp32 value is an online softmax: q . k in fp32 (128 products), exp2 of score differences, and a P.V sum
    rescaled at every new maximum and merged over warps, groups and contributors.  Its error is a few fp32 ulps of the
    scores (relative ~1e-6 on each weight, also at |s| ~ 80) and of the accumulated sum, which is a convex combination
    of V: far below 1e-4 max|V|.  That term also covers the output's rounding where half an ulp equals 2^-8 |x|.
q, k_new and v_new are not part of the error: the reference restates their rounding op for op, and the new cache column
must hold them bit for bit.

Teeth: every case also asserts, on the reference side, that dropping any single boundary token (the first valid column,
the edges of its tile, the first column of the last tile, pos - 1, alias_P - 1 / alias_P, the new token) moves some
output of the item outside this tolerance.  Keys aligned with q are planted on those columns (or, with all-equal scores,
large values), so a kernel that lost one of them fails.

Integrity on every launch: left-pad columns [0, kv_start), column pos and the columns after it are NaN before the
launch (a masked ring slot still enters o += 0 * v, so an over-read shows as NaN); the output must be finite; the cache is
bitwise unchanged except column pos, which holds exactly the reference's k_new / v_new; v5's hand-off records are all
zero afterwards and a guard region after them is untouched; a second launch gives a bitwise-equal output."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200.config import Dims
from plangen_b200.weights import rope_tables
from tests import attn_ref as A
from tests.gpu_util import assert_close, get_engine

pytestmark = pytest.mark.gpu

REL = A.ROPE_REL
WS_REC = A.AT_MAX_SLOTS * (A.HEAD_DIM + 2)           # hand-off words per item
GUARD = 4096
DEVICE = "cuda"


def _eng(dtype):
    if dtype == "bf16":                                 # up to 256 rows, positions up to 2239 (RoPE tables)
        return get_engine(O.TINY, "bf16", max_batch=128, max_prompt=2176, with_vq=False)
    return get_engine(O.TINY, "fp32", max_batch=32, max_prompt=1024, with_vq=False)


def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _launch(eng, impl, splits, part, R, H, kc, vc, ks, src, alias_P, pos_arg, step, rope, ctas, out, ws):
    from plangen_b200 import _lib
    _lib.check(eng._lib.pg_test_attn_decode_io(eng._h, impl, splits, _p(part), part.shape[0], R, H, _p(kc), _p(vc), kc.shape[2],
                                               _p(ks), _p(src), alias_P, pos_arg, _p(step), rope, ctas, _p(out), _p(ws),
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream)))


def _starts(kind, R, pos, g):
    if isinstance(kind, list):
        return kind
    if kind == "edges":                                 # 0, 31, 32, 33, one cached token, an empty row, ...
        base = [0, 31, 32, 33, pos - 1, pos, 17, pos // 2]
        return [min(base[r % len(base)], pos) for r in range(R)]
    if kind == "cfg":                                   # long cond rows, short uncond rows
        return [0 if r % 2 == 0 else max(pos - 29, 0) for r in range(R)]
    if kind == "ragged":                                # any start in [0, pos], empty rows included
        return torch.randint(0, pos + 1, (R,), generator=g).tolist()
    assert kind == "dense"
    return [0] * R


def _case(impl=3, R=2, H=2, starts="ragged", pos=100, S=1, ctas=0, rope=1, step=None, mode="rand", alias=None,
          splits=0, dtype="bf16", seed=0):
    return dict(impl=impl, R=R, H=H, starts=starts, pos=pos, S=S, ctas=ctas, rope=rope, step=step, mode=mode, alias=alias,
                splits=splits, dtype=dtype, seed=seed)


def _run(c):
    """Build the operands of case c, plant the boundary tokens, launch twice (and once more without aliasing when the
    duplicates are real copies) and check everything."""
    eng = _eng(c["dtype"])
    bf = c["dtype"] == "bf16"
    cdt = torch.bfloat16 if bf else torch.float32
    R, H, pos, S = c["R"], c["H"], c["pos"], c["S"]
    HD = H * A.HEAD_DIM
    g = torch.Generator().manual_seed(1000 + c["seed"])
    ks = _starts(c["starts"], R, pos, g)
    Tmax = pos + 6                                      # any Tmax; columns after pos exist and are poisoned
    alias = c["alias"]
    src = list(alias["src"]) if alias else None
    aP = alias["P"] if alias else 0
    sq, sk = {"rand": (math.sqrt(3.0),) * 2, "peak": (math.sqrt(80.0),) * 2, "equal": (0.0, 1.0)}[c["mode"]]
    part = torch.randn(S, R, 3, H, A.HEAD_DIM, generator=g) / math.sqrt(S)
    part[:, :, 0] *= sq
    part[:, :, 1] *= sk
    kc = (torch.randn(R, H, Tmax, A.HEAD_DIM, generator=g) * sk).to(cdt).float()
    vc = torch.randn(R, H, Tmax, A.HEAD_DIM, generator=g).to(cdt).float()
    if alias:
        for r, s in enumerate(src):
            if s != r:
                assert ks[r] == ks[s]
                part[:, r, 0] = part[:, s, 0]           # duplicates ask the same query of the same prompt
    cos, sin = rope_tables(Dims.from_any(O.TINY), eng.counter("tmax"))
    part = part.view(S, R, 3 * HD)
    q, _, _ = A.qkv_new(part, H, cos, sin, pos, ks, c["rope"], bf)

    # ---- plant the boundary tokens: keys aligned with q half a nat above the item's best random score (or, when every
    #      score is equal, large values), so that losing any one of them is visible
    K0 = A.effective_cache(kc, src, aP)
    pv = part.view(S, R, 3, H, A.HEAD_DIM)
    for r in range(R):
        st = ks[r]
        cols = A.boundary_columns(st, pos, aP)
        owner = lambda j: src[r] if (alias and j < aP) else r
        if c["mode"] == "equal":
            for j in cols:
                vc[owner(j), :, j] = (8.0 * torch.randn(H, A.HEAD_DIM, generator=g)).to(cdt).float()
            pv[:, r, 2] *= 8.0
            continue
        qn2 = (q[r].double() ** 2).sum(-1)                                        # [H]
        s_rand = torch.einsum("hnd,hd->hn", K0[r, :, st:pos].double(), q[r].double()) / math.sqrt(A.HEAD_DIM)
        t = (s_rand.amax(-1) if pos > st else torch.zeros(H, dtype=torch.float64)) + 0.5
        coef = t * math.sqrt(A.HEAD_DIM) / qn2                                    # k = coef * q  =>  score = t
        for j in cols:
            kc[owner(j), :, j] = (q[r].double() * coef[:, None]).to(cdt).float()
        pv[:, r, 1] = pv[:, r, 0] * coef[None, :, None].float()                   # k_new ~ coef * q
    q, k_new, v_new = A.qkv_new(part, H, cos, sin, pos, ks, c["rope"], bf)
    if alias and alias.get("copies"):                   # real copies: reading the source row changes nothing
        for r, s in enumerate(src):
            kc[r, :, :aP] = kc[s, :, :aP]
            vc[r, :, :aP] = vc[s, :, :aP]

    # ---- poison what the kernel must not read
    for r in range(R):
        kc[r, :, :ks[r]] = float("nan"); vc[r, :, :ks[r]] = float("nan")
        kc[r, :, pos:] = float("nan"); vc[r, :, pos:] = float("nan")
        if alias and alias.get("poison") and src[r] != r:
            kc[r, :, ks[r]:aP] = float("nan"); vc[r, :, ks[r]:aP] = float("nan")

    ref, vmax = A.attention(q, k_new, v_new, kc, vc, ks, pos, src, aP)
    assert torch.isfinite(ref).all()
    assert A.undetected_drops(q, k_new, v_new, kc, vc, ks, pos, src, aP) == []

    # ---- the launch
    dev = torch.device(DEVICE)
    kd, vd = kc.to(cdt).to(dev), vc.to(cdt).to(dev)
    k_before, v_before = kd.clone(), vd.clone()
    ksd = torch.tensor(ks, dtype=torch.int32, device=dev)
    srcd = torch.tensor(src, dtype=torch.int32, device=dev) if alias else None
    partd = part.to(dev).contiguous()
    stepd = torch.tensor([c["step"]], dtype=torch.int32, device=dev) if c["step"] is not None else None
    pos_arg = pos - (c["step"] or 0)
    n_ws = R * H * WS_REC
    ws = None
    if c["impl"] == 3:
        ws = torch.zeros(n_ws + GUARD, dtype=torch.int64, device=dev)
        ws[n_ws:] = 0x5A5A5A5A5A5A5A5A
    outs = []
    runs = [(srcd, aP)] * 2
    if alias and alias.get("copies"):
        runs.append((None, 0))                          # the same rows without aliasing
    for sr, ap in runs:
        out = torch.full((R, HD), float("nan"), dtype=cdt, device=dev)
        _launch(eng, c["impl"], c["splits"], partd, R, H, kd, vd, ksd, sr, ap, pos_arg, stepd, c["rope"], c["ctas"], out, ws)
        torch.cuda.synchronize()
        outs.append(out)
        if ws is not None:
            assert int(torch.count_nonzero(ws[:n_ws])) == 0, "hand-off records left set"
            assert bool((ws[n_ws:] == 0x5A5A5A5A5A5A5A5A).all()), "hand-off guard overwritten"
    iv = torch.int16 if bf else torch.int32
    assert torch.equal(outs[0].view(iv), outs[1].view(iv)), "two launches differ"
    for before, after, new in ((k_before, kd, k_new), (v_before, vd, v_new)):
        a, b = after.view(iv), before.view(iv)
        keep = torch.ones(Tmax, dtype=torch.bool, device=dev)
        keep[pos] = False
        assert torch.equal(a[:, :, keep], b[:, :, keep]), "cache written outside column pos"
        assert torch.equal(after[:, :, pos].cpu().float(), new), "new cache column is not the reference k_new / v_new"
    for k, out in enumerate(outs[:1] + outs[2:]):
        got = out.view(R, H, A.HEAD_DIM).double().cpu()
        what = "aliasing off: " if k else ""
        assert torch.isfinite(got).all(), what + "non-finite output (a poisoned column was read, or an output was never written)"
        bad = (got - ref).abs() > A.tolerance(ref, vmax)
        if bad.any():
            i = tuple(int(x) for x in bad.nonzero()[0])
            raise AssertionError(f"{what}{int(bad.sum())}/{bad.numel()} outputs off; first at (r, h, d) = {i}: got {got[i]:.6g} "
                                 f"want {ref[i]:.6g} (kv_start {ks[i[0]]}, pos {pos})")


SMS = 148                                              # contributor counts below are for a full B200 grid

V5_CASES = {
    # kv_start 0, 31, 32, 33, pos - 1, pos (empty rows) at pos = 32k - 1, 32k, 32k + 1; S below, at and above A5_PF
    "edges_pos95_S1": _case(R=8, starts="edges", pos=95, S=1),
    "edges_pos96_S3": _case(R=8, starts="edges", pos=96, S=3, seed=1),
    "edges_pos97_S4": _case(R=8, starts="edges", pos=97, S=4, seed=2),
    "edges_pos64_S5_rel": _case(R=8, starts="edges", pos=64, S=5, rope=REL, seed=3),
    "edges_pos65_S9_step": _case(R=8, starts="edges", pos=65, S=9, step=4, seed=4),
    "R1_H32": _case(R=1, H=32, starts="dense", pos=1023, S=5, seed=5),
    "R2_H16_cfg": _case(R=2, H=16, starts="cfg", pos=600, S=3, seed=6),
    "R3_H16_ctas3": _case(R=3, H=16, starts=[0, 700, 1023], pos=1024, S=9, ctas=3, seed=7),
    "R31_H4_ragged": _case(R=31, H=4, pos=257, seed=8),
    "R32_H4_cfg": _case(R=32, H=4, starts="cfg", pos=256, S=3, seed=9),
    "R33_H2_rel": _case(R=33, H=2, pos=289, S=5, rope=REL, seed=10),
    "R64_H2_short_items": _case(R=64, H=2, pos=20, seed=11),                     # U <= ctas: per = sub = 1, empty CTAs
    "R65_H4_ctas1": _case(R=65, H=4, pos=161, S=4, ctas=1, seed=12),
    "R256_H2_ragged": _case(R=256, H=2, pos=33, S=3, seed=13),
    "R256_H4_step": _case(R=256, H=4, starts="edges", pos=64, S=3, step=7, seed=14),
    # few long items over many contributors
    "long_32_contributors": _case(R=2, H=4, starts="dense", pos=1000, seed=15),
    "long_64_contributors": _case(R=1, H=2, starts="dense", pos=2048, S=3, seed=16),
    "long_was_65_small": _case(R=2, H=4, starts=[0, 1470], pos=2075, seed=17),
    "long_was_66_tiny": _case(R=1, H=2, starts="dense", pos=2100, S=5, rope=REL, seed=18),
    # scores
    "peaked": _case(R=4, H=4, pos=500, mode="peak", seed=19),
    "peaked_ctas1": _case(R=3, H=2, starts="edges", pos=300, mode="peak", ctas=1, seed=20),
    "all_equal": _case(R=4, H=2, starts="edges", pos=300, mode="equal", seed=21),
    # prompt columns read from a source row; the duplicates' own prompt strips are NaN
    "alias_straddles_tile": _case(R=4, starts=[3, 10, 3, 10], pos=100, alias=dict(src=[0, 1, 0, 1], P=45, poison=True), seed=22),
    "alias_below_kv_start": _case(R=4, starts=[50, 60, 50, 60], pos=90, alias=dict(src=[0, 1, 0, 1], P=40, poison=True), seed=23),
    "alias_P_is_pos": _case(R=2, starts=[5, 5], pos=77, alias=dict(src=[0, 0], P=77, poison=True), seed=24),
    "alias_cfg_batch": _case(R=32, H=4, starts=[0 if r % 2 == 0 else 171 for r in range(32)], pos=230, S=3,
                             alias=dict(src=[r if r < 2 or r % 2 == 0 else 1 for r in range(32)], P=200, poison=True), seed=25),
}

PLAIN_CASES = {
    "bf16_edges_splits7": _case(impl=0, R=8, starts="edges", pos=95, splits=7),
    "bf16_H16_splits64_S9": _case(impl=0, R=3, H=16, starts=[0, 700, 1023], pos=1024, S=9, splits=64, seed=1),
    "bf16_more_splits_than_tokens": _case(impl=0, R=4, starts=[0, 39, 40, 20], pos=40, splits=64, seed=2),
    "bf16_H32_splits2_rel_step": _case(impl=0, R=2, H=32, pos=97, splits=2, rope=REL, step=5, seed=3),
    "bf16_R33_splits1": _case(impl=0, R=33, H=4, pos=289, S=4, splits=1, seed=4),
    "bf16_rule_peaked": _case(impl=0, R=4, H=4, pos=500, mode="peak", seed=5),
    "fp32_edges_splits7": _case(impl=0, R=8, starts="edges", pos=96, S=3, splits=7, rope=0, dtype="fp32", seed=6),
    "fp32_more_splits_than_tokens": _case(impl=0, R=4, starts=[0, 39, 40, 20], pos=40, splits=64, rope=0, dtype="fp32", seed=7),
    "fp32_rel_step_equal": _case(impl=0, R=5, starts="edges", pos=130, S=5, splits=2, rope=REL, step=3, mode="equal",
                                 dtype="fp32", seed=8),
}


@pytest.mark.parametrize("name", list(V5_CASES))
def test_v5_matches_fp64_reference(name):
    _run(V5_CASES[name])


def test_v5_contributor_regimes_are_the_intended_ones():
    """The long-item cases reach what they are named for on a full grid: exactly AT_MAX_SLOTS contributors, and shapes
    the even cut alone would have given 65 and 66."""
    if _num_sms() != SMS:
        pytest.skip(f"contributor counts are laid out for {SMS} SMs")
    for name, old, new in (("long_32_contributors", 32, 32), ("long_64_contributors", 64, 64),
                           ("long_was_65_small", 65, None), ("long_was_66_tiny", 66, None)):
        c = V5_CASES[name]
        ks = _starts(c["starts"], c["R"], c["pos"], None)
        assert A.contributors(ks, c["H"], c["pos"], SMS, fixed=False).max() == old, name
        n = A.contributors(ks, c["H"], c["pos"], SMS).max()
        assert n == new if new is not None else n <= A.AT_MAX_SLOTS, name
    c = V5_CASES["R64_H2_short_items"]
    ks = _starts(c["starts"], c["R"], c["pos"], torch.Generator().manual_seed(1000 + c["seed"]))
    assert A.cut_params(ks, c["H"], c["pos"], SMS) == (1, 1)


@pytest.mark.parametrize("alias_P", [45, 100])
def test_v5_alias_on_equals_alias_off_when_the_rows_are_real_copies(alias_P):
    """Duplicate rows whose prompt columns really are copies of their source rows: the launch with src_row and the one
    without both match the reference."""
    _run(_case(R=4, starts=[3, 10, 3, 10], pos=100, alias=dict(src=[0, 1, 0, 1], P=alias_P, copies=True), seed=26))


@pytest.mark.parametrize("name", list(PLAIN_CASES))
def test_plain_kernel_matches_fp64_reference(name):
    _run(PLAIN_CASES[name])


def test_attn_decode_io_rejects_bad_arguments_by_name():
    from plangen_b200 import _lib
    eng = _eng("bf16")
    dev = torch.device("cuda")
    R, H, pos, Tmax = 2, 2, 10, 16
    part = torch.zeros(1, R, 3 * H * 128, device=dev)
    kc = torch.zeros(R, H, Tmax, 128, dtype=torch.bfloat16, device=dev)
    ks = torch.zeros(R, dtype=torch.int32, device=dev)
    out = torch.zeros(R, H * 128, dtype=torch.bfloat16, device=dev)
    ws = torch.zeros(R * H * WS_REC, dtype=torch.int64, device=dev)
    src = torch.zeros(R, dtype=torch.int32, device=dev)
    bad = {
        "impl": dict(impl=2), "ctas": dict(ctas=_num_sms() + 1), "pos": dict(pos=Tmax), "rope_flags": dict(rope=3),
        "ws": dict(ws=None), "src_row": dict(impl=0, src=src, aP=4), "splits": dict(impl=0, splits=65),
        "R=": dict(R=257),
    }
    for word, kw in bad.items():
        a = dict(impl=3, splits=0, part=part, R=R, H=H, kc=kc, vc=kc, ks=ks, src=None, aP=0, pos=pos, step=None, rope=1,
                 ctas=0, out=out, ws=ws)
        a.update(kw)
        with pytest.raises(_lib.PgError, match=word):
            _launch(eng, a["impl"], a["splits"], a["part"], a["R"], a["H"], a["kc"], a["vc"], a["ks"], a["src"], a["aP"],
                    a["pos"], a["step"], a["rope"], a["ctas"], a["out"], a["ws"])
    with pytest.raises(_lib.PgError, match="bf16"):
        e32 = _eng("fp32")
        _launch(e32, 3, 0, part, R, H, kc, kc, ks, None, 0, pos, None, 1, 0, out, ws)


@pytest.mark.parametrize("attn_impl", [3, 0])
def test_decode_after_prefill_with_an_all_padding_row_matches_autocast_oracle(attn_impl):
    """language_model.model prefill over a batch with an all-padding prompt row, then 3 decode steps: every row's
    decode hidden states match the reference under autocast (the empty row's new token attends only to itself), and
    the prefill output matches at the valid positions."""
    d = O.SMALL
    lens, P, steps = [60, 0, 37, 100], 100, 3
    R = len(lens)
    g = torch.Generator().manual_seed(31)
    ids = torch.randint(0, d.pad_id, (R, P), generator=g)
    mask = torch.zeros(R, P + steps, dtype=torch.long)
    for r, n in enumerate(lens):
        mask[r, P - n:] = 1
        ids[r, :P - n] = d.pad_id
    mask[:, P:] = 1
    ids, mask = ids.cuda(), mask.cuda()
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    sdc = {k: v.cuda() for k, v in sd.items()}
    toks = torch.randint(0, d.img_vocab, (steps, R), generator=g).cuda()
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        ref = [O.llama_model_forward(sdc, d, O.embed_tokens(sdc, ids), attention_mask=mask)]
        xs = [O.prepare_gen_img_embeds(sdc, toks[i]).unsqueeze(1) for i in range(steps)]
        for i in range(steps):
            ref.append(O.llama_model_forward(sdc, d, xs[i], attention_mask=mask, past_key_values=ref[-1].past_key_values))
    eng = get_engine(d, "bf16", max_batch=2, max_prompt=128, with_vq=False)
    eng.set_option("attn_impl", attn_impl)
    try:
        emb = eng.language_model.get_input_embeddings()(ids)
        out = eng.language_model.model(inputs_embeds=emb, attention_mask=mask, use_cache=True)
        hs = [out.last_hidden_state.clone()]
        for i in range(steps):
            out = eng.language_model.model(inputs_embeds=xs[i].float(), attention_mask=mask, use_cache=True,
                                           past_key_values=out.past_key_values)
            hs.append(out.last_hidden_state.clone())
        torch.cuda.synchronize()
    finally:
        eng.set_option("attn_impl", 3)
    valid = mask[:, :P] != 0
    assert_close(hs[0][valid].cpu().numpy(), ref[0].last_hidden_state.float()[valid].cpu().numpy(), 2e-2, 3e-2,
                 "prefill hidden states (valid positions)")
    for i in range(1, steps + 1):
        got = hs[i].cpu().numpy()
        assert np.isfinite(got).all(), f"decode step {i}"
        assert_close(got, ref[i].last_hidden_state.float().cpu().numpy(), 2e-2, 2e-2, f"decode step {i} hidden states")
