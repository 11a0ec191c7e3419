"""CPU tests of the guidance-schedule reference (tests/cfg_schedule_ref.py) and of the schedule argument
(plangen_b200.engine.guidance_schedule)."""
import ctypes
import math
import re

import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200.engine import guidance_schedule, sampling_plan
from tests import cfg_schedule_ref as SR
from tests import logprob_ref as LR
from tests import per_image_ref as PR

S = dict(temperature=[1.0, 0.7], top_k=[0, 50], top_p=[0.9, 1.0])


def _batch(d, B, n):
    cond, neg = O.synthetic_prompts(d, B, seed=5, lo=5, hi=12, neg_len=4)
    return O.t2i_infer_collate_batch(cond, neg, d.pad_id, n)


def test_constant_schedule_is_the_per_image_reference():
    d, B, n = O.TINY, 2, 5
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    ids, mask = _batch(d, B, n)
    w = [3.0, 7.5]
    sched = torch.tensor(w)[:, None].expand(B, n)
    gens = lambda: [torch.Generator().manual_seed(10 + b) for b in range(B)]
    toks, lps = SR.loop_ref(sd, d, ids, mask, n, sched, generator=gens(), **S)
    assert torch.equal(toks, PR.t2i_tokens(sd, d, ids, mask, n, w, S["temperature"], S["top_k"], S["top_p"], gens()))
    want_t, want_lp = LR.loop_ref(sd, d, ids, mask, n, w, generator=gens(), **S)
    assert torch.equal(toks, want_t) and torch.equal(lps, want_lp)
    # the scorer's reference too, on the loop's tokens
    img = toks.long()
    assert torch.equal(SR.score_ref(sd, d, ids, mask, img, sched, **S), LR.score_ref(sd, d, ids, mask, img, w, **S))


def test_varying_schedule_changes_the_tokens_from_the_step_it_differs():
    d, B, n = O.TINY, 2, 6
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    ids, mask = _batch(d, B, n)
    flat = torch.full((B, n), 5.0)
    ramp = 1.0 + 4.0 * torch.linspace(0, 1, n)[None, :].expand(B, n)
    a, _ = SR.loop_ref(sd, d, ids, mask, n, flat, generator=torch.Generator().manual_seed(1), **S)
    b, _ = SR.loop_ref(sd, d, ids, mask, n, ramp, generator=torch.Generator().manual_seed(1), **S)
    assert not torch.equal(a, b)
    # agreeing on the first k columns, the tokens agree there
    k = 3
    mixed = torch.where(torch.arange(n) < k, flat, ramp)
    c, _ = SR.loop_ref(sd, d, ids, mask, n, mixed, generator=torch.Generator().manual_seed(1), **S)
    assert torch.equal(a[:, :k], c[:, :k])


def test_guidance_schedule_takes_tensors_and_nested_sequences():
    want = torch.tensor([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]])
    for arg in (want, want.double(), want.tolist(), tuple(tuple(r) for r in want.tolist()), [want[0], want[1]],
                [[1, 2, 3], torch.tensor([4.0, 5.0, 6.0])]):
        got = guidance_schedule(arg, 2, 3)
        assert got.dtype == torch.float32 and got.device.type == "cpu" and got.is_contiguous()
        assert torch.equal(got, want)
    # scalars and one value per image stay with sampling_plan, exactly as before
    for arg in (5.0, torch.tensor(5.0), [3.0, 5.0], (3.0, 5.0), torch.tensor([3.0, 5.0])):
        assert guidance_schedule(arg, 2, 3) is None
    p = sampling_plan(2, [3.0, 5.0], 1.0, 0, 1.0, None, 0)
    assert p.cfg_weight == [3.0, 5.0]


def test_guidance_schedule_rejects_wrong_shapes_and_non_finite_entries_naming_them():
    with pytest.raises(ValueError, match="3 rows for 2"):
        guidance_schedule(torch.ones(3, 4), 2, 4)
    with pytest.raises(ValueError, match=r"cfg_weight\[0\]` has 5 steps for 4"):
        guidance_schedule(torch.ones(2, 5), 2, 4)
    with pytest.raises(ValueError, match=r"cfg_weight\[1\]` has 3 steps for 4"):
        guidance_schedule([[1.0] * 4, [1.0] * 3], 2, 4)
    with pytest.raises(ValueError, match="shape \\(2, 4, 1\\)"):
        guidance_schedule(torch.ones(2, 4, 1), 2, 4)
    with pytest.raises(ValueError, match=r"cfg_weight\[0, 2\]"):
        guidance_schedule([[1.0, 1.0, [1.0], 1.0], [1.0] * 4], 2, 4)
    with pytest.raises(ValueError, match=r"cfg_weight\[0\]` is a scalar"):
        guidance_schedule([5.0, [1.0] * 4], 2, 4)
    for bad in (math.nan, math.inf, -math.inf, 1e39):          # 1e39 overflows fp32
        t = torch.ones(2, 4, dtype=torch.float64)
        t[1, 3] = bad
        with pytest.raises(ValueError, match=r"cfg_weight\[1, 3\]"):
            guidance_schedule(t, 2, 4)
        with pytest.raises(ValueError, match=r"cfg_weight\[1, 3\]"):
            guidance_schedule(t.tolist(), 2, 4)
    # sampling_plan keeps rejecting 2-D input on its own (cfg_sample_embed takes no schedule)
    with pytest.raises(ValueError, match="1-D"):
        sampling_plan(2, torch.ones(2, 3), 1.0, 0, 1.0, None, 0)


def test_library_has_one_sampling_entry_point_per_job():
    from plangen_b200 import _lib, build, ops
    cdll = ctypes.CDLL(build.build())
    with open(build.os.path.join(build.HERE, "..", "include", "plangen_b200.h")) as f:
        header = f.read()
    # the loop and the scorer take the schedule as an optional argument of their one entry point each
    for name in ("pg_sample_image", "pg_score_image_tokens"):
        assert name in _lib.EXPORTS
        getattr(cdll, name)
        decl = re.search(rf"\b{name}\(([^;]*)\);", header)
        assert decl and "cfg_schedule_host" in decl.group(1), name
    for name in ("sample_image", "score_image_tokens"):
        assert name in ops.OP_NAMES
        assert "cfg_schedule" in str(getattr(torch.ops.plangen_b200, name).default._schema), name
    # one entry point per job: no variants with a suffix for per-image settings, log-probs or schedules
    jobs = ("pg_cfg_sample_embed", "pg_sample_image", "pg_score_image_tokens")
    sampling = re.compile(r"\b(?:%s)\w*(?=\s*\()" % "|".join(jobs))
    assert set(sampling.findall(header)) == set(jobs)
    assert {n for n in _lib.EXPORTS if sampling.match(n + "(")} == set(jobs)
    for job in jobs:
        for suffix in ("_per_image", "_logprobs", "_scheduled"):
            assert not hasattr(cdll, job + suffix), job + suffix
