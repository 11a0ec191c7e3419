"""CPU: the log-probability references (tests/logprob_ref.py) and the scorer's argument checks."""
import math

import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200.engine import check_score_args, sampling_plan
from tests import logprob_ref as LR
from tests import per_image_ref as PR


def test_removed_tokens_are_minus_inf_and_kept_tail_tokens_finite():
    V = 64
    g = torch.Generator().manual_seed(3)
    t = torch.randn(2, V, generator=g)
    t[0, 5] = t[0].max() + 1.0                 # the maximum of row 0
    t[0, 9] = t[0, 5] - 200.0                  # kept (no filter on row 0) but exp underflows in fp32
    filt = PR.filter_rows(t, [0, 10], [1.0, 0.8])
    lp_all = torch.log_softmax(filt, dim=-1)
    removed = torch.isinf(filt)
    assert not removed[0].any() and removed[1].any()
    assert torch.isneginf(lp_all[removed]).all()
    assert torch.isfinite(lp_all[~removed]).all()
    lp = LR.logprobs_of(filt, torch.tensor([9, int(removed[1].nonzero()[0])]))
    assert math.isfinite(lp[0].item()) and lp[0].item() < -199.0
    assert torch.isneginf(lp[1])
    assert float(torch.exp(filt[0, 9] - filt[0].max())) == 0.0          # log(e / sum) would be -inf here


@pytest.mark.parametrize("top_k,top_p", [(0, 1.0), (50, 0.9)])
def test_scorer_reference_equals_the_cached_teacher_forced_loop(top_k, top_p):
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    B, n = 2, 6
    cond, neg = O.synthetic_prompts(d, B, seed=5, lo=5, hi=12, neg_len=4)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, n)
    img = torch.randint(0, d.img_vocab, (B, n), generator=torch.Generator().manual_seed(1))
    s = dict(cfg_weight=[3.0, 5.0], temperature=[1.0, 0.7], top_k=[top_k, 0], top_p=[top_p, 1.0])
    _, want = LR.loop_ref(sd, d, ids, mask, n, forced=img, **s)
    got = LR.score_ref(sd, d, ids, mask, img, **s)
    fin = torch.isfinite(want)
    assert torch.equal(fin, torch.isfinite(got))
    assert (got[fin] - want[fin]).abs().max().item() <= 1e-5


def test_score_argument_checks_name_the_argument():
    ok = torch.zeros(2, 5, dtype=torch.int64)
    mask = torch.ones(4, 7 + 5)
    assert check_score_args(2, 7, ok, mask, 100, 8) == 5
    with pytest.raises(ValueError, match="image_tokens.*rows"):
        check_score_args(3, 7, ok, torch.ones(6, 12), 100, 8)
    with pytest.raises(ValueError, match=r"image_tokens.*\[0, 100\)"):
        check_score_args(2, 7, torch.full((2, 5), 100), mask, 100, 8)
    with pytest.raises(ValueError, match=r"image_tokens.*\[0, 100\)"):
        check_score_args(2, 7, torch.full((2, 5), -1), mask, 100, 8)
    with pytest.raises(ValueError, match="max_steps"):
        check_score_args(2, 7, torch.zeros(2, 9, dtype=torch.int64), torch.ones(4, 16), 100, 8)
    with pytest.raises(ValueError, match="mask"):
        check_score_args(2, 7, ok, torch.ones(4, 11), 100, 8)
    with pytest.raises(ValueError, match="integer"):
        check_score_args(2, 7, ok.float(), mask, 100, 8)
    with pytest.raises(ValueError, match="image_tokens"):
        check_score_args(2, 7, ok.view(-1), mask, 100, 8)
    # per-image settings are normalised (and rejected) by the same helper as sample_image's
    with pytest.raises(ValueError, match="top_k"):
        sampling_plan(2, 5.0, 1.0, [1, 2, 3], 1.0, None, 0)
    with pytest.raises(ValueError, match=r"top_p\[1\]"):
        sampling_plan(2, 5.0, 1.0, 0, [1.0, 1.5], None, 0)
