"""CPU tests of the per-image sampling reference (tests/per_image_ref.py) and of the argument normalisation
(plangen_b200.engine.sampling_plan)."""
import math

import pytest
import torch

from oracle import janus_oracle as O
from tests import per_image_ref as PR
from tests import top_p_ref as TP


def test_reference_loop_with_uniform_settings_is_the_top_p_reference():
    d, B, steps = O.TINY, 2, 4
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    cond, neg = O.synthetic_prompts(d, B, lo=5, hi=12, neg_len=4)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    for cfg, k, p in ((5.0, 100, 0.8), (3.0, 0, 0.5), (7.5, 20, 1.0)):
        want = TP.t2i_tokens(sd, d, ids, mask, steps, top_k=k, top_p=p, cfg_weight=cfg, temperature=1.0,
                             sampler=O.make_torch_sampler(torch.Generator().manual_seed(3)))
        got = PR.t2i_tokens(sd, d, ids, mask, steps, [cfg] * B, [1.0] * B, [k] * B, [p] * B, torch.Generator().manual_seed(3))
        assert torch.equal(got, want), (cfg, k, p)


def test_per_row_reference_treats_each_row_as_its_own_batch():
    g = torch.Generator().manual_seed(1)
    logits = torch.randn(6, 512, generator=g)
    cfg, temp, ks, ps = [1.0, 5.0, 7.5], [1.0, 0.7, 1.3], [0, 50, 10], [0.9, 1.0, 0.5]
    t = PR.filter_rows(PR.scaled_cfg(logits, "fp32", cfg, temp), ks, ps)
    for b in range(3):
        tb = PR.filter_rows(PR.scaled_cfg(logits[2 * b: 2 * b + 2], "fp32", [cfg[b]], [temp[b]]), [ks[b]], [ps[b]])
        assert torch.equal(t[b:b + 1], tb)
    gens = [torch.Generator().manual_seed(10 + b) for b in range(3)]
    tok = PR.draw(t, gens)
    for b in range(3):
        alone = torch.multinomial(torch.softmax(t[b:b + 1], -1), 1, generator=torch.Generator().manual_seed(10 + b))
        assert int(tok[b]) == int(alone)


def test_sampling_plan_gives_one_entry_per_image_for_scalars_sequences_and_tensors():
    from plangen_b200.engine import sampling_plan
    p = sampling_plan(3, 5.0, 1.0, 0, 1.0, None, 42)
    assert not p.rng_per_image
    assert p.cfg_weight == [5.0] * 3 and p.seed == [42] * 3 and p.offset == [0] * 3 and p.generators == []
    p = sampling_plan(3, [1, 3, 5], torch.tensor([1.0, 0.5, 2.0]), torch.tensor(7), (1.0, 0.9, 0.5), 11, 0)
    assert not p.rng_per_image
    assert p.cfg_weight == [1.0, 3.0, 5.0] and p.temperature == [1.0, 0.5, 2.0] and p.top_k == [7] * 3
    assert p.top_p == [1.0, 0.9, 0.5] and p.seed == [11] * 3
    p = sampling_plan(2, 5.0, 1.0, 0, 1.0, [5, 2 ** 64 - 1], 0)
    assert p.rng_per_image and p.seed == [5, -1] and p.offset == [0, 0]


def test_sampling_plan_rejects_bad_arguments():
    from plangen_b200.engine import sampling_plan
    with pytest.raises(ValueError, match="2 values for 3"):
        sampling_plan(3, [1.0, 2.0], 1.0, 0, 1.0, None, 0)
    with pytest.raises(ValueError, match="1-D"):
        sampling_plan(2, 5.0, torch.ones(2, 1), 0, 1.0, None, 0)
    with pytest.raises(ValueError, match="2 entries for 3"):
        sampling_plan(3, 5.0, 1.0, 0, 1.0, [1, 2], 0)
    with pytest.raises(ValueError, match=r"generator\[1\].*cpu"):
        sampling_plan(2, 5.0, 1.0, 0, 1.0, [1, torch.Generator()], 0)
    g = torch.Generator()
    with pytest.raises(ValueError, match=r"generator\[1\].*twice"):
        sampling_plan(2, 5.0, 1.0, 0, 1.0, [g, g], 0)
    for bad in (1.5, -0.1, math.nan):
        with pytest.raises(ValueError, match=r"top_p\[2\]"):
            sampling_plan(3, 5.0, 1.0, 0, [1.0, 0.9, bad], None, 0)
    with pytest.raises(ValueError, match=r"top_k\[0\]"):
        sampling_plan(2, 5.0, 1.0, [-1, 0], 1.0, None, 0)
