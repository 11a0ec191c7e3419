"""CPU tests of the top-k / top-p torch reference (tests/top_p_ref.py) against the installed transformers warpers."""
import os

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from oracle import philox as PX
from tests import top_p_ref as R


def _hf(scores, k, p):
    tf = pytest.importorskip("transformers")
    from transformers.generation.logits_process import LogitsProcessorList, TopKLogitsWarper, TopPLogitsWarper
    procs = LogitsProcessorList()
    if k > 0:                                    # GenerationMixin._get_logits_processor adds each only when it is on
        procs.append(TopKLogitsWarper(k))
    if p < 1.0:
        procs.append(TopPLogitsWarper(p))
    return procs(torch.zeros(scores.shape[0], 1, dtype=torch.long), scores.clone())


def _rows(kind, B=6, V=4096):
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, V, generator=g) * 3.0
    if kind == "bf16":                           # bf16-rounded CFG logits: ties everywhere
        x = (x.bfloat16() * 2).float()
    elif kind == "tied_max":                     # several tied maxima
        x[:, [5, 900, 3001]] = x.max(dim=-1, keepdim=True).values
    return x


@pytest.mark.parametrize("kind", ["randn", "bf16", "tied_max"])
@pytest.mark.parametrize("k", [0, 50])
@pytest.mark.parametrize("p", [0.0, 0.3, 0.9, 0.999, 1.0])
def test_filter_matches_hf_warpers(kind, k, p):
    x = _rows(kind)
    got = R.top_k_top_p_filter(x, k, p)
    want = _hf(x, k, p)
    assert torch.equal(torch.isinf(got), torch.isinf(want))
    assert torch.equal(got[~torch.isinf(got)], x[~torch.isinf(got)])          # kept logits are untouched
    assert bool((~torch.isinf(got)).any(dim=-1).all())                          # at least one token survives


def test_top_p_zero_keeps_one_of_tied_maxima():
    x = _rows("tied_max")
    kept = ~torch.isinf(R.top_k_top_p_filter(x, 0, 0.0))
    assert kept.sum(dim=-1).tolist() == [1] * x.shape[0]
    assert bool((x[kept] == x.max(dim=-1).values).all())


def test_reference_loop_without_filters_is_the_oracle_t2i(golden_dir):
    g = np.load(os.path.join(golden_dir, "lm_tiny_fp32.npz"))
    sd = O.init_state_dict(O.TINY, seed=0, with_vq=False)
    ids, mask = torch.from_numpy(g["ids"]), torch.from_numpy(g["mask"])
    toks = R.t2i_tokens(sd, O.TINY, ids, mask, 8, sampler=PX.PhiloxSampler(int(g["seed"]), int(g["num_sms"])))
    assert np.array_equal(toks.numpy(), g["tokens"])


def test_reference_loop_samples_inside_the_nucleus():
    d = O.TINY
    sd = O.init_state_dict(d, seed=0, with_vq=False)
    cond, neg = O.synthetic_prompts(d, 2, lo=5, hi=12, neg_len=4)
    ids, mask = O.t2i_infer_collate_batch(cond, neg, d.pad_id, d.n_img_tokens)
    trace = []
    toks = R.t2i_tokens(sd, d, ids, mask, 4, top_k=100, top_p=0.8, sampler=PX.PhiloxSampler(0, 148), trace=trace)
    for step, t in enumerate(trace):
        kept = ~torch.isinf(t)
        assert bool(kept.gather(1, toks[:, step:step + 1].long()).all())
        assert 1 <= int(kept.sum(dim=-1).min()) and int(kept.sum(dim=-1).max()) <= 100
