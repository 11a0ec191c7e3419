"""CPU tests of the decode-attention reference (tests/attn_ref.py): the reference against the oracle's eager attention, and
the restated work cut of attn_decode_v5_kernel (no item over AT_MAX_SLOTS contributors, the even cut kept elsewhere)."""
import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200.weights import rope_tables
from plangen_b200.config import Dims
from tests import attn_ref as A


@pytest.mark.parametrize("rope_flags", [0, A.ROPE_REL])
def test_reference_is_eager_attention_of_a_left_padded_decode_step(rope_flags):
    """fp32: the reference's q / k_new / v_new and attention equal the oracle's apply_rope + build_additive_mask + eager
    softmax for one decode step over left-padded rows, including an all-padding row (kv_start == pos), whose output is
    exactly v_new: the new token attends only to itself."""
    d = O.TINY
    R, H, S, pos, Tmax = 5, d.H, 3, 40, 64
    kv_start = [0, 7, 33, 39, 40]
    g = torch.Generator().manual_seed(5)
    part = torch.randn(S, R, 3 * H * 128, generator=g)
    kc = torch.randn(R, H, Tmax, 128, generator=g)
    vc = torch.randn(R, H, Tmax, 128, generator=g)
    cos, sin = rope_tables(Dims.from_any(d), Tmax)
    q, k_new, v_new = A.qkv_new(part, H, cos, sin, pos, kv_start, rope_flags, bf16=False)
    ref, _ = A.attention(q, k_new, v_new, kc, vc, kv_start, pos)
    assert torch.equal(ref[4], v_new[4].double())

    # the oracle: HF's eager attention of the new token over cache columns [0, pos] with the 0/1 padding mask
    x = (part[0] + part[1] + part[2]).view(R, 1, 3, H, 128)
    qs, ks, vs = (x[:, :, i].transpose(1, 2) for i in range(3))                 # (R, H, 1, 128)
    rope_pos = [[max(pos - s, 0)] for s in kv_start] if rope_flags & A.ROPE_REL else [[pos]] * R
    cs, sn = O.rope_cos_sin(torch.tensor(rope_pos), d, torch.float32)
    qs, ks = O.apply_rope(qs, ks, cs, sn)
    keys = torch.cat([kc[:, :, :pos], ks], dim=2)
    vals = torch.cat([vc[:, :, :pos], vs], dim=2)
    mask = (torch.arange(pos + 1)[None, :] >= torch.tensor(kv_start)[:, None]).long()
    aw = torch.matmul(qs, keys.transpose(2, 3)) * 128 ** -0.5
    aw = aw + O.build_additive_mask(mask, torch.tensor([pos]), pos + 1, torch.float32, R)
    want = torch.matmul(torch.softmax(aw, dim=-1), vals)[:, :, 0]
    assert torch.allclose(q, qs[:, :, 0], rtol=1e-5, atol=1e-5)
    assert torch.allclose(k_new, ks[:, :, 0], rtol=1e-5, atol=1e-5)
    assert torch.equal(v_new, vs[:, :, 0])
    torch.testing.assert_close(ref.float(), want, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(want[4], v_new[4])


def test_reference_reads_aliased_prompt_columns_from_the_source_row():
    R, H, pos, Tmax, P = 3, 2, 70, 96, 45
    g = torch.Generator().manual_seed(2)
    kc = torch.randn(R, H, Tmax, 128, generator=g)
    vc = torch.randn(R, H, Tmax, 128, generator=g)
    q, k_new, v_new = (torch.randn(R, H, 128, generator=g) for _ in range(3))
    poisoned_k, poisoned_v = kc.clone(), vc.clone()
    poisoned_k[2, :, :P] = float("nan")
    poisoned_v[2, :, :P] = float("nan")
    copy_k, copy_v = kc.clone(), vc.clone()
    copy_k[2, :, :P] = kc[0, :, :P]
    copy_v[2, :, :P] = vc[0, :, :P]
    ks = [3, 10, 3]
    want, _ = A.attention(q, k_new, v_new, copy_k, copy_v, ks, pos)
    got, _ = A.attention(q, k_new, v_new, poisoned_k, poisoned_v, ks, pos, src_row=[0, 1, 0], alias_P=P)
    assert torch.equal(got, want)


def test_dropping_a_token_is_what_the_teeth_check_measures():
    R, H, pos, Tmax = 1, 1, 5, 8
    g = torch.Generator().manual_seed(0)
    kc, vc = torch.randn(R, H, Tmax, 128, generator=g), torch.randn(R, H, Tmax, 128, generator=g)
    q, k_new, v_new = (torch.randn(R, H, 128, generator=g) for _ in range(3))
    full, _ = A.attention(q, k_new, v_new, kc, vc, [2], pos)
    cut, _ = A.attention(q, k_new, v_new, kc, vc, [3], pos)
    dropped, _ = A.attention(q, k_new, v_new, kc, vc, [2], pos, drop={(0, 2)})
    assert torch.equal(cut, dropped) and not torch.equal(full, dropped)


# ------------------------------------------------------------------------------------------------------- the cut
def _starts(R, pos, pattern, rng):
    if pattern == "dense":
        return [0] * R
    if pattern == "cfg":                      # long cond rows, short uncond rows
        return [0 if r % 2 == 0 else max(pos - 37, 0) for r in range(R)]
    if pattern == "ragged":                   # every row with at least one cached token
        return list(rng.integers(0, pos, R))
    return list(rng.integers(0, pos + 1, R))  # "empty": some rows may have no cached token


R_GRID = sorted(set(range(1, 34)) | set(range(34, 257, 7)) | {63, 64, 65, 127, 128, 129, 255, 256})


@pytest.mark.parametrize("H", [1, 2, 4, 16, 32])
def test_cut_gives_no_item_more_than_64_contributors_and_keeps_the_even_cut_elsewhere(H):
    """Over R, ragged kv_start, pos up to 8192 and 1, 7 or 148 CTAs: the cut gives no item more contributors than it has
    hand-off records (AT_MAX_SLOTS), and, where every row has a cached token, it is the parent's even cut wherever that one
    gave every item fewer than 64.
    (The bound is exact over alignments, not over the items' actual offsets, so a shape whose worst item met exactly 64
    slots may be widened.)  Every Janus head count at 148 CTAs keeps the even cut."""
    rng = np.random.default_rng(H)
    widened = 0
    for R in R_GRID:
        for pos in (1, 31, 32, 33, 1088, 2100, 4097, 8192):
            for pattern in ("dense", "cfg", "ragged", "empty"):
                ks = _starts(R, pos, pattern, rng)
                for ctas in (1, 7, 148):
                    n = A.contributors(ks, H, pos, ctas)
                    assert n.max() <= A.AT_MAX_SLOTS, (R, H, pos, pattern, ctas, n.max())
                    assert n.min() >= 1
                    if pattern != "empty" and A.cut_params(ks, H, pos, ctas) != A.cut_params(ks, H, pos, ctas, fixed=False):
                        widened += 1
                        assert A.contributors(ks, H, pos, ctas, fixed=False).max() >= A.AT_MAX_SLOTS
                        assert H < 16 or ctas < 148, (R, H, pos, pattern, ctas)
    if H <= 2:
        assert widened > 0                    # the grid reaches the widened regime


def test_cut_fixes_the_known_overflows_and_empty_rows():
    # SMALL dims (H = 4), one image (cond + uncond rows), 1500-token prompt at its last step; TINY, one row at 2100
    for ks, H, pos, old in (([0, 1470], 4, 1500 + 575, 65), ([0], 2, 2100, 66)):
        assert A.contributors(ks, H, pos, 148, fixed=False).max() == old
        assert A.contributors(ks, H, pos, 148).max() <= A.AT_MAX_SLOTS
    # a row without cached tokens owned no unit, so nothing wrote its output or its new cache column
    assert A.contributors([0, 40], 4, 40, 148, fixed=False)[1].tolist() == [0] * 4
    assert A.contributors([0, 40], 4, 40, 148)[1].tolist() == [1] * 4
    assert A.row_units([40, 40], 40).tolist() == [0, 1, 2]
