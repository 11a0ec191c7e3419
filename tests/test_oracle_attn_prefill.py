"""CPU tests of the prefill / SigLIP attention reference (tests/attn_prefill_ref.py): with every rounding off it is the
oracle's eager attention; its acceptance criterion rejects plausible kernel faults, each by name, and accepts fp32
restatements of the kernels; and the planted boundary keys are ones whose loss the criterion would see."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import janus_oracle as O
from tests import attn_prefill_ref as A

LOG2E = float(torch.tensor(1.4426950408889634, dtype=torch.float32))


def _prefill_case(bf16=True, R=4, P=300, H=2, starts=(0, 5, 130, 257), mode="rand", seed=0):
    g = torch.Generator().manual_seed(seed)
    rnd = A.bf if bf16 else (lambda t: t.float())
    a = math.sqrt(80.0) if mode == "peak" else math.sqrt(3.0)
    q = rnd(torch.randn(R, P, H, 128, generator=g) * (0.0 if mode == "equal" else a))
    K = rnd(torch.randn(R, H, P, 128, generator=g) * a)
    V = rnd(torch.randn(R, H, P, 128, generator=g))
    ks = list(starts)
    A.plant_prefill(q, K, V, ks, mode, g, rnd)
    return q, K, V, ks


def _vit_case(bf16=True, n=2, NP=400, heads=2, hd=64, mode="rand", seed=0):
    g = torch.Generator().manual_seed(seed)
    rnd = A.bf if bf16 else (lambda t: t.float())
    W = heads * hd
    qkv = torch.randn(n * NP, 3 * W, generator=g) * math.sqrt(3.0)
    if mode == "peak":
        qkv[:, :2 * W] *= math.sqrt(80.0 / 3.0)
    if mode == "equal":
        qkv[:, :W] = 0.0
    qkv = rnd(qkv)
    A.plant_vit(qkv, n, NP, W, heads, mode, g, rnd)
    return qkv, W


def _rejected(got, ref, tol):
    return bool(((got.double() - ref).abs() > tol).any())


# ------------------------------------------------------------------------------------------------ against the oracle
def test_prefill_reference_without_rounding_is_eager_attention_over_a_left_padded_batch():
    """Rounding off, the prefill reference is HF's eager attention with the 0/1 padding mask and the causal mask at every
    valid query; pad queries, and every query of an all-padding row, give exact zeros (the kernels' convention; eager
    attention gives a meaningless uniform average there)."""
    R, P, H = 4, 150, 2
    ks = [0, 7, 129, P]
    g = torch.Generator().manual_seed(3)
    q = torch.randn(R, P, H, 128, generator=g)
    K = torch.randn(R, H, P + 5, 128, generator=g)
    V = torch.randn(R, H, P + 5, 128, generator=g)
    ref, _, _ = A.prefill(q, K, V, ks, "tc", exact=True)
    mask = (torch.arange(P)[None, :] >= torch.tensor(ks)[:, None]).long()
    qs = q.permute(0, 2, 1, 3).double()
    aw = qs @ K[:, :, :P].double().transpose(2, 3) * 128 ** -0.5
    aw = aw + O.build_additive_mask(mask, torch.arange(P), P, torch.float64, R)
    want = (torch.softmax(aw, dim=-1) @ V[:, :, :P].double()).permute(0, 2, 1, 3)
    for r in range(R):
        torch.testing.assert_close(ref[r, ks[r]:], want[r, ks[r]:], rtol=1e-12, atol=1e-12)
        assert bool((ref[r, :ks[r]] == 0).all())
    assert bool((ref[3] == 0).all())


def test_vit_reference_without_rounding_is_sdpa():
    qkv, W = _vit_case(bf16=False, n=2, NP=50, heads=2, hd=64)
    ref, _, _ = A.vit(qkv, 2, 50, W, 2, "tc", exact=True)
    x = qkv.double().view(2, 50, 3, 2, 64)
    q, k, v = (x[:, :, i].transpose(1, 2) for i in range(3))
    want = F.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(100, 2, 64)
    torch.testing.assert_close(ref, want, rtol=1e-12, atol=1e-12)


# --------------------------------------------------------------------------------------------------------- the teeth
@pytest.mark.parametrize("kernel", ["tc", "cc_bf16"])
@pytest.mark.parametrize("fault", list(A.PREFILL_FAULTS) + ["packed_neighbour"])
def test_prefill_criterion_rejects_the_fault(kernel, fault):
    q, K, V, ks = _prefill_case(seed=1)
    ref, tol, _ = A.prefill(q, K, V, ks, kernel)
    if fault == "packed_neighbour":                    # packed_row_of off by one: row r's tokens use row r - 1's keys
        bad, _, _ = A.prefill(q, K, V, ks, kernel, row_kv=[1] + list(range(len(ks) - 1)))
    else:
        bad, _, _ = A.prefill(q, K, V, ks, kernel, fault=fault)
    assert _rejected(A.bf(bad), ref, tol), f"{kernel}: the criterion accepts the fault {fault}"


@pytest.mark.parametrize("kernel,fault", [("tc", f) for f in A.VIT_FAULTS] + [("cc_bf16", "keys_past_np")])
def test_vit_criterion_rejects_the_fault(kernel, fault):
    qkv, W = _vit_case(n=2, NP=400, seed=2)
    ref, tol, _ = A.vit(qkv, 2, 400, W, 2, kernel)
    if kernel == "tc":
        bad, _, _ = A.vit(qkv, 2, 400, W, 2, kernel, fault=fault)
    else:                                              # keys >= NP valid: the whole row of 32 * VA_MAXI slots
        bad, _, _ = A.vit(qkv, 1, 400 + 32, W, 2, kernel)
        bad, ref, tol = bad[:400], ref[:400], tol[:400]
    assert _rejected(A.bf(bad), ref, tol), f"{kernel}: the criterion accepts the fault {fault}"


# ------------------------------------------------------------------------------- fp32 restatements are accepted
def _prefill_tc_fp32(q, K, V, ks):
    """attn_prefill_tc_kernel in fp32, block by block: fp32 q.k, exp2 of the fp32 product (s - m) * log2e."""
    R, P, H, D = q.shape
    scale = A.f32_scale(D)
    out = torch.zeros(R, P, H, D)
    for r in range(R):
        st = ks[r]
        for h in range(H):
            S = A.bf(A.bf(q[r, :, h] @ K[r, h, :P].T) * scale)
            i, j = torch.arange(P)[:, None], torch.arange(P)[None, :]
            vis = (j >= st) & (j <= i)
            m = torch.full((P, 1), -math.inf)
            l = torch.zeros(P, 1)
            o = torch.zeros(P, D)
            for kb in range(st // A.PA_BK, (P - 1) // A.PA_BK + 1):
                cols = slice(kb * A.PA_BK, min(P, (kb + 1) * A.PA_BK))
                s, vb = S[:, cols], vis[:, cols]
                m_new = torch.maximum(m, torch.where(vb, s, -math.inf).amax(-1, keepdim=True))
                alpha = torch.where(m_new == -math.inf, torch.ones(()), torch.exp2((m - m_new) * LOG2E))
                p = torch.where(vb, torch.exp2((s - torch.where(m_new == -math.inf, 0.0, m_new)) * LOG2E), 0.0)
                l = l * alpha + p.sum(-1, keepdim=True)
                o = o * alpha + A.bf(p) @ V[r, h, cols]
                m = m_new
            out[r, :, h] = A.bf(o * torch.where(l > 0, 1.0 / l, 0.0))
    return out


def _vit_tc_fp32(qkv, n, NP, W, heads):
    hd = W // heads
    sl2 = float(torch.tensor(A.f32_scale(hd), dtype=torch.float32) * LOG2E)
    out = torch.zeros(n * NP, heads, hd)
    for img in range(n):
        x = qkv[img * NP:(img + 1) * NP].view(NP, 3, heads, hd)
        for h in range(heads):
            S = x[:, 0, h] @ x[:, 1, h].T
            m = torch.full((NP, 1), -math.inf)
            l = torch.zeros(NP, 1)
            o = torch.zeros(NP, hd)
            for k0 in range(0, NP, A.VT_BK):
                s = S[:, k0:k0 + A.VT_BK]
                m_new = torch.maximum(m, s.amax(-1, keepdim=True) * sl2)
                alpha = torch.exp2(m - m_new)
                p = torch.exp2((s.double() * sl2 - m_new.double()).float())          # fma: one rounding
                l = l * alpha + p.sum(-1, keepdim=True)
                o = o * alpha + A.bf(p) @ x[k0:k0 + A.VT_BK, 2, h]
                m = m_new
            out[img * NP:(img + 1) * NP, h] = A.bf(o / l)
    return out


@pytest.mark.parametrize("mode", ["rand", "peak", "equal"])
def test_criterion_accepts_fp32_restatements_of_the_kernels(mode):
    q, K, V, ks = _prefill_case(mode=mode, seed=4)
    ref, tol, allow = A.prefill(q, K, V, ks, "tc")
    got = _prefill_tc_fp32(q, K, V, ks)
    assert not _rejected(got, ref, tol), f"tcgen05 prefill, {mode}"
    for kernel, rnd in (("cc_bf16", A.bf), ("cc_fp32", lambda t: t.float())):
        ref, tol, _ = A.prefill(q, K, V, ks, kernel)
        want = torch.zeros_like(ref)
        for r, st in enumerate(ks):
            s = torch.einsum("phd,hkd->hpk", q[r] * A.f32_scale(128), K[r, :, :q.shape[1]])
            i, j = torch.arange(q.shape[1])[:, None], torch.arange(q.shape[1])[None, :]
            s = torch.where((j >= st) & (j <= i), s, -math.inf)
            w = torch.nan_to_num(torch.softmax(s, -1))
            want[r] = (w @ V[r, :, :q.shape[1]]).permute(1, 0, 2).double()
        assert not _rejected(rnd(want), ref, tol), f"{kernel} prefill, {mode}"
    qkv, W = _vit_case(n=2, NP=400, mode=mode, seed=5)
    ref, tol, _ = A.vit(qkv, 2, 400, W, 2, "tc")
    assert not _rejected(_vit_tc_fp32(qkv, 2, 400, W, 2), ref, tol), f"tcgen05 ViT, {mode}"
    ref, tol, _ = A.vit(qkv, 2, 400, W, 2, "cc_bf16")
    x = qkv.view(2, 400, 3, 2, 64)
    s = torch.einsum("iqhd,ikhd->ihqk", x[:, :, 0], x[:, :, 1])
    p = A.bf(torch.softmax(A.bf(s) * A.f32_scale(64), -1))
    want = torch.einsum("ihqk,ikhd->iqhd", p, x[:, :, 2]).reshape(800, 2, 64)
    assert not _rejected(A.bf(want), ref, tol), f"CUDA-core ViT, {mode}"


# ----------------------------------------------------------------------------------------------- planted keys
@pytest.mark.parametrize("mode", ["rand", "peak", "equal"])
def test_dropping_any_planted_boundary_key_breaks_the_tolerance(mode):
    q, K, V, ks = _prefill_case(mode=mode, seed=6)
    for kernel in ("tc", "cc_bf16"):
        ref, tol, _ = A.prefill(q, K, V, ks, kernel)
        missed = A.undetected_drops(ref, tol, lambda r, h, c: A.prefill_weight(q, K, V, ks, r, h, c),
                                    lambda r: A.boundary_columns(ks[r], q.shape[1]))
        assert missed == [], (kernel, missed)
    qkv, W = _vit_case(n=2, NP=400, mode=mode, seed=7)
    ref, tol, _ = A.vit(qkv, 2, 400, W, 2, "tc")
    refi, toli = ref.view(2, 400, 2, 64), tol.view(2, 400, 2, 64)
    missed = A.undetected_drops(refi, toli, lambda i, h, c: A.vit_weight(qkv, 400, W, 2, i, h, c),
                                lambda i: A.vit_boundary_columns(400))
    assert missed == [], missed
