"""CPU: the contraction reference (tests/gemm_ref.py) and the acceptance criteria of tests/test_gpu_gemm_epi.py.

* Teeth: on data shaped like the GPU tests', each criterion rejects a plausible fault of the kernel it checks (silu
  without the bf16 rounding of g, gate and up swapped, a bias off by one column, GELU with the tanh approximation, add16
  added before the first rounding, the residual add without bf16(acc + bias), a RoPE position off by one, rope_start
  ignored, a packed token assigned to the neighbouring row, the last k-block dropped), and accepts fp32 restatements of
  the kernels' approximations (erf_fast, the ex2 / rcp silu), so the near-midpoint allowance is neither too tight nor
  the reason a fault passes.
* The tile-major restatement against a literal transcription of tile_weight_kernel's loop, and its inverse.
* The stream-K cut (skg_u0 / skg_owner): every unit owned once, fragments, contributor ranks within the scratch, the
  finisher of each tile, and the host guard on fragments per CTA over tile counts, k-block counts and CTA counts."""
import math

import numpy as np
import pytest
import torch

from tests import gemm_ref as G
from tests.gpu_util import assert_close


def _data(M, N, K, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(M, K, generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(torch.bfloat16)
    return X, W, G.acc64(X, W).float(), g


def _erf_fast32(x):
    """gemm.cuh erf_fast in fp32 (exact exp2 / division stand in for ex2.approx / rcp.approx)."""
    x = x.astype(np.float32)
    ax = np.abs(x)
    t = np.float32(1.0) / (np.float32(0.3275911) * ax + np.float32(1.0))
    ex = np.exp2(-ax * ax * np.float32(1.4426950408889634)).astype(np.float32)
    poly = t * (t * (t * (t * (t * np.float32(1.061405429) - np.float32(1.453152027)) + np.float32(1.421413741))
                     - np.float32(0.284496736)) + np.float32(0.254829592))
    return np.copysign(np.float32(1.0) - poly * ex, x).astype(np.float32)


def test_rows_criteria_reject_faults():
    M, N, K = 100, 264, 200
    X, W, acc, g = _data(M, N, K, 1)
    bias = 0.5 * torch.randn(N, generator=g)
    add16 = torch.randn(M, N, generator=g).to(torch.bfloat16)
    want = G.rows(acc, bias)
    assert not torch.equal(G.rows(acc, torch.roll(bias, 1)), want), "bias off by one column passes"
    want_add = G.rows(acc, bias, add16)
    assert not torch.equal(G.bf(acc + bias + add16.float()), want_add), "add16 before the first rounding passes"
    res = torch.randn(M, N, generator=g)
    assert not torch.equal(res + (acc + bias), G.resid(res, acc, bias)), "residual without bf16(acc + bias) passes"
    # GELU: erf_fast in fp32 is accepted, the tanh approximation is not
    lo, hi = G.gelu_rows(acc, bias)
    t = G.bf(acc + bias).numpy()
    fast = G.bf(torch.from_numpy((t * np.float32(0.5)) * (np.float32(1.0) + _erf_fast32(t * np.float32(0.70710678118654752440)))))
    assert bool(G.in_interval(fast, lo, hi).all()), "the criterion rejects erf_fast"
    assert float((lo != hi).float().mean()) < 0.01
    bad = ~G.in_interval(G.gelu_tanh_rows(acc, bias), lo, hi)
    assert int(bad.sum()) > 0, "GELU with the tanh approximation passes"


def test_accumulator_criterion_rejects_dropped_k_block():
    for K in (72, 200, 2048):
        X, W, acc, _ = _data(33, 136, K, K)
        want = G.acc64(X, W)
        assert_close(acc.numpy(), want.numpy(), 1e-4, 2e-6, "fp32 of fp64")
        with pytest.raises(AssertionError):
            assert_close(G.acc64(X, W, drop_last_kb=True).numpy(), want.numpy(), 1e-4, 2e-6, "last k-block dropped")


def _silu_fast32(gv):
    """The decode / stream-K silu in fp32: g * 1 / (1 + 2^(-g log2 e))."""
    gv = gv.float().numpy()
    ex = np.exp2((-gv * np.float32(1.4426950408889634)).astype(np.float32)).astype(np.float32)
    return torch.from_numpy((gv * (np.float32(1.0) / (np.float32(1.0) + ex))).astype(np.float32))


@pytest.mark.parametrize("K", [64, 512, 2048])
def test_swiglu_criteria_reject_faults(K):
    M, F = 33, 320
    g_ = torch.Generator().manual_seed(K)
    X = torch.randn(M, K, generator=g_).to(torch.bfloat16)
    Wg = (torch.randn(F, K, generator=g_) / math.sqrt(K)).to(torch.bfloat16)
    Wu = (torch.randn(F, K, generator=g_) / math.sqrt(K)).to(torch.bfloat16)
    W = G.pack_gate_up(Wg, Wu)
    assert torch.equal(W.view(2 * F // 128, 2, 64, K)[:, 0].reshape(F, K), Wg)
    a64 = G.acc64(X, W)
    acc = a64.float()
    ga, ua = G.split_gate_up(acc)
    assert torch.equal(ga, (X.double() @ Wg.double().T).float())
    gb, ub = G.bf(ga), G.bf(ua)
    kernel_like = G.bf(G.bf(_silu_fast32(gb)) * ub)
    lo, hi = G.swiglu(acc, fast=True)
    assert bool(G.in_interval(kernel_like, lo, hi).all()), "the criterion rejects the ex2 / rcp silu"
    assert float((lo != hi).float().mean()) < 0.01
    faults = {
        "silu without bf16(g)": G.bf(G.bf(_silu_fast32(ga)) * ub),
        "gate and up swapped": G.bf(G.bf(_silu_fast32(ub)) * gb),
        "no rounding of silu": G.bf(_silu_fast32(gb) * ub),
    }
    lo64, hi64 = G.swiglu64(a64, G.sum_bound(X, W))
    assert bool(G.in_interval(kernel_like, lo64, hi64).all()), "the fp64 criterion rejects the kernel's own restatement"
    assert float((lo64 != hi64).float().mean()) < (0.25 if K <= 512 else 0.75)   # a worst-case summation bound: wide
    for name, h in faults.items():
        assert int((~G.in_interval(h, lo, hi)).sum()) > 0, f"{name} passes the same-kernel criterion"
        assert int((~G.in_interval(h, lo64, hi64)).sum()) > 0, f"{name} passes the fp64 criterion"
    # the pair kernel's expf / IEEE-division silu
    pair_like = G.bf(G.bf(gb / (1.0 + torch.exp(-gb))) * ub)
    assert bool(G.in_interval(pair_like, *G.swiglu(acc, fast=False)).all())


def test_qkv_criteria_reject_faults():
    H, R, K = 2, 4, 128
    row_off = [0, 70, 70, 71]                   # row 1 empty (deduplicated), row 2 one token, row 3 the rest
    kv_start = [3, 9, 40, 0]
    rope_start = [3, 0, 30, 0]
    M, Tmax = 200, 256
    X, W, acc, g = _data(M, 3 * H * 128, K, 7)
    cos, sin = (t.float() for t in (torch.rand(Tmax, 64, generator=g), torch.rand(Tmax, 64, generator=g)))
    kc0 = torch.randn(R, H, Tmax, 128, generator=g).to(torch.bfloat16).float()
    vc0 = torch.randn(R, H, Tmax, 128, generator=g).to(torch.bfloat16).float()
    rw, col, pr = G.qkv_positions(M, R, 0, row_off, kv_start, rope_start)
    assert rw[69] == 0 and rw[70] == 2 and rw[71] == 3 and col[70] == 40 and col[71] == 0 and pr[70] == 10
    q, kc, vc = G.qkv(acc, H, cos, sin, rw, col, pr, kc0, vc0)
    q1, kc1, _ = G.qkv(acc, H, cos, sin, rw, col, pr + 1, kc0, vc0)
    assert not torch.equal(q1, q) and not torch.equal(kc1, kc), "RoPE position off by one passes"
    _, _, pr_nors = G.qkv_positions(M, R, 0, row_off, kv_start, None)
    q2, _, _ = G.qkv(acc, H, cos, sin, rw, col, pr_nors, kc0, vc0)
    assert not torch.equal(q2, q), "rope_start ignored passes"
    rw3, col3 = rw.copy(), col.copy()
    rw3[71], col3[71] = 2, kv_start[2] + 1      # the first token of row 3 given to row 2
    pr3 = np.maximum(col3 - np.asarray(rope_start)[rw3], 0)
    _, kc3, vc3 = G.qkv(acc, H, cos, sin, rw3, col3, pr3, kc0, vc0)
    assert not torch.equal(kc3, kc) and not torch.equal(vc3, vc), "a packed token in the neighbouring row passes"
    # padded block: position m % P, row m // P
    rwp, colp, prp = G.qkv_positions(300, 3, 100, None, [0, 0, 0], None)
    assert rwp[199] == 1 and colp[199] == 99 and prp[200] == 0


@pytest.mark.parametrize("N,K", [(128, 64), (200, 72), (5, 8), (300, 200), (384, 5632)])
def test_tile_major_restatement(N, K):
    g = torch.Generator().manual_seed(N + K)
    W = torch.randn(N, K, generator=g).to(torch.bfloat16)
    buf = G.tile_major(W)
    nkb = -(-K // 64)
    assert buf.size == -(-N // 128) * nkb * G.TILE_BYTES
    # a literal transcription of tile_weight_kernel's loop
    w16 = W.view(torch.int16).numpy().view(np.uint16)
    lit = np.zeros(buf.size // 2, dtype=np.uint16)
    n_chunks = buf.size // 16
    for idx in range(0, n_chunks, max(1, n_chunks // 4096)):
        c, r, tile = idx & 7, (idx >> 3) & 127, idx >> 10
        kb, nt = tile % nkb, tile // nkb
        n, k = nt * 128 + r, kb * 64 + c * 8
        dst = (tile * G.TILE_BYTES + r * 128 + ((c ^ (r & 7)) * 16)) // 2
        lit[dst:dst + 8] = w16[n, k:k + 8] if (n < N and k + 8 <= K) else 0
        assert np.array_equal(buf.view(np.uint16)[dst:dst + 8], lit[dst:dst + 8]), (idx, n, k)
    assert np.array_equal(G.untile(buf, N, K), w16)
    # everything outside the real elements is zero
    ones = torch.full((N, K), 1.0).to(torch.bfloat16)
    assert int((G.tile_major(ones).view(np.uint16) != 0).sum()) == N * K


@pytest.mark.parametrize("n_tiles", [1, 2, 5, 22, 88, 172])
@pytest.mark.parametrize("num_kb", [1, 4, 8, 32, 64])
def test_stream_k_cut(n_tiles, num_kb):
    U = n_tiles * num_kb
    for ctas in (1, 5, 7, 16, 148, 0):
        Gc = G.skg_grid(n_tiles, num_kb, ctas, 148)
        mc = G.skg_max_contrib(n_tiles, num_kb, Gc)
        seen = np.zeros(U, dtype=np.int64)
        finisher = {}
        for c in range(Gc):
            u0, u1 = G.skg_u0(c, U, Gc), G.skg_u0(c + 1, U, Gc)
            for u in range(u0, u1):
                assert G.skg_owner(u, U, Gc) == c
            frs = G.skg_fragments(c, n_tiles, num_kb, Gc)
            assert [t for t, _, _ in frs] == sorted((t for t, _, _ in frs), reverse=True)
            for t, lo, hi in frs:
                assert 0 <= lo < hi <= num_kb
                seen[t * num_kb + lo:t * num_kb + hi] += 1
                rank = c - G.skg_owner(t * num_kb, U, Gc)
                assert 0 <= rank < mc, (c, t, rank, mc)        # the partial's scratch slot / the finisher's nc
                if hi == num_kb:
                    finisher[t] = c
        assert (seen == 1).all()                                # every (tile, k-block) unit owned exactly once
        assert sorted(finisher) == list(range(n_tiles))
        for t, c in finisher.items():
            assert c == G.skg_owner(t * num_kb + num_kb - 1, U, Gc)
        contrib = G.skg_contributors(n_tiles, num_kb, Gc)
        assert contrib.min() >= 1 and contrib.max() <= mc
        refused = G.skg_refused(n_tiles, num_kb, Gc)
        assert refused == any(len(G.skg_fragments(c, n_tiles, num_kb, Gc)) > G.SKG_MAX_FRAGS for c in range(Gc))
        if ctas == 0 and n_tiles in (88, 172):
            assert not refused


def test_stream_k_guard_cases():
    # Janus-1.3B (D 2048, F 5632) and Janus-Pro-7B (D 4096, F 11008) gate|up on 148 SMs: at most three tiles per CTA
    for n_tiles, num_kb in ((88, 32), (172, 64)):
        Gc = G.skg_grid(n_tiles, num_kb, 0, 148)
        assert max(len(G.skg_fragments(c, n_tiles, num_kb, Gc)) for c in range(Gc)) <= 3
    # one CTA over five tiles (or 30 one-k-block tiles over 7 CTAs): the kernel would drop fragments, the host refuses
    assert G.skg_refused(5, 8, 1)
    assert G.skg_refused(30, 1, 7) and not G.skg_refused(28, 1, 7)
    assert not G.skg_refused(4, 8, 1)
