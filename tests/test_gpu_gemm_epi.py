"""-m gpu: the tcgen05 contractions and their fused epilogues against tests/gemm_ref.py.

Each case runs one contraction exactly as the engine issues it (pg_test_contraction_run: run_gemm, run_conv_gemm, the
stream-K gate|up launch; PDL off) on operands the test owns, and asserts the kernel it reached: gemm_tc_kernel<NT>, the
CTA pair (gemm_tc2_kernel), stream-K (gemm_swiglu_sk_kernel<NT>), the implicit convolution, or im2col when the
convolution does not qualify.

Acceptance criteria:
  A. Accumulators.  Each kernel's plain fp32 store (split-K partials summed) is within rtol 1e-4, atol 2e-6 max|ref| of
     fp64 X.W^T (bf16 products are exact; only the fp32 summation order differs), also for tile-major weights and the
     convolution geometries.  Tile-major and TMA weights give bitwise-equal accumulators: the same MMAs on the same bytes.
  B. Epilogues of gemm_tc / gemm_tc2 / the convolution.  The plain store with splits = 1 runs the same kernel with the
     same MMA order (the reported path shows it), so its fp32 values are exactly what the fused epilogue reads from
     TMEM.  The fused output must equal the restatement (gemm_ref: bf16(acc + bias), bf16(bf16(acc + bias) + add16),
     resid + bf16(acc + bias), the QKV RoPE / scatter) on those accumulators bit for bit.  The documented approximations
     are the exception: erf_fast in GELU, the ex2 / rcp silu of the decode SwiGLU and expf in the pair's.  There the
     restatement computes the exact value v before the bf16 rounding and the kernel's fp32 value lies within
     delta = 2^-18 |v| (plus erf_fast's absolute error times |t| / 2 for GELU, |g| 2^-22 |v| for ex2 / rcp) of it; rounding
     is monotone, so the result must lie in [bf16(v - delta), bf16(v + delta)].  That is one value, or the two
     neighbours of a midpoint within delta of v (one ulp); the test reports how many elements that covers and bounds
     the fraction below 1 %.
  C. Stream-K.  It has no accumulators of its own to restate, so the restatement runs on the fp64 accumulators: g and u
     may round either way where they lie within the fp32 summation bound (gemm_ref.sum_bound: one rounding of at most an
     ulp of sum |x w| per 16-deep MMA step plus 16 merges) of a midpoint, silu as in B.  The decode SwiGLU epilogue on
     the same operands meets the same rule.  The bound is a worst case, so the ambiguous share is reported, not bounded
     tightly; tests/test_oracle_gemm_epi.py shows each criterion still rejects the plausible faults on such data.

Integrity on every launch: outputs sit in NaN-poisoned buffers with a guard after them, and rows >= M and the guard
stay bitwise untouched; QKV leaves every cache column but those its tokens own, and every q row >= M, bitwise unchanged;
stream-K's counters are zero again afterwards; a second launch gives bitwise-equal results."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import janus_oracle as O
from plangen_b200.config import Dims
from plangen_b200.weights import rope_tables
from tests import gemm_ref as G
from tests.gpu_util import assert_close, get_engine

pytestmark = pytest.mark.gpu

PLAIN, ROWS, RESID, SWIGLU, QKV, SWIGLU_SK, CONV = range(7)
P_TC, P_TC2, P_SK, P_CONV, P_IM2COL = 2, 3, 4, 5, 6
GUARD = 4096
NEAR_MAX = 0.01


def _eng():
    # the engine of test_gpu_attn_decode.py (cached): RoPE tables up to position 2239
    return get_engine(O.TINY, "bf16", max_batch=128, max_prompt=2176, with_vq=False)


def _nt(M):
    return 16 if M <= 16 else 32 if M <= 32 else 64 if M <= 64 else 128 if M <= 128 else 256


def _run(eng, **kw):
    from plangen_b200 import _lib
    p = _lib.PgTestContraction()
    for k, v in kw.items():
        if isinstance(v, torch.Tensor):
            v = v.data_ptr()
        setattr(p, k, v)
    _lib.check(eng._lib.pg_test_contraction_run(eng._h, C.byref(p), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    return p.path, p.path_nt


def _poisoned(rows, cols, dtype):
    """(flat buffer, [rows][cols] view): NaN everywhere, `GUARD` elements after the view."""
    buf = torch.full((rows * cols + GUARD,), float("nan"), dtype=dtype, device="cuda")
    return buf, buf[:rows * cols].view(rows, cols)


def _untouched(buf, start):
    ref = torch.full_like(buf[start:], float("nan"))
    bits = torch.int16 if buf.dtype == torch.bfloat16 else torch.int32
    return torch.equal(buf[start:].view(bits), ref.view(bits))


def _operands(M, N, K, seed, w=None):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(M, K, generator=g).to(torch.bfloat16)
    W = w if w is not None else (torch.randn(N, K, generator=g) / math.sqrt(K)).to(torch.bfloat16)
    return X, W, g


def _plain(eng, X, W, splits=1, weights=0, conv=None):
    """fp32 accumulators of the plain store (summed over splits), the path, and the tile-major buffer (weights=1)."""
    M, N, K = X.shape[0] if conv is None else conv[0] * conv[1] * conv[2], W.shape[0], W.shape[1]
    buf, Cv = _poisoned(splits * M, N, torch.float32)
    kw = dict(X=X.cuda() if not X.is_cuda else X, W=W.cuda() if not W.is_cuda else W, M=M, N=N, K=K, splits=splits, C=Cv,
              c_bytes=splits * M * N * 4, weights=weights)
    wt = None
    if weights:
        wt = torch.zeros((-(-N // 128)) * (-(-K // 64)) * G.TILE_BYTES, dtype=torch.uint8, device="cuda")
        kw.update(w_tiled=wt, w_tiled_bytes=wt.numel())
    if conv is not None:
        kw.update(mode=CONV, img_b=conv[0], img_h=conv[1], img_w=conv[2])
    path = _run(eng, **kw)
    assert _untouched(buf, splits * M * N), "plain store wrote past its partials"
    assert torch.isfinite(Cv).all(), "plain store left NaN in its partials"
    acc = Cv.view(splits, M, N).sum(0).cpu()
    return acc, path, wt


def _check_acc(acc, want, what):
    assert_close(acc.numpy(), want.numpy(), rtol=1e-4, atol_frac=2e-6, what=what)


def _rows_launch(eng, X, W, M, N, K, weights=0, bias=None, gelu=0, add16=None, alias=False, conv=None, twice=True):
    """Fused bf16 rows; returns ([M][N] fp32 values, path).  alias: add16 is the output buffer itself."""
    buf, out = _poisoned(M, N, torch.bfloat16)
    if alias:
        out.copy_(add16)
    kw = dict(mode=ROWS if conv is None else CONV, X=X.cuda(), W=W.cuda(), M=M, N=N, K=K, out=out, gelu=gelu, weights=weights,
              bias=bias.cuda() if bias is not None else None, add16=(out if alias else add16.cuda()) if add16 is not None else None)
    if weights:
        wt = torch.zeros((-(-N // 128)) * (-(-K // 64)) * G.TILE_BYTES, dtype=torch.uint8, device="cuda")
        kw.update(w_tiled=wt, w_tiled_bytes=wt.numel())
    if conv is not None:
        kw.update(img_b=conv[0], img_h=conv[1], img_w=conv[2])
    if kw["bias"] is None:
        kw.pop("bias")
    if kw["add16"] is None:
        kw.pop("add16")
    bias_dev, add_dev = kw.get("bias"), kw.get("add16")      # keep them alive through the launch
    path = _run(eng, **kw)
    got = out.clone()
    assert _untouched(buf, M * N), "fused rows wrote past row M"
    if twice:
        if alias:
            out.copy_(add16)
        _run(eng, **kw)
        assert torch.equal(out.view(torch.int16), got.view(torch.int16)), "two launches differ"
    del bias_dev, add_dev
    return got.float().cpu(), path


def _resid_launch(eng, X, W, M, N, K, bias, res0, weights=0):
    buf, res = _poisoned(M, N, torch.float32)
    res.copy_(res0)
    kw = dict(mode=RESID, X=X.cuda(), W=W.cuda(), M=M, N=N, K=K, resid=res, bias=bias.cuda(), weights=weights)
    if weights:
        wt = torch.zeros((-(-N // 128)) * (-(-K // 64)) * G.TILE_BYTES, dtype=torch.uint8, device="cuda")
        kw.update(w_tiled=wt, w_tiled_bytes=wt.numel())
    path = _run(eng, **kw)
    got = res.clone()
    assert _untouched(buf, M * N), "residual add wrote past row M"
    res.copy_(res0)
    _run(eng, **kw)
    assert torch.equal(res.view(torch.int32), got.view(torch.int32)), "two launches differ"
    return got.cpu(), path


def _report(what, lo, hi):
    amb = int((lo != hi).sum())
    frac = amb / lo.numel()
    print(f"{what}: {amb} of {lo.numel()} elements ({100 * frac:.3f} %) within the approximation's reach of a midpoint")
    return frac


def _assert_epilogue_rows(eng, X, W, M, N, K, path_want, g, weights=0, conv=None):
    """criterion B for the four row epilogues, on the plain store's accumulators of the same kernel."""
    acc, path, _ = _plain(eng, X, W, weights=weights, conv=conv)
    assert path == path_want, f"plain store ran {path}, expected {path_want}"
    bias = 0.5 * torch.randn(N, generator=g)
    add16 = torch.randn(M, N, generator=g).to(torch.bfloat16)
    got, path = _rows_launch(eng, X, W, M, N, K, weights, bias=bias, conv=conv)
    assert path == path_want
    assert torch.equal(got, G.rows(acc, bias)), "bias -> bf16 rows differ from bf16(acc + bias)"
    got, path = _rows_launch(eng, X, W, M, N, K, weights, bias=bias, add16=add16, conv=conv)
    assert path == path_want
    assert torch.equal(got, G.rows(acc, bias, add16)), "add16 rows differ from bf16(bf16(acc + bias) + add16)"
    got, path = _rows_launch(eng, X, W, M, N, K, weights, bias=bias, add16=add16, alias=True, conv=conv)
    assert path == path_want
    assert torch.equal(got, G.rows(acc, bias, add16)), "add16 aliasing out differs"
    if conv is not None:
        return acc
    got, path = _rows_launch(eng, X, W, M, N, K, weights, bias=bias, gelu=1)
    assert path == path_want
    lo, hi = G.gelu_rows(acc, bias)
    bad = ~G.in_interval(got, lo, hi)
    assert not bad.any(), f"GELU rows: {int(bad.sum())} elements outside the erf_fast interval"
    assert _report(f"GELU M={M} N={N} K={K} path={path}", lo, hi) < NEAR_MAX
    res0 = torch.randn(M, N, generator=g).cuda()
    got, path = _resid_launch(eng, X, W, M, N, K, bias, res0, weights)
    assert path == path_want
    assert torch.equal(got, G.resid(res0.cpu(), acc, bias)), "residual add differs from resid + bf16(acc + bias)"
    return acc


# ------------------------------------------------------------------------------------------------ gemm_tc<NT>
TC_CASES = [  # (M, N, K): every token-tile width, N = 8 (mod 128) and multiples of 128, a single k-block, ragged K, ring reuse
    (1, 136, 64), (15, 256, 72), (17, 136, 200), (33, 384, 2048), (64, 520, 200), (100, 264, 5632), (128, 128, 2048),
    (129, 128, 200), (300, 8, 72), (200, 120, 2048),
]


@pytest.mark.parametrize("M,N,K", TC_CASES)
def test_gemm_tc_epilogues(M, N, K):
    eng = _eng()
    X, W, g = _operands(M, N, K, M * 131 + N + K)
    want = G.acc64(X, W)
    acc0, path0, _ = _plain(eng, X, W)
    acc1, path1, wt = _plain(eng, X, W, weights=1)
    assert path0 == path1 == (P_TC, _nt(M)), (path0, path1)
    _check_acc(acc0, want, f"gemm_tc<{_nt(M)}> {M}x{N}x{K}")
    assert torch.equal(acc0.view(torch.int32), acc1.view(torch.int32)), "tile-major and TMA weights give different accumulators"
    assert np.array_equal(wt.cpu().numpy(), G.tile_major(W)), "tile-major copy differs from the SWIZZLE_128B restatement"
    accs, paths, _ = _plain(eng, X, W, splits=3)
    assert paths[0] == P_TC
    _check_acc(accs, want, f"gemm_tc<{_nt(M)}> {M}x{N}x{K} / 3 splits")
    for weights in (0, 1):
        _assert_epilogue_rows(eng, X, W, M, N, K, (P_TC, _nt(M)), g, weights)


def _swiglu_launch(eng, X, W, M, F, K, weights, mode=SWIGLU, **kw):
    buf, out = _poisoned(M, F, torch.bfloat16)
    args = dict(mode=mode, X=X.cuda(), W=W.cuda(), M=M, N=2 * F, K=K, out=out, weights=weights, **kw)
    if weights:
        wt = torch.zeros((-(-2 * F // 128)) * (-(-K // 64)) * G.TILE_BYTES, dtype=torch.uint8, device="cuda")
        args.update(w_tiled=wt, w_tiled_bytes=wt.numel())
    path = _run(eng, **args)
    got = out.clone()
    assert _untouched(buf, M * F), "SwiGLU wrote past row M"
    _run(eng, **args)
    assert torch.equal(out.view(torch.int16), got.view(torch.int16)), "two launches differ"
    return got.float().cpu(), path, args


def _gate_up(M, F, K, seed):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(M, K, generator=g).to(torch.bfloat16)
    Wg = (torch.randn(F, K, generator=g) / math.sqrt(K)).to(torch.bfloat16)
    Wu = (torch.randn(F, K, generator=g) / math.sqrt(K)).to(torch.bfloat16)
    return X, G.pack_gate_up(Wg, Wu)


@pytest.mark.parametrize("M", [1, 17, 64, 100, 128])
@pytest.mark.parametrize("F,K", [(64, 200), (320, 2048), (1408, 512)])
def test_gemm_tc_swiglu_decode(M, F, K):
    eng = _eng()
    X, W = _gate_up(M, F, K, M + F + K)
    for weights in (0, 1):
        acc, path, _ = _plain(eng, X, W, weights=weights)
        assert path == (P_TC, _nt(M))
        _check_acc(acc, G.acc64(X, W), "gate|up accumulators")
        got, path, _ = _swiglu_launch(eng, X, W, M, F, K, weights)
        assert path == (P_TC, _nt(M))
        lo, hi = G.swiglu(acc, fast=True)
        bad = ~G.in_interval(got, lo, hi)
        assert not bad.any(), f"decode SwiGLU: {int(bad.sum())} elements outside bf16(bf16(silu(bf16 g)) * bf16 u)"
        assert _report(f"decode SwiGLU M={M} F={F} K={K} weights={weights}", lo, hi) < NEAR_MAX


# ------------------------------------------------------------------------------------------------ CTA pair
PAIR_CASES = [  # (M, N, K): odd weight-tile counts (the last pair's second CTA has no rows), ragged M, N = 8 (mod 128)
    (129, 384, 200), (255, 136, 72), (257, 640, 1024), (513, 1160, 200), (2048, 384, 1024),
]


@pytest.mark.parametrize("M,N,K", PAIR_CASES)
def test_gemm_tc2_epilogues(M, N, K):
    eng = _eng()
    X, W, g = _operands(M, N, K, M * 7 + N + K)
    acc, path, _ = _plain(eng, X, W)
    assert path == (P_TC2, 256)
    _check_acc(acc, G.acc64(X, W), f"CTA pair {M}x{N}x{K}")
    _assert_epilogue_rows(eng, X, W, M, N, K, (P_TC2, 256), g)


@pytest.mark.parametrize("M", [129, 257, 2048])
@pytest.mark.parametrize("F", [192, 320, 1408])
def test_gemm_tc2_swiglu(M, F):
    eng = _eng()
    K = 512
    X, W = _gate_up(M, F, K, M * 3 + F)
    acc, path, _ = _plain(eng, X, W)
    assert path == (P_TC2, 256)
    got, path, _ = _swiglu_launch(eng, X, W, M, F, K, 0)
    assert path == (P_TC2, 256)
    lo, hi = G.swiglu(acc, fast=False)
    bad = ~G.in_interval(got, lo, hi)
    assert not bad.any(), f"pair SwiGLU: {int(bad.sum())} elements outside bf16(bf16(silu(bf16 g)) * bf16 u)"
    assert _report(f"pair SwiGLU M={M} F={F}", lo, hi) < NEAR_MAX


QKV_CASES = [  # (H, layout, rope_start): padded [R][P] blocks, packed streams with a deduplicated (empty) row and a one-token row
    (1, "padded", False), (2, "padded", True), (4, "packed", False), (16, "packed", True), (2, "packed_long", False),
    (4, "packed_long", True),
]


def _qkv_layout(layout):
    if layout == "padded":
        R, P = 3, 100
        return R, P, 3 * 100, None, [0, 37, 99], None
    if layout == "packed":                # rows: 70 tokens, empty, one token, the rest
        R, P = 4, 0
        return R, P, 200, [0, 70, 70, 71], [3, 9, 40, 0], None
    R, P = 3, 0                           # long positions: up to the RoPE tables' end
    return R, P, 400, [0, 1, 1], [2000, 5, 1800], None


@pytest.mark.parametrize("H,layout,with_rs", QKV_CASES)
def test_gemm_tc2_qkv(H, layout, with_rs):
    eng = _eng()
    K = 256
    N = 3 * H * 128
    R, P, M, row_off, kv_start, _ = _qkv_layout(layout)
    rope_start = [max(s - 3 * r, 0) for r, s in enumerate(kv_start)] if with_rs else None
    if layout == "padded" and with_rs:
        rope_start = [0, 37, 99]
    Tmax = 2240 if layout == "packed_long" else 256
    X, W, g = _operands(M, N, K, H * 1000 + M)
    acc, path, _ = _plain(eng, X, W)
    assert path == (P_TC2, 256)
    tmax_eng = eng.counter("tmax")
    assert Tmax <= tmax_eng
    cos, sin = rope_tables(Dims.from_any(O.TINY), tmax_eng)
    rw, col, pr = G.qkv_positions(M, R, P, row_off, kv_start, rope_start)
    kc0 = torch.full((R, H, Tmax, 128), float("nan"), dtype=torch.bfloat16)
    vc0 = kc0.clone()
    q_ref, kc_ref, vc_ref = G.qkv(acc, H, cos, sin, rw, col, pr, kc0.float(), vc0.float())
    qbuf, q = _poisoned(M, H * 128, torch.bfloat16)
    kc, vc = kc0.cuda(), vc0.cuda()
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device="cuda") if v is not None else None
    ro_d, ks_d, rs_d = i32(row_off), i32(kv_start), i32(rope_start)
    args = dict(mode=QKV, X=X.cuda(), W=W.cuda(), M=M, N=N, K=K, q_out=q, kcache=kc, vcache=vc, kv_start=ks_d, R=R, P=P, H=H,
                Tmax=Tmax)
    if ro_d is not None:
        args["row_off"] = ro_d
    if rs_d is not None:
        args["rope_start"] = rs_d
    for rep in range(2):
        path = _run(eng, **args)
        assert path == (P_TC2, 256)
        assert _untouched(qbuf, M * H * 128), "q rows >= M written"
        assert torch.equal(q.cpu().float(), q_ref), f"q differs from bf16(acc) rotated at its RoPE position (launch {rep})"
        assert torch.equal(kc.cpu().view(torch.int16), _cache_bits(kc0, kc_ref, rw, col)), "K cache differs"
        assert torch.equal(vc.cpu().view(torch.int16), _cache_bits(vc0, vc_ref, rw, col)), "V cache differs"


def _cache_bits(c0, ref, rw, col):
    """Expected cache bits: the initial (poisoned) bits everywhere except the columns the tokens own, which hold the
    reference's values.  Taken from c0 itself, since a NaN's bits do not survive a float round trip."""
    bits = c0.view(torch.int16).clone()
    rw_t, col_t = torch.as_tensor(rw, dtype=torch.int64), torch.as_tensor(col, dtype=torch.int64)
    bits[rw_t, :, col_t] = ref[rw_t, :, col_t].to(torch.bfloat16).view(torch.int16)
    return bits


# ------------------------------------------------------------------------------------------------ stream-K
SK_CASES = [  # (M, F, D, ctas): -1 = every SM, 0 = the production rule
    (1, 256, 512, 1),        # one CTA, four whole tiles: one contributor each
    (16, 320, 1024, 7),      # ranges shorter than a tile
    (33, 320, 1024, 5),      # exactly one tile per CTA
    (17, 1408, 2048, -1),    # all SMs
    (64, 128, 512, 0),       # production rule, U < SMs: one k-block per CTA, eight contributors per tile
    (64, 1408, 256, 7),      # a whole tile plus a head and a tail
    (33, 704, 512, 0),
]


@pytest.mark.parametrize("M,F,D,ctas", SK_CASES)
def test_stream_k_swiglu(M, F, D, ctas):
    eng = _eng()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ctas = sms if ctas == -1 else ctas
    n_tiles, num_kb = 2 * F // 128, D // 64
    Gc = G.skg_grid(n_tiles, num_kb, ctas, sms)
    assert not G.skg_refused(n_tiles, num_kb, Gc)
    contrib = G.skg_contributors(n_tiles, num_kb, Gc)
    print(f"stream-K M={M} F={F} D={D}: {Gc} CTAs, contributors per tile {contrib.min()}..{contrib.max()}")
    mc = G.skg_max_contrib(n_tiles, num_kb, Gc)
    NT = 16 if M <= 16 else 32 if M <= 32 else 64
    scratch = torch.full((n_tiles * mc * NT * 128,), float("nan"), dtype=torch.float32, device="cuda")
    counters = torch.zeros(n_tiles + 64, dtype=torch.int32, device="cuda")
    X, W = _gate_up(M, F, D, M * 5 + F + D)
    got, path, _ = _swiglu_launch(eng, X, W, M, F, D, 1, mode=SWIGLU_SK, ctas=ctas, scratch=scratch,
                                  scratch_bytes=scratch.numel() * 4, counters=counters, n_counters=n_tiles)
    assert path == (P_SK, NT)
    assert int(counters.abs().sum()) == 0, "stream-K counters not re-armed"
    a64 = G.acc64(X, W)
    lo, hi = G.swiglu64(a64, G.sum_bound(X, W))
    bad = ~G.in_interval(got, lo, hi)
    assert not bad.any(), f"stream-K SwiGLU: {int(bad.sum())} elements outside the fp64 restatement's reach"
    _report(f"stream-K SwiGLU M={M} F={F} D={D} ctas={ctas}", lo, hi)
    dec, path, _ = _swiglu_launch(eng, X, W, M, F, D, 1)
    assert path == (P_TC, _nt(M))
    assert G.in_interval(dec, lo, hi).all(), "decode SwiGLU outside the fp64 restatement's reach"
    print(f"  stream-K and decode SwiGLU differ at {int((dec != got).sum())} of {got.numel()} elements")


def test_stream_k_refuses_cut_beyond_fragments():
    """A CTA whose range touches more than SKG_MAX_FRAGS tiles is refused on the host, before any launch."""
    from plangen_b200 import _lib
    eng = _eng()
    M, F, D = 1, 320, 512                    # five tiles of eight k-blocks on one CTA
    assert G.skg_refused(5, 8, 1)
    X, W = _gate_up(M, F, D, 3)
    scratch = torch.zeros(5 * 9 * 16 * 128, dtype=torch.float32, device="cuda")
    counters = torch.zeros(5, dtype=torch.int32, device="cuda")
    with pytest.raises(_lib.PgError, match="fragments"):
        _swiglu_launch(eng, X, W, M, F, D, 1, mode=SWIGLU_SK, ctas=1, scratch=scratch, scratch_bytes=scratch.numel() * 4,
                       counters=counters, n_counters=5)


# ------------------------------------------------------------------------------------------------ convolution
CONV_CASES = [  # (B, H, W, Cin, Cout): bw == W with a partial bottom block, bw == 192, several images per launch
    (1, 70, 3, 64, 8), (3, 10, 24, 192, 72), (1, 6, 48, 64, 128), (3, 3, 96, 64, 256), (1, 2, 192, 512, 72),
    (1, 3, 384, 192, 8), (3, 5, 24, 64, 128),
]


@pytest.mark.parametrize("B,H,W,Cin,Cout", CONV_CASES)
def test_conv_implicit(B, H, W, Cin, Cout):
    eng = _eng()
    g = torch.Generator().manual_seed(B * H * W + Cin + Cout)
    act = torch.randn(B, H, W, Cin, generator=g).to(torch.bfloat16)
    Wc = (torch.randn(Cout, 9 * Cin, generator=g) / math.sqrt(9 * Cin)).to(torch.bfloat16)
    M = B * H * W
    X = act.reshape(M, Cin)
    acc, path, _ = _plain(eng, X.cuda(), Wc, conv=(B, H, W))
    assert path == (P_CONV, 192), path
    _check_acc(acc, G.conv_cols(act).double() @ Wc.double().T, f"conv {B}x{H}x{W}x{Cin}->{Cout}")
    _assert_epilogue_rows(eng, X, Wc, M, Cout, 9 * Cin, (P_CONV, 192), g, conv=(B, H, W))


@pytest.mark.parametrize("W,Cin", [(5, 64), (24, 32)])
def test_conv_not_taken(W, Cin):
    eng = _eng()
    X = torch.zeros(2 * W, Cin, dtype=torch.bfloat16, device="cuda")
    Wc = torch.zeros(8, 9 * Cin, dtype=torch.bfloat16, device="cuda")
    C_ = torch.zeros(2 * W, 8, device="cuda")
    assert _run(eng, mode=CONV, X=X, W=Wc, M=2 * W, N=8, K=9 * Cin, C=C_, c_bytes=C_.numel() * 4, img_b=1, img_h=2,
                img_w=W) == (P_IM2COL, 0)


def test_contraction_bounds_fail_by_name():
    from plangen_b200 import _lib
    eng = _eng()
    X = torch.zeros(300, 256, dtype=torch.bfloat16, device="cuda")
    W = torch.zeros(768, 256, dtype=torch.bfloat16, device="cuda")
    out = torch.zeros(300 * 768, dtype=torch.bfloat16, device="cuda")
    ks = torch.zeros(3, dtype=torch.int32, device="cuda")
    ks_far = torch.tensor([2100], dtype=torch.int32, device="cuda")
    ro = torch.zeros(1, dtype=torch.int32, device="cuda")
    cases = [
        (dict(mode=SWIGLU, M=4, N=200, out=out), "N % 128"),
        (dict(mode=QKV, M=300, N=768, q_out=out, kcache=out, vcache=out, kv_start=ks, R=3, P=100, H=1, Tmax=128), "3\\*H\\*128"),
        (dict(mode=QKV, M=100, N=768, q_out=out, kcache=out, vcache=out, kv_start=ks, R=1, P=100, H=2, Tmax=128), "CTA pair"),
        (dict(mode=QKV, M=300, N=768, q_out=out, kcache=out, vcache=out, kv_start=ks, R=3, P=100, H=2, Tmax=50), "Tmax=50"),
        (dict(mode=QKV, M=300, N=768, q_out=out, kcache=out, vcache=out, kv_start=ks_far, row_off=ro, R=1, H=2, Tmax=4000),
         "engine's Tmax"),
        (dict(mode=ROWS, M=300, N=768, out=out, weights=1, w_tiled=out, w_tiled_bytes=out.numel() * 2), "CTA pair"),
        (dict(mode=SWIGLU_SK, M=65, N=256, out=out, weights=1, w_tiled=out, w_tiled_bytes=out.numel() * 2, scratch=out,
              scratch_bytes=out.numel() * 2, counters=ks, n_counters=3), "M=65"),
        (dict(mode=SWIGLU_SK, M=8, N=256, out=out, weights=0), "tile-major"),
        (dict(mode=ROWS, M=8, N=768, out=out, gelu=2), "gelu=2"),
    ]
    for kw, msg in cases:
        kw.setdefault("K", 256)
        with pytest.raises(_lib.PgError, match=msg):
            _run(eng, X=X, W=W, **kw)
