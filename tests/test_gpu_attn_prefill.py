"""-m gpu: the prefill and SigLIP attention kernels against an fp64 reference of their own operation
(tests/attn_prefill_ref.py).

Each case launches one attention exactly as the engine does (pg_test_attn_prefill_io / pg_test_vit_attn_io: the engine's
launch_prefill_attn / launch_vit_attn, PDL off) on operands the test owns.  Compared: attn_prefill_tc_kernel (impl 1, bf16,
padded block and packed stream), attn_prefill_kernel (impl 0, bf16 and fp32), vit_attn_tc_kernel (impl 1) and
vit_attn_kernel (impl 0, bf16 and fp32).

Tolerance, |got - ref| <= out_rel |ref| + (expm1(2 E) + 8 * 2^-24 (keys + 16)) * sum_k w_k (|v_k| + |ref|) + allowance:
  * out_rel: the output is an fp32 value rounded to the engine's dtype with RNE, which moves x by at most half an ulp:
    2^-8 |x| in bf16 (2^-23 |x| in fp32);
  * the fp32 accumulations - P.V over at most `keys` keys in tcgen05 MMAs or FMA chains, the row sum, the rescales by
    exp(m_old - m_new) (which multiply numerator and sum alike and cancel in o / l) and the final 1 / l - each add at
    most one ulp (truncating tensor-core adds included) of a partial sum bounded by sum_k p_k |v_k|, so together at most
    a few times 2^-24 * keys of the weighted sum; 8 * (keys + 16) covers them with room for the 1 / l product;
  * E bounds the error of one exp argument that no rounding of the restatement absorbs: fp32 scores that are not
    rounded (CUDA-core prefill: 130 FMA steps of |q||k| * scale; tcgen05 ViT: 12 * 2^-24 of |q||k| for the 4 MMA steps
    plus the fp32 scale * log2e and the rounded maximum), the fp32 product (s - m) * log2e (1.5 * 2^-24 |s - m|) and
    exp2f / expf (2 ulp).  A weight exp(s_k - m) / l then changes by at most a factor exp(+-2E) (numerator and sum);
  * the allowance: the tcgen05 prefill rounds q.k to bf16 (and the bf16 CUDA-core ViT rnd(q.k)) after an fp32 sum whose
    error is at most 20 * 2^-24 (tcgen05: 8 MMA steps of 16, rounded or truncated, plus merges) or (hd + 2) * 2^-24 (FMA)
    times sum_d |q_d k_d|; where the fp64 value lies within that window of a bf16 midpoint, the kernel may take the other
    neighbour, which changes that key's weight by at most |expm1(ds) w / (1 + expm1(ds) w)| and the output by that times
    |v - ref|; when the key may be its block's maximum, every p of the row is rounded relative to a shifted maximum, so
    the p windows below widen by |ds|.  p itself is rounded to bf16 (tcgen05 kernels, bf16 CUDA-core ViT) after an error
    of at most E (plus the widening); a p within that window of a midpoint may round the other way, which changes the
    numerator by one bf16 ulp of p, so the output by that times |v| / l.
The share of outputs that use an allowance is printed for every case (run with -s).

Teeth: every case also asserts, on the reference side, that dropping any single boundary key (the first visible column,
63 / 64 / 127 / 128 / 255 / 256 around block edges, the first column of the last block, the last column; for SigLIP
0, 191 / 192, 383 / 384 and NP - 1) moves the output of its query outside this tolerance.  Keys aligned with that query
are planted on those columns (with all-equal scores, large values), so a kernel that lost one of them fails.  The CPU
tests (test_oracle_attn_prefill.py) show the criterion rejects restated faults by name.

Integrity on every launch: the output is NaN-poisoned with guard rows before and after it; afterwards every owned row is
finite, pad queries of the padded layout are exactly 0, and the guards keep their bits.  In the packed stream duplicate
rows and the columns before kv_start have no output rows, and the real tokens equal the padded launch's bit for bit (the
tiles are in column space in both).  Cache columns outside [kv_start, P) and the rows after the last image hold +-2^100:
finite (a masked key still enters P.V with weight 0, so NaN there would be a false failure), and large enough that a
leaked key blows up the output.  The inputs keep their bits and a second launch agrees bitwise."""
import ctypes as C
import math

import pytest
import torch

from oracle import janus_oracle as O
from tests import attn_prefill_ref as A
from tests.gpu_util import get_engine

pytestmark = pytest.mark.gpu

GUARD = 48
DEV = "cuda"


def _eng(dtype):
    return get_engine(O.TINY, dtype, max_batch=2, max_prompt=64, with_vq=False)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _poisoned(rows, cols, dtype):
    big = torch.full((rows + 2 * GUARD, cols), float("nan"), dtype=dtype, device=DEV)
    return big, big[GUARD:GUARD + rows], big.clone()


def _check_guard(big, before):
    assert torch.equal(_bits(big[:GUARD]), _bits(before[:GUARD])), "guard before the output written"
    assert torch.equal(_bits(big[-GUARD:]), _bits(before[-GUARD:])), "guard after the output written"


def _sentinel(shape, g):
    return (torch.randint(0, 2, shape, generator=g, device=DEV).float() * 2 - 1) * A.SENTINEL


def _compare(got, ref, tol, what):
    got = got.double()
    assert torch.isfinite(got).all(), f"{what}: non-finite output (a row was never written, or a masked key leaked)"
    bad = (got - ref).abs() > tol
    if bad.any():
        i = tuple(int(x) for x in bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} outputs off; first at {i}: got {got[i]:.6g} "
                             f"want {ref[i]:.6g} (tol {tol[i]:.3g})")


def _share(what, allow):
    print(f"\n{what}: {100.0 * float(allow.float().mean()):.3f} % of outputs use the near-midpoint allowance")


# --------------------------------------------------------------------------------------------------------- prefill
def _launch_prefill(eng, impl, q, kc, vc, ks, ro, R, P, H, out):
    from plangen_b200 import _lib
    _lib.check(eng._lib.pg_test_attn_prefill_io(eng._h, impl, _p(q), _p(kc), _p(vc), _p(ks), _p(ro), R, P, H, kc.shape[2],
                                                _p(out), _stream()))


def _run_prefill(kernel, R, H, P, starts, mode="rand", dups=None, seed=0):
    """kernel "tc" | "cc_bf16" | "cc_fp32"; dups: rows with no tokens of their own in a packed launch (tcgen05 only)."""
    bf16 = kernel != "cc_fp32"
    dt = torch.bfloat16 if bf16 else torch.float32
    rnd = A.bf if bf16 else (lambda t: t.float())
    eng = _eng("bf16" if bf16 else "fp32")
    Tmax = P + 5 if (P + 5) % 128 else P + 6         # not a multiple of 128: the last strip's last block leaves the map
    ks = list(starts)
    g = torch.Generator(device=DEV).manual_seed(100 + seed)
    a = math.sqrt(80.0) if mode == "peak" else math.sqrt(3.0)
    q = rnd(torch.randn(R, P, H, 128, generator=g, device=DEV) * (0.0 if mode == "equal" else a))
    K = rnd(torch.randn(R, H, Tmax, 128, generator=g, device=DEV) * a)
    V = rnd(torch.randn(R, H, Tmax, 128, generator=g, device=DEV))
    A.plant_prefill(q, K, V, ks, mode, torch.Generator().manual_seed(seed), rnd)
    for r, st in enumerate(ks):
        for X in (K, V):
            X[r, :, :st] = _sentinel(X[r, :, :st].shape, g)
            X[r, :, P:] = _sentinel(X[r, :, P:].shape, g)
    ref, tol, allow = A.prefill(q, K, V, ks, kernel, elems=1 << 25)
    assert A.undetected_drops(ref, tol, lambda r, h, c: A.prefill_weight(q, K, V, ks, r, h, c),
                              lambda r: A.boundary_columns(ks[r], P)) == []
    _share(f"prefill {kernel} R={R} H={H} P={P} {mode}", allow)

    impl = 1 if kernel == "tc" else 0
    qd, kd, vd = q.to(dt).reshape(R * P, H * 128), K.to(dt), V.to(dt)
    ksd = torch.tensor(ks, dtype=torch.int32, device=DEV)
    before = [t.clone() for t in (qd, kd, vd, ksd)]
    outs = []
    for _ in range(2):
        big, out, snap = _poisoned(R * P, H * 128, dt)
        _launch_prefill(eng, impl, qd, kd, vd, ksd, None, R, P, H, out)
        torch.cuda.synchronize()
        _check_guard(big, snap)
        outs.append(out)
    assert torch.equal(_bits(outs[0]), _bits(outs[1])), "two launches differ"
    got = outs[0].view(R, P, H, 128)
    for r, st in enumerate(ks):
        assert bool((got[r, :st] == 0).all()), f"row {r}: pad queries are not exactly 0"
    _compare(got.float(), ref, tol, f"prefill {kernel}")

    if dups is not None:                               # the packed stream of the same rows
        own = [r for r in range(R) if r not in dups]
        ro = [0]
        for r in range(R):
            ro.append(ro[-1] + (P - ks[r] if r in own else 0))
        rod = torch.tensor(ro, dtype=torch.int32, device=DEV)
        qp = torch.cat([qd.view(R, P, -1)[r, ks[r]:] for r in own]).contiguous()
        before += [qp.clone(), rod.clone()]
        packs = []
        for _ in range(2):
            big, out, snap = _poisoned(ro[-1], H * 128, dt)
            _launch_prefill(eng, 1, qp, kd, vd, ksd, rod, R, P, H, out)
            torch.cuda.synchronize()
            _check_guard(big, snap)
            packs.append(out)
        assert torch.equal(_bits(packs[0]), _bits(packs[1])), "two packed launches differ"
        assert torch.isfinite(packs[0].float()).all(), "a packed row was never written"
        want = torch.cat([outs[0].view(R, P, -1)[r, ks[r]:] for r in own])
        assert torch.equal(_bits(packs[0]), _bits(want)), "packed stream differs from the padded block"
        after = [qd, kd, vd, ksd, qp, rod]
    else:
        after = [qd, kd, vd, ksd]
    for b, a_ in zip(before, after):
        assert torch.equal(_bits(b) if b.is_floating_point() else b, _bits(a_) if a_.is_floating_point() else a_), "an input changed"


def _pc(R, H, P, starts, mode="rand", dups=None, seed=0):
    return dict(R=R, H=H, P=P, starts=starts, mode=mode, dups=dups, seed=seed)


PREFILL_CASES = {
    "P1": _pc(2, 2, 1, [0, 1]),
    "P2": _pc(3, 2, 2, [0, 1, 2], seed=1),
    "P127": _pc(4, 2, 127, [0, 1, 126, 127], seed=2),
    "P128": _pc(4, 2, 128, [0, 64, 127, 128], seed=3),
    "P129": _pc(4, 1, 129, [0, 127, 128, 129], seed=4),
    "P255_H16": _pc(3, 16, 255, [0, 127, 254], seed=5),
    "P256_H32": _pc(2, 32, 256, [128, 255], seed=6),
    "P383_R32": _pc(32, 1, 383, [[0, 127, 128, 129, 200, 255, 256, 382, 383][r % 9] for r in range(32)], seed=7),
    "P385": _pc(4, 2, 385, [0, 129, 256, 384], seed=8),
    "P512_peak": _pc(4, 2, 512, [0, 127, 300, 511], mode="peak", seed=9),
    "P600_equal": _pc(3, 2, 600, [0, 128, 599], mode="equal", seed=10),
    "P1100_H16": _pc(2, 16, 1100, [0, 700], seed=11),
    "P1100_R8_peak": _pc(8, 2, 1100, [0, 1, 127, 128, 129, 640, 1023, 1099], mode="peak", seed=12),
}

PACKED_CASES = {
    "P129_dup": _pc(4, 2, 129, [0, 127, 0, 128], dups={2}, seed=13),
    "P385_all_pad_and_dup": _pc(5, 2, 385, [1, 129, 385, 1, 384], dups={3}, seed=14),
    "P600_H16": _pc(4, 16, 600, [0, 300, 0, 599], dups={2}, seed=15),
    "P1100": _pc(3, 2, 1100, [1, 1000, 129], dups=set(), seed=16),
    "P256_R32": _pc(32, 1, 256, [[0, 127, 128, 255][r % 4] for r in range(32)], dups={5, 6, 7, 20}, seed=17),
}


@pytest.mark.parametrize("kernel", ["tc", "cc_bf16", "cc_fp32"])
@pytest.mark.parametrize("name", list(PREFILL_CASES))
def test_prefill_attention_matches_fp64_reference(name, kernel):
    _run_prefill(kernel, **PREFILL_CASES[name])


@pytest.mark.parametrize("name", list(PACKED_CASES))
def test_prefill_tc_packed_stream_matches_reference_and_padded_block(name):
    _run_prefill("tc", **PACKED_CASES[name])


# ------------------------------------------------------------------------------------------------------------ SigLIP
def _launch_vit(eng, impl, qkv, n, NP, W, heads, out):
    from plangen_b200 import _lib
    _lib.check(eng._lib.pg_test_vit_attn_io(eng._h, impl, _p(qkv), qkv.shape[0], n, NP, W, heads, _p(out), _stream()))


def _run_vit(kernel, NP, n, heads, mode="rand", hd=64, seed=0):
    bf16 = kernel != "cc_fp32"
    dt = torch.bfloat16 if bf16 else torch.float32
    rnd = A.bf if bf16 else (lambda t: t.float())
    eng = _eng("bf16" if bf16 else "fp32")
    W = heads * hd
    g = torch.Generator(device=DEV).manual_seed(200 + seed)
    qkv = torch.randn((n + 1) * NP, 3 * W, generator=g, device=DEV) * math.sqrt(3.0)
    if mode == "peak":
        qkv[:, :2 * W] *= math.sqrt(80.0 / 3.0)
    if mode == "equal":
        qkv[:, :W] = 0.0
    qkv = rnd(qkv)
    A.plant_vit(qkv, n, NP, W, heads, mode, torch.Generator().manual_seed(seed), rnd)
    qkv[n * NP:] = _sentinel(qkv[n * NP:].shape, g)    # the image after the last one
    ref, tol, allow = A.vit(qkv, n, NP, W, heads, kernel)
    R4, T4 = ref.view(n, NP, heads, hd), tol.view(n, NP, heads, hd)
    assert A.undetected_drops(R4, T4, lambda i, h, c: A.vit_weight(qkv, NP, W, heads, i, h, c),
                              lambda i: A.vit_boundary_columns(NP)) == []
    _share(f"SigLIP {kernel} NP={NP} n={n} heads={heads} {mode}", allow)

    impl = 1 if kernel == "tc" else 0
    qd = qkv.to(dt)
    before = qd.clone()
    outs = []
    for rows in ((n + 1) * NP, (n + 1) * NP, n * NP):  # the maps cover the extra image, twice; then only the n images
        big, out, snap = _poisoned(n * NP, W, dt)
        _launch_vit(eng, impl, qd[:rows], n, NP, W, heads, out)
        torch.cuda.synchronize()
        _check_guard(big, snap)
        outs.append(out)
    assert torch.equal(_bits(outs[0]), _bits(outs[1])), "two launches differ"
    assert torch.equal(_bits(outs[0]), _bits(outs[2])), "the rows after the last image changed the result"
    assert torch.equal(_bits(before), _bits(qd)), "qkv changed"
    _compare(outs[0].view(n * NP, heads, hd).float(), ref, tol, f"SigLIP {kernel}")


VIT_CASES = {
    "NP2": dict(NP=2, n=1, heads=1),
    "NP36_n3": dict(NP=36, n=3, heads=2, seed=1),
    "NP128_H16_peak": dict(NP=128, n=1, heads=16, mode="peak", seed=2),
    "NP190_n3": dict(NP=190, n=3, heads=2, seed=3),
    "NP192_equal": dict(NP=192, n=1, heads=2, mode="equal", seed=4),
    "NP194_n3": dict(NP=194, n=3, heads=1, seed=5),
    "NP384_peak": dict(NP=384, n=1, heads=2, mode="peak", seed=6),
    "NP576_n3_H16": dict(NP=576, n=3, heads=16, seed=7),
    "NP1024": dict(NP=1024, n=1, heads=2, seed=8),
}


@pytest.mark.parametrize("kernel", ["tc", "cc_bf16", "cc_fp32"])
@pytest.mark.parametrize("name", list(VIT_CASES))
def test_vit_attention_matches_fp64_reference(name, kernel):
    _run_vit(kernel, **VIT_CASES[name])


def test_vit_cuda_core_kernel_with_head_dim_128():
    _run_vit("cc_bf16", NP=100, n=2, heads=2, hd=128, seed=9)


# ------------------------------------------------------------------------------------------------------- bad input
def test_test_entries_reject_bad_arguments_by_name():
    from plangen_b200 import _lib
    eng, e32 = _eng("bf16"), _eng("fp32")
    R, P, H, Tmax = 2, 8, 1, 16
    q = torch.zeros(R * P, H * 128, dtype=torch.bfloat16, device=DEV)
    kc = torch.zeros(R, H, Tmax, 128, dtype=torch.bfloat16, device=DEV)
    out = torch.zeros_like(q)
    ks = torch.tensor([0, 3], dtype=torch.int32, device=DEV)
    ro_bad = torch.tensor([0, 8, 12], dtype=torch.int32, device=DEV)          # row 1 has 5 tokens, not 4
    ks_bad = torch.tensor([0, 9], dtype=torch.int32, device=DEV)
    bad = [
        ("impl", dict(impl=2)), ("row_off", dict(impl=0, ro=ro_bad)), ("null operand", dict(q=None)),
        ("Tmax", dict(P=Tmax + 1)), ("kv_start", dict(ks=ks_bad)), ("row_off", dict(ro=ro_bad)),
    ]
    for word, kw in bad:
        a = dict(eng=eng, impl=1, q=q, ks=ks, ro=None, P=P)
        a.update(kw)
        with pytest.raises(_lib.PgError, match=word):
            _launch_prefill(a["eng"], a["impl"], a["q"], kc, kc, a["ks"], a["ro"], R, a["P"], H, out)
    q32 = torch.zeros(R * P, H * 128, device=DEV)
    with pytest.raises(_lib.PgError, match="tcgen05"):
        _launch_prefill(e32, 1, q32, kc, kc, ks, None, R, P, H, q32)
    qkv = torch.zeros(2048, 3 * 128, dtype=torch.bfloat16, device=DEV)
    vo = torch.zeros(64, 128, dtype=torch.bfloat16, device=DEV)
    for word, (impl, rows, n, NP, heads) in {"hd": (1, 64, 1, 64, 1), "qkv_rows": (0, 32, 1, 64, 2),
                                             "NP": (0, 64, 1, 2000, 2), "impl": (3, 64, 1, 64, 2)}.items():
        with pytest.raises(_lib.PgError, match=word):
            _launch_vit(eng, impl, qkv[:rows], n, NP, 128, heads, vo)
    with pytest.raises(_lib.PgError, match="hd"):
        _launch_vit(eng, 0, torch.zeros(8, 3 * 256, dtype=torch.bfloat16, device=DEV), 1, 8, 256, 1, vo)
