"""Reference of one prefill-attention launch (attn_prefill_tc.cuh attn_prefill_tc_kernel, lm_kernels.cuh
attn_prefill_kernel) and of one SigLIP attention launch (vit_kernels.cuh vit_attn_tc_kernel, vit_attn_kernel).

Each kernel is restated in fp64 at its own rounding points, with its own key blocks:
  * tcgen05 prefill: s = bf16(bf16(q.k) * scale) (fp32 product); 128-key blocks from kv_start // 128; per block the running
    maximum m, p = bf16(exp(s - m)) into the numerator and the unrounded p into the row sum; the numerator and the sum
    are rescaled by exp(m_old - m_new) when a later block raises the maximum; output bf16(o / l).
  * CUDA-core prefill: scores q.k * scale unrounded, 64-key blocks from (kv_start // 64) * 64, unrounded p; output in the
    engine's dtype.  (Its block structure only shows through the faults the CPU tests restate.)
  * tcgen05 ViT: fp32 scores, 192-key blocks, p = bf16(exp(s * scale - m)), fp32 sum, output bf16(o / l).
  * CUDA-core ViT: s = rnd(q.k) * scale (fp32 product), exact two-pass softmax, p = rnd(e / sum), output rnd(sum p v).
Key visibility: key j is visible to the query at column i of row r iff kv_start[r] <= j <= i (causal attention with LEFT
padding); a pad query (i < kv_start[r]) sees nothing and its output is exactly 0.  SigLIP attention is unmasked over the
NP patches of one image.

Tolerance |got - ref| <= tol (derived in tests/test_gpu_attn_prefill.py):
  tol = out_rel |ref| + (expm1(2 E) + 8 * 2^-24 (keys + 16)) * sum_k w_k (|v_k| + |ref|) + allowance
with w the normalized softmax weights, E the largest continuous error of one exp argument (fp32 scores that are not
rounded, the fp32 exp argument, exp2f / expf), and the allowance covering the keys whose rounding the kernel may resolve
the other way: a bf16 rounding of q.k (tcgen05 prefill, bf16 CUDA-core ViT) or of p whose fp64 value lies within the
derived error window of a rounding midpoint.  Such a key adds its worst-case weight change times |v - ref| (bounded by
|v| + |ref|), or, for a flip of p, which enters the numerator only, one bf16 ulp of p times |v| / l."""
import math
from typing import Optional, Sequence

import torch

HEAD_DIM = 128
PA_BK = 128                  # attn_prefill_tc.cuh: keys per block (and queries per tile)
CC_BK = 64                   # lm_kernels.cuh attn_prefill_kernel: keys per block (and queries per tile)
VT_BK = 192                  # vit_kernels.cuh: keys per block of vit_attn_tc_kernel
VA_MAX_NP = 32 * 32          # vit_attn_kernel: 32 * VA_MAXI keys in registers
U = 2.0 ** -24
EXP_REL = 2.0 ** -22         # exp2f / expf: 2 ulp
SENTINEL = 2.0 ** 100        # a large finite value for columns the kernels must not use

PREFILL_FAULTS = ("diag_exclusive", "kv_start_exclusive", "kb_lo_early", "kb_lo_late", "last_block_dropped",
                  "no_rescale", "scale_twice", "scale_omitted")
VIT_FAULTS = ("keys_past_np", "block191", "block193")


def bf(x: torch.Tensor) -> torch.Tensor:
    """fp32 value rounded to bf16 with RNE, kept as fp32 (an fp64 input is first rounded to fp32, as the kernels hold it)."""
    return x.float().to(torch.bfloat16).float()


def f32_scale(n: int) -> float:
    """1.0f / sqrtf((float)n), both correctly rounded in fp32."""
    return float(1.0 / torch.tensor(float(n), dtype=torch.float32).sqrt())


def _core(s, vis, blk, v, *, round_p: bool, out_rel: float, normalize_first: bool = False, rescale: bool = True,
          e_score=0.0, e_extra: float = 0.0, s_alts: Sequence[torch.Tensor] = ()):
    """Blocked online softmax in fp64.  s [B][Q][N] the kernel's scores in natural-log units (column n of key block
    blk[n]); vis [B or 1][Q][N]; v [B][N][D].  Returns ref [B][Q][D], tol and the mask of outputs with an allowance."""
    vis = vis.expand_as(s)
    z = torch.zeros((), dtype=s.dtype, device=s.device)
    sm = torch.where(vis, s, z - math.inf)
    idx = blk.view(1, 1, -1).expand_as(s)
    nb = int(blk.max()) + 1
    bm = torch.full(s.shape[:-1] + (nb,), -math.inf, dtype=s.dtype, device=s.device).scatter_reduce(-1, idx, sm, "amax")
    run = torch.cummax(bm, -1).values                      # running maximum after each block
    mk = run.gather(-1, idx)                               # ... at the block of each column
    mfin = run[..., -1:]
    p = torch.where(vis, torch.exp(torch.where(vis, s - mk, z)), z)
    fac = torch.where(vis, torch.exp(torch.where(vis, mk - mfin, z)), z) if rescale else vis.to(s.dtype)
    d = p * fac
    linv = torch.where(d.sum(-1, keepdim=True) > 0, 1.0 / d.sum(-1, keepdim=True), z)
    w = d * linv
    if normalize_first:                                    # p = rnd(e / sum), o = sum p v
        base, to_num = w, torch.ones_like(w)
    else:                                                  # o = sum rnd(p) v (rescaled), / l
        base, to_num = p, fac * linv
    num = (bf(base).double() if round_p else base) * to_num
    ref = num @ v
    av = v.abs()
    sv = w @ av + ref.abs()                                # sum_k w_k (|v_k| + |ref|)
    E = e_score + e_extra + EXP_REL + 1.5 * U * torch.where(vis, (s - mk).abs(), z)
    Eq = torch.where(vis, E, z).amax(-1, keepdim=True)
    n = vis.sum(-1, keepdim=True).to(s.dtype)
    tol = out_rel * ref.abs() + (torch.expm1(2 * Eq) + 8 * U * (n + 16) * (n > 0)) * sv
    allow = torch.zeros_like(ref)
    c = torch.zeros_like(Eq)                               # common-factor change of p when a normalizer may move
    if s_alts:
        t = torch.zeros_like(s)
        for sa in s_alts:
            dlt = torch.where(vis, sa - s, z)
            g = torch.expm1(dlt) * w
            t = torch.maximum(t, (g / (1 + g)).abs() + (2.0 ** -8 * w if round_p else z) * (dlt != 0))
            if round_p and normalize_first:                # the sum moves: every p = e / sum by the same factor
                c = torch.maximum(c, 1.01 * g.abs().amax(-1, keepdim=True))
            elif round_p:                                  # a block maximum may move: every p of the row is rescaled
                may_be_max = (dlt != 0) & (torch.maximum(sa, s) >= mk)
                c = torch.maximum(c, torch.where(may_be_max, dlt.abs(), z).amax(-1, keepdim=True))
        allow = allow + t @ av + t.sum(-1, keepdim=True) * ref.abs()
    if round_p:
        win = E + c
        b0 = bf(base).double()
        dp = torch.maximum((bf(base * torch.exp(win)).double() - b0).abs(), (bf(base * torch.exp(-win)).double() - b0).abs())
        allow = allow + torch.where(vis, dp * to_num, z) @ av
    return ref, tol + allow, allow > 0


def _flip_alts(x, delta, chain):
    """Scores the kernel may produce when its fp32 sum of q.k, within delta of the fp64 value x, rounds the other way."""
    return [chain(x - delta), chain(x + delta)]


# --------------------------------------------------------------------------------------------------------- prefill
def prefill(q: torch.Tensor, K: torch.Tensor, V: torch.Tensor, kv_start: Sequence[int], kernel: str, *,
            exact: bool = False, fault: Optional[str] = None, row_kv: Optional[Sequence[int]] = None, elems: int = 1 << 22):
    """q [R][P][H][128] (the padded block), K / V [R][H][Tmax][128], fp32 tensors holding the kernel's operand values.
    kernel: "tc" (attn_prefill_tc_kernel), "cc_bf16" / "cc_fp32" (attn_prefill_kernel<T>).  exact: every rounding off
    (plain fp64 causal softmax).  fault: one of PREFILL_FAULTS, restated; row_kv[r]: the row whose K / V row r reads (a
    packed token given to the neighbouring row).  Returns ref, tol [R][P][H][128] fp64 and the allowance mask."""
    R, P, H, _ = q.shape
    dev = q.device
    tc = kernel == "tc"
    BK = PA_BK if tc else CC_BK
    scale = f32_scale(HEAD_DIM)
    if fault == "scale_twice":
        scale_k = scale * scale
    elif fault == "scale_omitted":
        scale_k = 1.0
    else:
        scale_k = scale
    out_rel = 2.0 ** -23 if kernel == "cc_fp32" else 2.0 ** -8
    ref = torch.zeros(R, P, H, HEAD_DIM, dtype=torch.float64, device=dev)
    tol, allow = torch.zeros_like(ref), torch.zeros(ref.shape, dtype=torch.bool, device=dev)
    i = torch.arange(P, device=dev)[:, None]
    j = torch.arange(P, device=dev)[None, :]
    blk = torch.arange(P, device=dev) // BK
    hc = max(1, elems // (P * P))
    for r in range(R):
        st = int(kv_start[r])
        kr = int(row_kv[r]) if row_kv is not None else r
        lo = st
        if fault == "kb_lo_late":                          # the block holding kv_start skipped
            lo = (st // BK + 1) * BK
        elif fault == "kb_lo_early":                       # walk from one block early and mask against its first key
            lo = max(0, (st // BK - 1) * BK)
        elif fault == "kv_start_exclusive":
            lo = st + 1
        vis = (j >= lo) & ((j < i) if fault == "diag_exclusive" else (j <= i)) & (i >= st)
        if fault == "last_block_dropped":                  # the tile's last block is the query's own (tile = block)
            vis = vis & (j // BK != i // BK)
        for h0 in range(0, H, hc):
            h1 = min(H, h0 + hc)
            qh = q[r, :, h0:h1].permute(1, 0, 2).double()
            kh, vh = K[kr, h0:h1, :P].double(), V[kr, h0:h1, :P].double()
            x = qh @ kh.transpose(1, 2)
            ax = qh.abs() @ kh.abs().transpose(1, 2)
            kw = dict(out_rel=out_rel, rescale=fault != "no_rescale")
            if exact:
                o = _core(x * (1 / math.sqrt(HEAD_DIM)), vis[None], blk, vh, round_p=False, out_rel=0.0)
            elif tc:
                chain = lambda y: bf(bf(y) * scale_k).double()           # noqa: E731  fp32 product, two bf16 roundings
                o = _core(chain(x), vis[None], blk, vh, round_p=True, s_alts=_flip_alts(x, 20 * U * ax, chain), **kw)
            else:                                          # fp32 q * scale, 128 FMAs
                o = _core(x * scale_k, vis[None], blk, vh, round_p=False, e_score=130 * U * ax * scale_k, **kw)
            ref[r, :, h0:h1] = o[0].permute(1, 0, 2)
            tol[r, :, h0:h1] = o[1].permute(1, 0, 2)
            allow[r, :, h0:h1] = o[2].permute(1, 0, 2)
    return ref, tol, allow


def boundary_columns(st: int, P: int) -> list:
    """Columns where a prefill kernel goes wrong first: the first visible one, 127 / 128 / 255 / 256 around block edges,
    the first column of the last block, and P - 1.  Only those inside [st, P)."""
    cols = {st, st + 1, 63, 64, 127, 128, 255, 256, ((P - 1) // PA_BK) * PA_BK, P - 1}
    return sorted(c for c in cols if st <= c < P)


def vit_boundary_columns(NP: int) -> list:
    return sorted(c for c in {0, 191, 192, 383, 384, NP - 1} if 0 <= c < NP)


def undetected_drops(ref: torch.Tensor, tol: torch.Tensor, w_of, cols_of) -> list:
    """(row, head, column) of every planted column c whose removal leaves the output of query c within the tolerance: an
    error the comparison could not see.  Removing key c with weight w changes the output to (out - w v_c) / (1 - w).
    w_of(r, h, c) -> (w, v_c) in fp64; cols_of(r) -> columns; ref / tol [R][Q][H][D]."""
    missed = []
    for r in range(ref.shape[0]):
        for c in cols_of(r):
            for h in range(ref.shape[2]):
                w, vc = w_of(r, h, c)
                if w >= 1.0:                               # the only visible key: nothing would be left
                    continue
                out = ref[r, c, h]
                moved = (out - w * vc) / (1.0 - w)
                if not bool(((moved - out).abs() > tol[r, c, h]).any()):
                    missed.append((r, h, c))
    return missed


def prefill_weight(q, K, V, kv_start, r, h, c):
    """fp64 softmax weight of key c for the query at column c of row r, and v_c."""
    st = int(kv_start[r])
    qc = q[r, c, h].double()
    s = K[r, h, st:c + 1].double() @ qc / math.sqrt(HEAD_DIM)
    return float(torch.softmax(s, 0)[-1]), V[r, h, c].double()


# ------------------------------------------------------------------------------------------------------------ SigLIP
def _vit_columns(NP: int, rows_avail: int, tc: bool, fault: Optional[str], dev):
    """(key index within the image, block) of every column the kernel combines."""
    if not tc:
        key = torch.arange(NP, device=dev)
        return key, torch.zeros_like(key)
    if fault in ("block191", "block193"):                  # 192-key tiles at a stride of 191 / 193, masked by NP
        stride = int(fault[5:])
        keys, blks = [], []
        for kb in range(-(-NP // stride)):
            for t in range(VT_BK):
                if kb * stride + t < NP:
                    keys.append(kb * stride + t)
                    blks.append(kb)
        return torch.tensor(keys, device=dev), torch.tensor(blks, device=dev)
    n = -(-NP // VT_BK) * VT_BK if fault == "keys_past_np" else NP
    key = torch.arange(n, device=dev)
    return key, key // VT_BK


def vit(qkv: torch.Tensor, n: int, NP: int, W: int, heads: int, kernel: str, *, exact: bool = False,
        fault: Optional[str] = None):
    """qkv [rows][3W] fp32 holding the kernel's operand values; image i is rows [i*NP, (i+1)*NP).  kernel: "tc"
    (vit_attn_tc_kernel), "cc_bf16" / "cc_fp32" (vit_attn_kernel<T>).  fault: one of VIT_FAULTS ("keys_past_np" reads
    the rows after the image, zeros past the buffer, as TMA does).  Returns ref, tol [n*NP][heads][hd] and the mask."""
    hd = W // heads
    dev = qkv.device
    tc = kernel == "tc"
    scale = f32_scale(hd)
    rows = qkv.shape[0]
    key, blk = _vit_columns(NP, rows, tc, fault, dev)
    ref = torch.zeros(n * NP, heads, hd, dtype=torch.float64, device=dev)
    tol, allow = torch.zeros_like(ref), torch.zeros(ref.shape, dtype=torch.bool, device=dev)
    vis = torch.ones(1, NP, key.numel(), dtype=torch.bool, device=dev)
    for img in range(n):
        rk = img * NP + key
        kk = torch.zeros(key.numel(), 3 * W, dtype=qkv.dtype, device=dev)
        ok = rk < rows
        kk[ok] = qkv[rk[ok]]
        q = qkv[img * NP:(img + 1) * NP, :W].view(NP, heads, hd).permute(1, 0, 2).double()
        k = kk[:, W:2 * W].view(-1, heads, hd).permute(1, 0, 2).double()
        v = kk[:, 2 * W:].view(-1, heads, hd).permute(1, 0, 2).double()
        x = q @ k.transpose(1, 2)
        ax = q.abs() @ k.abs().transpose(1, 2)
        if exact:
            o = _core(x / math.sqrt(hd), vis, blk, v, round_p=False, out_rel=0.0)
        elif tc:
            s = x * scale
            m = s.amax(-1, keepdim=True).abs()
            o = _core(s, vis, blk, v, round_p=True, out_rel=2.0 ** -8, e_score=U * scale * (12 * ax + 4 * x.abs()) + 2 * U * m)
        elif kernel == "cc_bf16":
            chain = lambda y: (bf(y) * scale).double()                  # noqa: E731  rnd(q.k) * scale in fp32
            s = chain(x)
            o = _core(s, vis, blk, v, round_p=True, normalize_first=True, out_rel=2.0 ** -8, e_score=2 * U * s.abs(),
                      e_extra=(NP + 4) * U, s_alts=_flip_alts(x, (hd + 2) * U * ax, chain))
        else:
            s = x * scale
            o = _core(s, vis, blk, v, round_p=False, normalize_first=True, out_rel=2.0 ** -23,
                      e_score=(hd + 2) * U * ax * scale + 2 * U * s.abs(), e_extra=(NP + 4) * U)
        sl = slice(img * NP, (img + 1) * NP)
        ref[sl], tol[sl], allow[sl] = (t.permute(1, 0, 2) for t in o)
    return ref, tol, allow


def vit_weight(qkv, NP, W, heads, img, h, c):
    """fp64 softmax weight of key c for query c of image img, and v_c."""
    hd = W // heads
    rows = qkv[img * NP:(img + 1) * NP].double()
    qc = rows[c, h * hd:(h + 1) * hd]
    s = rows[:, W + h * hd:W + (h + 1) * hd] @ qc / math.sqrt(hd)
    return float(torch.softmax(s, 0)[c]), rows[c, 2 * W + h * hd:2 * W + (h + 1) * hd]


# ------------------------------------------------------------------------------------------------ planted keys
def plant_prefill(q, K, V, kv_start, mode, g, rnd):
    """In place: on every boundary column c of each row, a key aligned with the query at column c, its score half a nat
    above the best earlier key of that query; with all-equal scores (mode "equal") large values instead.  rnd rounds to
    the operand dtype."""
    R, P, H, D = q.shape
    for r in range(R):
        st = int(kv_start[r])
        for c in boundary_columns(st, P):
            if mode == "equal":
                V[r, :, c] = rnd(16.0 * torch.randn(H, D, generator=g)).to(V.device)
                continue
            qc = q[r, c].double()
            s = torch.einsum("hnd,hd->hn", K[r, :, st:c].double(), qc) / math.sqrt(D)
            t = (s.amax(-1) if c > st else torch.zeros(H, dtype=torch.float64, device=q.device)) + 0.5
            K[r, :, c] = rnd((qc * (t * math.sqrt(D) / (qc ** 2).sum(-1))[:, None]).float())


def plant_vit(qkv, n, NP, W, heads, mode, g, rnd):
    """In place, per image and head: on every boundary column c a key aligned with query c, its score half a nat above the
    best other key of that query (mode "equal": large values)."""
    hd = W // heads
    for img in range(n):
        rows = slice(img * NP, (img + 1) * NP)
        for c in vit_boundary_columns(NP):
            rc = img * NP + c
            for h in range(heads):
                qs, ks, vs = (slice(o + h * hd, o + (h + 1) * hd) for o in (0, W, 2 * W))
                if mode == "equal":
                    qkv[rc, vs] = rnd(16.0 * torch.randn(hd, generator=g)).to(qkv.device)
                    continue
                qc = qkv[rc, qs].double()
                s = qkv[rows, ks].double() @ qc / math.sqrt(hd)
                s[c] = -math.inf
                t = s.max() + 0.5
                qkv[rc, ks] = rnd((qc * (t * math.sqrt(hd) / (qc ** 2).sum())).float())
