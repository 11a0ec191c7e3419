"""Reference of the tcgen05 contractions (gemm.cuh gemm_tc_kernel, gemm_tc2.cuh gemm_tc2_kernel, gemm_sk.cuh
gemm_swiglu_sk_kernel, the implicit 3x3 convolution) and their fused epilogues, plus host restatements of the tile-major
weight layout (tile_weight_kernel) and of the stream-K cut (skg_u0 / skg_owner).

Accumulators are fp64 (bf16 products are exact).  The epilogues are restated op for op in torch fp32 / bf16 with RNE at
the kernels' rounding points, applied either to the fp32 accumulators of the same kernel (bit-exact comparisons) or to
the fp64 ones (stream-K).  Where a kernel uses a documented approximation (erf_fast, ex2 / rcp silu, expf) the
restatement computes the exact value before the rounding and `interval` gives the bf16 values the kernel may produce."""
import math
from typing import Optional, Sequence

import numpy as np
import torch

from tests import attn_ref as A

TC_BM, TC_BK, TILE_BYTES = 128, 64, 128 * 64 * 2
SKG_MAX_FRAGS = 4
HEAD_DIM = 128
MID_REL = 2.0 ** -18                 # near-midpoint window of the approximated epilogues (see test_gpu_gemm_epi.py)
ERF_FAST_ABS = 4e-7                  # |erf_fast - erf|: A&S 7.1.26 (1.5e-7) plus its ex2 / rcp / fp32 roundings


def bf(x: torch.Tensor) -> torch.Tensor:
    """RNE to bf16, kept as fp32."""
    return x.float().to(torch.bfloat16).float()


# ------------------------------------------------------------------------------------------------------- accumulators
def acc64(X: torch.Tensor, W: torch.Tensor, drop_last_kb: bool = False) -> torch.Tensor:
    """X [M][K] . W [N][K]^T in fp64.  drop_last_kb: the same without the last 64-wide k-block (a fault the teeth use)."""
    X, W = X.double(), W.double()
    if drop_last_kb:
        k_end = ((X.shape[1] - 1) // TC_BK) * TC_BK
        X, W = X[:, :k_end], W[:, :k_end]
    return X @ W.T


def absacc64(X: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    return X.double().abs() @ W.double().abs().T


def conv_cols(act: torch.Tensor) -> torch.Tensor:
    """NHWC [B][H][W][Cin] -> [B*H*W][9*Cin], k = tap*Cin + cin with tap = 3*(dy+1) + (dx+1), zero padding 1 (the k order of
    run_conv_gemm's weight [Cout][9*Cin] and of its TMA boxes)."""
    B, H, W, Cin = act.shape
    p = torch.zeros(B, H + 2, W + 2, Cin, dtype=act.dtype)
    p[:, 1:H + 1, 1:W + 1] = act
    taps = [p[:, dy:dy + H, dx:dx + W] for dy in range(3) for dx in range(3)]
    return torch.stack(taps, dim=3).reshape(B * H * W, 9 * Cin)


def sum_bound(X: torch.Tensor, W: torch.Tensor) -> torch.Tensor:
    """Bound on |fp32 accumulator - fp64| for any of the contractions: one fp32 rounding (at most 1 ulp, whatever the
    tensor core's rounding mode) per 16-deep MMA step, plus 16 for the merges of accumulator blocks and stream-K partials,
    each at most 2^-24 of sum |x w|."""
    K = X.shape[1]
    return 2.0 * (K / 16 + 16) * 2.0 ** -24 * absacc64(X, W)


# ------------------------------------------------------------------------------------------ intervals of bf16 values
# Rounding is monotone: a kernel value within delta of v rounds to a bf16 value in [bf16(v - delta), bf16(v + delta)].
# Where delta is far below half an ulp (the body of every epilogue) that interval is one value, or the two neighbours
# of a rounding midpoint lying within delta of v: the one-ulp allowance.  In erf_fast's far negative tail, where its
# absolute error bound exceeds the bf16 spacing of GELU's tiny values, it is wider.
def interval(v: torch.Tensor, delta: torch.Tensor):
    """(lo, hi) bf16 values (as fp32) the rounding of any value within delta of v (fp64) can give."""
    v, delta = v.double(), delta.double()
    return bf((v - delta).float()), bf((v + delta).float())


def in_interval(got: torch.Tensor, lo: torch.Tensor, hi: torch.Tensor) -> torch.Tensor:
    g = got.float()
    return (g >= lo) & (g <= hi)


def _mul_interval(alo, ahi, blo, bhi):
    c = torch.stack([alo.double() * blo.double(), alo.double() * bhi.double(), ahi.double() * blo.double(), ahi.double() * bhi.double()])
    return c.amin(0), c.amax(0)


# -------------------------------------------------------------------------------------------------- row epilogues
def rows(acc32: torch.Tensor, bias: Optional[torch.Tensor] = None, add16: Optional[torch.Tensor] = None) -> torch.Tensor:
    """bf16(acc + bias), or bf16(bf16(acc + bias) + add16): exact (fp32 adds, RNE)."""
    b = bias.float() if bias is not None else torch.zeros(acc32.shape[1])
    t = bf(acc32.float() + b)
    if add16 is not None:
        t = bf(t + add16.float())
    return t


def gelu_rows(acc32: torch.Tensor, bias: Optional[torch.Tensor] = None):
    """bf16(gelu(bf16(acc + bias))) with the exact erf: the interval (lo, hi) the kernel's erf_fast may give."""
    b = bias.float() if bias is not None else torch.zeros(acc32.shape[1])
    t = bf(acc32.float() + b).double()
    v = t * 0.5 * (1.0 + torch.erf(t / math.sqrt(2.0)))
    return interval(v, MID_REL * v.abs() + 0.5 * t.abs() * ERF_FAST_ABS)


def gelu_tanh_rows(acc32: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The tanh approximation of GELU (a fault the teeth use)."""
    b = bias.float() if bias is not None else torch.zeros(acc32.shape[1])
    t = bf(acc32.float() + b).double()
    return bf(0.5 * t * (1 + torch.tanh(math.sqrt(2 / math.pi) * (t + 0.044715 * t ** 3))))


def resid(res: torch.Tensor, acc32: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """resid + bf16(acc + bias) in fp32."""
    b = bias.float() if bias is not None else torch.zeros(acc32.shape[1])
    return res.float() + bf(acc32.float() + b)


# ---------------------------------------------------------------------------------------------------------- SwiGLU
def pack_gate_up(g: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """Gate / up weights [F][D] packed as the engine packs them (plangen_b200/weights.py, bf16, F % 64 == 0)."""
    F, D = g.shape
    return torch.stack([g.reshape(F // 64, 64, D), u.reshape(F // 64, 64, D)], dim=1).reshape(2 * F, D)


def split_gate_up(acc: torch.Tensor):
    """[M][2F] accumulators of the packed weight -> gate [M][F], up [M][F]."""
    M, N = acc.shape
    a = acc.reshape(M, N // 128, 2, 64)
    return a[:, :, 0].reshape(M, N // 2), a[:, :, 1].reshape(M, N // 2)


SILU_ARGMIN, SILU_MIN = -1.2784645427610738, -0.2784645427610738


def _silu64(g: torch.Tensor) -> torch.Tensor:
    g = g.double()
    return g / (1.0 + torch.exp(-g))


def silu_delta(g: torch.Tensor, fast: bool) -> torch.Tensor:
    """How far the kernel's fp32 silu may be from the exact one: ex2.approx / rcp.approx (decode, stream-K), whose argument
    -g log2(e) is itself rounded, or expf + IEEE division (CTA pair)."""
    v = _silu64(g).abs()
    return (MID_REL + (g.double().abs() * 2.0 ** -22 if fast else 0.0)) * v


def swiglu_interval(glo, ghi, ulo, uhi, fast: bool):
    """h = bf16(bf16(silu(g)) * u), the product exact in fp32, for g in [glo, ghi] and u in [ulo, uhi] (bf16 values):
    the interval (lo, hi) of results."""
    s1, s2 = _silu64(glo), _silu64(ghi)
    smin, smax = torch.minimum(s1, s2), torch.maximum(s1, s2)
    inside = (glo.double() <= SILU_ARGMIN) & (ghi.double() >= SILU_ARGMIN)
    smin = torch.where(inside, torch.full_like(smin, SILU_MIN), smin)
    dg = torch.maximum(silu_delta(glo, fast), silu_delta(ghi, fast))
    sglo, sghi = bf((smin - dg).float()), bf((smax + dg).float())
    plo, phi = _mul_interval(sglo, sghi, ulo, uhi)
    return bf(plo.float()), bf(phi.float())


def swiglu(acc32: torch.Tensor, fast: bool):
    """SwiGLU epilogue on the kernel's own fp32 accumulators [M][2F] (packed rows): the interval (lo, hi)."""
    ga, ua = split_gate_up(acc32.float())
    g, u = bf(ga), bf(ua)
    return swiglu_interval(g, g, u, u, fast)


def swiglu64(a64: torch.Tensor, delta: torch.Tensor):
    """Stream-K / decode SwiGLU against the fp64 accumulators: g and u each anywhere their fp32 sums may round to (delta,
    the summation bound), silu as the kernels' ex2 / rcp form.  The interval (lo, hi)."""
    g64, u64 = split_gate_up(a64)
    dg, du = split_gate_up(delta)
    glo, ghi = interval(g64, dg)
    ulo, uhi = interval(u64, du)
    return swiglu_interval(glo, ghi, ulo, uhi, fast=True)


# ------------------------------------------------------------------------------------------------------------- QKV
def qkv_positions(M: int, R: int, P: int, row_off: Optional[Sequence[int]], kv_start: Sequence[int],
                  rope_start: Optional[Sequence[int]]):
    """(row, cache column, RoPE position) of every token of the QKV epilogue: packed stream (row_off) or padded [R][P]."""
    m = np.arange(M)
    if row_off is not None:
        ro = np.asarray(row_off, dtype=np.int64)
        rw = np.searchsorted(ro, m, side="right") - 1
        col = np.asarray(kv_start, dtype=np.int64)[rw] + (m - ro[rw])
    else:
        rw, col = m // P, m % P
    pr = np.maximum(col - np.asarray(rope_start, dtype=np.int64)[rw], 0) if rope_start is not None else col
    return rw, col, pr


def qkv(acc32: torch.Tensor, H: int, cos: torch.Tensor, sin: torch.Tensor, rw, col, pr, kcache: torch.Tensor,
        vcache: torch.Tensor):
    """q [M][H*128], and the caches [R][H][Tmax][128] after the epilogue's scatter (bf16 values as fp32)."""
    M = acc32.shape[0]
    x = bf(acc32.float()).view(M, 3, H, HEAD_DIM)
    pr_t = torch.as_tensor(pr, dtype=torch.int64)
    c, s = cos[pr_t][:, None, :], sin[pr_t][:, None, :]
    out = []
    for w in (0, 1):
        a, b = A.rope_pair(x[:, w, :, :64], x[:, w, :, 64:], c, s, False, True)
        out.append(torch.cat([a, b], dim=-1))
    kc, vc = kcache.clone().float(), vcache.clone().float()
    rw_t, col_t = torch.as_tensor(rw, dtype=torch.int64), torch.as_tensor(col, dtype=torch.int64)
    for h in range(H):
        kc[rw_t, h, col_t] = out[1][:, h]
        vc[rw_t, h, col_t] = x[:, 2, h]
    return out[0].reshape(M, H * HEAD_DIM), kc, vc


# ------------------------------------------------------------------------------------------------------ tile-major
def tile_major(W: torch.Tensor) -> np.ndarray:
    """tile_weight_kernel restated: tile (nt, kb) of 128 rows x 64 k is 16 KB, chunk c (8 bf16) of row r at
    r*128 + ((c ^ (r & 7)) * 16); rows >= N and k >= K are zero.  Returns uint8 [tiles * 16384]."""
    N, K = W.shape
    nt, nkb = -(-N // TC_BM), -(-K // TC_BK)
    Wp = np.zeros((nt * TC_BM, nkb * TC_BK), dtype=np.uint16)
    Wp[:N, :K] = W.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    src = Wp.reshape(nt, TC_BM, nkb, 8, 8).transpose(0, 2, 1, 3, 4)          # [nt][kb][r][c][8]
    out = np.empty_like(src)
    r = np.arange(TC_BM)
    for c in range(8):
        out[:, :, r, c ^ (r & 7)] = src[:, :, r, c]
    return out.reshape(-1).view(np.uint8)


def untile(buf: np.ndarray, N: int, K: int) -> np.ndarray:
    """Inverse of tile_major by direct addressing (one element at a time over the formula): uint16 [N][K]."""
    nkb = -(-K // TC_BK)
    b16 = buf.view(np.uint16)
    n = np.arange(N)[:, None]
    k = np.arange(K)[None, :]
    r, c, e = n % TC_BM, (k % TC_BK) // 8, k % 8
    tile = (n // TC_BM) * nkb + k // TC_BK
    off = tile * TILE_BYTES + r * 128 + (c ^ (r & 7)) * 16 + e * 2
    return b16[off // 2]


# ------------------------------------------------------------------------------------------------- the stream-K cut
def skg_u0(c: int, U: int, G: int) -> int:
    return (c * U) // G


def skg_owner(u: int, U: int, G: int) -> int:
    c = (u * G) // U
    while c + 1 < G and skg_u0(c + 1, U, G) <= u:
        c += 1
    while c > 0 and skg_u0(c, U, G) > u:
        c -= 1
    return c


def skg_grid(n_tiles: int, num_kb: int, ctas: int, num_sms: int) -> int:
    U = n_tiles * num_kb
    return min(ctas if ctas > 0 else num_sms, U)


def skg_max_contrib(n_tiles: int, num_kb: int, G: int) -> int:
    per_min = max(1, (n_tiles * num_kb) // G)
    return -(-num_kb // per_min) + 1


def skg_fragments(c: int, n_tiles: int, num_kb: int, G: int):
    """CTA c's fragments in processing order (reverse range order), uncapped: [(tile, kb_lo, kb_hi)]."""
    U = n_tiles * num_kb
    u0, u1 = skg_u0(c, U, G), skg_u0(c + 1, U, G)
    if u1 <= u0:
        return []
    out = []
    for t in range((u1 - 1) // num_kb, u0 // num_kb - 1, -1):
        lo, hi = t * num_kb, (t + 1) * num_kb
        out.append((t, max(u0, lo) - lo, min(u1, hi) - lo))
    return out


def skg_refused(n_tiles: int, num_kb: int, G: int) -> bool:
    """launch_swiglu_sk's host guard: some CTA's range touches more tiles than it keeps fragments."""
    return any(len(skg_fragments(c, n_tiles, num_kb, G)) > SKG_MAX_FRAGS for c in range(G))


def skg_contributors(n_tiles: int, num_kb: int, G: int) -> np.ndarray:
    """CTAs whose range meets each tile, [n_tiles]."""
    U = n_tiles * num_kb
    return np.array([skg_owner(t * num_kb + num_kb - 1, U, G) - skg_owner(t * num_kb, U, G) + 1 for t in range(n_tiles)])
