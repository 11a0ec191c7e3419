"""Reference of one decode-attention launch (lm_kernels.cuh attn_decode_kernel, attn_v5.cuh attn_decode_v5_kernel), and a
host restatement of v5's work cut (attn_tma.cuh build_row_units / AttnCut).

q, k_new, v_new are restated op for op, so they are bit-identical to the kernel's: the split-K slabs are summed in fp32
left to right (the kernels' order), rounded to the engine's dtype with RNE, and rotated with `rope_pair`'s fp32 products
and roundings.  The attention itself is fp64: softmax(q . K^T / sqrt(128)) over the row's cached columns
[kv_start, pos) plus the new token, times V.  Columns below alias_P of a row with src_row[r] != r are read from the
source row (prefill de-duplication), as the kernel's producer reads them."""
import math
from typing import Optional, Sequence

import numpy as np
import torch

HEAD_DIM = 128
ROPE_BF16, ROPE_REL = 1, 2                       # the rope flags decode_layers passes (lm_kernels.cuh ROPE_REL)
AT_TILE, AT_NG, AT_MAX_SLOTS = 32, 4, 64         # attn_tma.cuh


def _rnd(x: torch.Tensor, bf16: bool) -> torch.Tensor:
    return x.to(torch.bfloat16).float() if bf16 else x


def rope_pair(x1, x2, c, s, bf16_trig: bool, bf16: bool):
    """lm_kernels.cuh rope_pair<T> on fp32 tensors: every product and sum is one correctly rounded fp32 op."""
    if bf16_trig:
        c, s = _rnd(c, bf16), _rnd(s, bf16)
        o1 = _rnd(_rnd(x1 * c, bf16) + _rnd(-x2 * s, bf16), bf16)
        o2 = _rnd(_rnd(x2 * c, bf16) + _rnd(x1 * s, bf16), bf16)
    else:
        o1 = _rnd(x1 * c + (-x2) * s, bf16)
        o2 = _rnd(x2 * c + x1 * s, bf16)
    return o1, o2


def qkv_new(part: torch.Tensor, H: int, cos: torch.Tensor, sin: torch.Tensor, pos: int, kv_start: Sequence[int],
            rope_flags: int, bf16: bool):
    """part fp32 [S][R][3*H*128] (CPU), cos / sin fp32 [Tmax][64] (weights.rope_tables).  Returns fp32 q, k_new, v_new
    [R][H][128] with exactly the kernel's values (q before the 1/sqrt(128) scale)."""
    S, R, _ = part.shape
    acc = part[0].clone()
    for k in range(1, S):                                      # fp32, left to right
        acc = acc + part[k]
    x = _rnd(acc, bf16).view(R, 3, H, HEAD_DIM)
    ks = torch.as_tensor(np.asarray(kv_start, dtype=np.int64))
    pr = (pos - ks).clamp(min=0) if rope_flags & ROPE_REL else torch.full((R,), pos, dtype=torch.int64)
    c, s = cos[pr][:, None, :], sin[pr][:, None, :]            # [R][1][64]
    bt = bool(rope_flags & ROPE_BF16)
    out = []
    for w in (0, 1):
        a, b = rope_pair(x[:, w, :, :64], x[:, w, :, 64:], c, s, bt, bf16)
        out.append(torch.cat([a, b], dim=-1))
    return out[0], out[1], x[:, 2].clone()


def effective_cache(cache: torch.Tensor, src_row: Optional[Sequence[int]], alias_P: int) -> torch.Tensor:
    """[R][H][T][128] as the kernel reads it: columns below alias_P of row r come from row src_row[r]."""
    if src_row is None or alias_P <= 0:
        return cache
    eff = cache.clone()
    src = torch.as_tensor(np.asarray(src_row, dtype=np.int64))
    eff[:, :, :alias_P] = cache[src][:, :, :alias_P]
    return eff


def attention(q, k_new, v_new, kcache, vcache, kv_start, pos, src_row=None, alias_P=0, drop=None):
    """fp64 attention of the new token of every (row, head).  kcache / vcache [R][H][Tmax][128] (any float dtype, CPU).
    drop: optional {(r, col)} of columns to leave out (col == pos is the new token) - the teeth checks.
    Returns out [R][H][128] fp64 and max|V| over each item's attended values [R][H]."""
    R, H = q.shape[0], q.shape[1]
    K = effective_cache(kcache, src_row, alias_P)
    V = effective_cache(vcache, src_row, alias_P)
    out = torch.zeros(R, H, HEAD_DIM, dtype=torch.float64)
    vmax = torch.zeros(R, H, dtype=torch.float64)
    for r in range(R):
        st = int(kv_start[r])
        keys = torch.cat([K[r, :, st:pos].double(), k_new[r, :, None].double()], dim=1)       # [H][n+1][128]
        vals = torch.cat([V[r, :, st:pos].double(), v_new[r, :, None].double()], dim=1)
        keep = torch.ones(keys.shape[1], dtype=torch.bool)
        for (rr, col) in (drop or ()):
            if rr == r:
                keep[col - st] = False
        keys, vals = keys[:, keep], vals[:, keep]
        sc = torch.einsum("hnd,hd->hn", keys, q[r].double()) / math.sqrt(HEAD_DIM)
        p = torch.softmax(sc, dim=-1)
        out[r] = torch.einsum("hn,hnd->hd", p, vals)
        vmax[r] = vals.abs().amax(dim=(1, 2)) if vals.shape[1] else 0.0
    return out, vmax


def tolerance(ref: torch.Tensor, vmax: torch.Tensor) -> torch.Tensor:
    """2^-8 |ref| + 1e-4 max|V of the item| (derived in tests/test_gpu_attn_decode.py)."""
    return 2.0 ** -8 * ref.abs() + 1e-4 * vmax[..., None]


# ---------------------------------------------------------------------------------------------- the work cut (v5)
def row_tiles(st: int, pos: int) -> int:
    return ((pos - 1) // AT_TILE - st // AT_TILE + 1) if pos > st else 0


def row_units(kv_start: Sequence[int], pos: int, fixed: bool = True) -> np.ndarray:
    """Exclusive prefix [R + 1] of units per row.  fixed=False restates the parent cut, in which a row without cached
    tokens had no unit."""
    st = np.asarray(kv_start, dtype=np.int64)
    u = np.where(pos > st, (pos - 1) // AT_TILE - st // AT_TILE + 1, 0)
    if fixed:
        u = np.maximum(u, 1)
    return np.concatenate([[0], np.cumsum(u)])


def max_contributors_bound(u: int, per: int, sub: int) -> int:
    """AttnCut::bound: the most slots an item of u units can meet under the cut (per, sub), over every alignment."""
    k = -(-per // sub)                                   # non-empty slots of a whole CTA
    g = per - (k - 1) * sub                              # its last slot's units (1 .. sub)
    w = u - 1                                            # slot starts strictly inside the item, periodic in per
    m, rem = divmod(w, per)
    inner = 0 if rem == 0 else min(k, 1 + (1 + (rem - 1 - g) // sub if rem - 1 >= g else 0))
    return 1 + k * m + inner


def cut(U: int, ctas: int, u_max: int, fixed: bool = True):
    """AttnCut::init: (per, sub).  fixed=False is the parent's even cut without the contributor bound."""
    per = max(1, (U + ctas - 1) // ctas)
    sub = (per + AT_NG - 1) // AT_NG
    if fixed and max_contributors_bound(u_max, per, sub) > AT_MAX_SLOTS:
        sub = max(sub, -(-(u_max - 1) // (AT_MAX_SLOTS - 1)))
        per = AT_NG * sub
    return per, sub


def contributors(kv_start: Sequence[int], H: int, pos: int, ctas: int, fixed: bool = True) -> np.ndarray:
    """Contributors (non-empty group slots intersecting the item's units) of every item, [R][H]; 0 for an item without
    units (the parent cut's empty rows)."""
    ru = row_units(kv_start, pos, fixed)
    R = len(kv_start)
    ur = np.diff(ru)
    U = int(ru[-1]) * H
    if U == 0:
        return np.zeros((R, H), dtype=np.int64)
    per, sub = cut(U, ctas, int(ur.max()), fixed)
    slots = np.arange(ctas * AT_NG)
    c, g = slots // AT_NG, slots % AT_NG
    cb = np.minimum(c * per, U)
    ce = np.minimum(cb + per, U)
    lo = np.minimum(cb + g * sub, ce)
    hi = np.minimum(lo + sub, ce)
    pref = np.concatenate([[0], np.cumsum(lo < hi)])
    item_lo = (ru[:-1, None] * H + np.arange(H)[None, :] * ur[:, None])
    item_hi = item_lo + ur[:, None]
    slot_of = lambda u: (u // per) * AT_NG + (u % per) // sub
    n = pref[slot_of(np.maximum(item_hi - 1, 0)) + 1] - pref[slot_of(item_lo)]
    return np.where(ur[:, None] > 0, n, 0)


def cut_params(kv_start: Sequence[int], H: int, pos: int, ctas: int, fixed: bool = True):
    ru = row_units(kv_start, pos, fixed)
    return cut(int(ru[-1]) * H, ctas, int(np.diff(ru).max()), fixed)


# ------------------------------------------------------------------------------------------------------ the teeth
def boundary_columns(st: int, pos: int, alias_P: int = 0) -> list:
    """Cached columns where a kernel goes wrong first: the row's first valid column, the edges of its first tile, the
    first column of its last tile, pos - 1, and alias_P - 1 / alias_P.  Only those inside [st, pos)."""
    t_end = (st // AT_TILE + 1) * AT_TILE
    cols = {st, t_end - 1, t_end, ((pos - 1) // AT_TILE) * AT_TILE, pos - 1}
    if alias_P > 0:
        cols |= {alias_P - 1, alias_P}
    return sorted(c for c in cols if st <= c < pos)


def undetected_drops(q, k_new, v_new, kcache, vcache, kv_start, pos, src_row=None, alias_P=0):
    """(row, head, column) of every boundary column (and the new token, column pos) whose removal leaves the reference
    within the test's tolerance for the whole item: an error the comparison could not see.  Removing token j changes
    the output to (out - p_j v_j) / (1 - p_j)."""
    K = effective_cache(kcache, src_row, alias_P)
    V = effective_cache(vcache, src_row, alias_P)
    missed = []
    for r in range(q.shape[0]):
        st = int(kv_start[r])
        keys = torch.cat([K[r, :, st:pos].double(), k_new[r, :, None].double()], dim=1)
        vals = torch.cat([V[r, :, st:pos].double(), v_new[r, :, None].double()], dim=1)
        p = torch.softmax(torch.einsum("hnd,hd->hn", keys, q[r].double()) / math.sqrt(HEAD_DIM), dim=-1)
        out = torch.einsum("hn,hnd->hd", p, vals)
        tol = tolerance(out, vals.abs().amax(dim=(1, 2)))
        for col in boundary_columns(st, pos, alias_P) + [pos]:
            j = col - st
            for h in range(q.shape[1]):
                if p[h, j] >= 1.0:                              # the only token: nothing would be left
                    continue
                moved = (out[h] - p[h, j] * vals[h, j]) / (1.0 - p[h, j])
                if not bool(((moved - out[h]).abs() > tol[h]).any()):
                    missed.append((r, h, col))
    return missed
