// KV-cache decode attention for the paired cond/uncond CFG batch, bf16 cache, one launch per layer: shared pieces
// (unit space, even cut over CTAs x groups, per-group TMA producer).  The kernel itself is attn_v5.cuh.
//
// Design (B200): the kernel is a persistent HBM streamer, one CTA per SM.  Work = "units" of 32 cached
// tokens of one (row, head) item.  The flat unit space [0, U) is cut into equal contiguous ranges, one per CTA,
// and every CTA range again into 4 contiguous sub-ranges, one per consumer GROUP (4 warps), so rows with long
// prompts (cond) and short prompts (uncond) are balanced exactly.  Each group is an independent stream:
//   * it owns private ring stages (K 8 KB + V 8 KB each) fed by its own producer warp with TMA bulk
//     copies (cp.async.bulk), in order;
//   * its 4 warps each take 8 of a tile's 32 tokens and keep their own fp32 online-softmax state (scores
//     by a transposed warp reduction, P.V with one row broadcast per token);
//   * item boundaries (RoPE'd q of the next item, merge of the 4 warps, hand-off to other contributors)
//     only synchronise the group's 128 threads - the other groups keep streaming.
// Because a stage always belongs to the same group, its warps observe every phase of the stage's
// mbarriers in order (TMA loads complete out of order; a consumer that skipped a phase would alias
// parities).  Cached tokens do not depend on the current step, so with PDL the rings are filled BEFORE
// griddepcontrol.wait (while the QKV contraction is still running); only q and the new k/v wait.
#pragma once
#include "common.cuh"
#include "lm_kernels.cuh"

namespace pg {

constexpr int AT_TILE = 32;                             // tokens per unit
constexpr int AT_TILE_BYTES = AT_TILE * HEAD_DIM * 2;   // 8 KB (K) and 8 KB (V)
constexpr int AT_NG = 4;                                // consumer groups per CTA
constexpr int AT_GW = 4;                                // warps per group
constexpr int AT_GT = AT_GW * 32;                       // threads per group
constexpr int AT_NW = AT_NG * AT_GW;
constexpr int AT_TW = AT_TILE / AT_GW;                  // tokens per warp per tile (8)
constexpr int AT_THREADS = 32 * (AT_NW + AT_NG);      // 16 consumer warps + one producer warp per group
constexpr int AT_MAX_ROWS = 256;
constexpr int AT_MAX_SLOTS = 64;                        // partial records per item
static_assert(AT_TW == 8, "the transposed reduction below is written for 8 tokens per warp");

PG_DEVINL void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}
// explicit shared-space 8-byte load (generic loads through a function-argument pointer are not proven to
// be shared memory by the compiler and take the slow generic path)
PG_DEVINL uint2 lds_v2(uint32_t saddr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
  return v;
}
PG_DEVINL void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
PG_DEVINL bool mbar_test_wait(uint64_t* bar, uint32_t parity) {       // non-blocking probe
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// debug timeline: stamp k of group g of this CTA (16 stamps per group); dbg == nullptr in production
PG_DEVINL void at_stamp(unsigned long long* dbg, int g, int k) {
  if (dbg) dbg[((size_t)blockIdx.x * AT_NG + g) * 16 + k] = global_timer_ns();
}

// tiles covering cached tokens [start, pos) on a 32-token grid
PG_DEVINL int row_tiles(int start, int pos) { return pos > start ? ((pos - 1) / AT_TILE - start / AT_TILE + 1) : 0; }

// exclusive prefix of units per row into row_units[0..R], and the largest row's unit count into *u_max (one warp).
// A row's units are its tiles; the token being decoded rides on the last one.  A row without cached tokens
// (kv_start == pos: an all-padding prompt) still gets one unit, which carries only the new token.
PG_DEVINL void build_row_units(int* row_units, const int32_t* kv_start, int R, int pos, int lane, int* row_start,
                                int* u_max) {
  int carry = 0, mx = 0;
  for (int r0 = 0; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    const int st = (r < R) ? kv_start[r] : 0;
    if (r < R) row_start[r] = st;
    int u = (r < R) ? max(row_tiles(st, pos), 1) : 0;
    mx = max(mx, u);
    int incl = u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (r < R) row_units[r] = carry + incl - u;
    carry += __shfl_sync(0xffffffffu, incl, 31);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) { row_units[R] = carry; *u_max = mx; }
}

// How the flat unit space is cut: CTA c gets [c*per, (c+1)*per), its group g gets [.. + g*sub, .. + (g+1)*sub)
// Invariant: no item gets more than AT_MAX_SLOTS contributors (non-empty group slots intersecting its units), because an
// item owns AT_MAX_SLOTS hand-off records.  The even cut keeps it unless few long items meet many CTAs: when bound() says
// an item of u_max units could meet more slots, sub is widened to at least ceil((u_max - 1) / (AT_MAX_SLOTS - 1)) and per
// to 4 * sub.  Every slot then holds sub units, so an item meets at most 1 + ceil((u - 1) / sub) <= AT_MAX_SLOTS slots,
// and per only grows, so the CTAs still cover U.  Elsewhere (every Janus shape) the cut is the even cut.
struct AttnCut {
  int U, per, sub;
  PG_DEVINL void init(int units, int ctas, int u_max) {
    U = units;
    per = max(1, (U + ctas - 1) / ctas);
    sub = (per + AT_NG - 1) / AT_NG;
    if (bound(u_max) > AT_MAX_SLOTS) {
      sub = max(sub, (u_max + AT_MAX_SLOTS - 3) / (AT_MAX_SLOTS - 1));
      per = AT_NG * sub;
    }
  }
  // the most slots an item of u >= 1 units can meet, over every alignment: 1 + the slot starts strictly inside it.  A
  // whole CTA has k non-empty slots, the last one of g <= sub units; starts repeat with period per.
  PG_DEVINL int bound(int u) const {
    const int k = (per + sub - 1) / sub, g = per - (k - 1) * sub;
    const int m = (u - 1) / per, rem = (u - 1) % per;
    const int inner = rem == 0 ? 0 : min(k, rem - 1 >= g ? 2 + (rem - 1 - g) / sub : 1);
    return 1 + k * m + inner;
  }
  PG_DEVINL void group_range(int c, int g, int& lo, int& hi) const {
    const int cb = min(c * per, U), ce = min(cb + per, U);
    lo = min(cb + g * sub, ce);
    hi = min(lo + sub, ce);
  }
  PG_DEVINL int slot_of(int u) const { return (u / per) * AT_NG + (u % per) / sub; }
  PG_DEVINL bool slot_nonempty(int slot) const {
    int lo, hi;
    group_range(slot / AT_NG, slot % AT_NG, lo, hi);
    return lo < hi;
  }
};

// Producer side of ONE group stream (one dedicated producer warp per group, lane 0): in-order TMA bulk
// copies of the group's K/V tiles into its private stages.  A single thread feeding all four groups
// (~1300 cycles of address arithmetic, barrier probe and two bulk-copy issues per tile) was the bottleneck
// of the kernel; four independent issuers are not.
// Only the VALID tokens of a tile are copied: the first tile of a row starts at the row's first real column (left
// padding is not a multiple of 32), the last one ends at the newest cached token.  The untouched token slots of the
// stage keep whatever an earlier tile left there (the kernel zero-fills its ring once at entry, so that is always a
// finite value); the consumer masks them.  Saves ~31 of the tokens read per (row, head): 8 of 146 MB per launch at configs[1].
// Shared prompts: when row r's prompt K / V are a copy of row src_row[r]'s (prefill de-duplication: PlanGen's unconditional
// rows all carry the same negative prompt) the prompt columns (< alias_P) are read from the SOURCE row's strips, so all
// copies ask for the same addresses and all but the first are served by L2 (kept there: pol_shared) instead of HBM.
template <int SPG>
PG_DEVINL void attn_produce_group(int gb, int ge, const int* row_units, int R, int H, int Tmax, int pos,
                                  const int32_t* __restrict__ kv_start, const bf16* __restrict__ kcache,
                                  const bf16* __restrict__ vcache, uint8_t* ring, int stage_stride_bytes,
                                  const int* stage_of, uint64_t* full_bar, uint64_t* empty_bar, int& kload,
                                  uint64_t pol, int r_hint = 0, const int32_t* __restrict__ src_row = nullptr, int alias_P = 0,
                                  uint64_t pol_shared = 0) {
  int r = r_hint;
  while (r + 1 < R && row_units[r + 1] * H <= gb) ++r;
  int ur = row_units[r + 1] - row_units[r];
  int local = gb - row_units[r] * H;
  int h = local / ur, k = local % ur;
  for (int u = gb; u < ge; ++u) {
    {
      const int s = stage_of[kload % SPG];
      mbar_wait(&empty_bar[s], (((uint32_t)(kload / SPG)) & 1u) ^ 1u, 11, kload);
      const int st = kv_start[r];
      const int t0k = (st / AT_TILE + k) * AT_TILE;
      const int a = k == 0 ? (st & (AT_TILE - 1)) : 0;                 // first valid token slot of the tile
      const int b = min(AT_TILE, pos - t0k);                           // one past the last cached token slot
      const uint32_t bytes = (uint32_t)max(b - a, 0) * (HEAD_DIM * 2);
      // a row without cached tokens copies nothing: its arrive with 0 bytes expected completes the stage's phase
      mbar_expect_tx(&full_bar[s], 2 * bytes);
      const size_t off = (((size_t)r * H + h) * Tmax + t0k + a) * HEAD_DIM;
      uint8_t* dst = ring + (size_t)s * stage_stride_bytes + (size_t)a * (HEAD_DIM * 2);
      const int rs = (src_row != nullptr && t0k + a < alias_P) ? src_row[r] : r;
      if (bytes == 0) {
        // no bulk copy of zero bytes
      } else if (rs != r) {
        // tokens [t0k + a, min(t0k + b, alias_P)) from the source row, the rest (generated tokens) from the row itself
        const int nb = min(b, alias_P - t0k) - a;
        const uint32_t sb = (uint32_t)nb * (HEAD_DIM * 2);
        const size_t soff = (((size_t)rs * H + h) * Tmax + t0k + a) * HEAD_DIM;
        bulk_load(dst, kcache + soff, sb, &full_bar[s], pol_shared);
        bulk_load(dst + AT_TILE_BYTES, vcache + soff, sb, &full_bar[s], pol_shared);
        if (sb < bytes) {
          bulk_load(dst + sb, kcache + off + (size_t)nb * HEAD_DIM, bytes - sb, &full_bar[s], pol);
          bulk_load(dst + AT_TILE_BYTES + sb, vcache + off + (size_t)nb * HEAD_DIM, bytes - sb, &full_bar[s], pol);
        }
      } else {
        bulk_load(dst, kcache + off, bytes, &full_bar[s], pol);
        bulk_load(dst + AT_TILE_BYTES, vcache + off, bytes, &full_bar[s], pol);
      }
      ++kload;
    }
    // advance (r, h, k) to the next unit without divisions
    if (++k == ur) {
      k = 0;
      if (++h == H) {
        h = 0;
        ++r;
        if (r < R) ur = row_units[r + 1] - row_units[r];
      }
    }
  }
}

}  // namespace pg
