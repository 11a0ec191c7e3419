// Decode attention: the group streams described in attn_tma.cuh with the item-boundary round trips taken off the
// stream.
//
// What the in-kernel timeline (tools/attn_timeline.py, %globaltimer stamps per group) showed for an earlier
// generation that merged hand-offs through threadfence + counter (round 1, removed):
// the kernel costs  t = ~15 us + bytes / 7.6 TB/s .  While the KV stream saturates the memory pipe (~20-28 MB
// of tile requests queued chip-wide) one L2 round trip takes 4-5 us instead of ~1 us, and every item boundary
// of a group paid several of them in sequence: the split-K QKV partials of the next item's q, then
// threadfence -> atomic -> last-arriver loads for the hand-off.  Groups whose range began with a lone
// new-token unit paid two boundaries before their first tile and finished last.
//
// Hence, on the consumer side:
//   * the token being decoded rides on the item's last tile (no unit of its own): no empty segments.  A row
//     without cached tokens has one unit that carries only the new token (build_row_units);
//   * the partials of the NEXT segment's q / k / v are loaded into registers before the current segment's
//     tile loop and only consumed at the boundary: the round trip overlaps the stream;
//   * hand-off without waiting: a contributor stores its record as 64-bit words {value, valid flag} (one
//     atomic store per word, no fence, no counter) and moves on.  The LAST contributor of an item (it meets
//     the item first in its range, and only ever waits for earlier groups) keeps its own record in
//     registers and, at the end of its stream, polls the other records word by word - data and flag arrive
//     in the same load - merges in rank order and clears the words for the next launch;
//   * 2 ring stages per group instead of 3: 19 MB in flight still covers bandwidth x latency and shortens
//     every queue; warp-parallel row lookup in the prologue.
// Results are deterministic (fixed merge order).
#pragma once
#include "attn_tma.cuh"

namespace pg {

#ifndef PG_A5_SPG
#define PG_A5_SPG 2
#endif
constexpr int A5_SPG = PG_A5_SPG;
constexpr int A5_STAGES = AT_NG * A5_SPG;
constexpr int A5_SMEM = A5_STAGES * 2 * AT_TILE_BYTES + 128;
constexpr int A5_REC = HEAD_DIM + 2;                       // (o[128], M, L) per contributor, one 64-bit word each

PG_DEVINL void a5_post(unsigned long long* p, float v) {   // {valid = 1, value} in one single-copy-atomic store
  const unsigned long long w = (1ull << 32) | (unsigned long long)__float_as_uint(v);
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
PG_DEVINL float a5_take(const unsigned long long* p, int tag) {      // spin until the word is valid (bounded)
  unsigned long long w, t0 = 0;
  for (;;) {
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
    if (w >> 32) break;
    if (t0 == 0) t0 = global_timer_ns();
    else if (global_timer_ns() - t0 > 4000000000ull) {
      printf("attn v5: hand-off word timeout (tag %d, cta %d, thread %d)\n", tag, (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
  return __uint_as_float((unsigned)w);
}
constexpr int A5_PF = 4;                                   // split-K slabs that can be prefetched in registers

struct A5Seg {
  int r, h, start, first_tile, n_tiles, owns_new, item_lo, item_hi;
};

// first row whose units reach past flat unit u (whole warp)
PG_DEVINL int a5_row_of(const int* row_units, int R, int H, int u, int lane) {
  int r = 0;
  for (int r0 = 0; r0 < R; r0 += 32) {
    const int rr = r0 + lane;
    const bool below = (rr + 1 < R) && (row_units[rr + 1] * H <= u);
    r += __popc(__ballot_sync(0xffffffffu, below));
  }
  return r;
}

PG_DEVINL A5Seg a5_next_segment(int& u, int& r, int ge, const int* row_units, int H, const int* row_start) {
  while (row_units[r + 1] * H <= u) ++r;
  const int ur = row_units[r + 1] - row_units[r];
  const int item_base = row_units[r] * H;
  A5Seg s;
  s.r = r;
  s.h = (u - item_base) / ur;
  s.item_lo = item_base + s.h * ur; s.item_hi = s.item_lo + ur;
  const int seg_hi = min(s.item_hi, ge);
  s.start = row_start[r];
  s.first_tile = u - s.item_lo;
  s.n_tiles = seg_hi - u;
  s.owns_new = (seg_hi == s.item_hi) ? 1 : 0;
  u = seg_hi;
  return s;
}

// The split-K slabs one thread needs for a segment: threads 0..63 the rotary pair (jj, jj + 64) of q,
// threads 64..127 the pair of k and the two values of v when the segment owns the new token.
struct A5Pref {
  float x[A5_PF][4];
};
PG_DEVINL void a5_issue(A5Pref& pf, const A5Seg& s, int tg, int H, const float* __restrict__ part, int S,
                        size_t split_stride) {
  const int HD = H * HEAD_DIM, jj = tg & 63;
  const float* row = part + (size_t)s.r * 3 * HD + s.h * HEAD_DIM + jj;
  const bool qthread = tg < 64, kv = !qthread && s.owns_new;
#pragma unroll
  for (int k = 0; k < A5_PF; ++k) {
    const float* p = row + (size_t)k * split_stride;
    const bool on = k < S;
    pf.x[k][0] = (on && qthread) ? __ldcg(p) : (on && kv) ? __ldcg(p + HD) : 0.f;
    pf.x[k][1] = (on && qthread) ? __ldcg(p + 64) : (on && kv) ? __ldcg(p + HD + 64) : 0.f;
    pf.x[k][2] = (on && kv) ? __ldcg(p + 2 * HD) : 0.f;
    pf.x[k][3] = (on && kv) ? __ldcg(p + 2 * HD + 64) : 0.f;
  }
}
// value v of the prefetched slabs, summed left to right; slabs beyond A5_PF are fetched now
PG_DEVINL float a5_sum(const A5Pref& pf, int v, int S, const float* p, size_t split_stride) {
  float a = pf.x[0][v];
#pragma unroll
  for (int k = 1; k < A5_PF; ++k) if (k < S) a += pf.x[k][v];
  for (int k = A5_PF; k < S; ++k) a += __ldcg(p + (size_t)k * split_stride);
  return a;
}

struct A5GroupSmem {
  float q[HEAD_DIM], k[HEAD_DIM], v[HEAD_DIM];
  float m[AT_GW], l[AT_GW], o[AT_GW][HEAD_DIM];
};

// One consumer group's whole stream: units [gb, ge).  All 128 threads of the group call this.
template <int SPG>
PG_DEVINL void a5_group_stream(int tg, int gb, int ge, int r0, const AttnCut& cut, const int* row_units,
                               const int* row_start, int H, int Tmax, int pos, const float* __restrict__ part, int S,
                               size_t split_stride, const float* __restrict__ cosT, const float* __restrict__ sinT,
                               bf16* __restrict__ kcache, bf16* __restrict__ vcache, bf16* __restrict__ out,
                               unsigned long long* __restrict__ ws_ll, float scale, int trig_flags,
                               uint8_t* ring, int stage_stride_bytes, const int* stage_of, uint64_t* full_bar,
                               uint64_t* empty_bar, A5GroupSmem& sm, int my_slot, int bar_id, int dbg_skip_math,
                               unsigned long long* dbg) {
  if (gb >= ge) return;
  const int lane = tg & 31, wig = tg >> 5, jj = tg & 63;
  const int HD = H * HEAD_DIM;
  const float LOG2E = 1.4426950408889634f;
  const uint32_t ring_s = smem_u32(ring);
  const bool bf16_trig = (trig_flags & 1) != 0, rope_rel = (trig_flags & ROPE_REL) != 0;
  float c = cosT[pos * 64 + jj], sn = sinT[pos * 64 + jj];
  int u = gb, r = r0, kc = 0;
  A5Seg cur = a5_next_segment(u, r, ge, row_units, H, row_start);
  A5Pref pf;
  a5_issue(pf, cur, tg, H, part, S, split_stride);
  // record kept for the end of the stream when this group is the last contributor of its first item
  float dfM = 0.f, dfL = 0.f, dfacc = 0.f;
  int df_it = -1, df_n = 0;
  for (bool first = true;; first = false) {
    // ---- q (all), k/v of the new token (owner) from the prefetched partials
    {
      const float* p = part + (size_t)cur.r * 3 * HD + cur.h * HEAD_DIM + jj;
      if (rope_rel) {                       // text decode: position relative to the row's first valid column
        const int pr = max(pos - cur.start, 0);
        c = cosT[pr * 64 + jj]; sn = sinT[pr * 64 + jj];
      }
      if (tg < 64) {
        const float x1 = bf16_round(a5_sum(pf, 0, S, p, split_stride));
        const float x2 = bf16_round(a5_sum(pf, 1, S, p + 64, split_stride));
        float a, b;
        rope_pair<bf16>(x1, x2, c, sn, bf16_trig, a, b);
        sm.q[jj] = a * (scale * LOG2E); sm.q[jj + 64] = b * (scale * LOG2E);
      } else if (cur.owns_new) {
        const float x1 = bf16_round(a5_sum(pf, 0, S, p + HD, split_stride));
        const float x2 = bf16_round(a5_sum(pf, 1, S, p + HD + 64, split_stride));
        const float v1 = bf16_round(a5_sum(pf, 2, S, p + 2 * HD, split_stride));
        const float v2 = bf16_round(a5_sum(pf, 3, S, p + 2 * HD + 64, split_stride));
        float a, b;
        rope_pair<bf16>(x1, x2, c, sn, bf16_trig, a, b);
        sm.k[jj] = a; sm.k[jj + 64] = b; sm.v[jj] = v1; sm.v[jj + 64] = v2;
        const size_t cidx = (((size_t)cur.r * H + cur.h) * Tmax + pos) * HEAD_DIM + jj;
        kcache[cidx] = __float2bfloat16_rn(a); kcache[cidx + 64] = __float2bfloat16_rn(b);
        vcache[cidx] = __float2bfloat16_rn(v1); vcache[cidx + 64] = __float2bfloat16_rn(v2);
      }
    }
    // ---- the next segment's partials go into the pipe now and are used after this segment's tiles
    const bool has_next = u < ge;
    A5Seg nxt = cur;
    if (has_next) {
      nxt = a5_next_segment(u, r, ge, row_units, H, row_start);
      a5_issue(pf, nxt, tg, H, part, S, split_stride);
    }
    named_bar_sync(bar_id, AT_GT);
    if (tg == 0 && first) at_stamp(dbg, bar_id - 1, 2);
    float qv[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) qv[i] = sm.q[lane * 4 + i];
    float m = -INFINITY, l = 0.f, o[4] = {0.f, 0.f, 0.f, 0.f};
    const int start = cur.start;
    for (int t = 0; t < cur.n_tiles; ++t, ++kc) {
      const int s = stage_of[kc % SPG];
      mbar_wait(&full_bar[s], (uint32_t)(kc / SPG) & 1u, 12, kc);
      if (tg == 0 && kc == 0) at_stamp(dbg, bar_id - 1, 3);
      if (dbg_skip_math) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
        continue;
      }
      const uint32_t kt = ring_s + (uint32_t)(s * stage_stride_bytes + wig * AT_TW * (HEAD_DIM * 2) + lane * 8);
      const uint32_t vt = kt + AT_TILE_BYTES;
      const int t0 = (start / AT_TILE + cur.first_tile + t) * AT_TILE + wig * AT_TW;
      float sc[AT_TW];
#pragma unroll
      for (int i = 0; i < AT_TW; ++i) {
        const uint2 kk = lds_v2(kt + i * (HEAD_DIM * 2));
        float d = bf16lo(kk.x) * qv[0];
        d = fmaf(bf16hi(kk.x), qv[1], d); d = fmaf(bf16lo(kk.y), qv[2], d); d = fmaf(bf16hi(kk.y), qv[3], d);
        sc[i] = d;
      }
      // transposed reduction over lane bits 4,3,2 (8 -> 1 value per lane), then butterflies over bits 1,0:
      // afterwards every lane holds the full dot product of token (lane >> 2)
#pragma unroll
      for (int off = 16, n = AT_TW; off >= 4; off >>= 1, n >>= 1) {
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n / 2; ++i) {
          const float send = upper ? sc[i] : sc[i + n / 2];
          const float recv = __shfl_xor_sync(0xffffffffu, send, off);
          sc[i] = (upper ? sc[i + n / 2] : sc[i]) + recv;
        }
      }
      sc[0] += __shfl_xor_sync(0xffffffffu, sc[0], 2);
      sc[0] += __shfl_xor_sync(0xffffffffu, sc[0], 1);
      const int tok = t0 + (lane >> 2);
      const bool valid = (tok >= start) && (tok < pos);
      const float sv = valid ? sc[0] : -INFINITY;
      const float mx = fmaxf(m, warp_max(sv));
      const float p = valid ? exp2f(sv - mx) : 0.f;
      const float corr = (mx == -INFINITY) ? 1.f : exp2f(m - mx);
      l = l * corr + 0.25f * warp_sum(p);                                 // every token's p sits on 4 lanes
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] *= corr;
#pragma unroll
      for (int i = 0; i < AT_TW; ++i) {
        const float pi = __shfl_sync(0xffffffffu, p, i * 4);
        const uint2 vv = lds_v2(vt + i * (HEAD_DIM * 2));
        o[0] = fmaf(pi, bf16lo(vv.x), o[0]); o[1] = fmaf(pi, bf16hi(vv.x), o[1]);
        o[2] = fmaf(pi, bf16lo(vv.y), o[2]); o[3] = fmaf(pi, bf16hi(vv.y), o[3]);
      }
      m = mx;
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty_bar[s]);                          // AT_GW arrivals free the stage
    }
    if (tg == 0 && !has_next) at_stamp(dbg, bar_id - 1, 4);
    // ---- the token being decoded (owner, warp 0 of the group), straight from shared memory
    if (cur.owns_new && wig == 0) {
      float d = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) d = fmaf(sm.k[lane * 4 + i], qv[i], d);
      d = warp_sum(d);
      const float mx = fmaxf(m, d);
      const float corr = (m == -INFINITY) ? 0.f : exp2f(m - mx);
      const float p = exp2f(d - mx);
      l = l * corr + p;
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = fmaf(p, sm.v[lane * 4 + i], o[i] * corr);
      m = mx;
    }
    // ---- merge the 4 warps of the group
    if (lane == 0) { sm.m[wig] = m; sm.l[wig] = l; }
#pragma unroll
    for (int i = 0; i < 4; ++i) sm.o[wig][lane * 4 + i] = o[i];
    named_bar_sync(bar_id, AT_GT);
    float M = -INFINITY, Ltot = 0.f, acc = 0.f;
#pragma unroll
    for (int w = 0; w < AT_GW; ++w) M = fmaxf(M, sm.m[w]);
#pragma unroll
    for (int w = 0; w < AT_GW; ++w) {
      const float f = (sm.m[w] == -INFINITY) ? 0.f : exp2f(sm.m[w] - M);
      Ltot += sm.l[w] * f;
      acc += sm.o[w][tg] * f;                                             // tg < 128: one output dim each
    }
    // contributors of this item = non-empty group slots intersecting [item_lo, item_hi)
    const int s_first = cut.slot_of(cur.item_lo), s_last = cut.slot_of(cur.item_hi - 1);
    int n_contrib = 0, my_rank = 0;
    for (int sl = s_first; sl <= s_last; ++sl) {
      if (cut.slot_nonempty(sl)) {
        if (sl < my_slot) ++my_rank;
        ++n_contrib;
      }
    }
    const int it = cur.r * H + cur.h;
    if (n_contrib == 1) {
      out[(size_t)it * HEAD_DIM + tg] = __float2bfloat16_rn(acc / Ltot);
    } else if (my_rank == n_contrib - 1) {
      dfM = M; dfL = Ltot; dfacc = acc; df_it = it; df_n = n_contrib;     // only possible for the first segment
    } else {
      unsigned long long* wp = ws_ll + ((size_t)it * AT_MAX_SLOTS + my_rank) * A5_REC;
      a5_post(wp + tg, acc);
      if (tg == 0) { a5_post(wp + HEAD_DIM, M); a5_post(wp + HEAD_DIM + 1, Ltot); }
    }
    named_bar_sync(bar_id, AT_GT);                                        // sm.* free for the next segment
    if (!has_next) break;
    cur = nxt;
  }
  // ---- deferred merge: take the records of ranks 0 .. n-2 as they become valid, combine in rank order
  //      (own record last), clear the words for the next launch.  With few rows an item is cut over many
  //      groups (n <= AT_MAX_SLOTS by the AttnCut invariant, so n-1 <= 63 and 2(n-1) < AT_GT): the (M, L) words are
  //      fetched by 2(n-1) threads at once into shared memory and the output words eight records at a time, instead
  //      of one dependent round trip per record.
  if (df_it >= 0) {
    const int n_other = df_n - 1;
    unsigned long long* wb = ws_ll + (size_t)df_it * AT_MAX_SLOTS * A5_REC;
    float* ml = sm.o[0];                                                  // [n_other][2], free since the last barrier
    if (tg < 2 * n_other) {
      unsigned long long* w = wb + (size_t)(tg >> 1) * A5_REC + HEAD_DIM + (tg & 1);
      ml[tg] = a5_take(w, 1);
      *w = 0ull;
    }
    named_bar_sync(bar_id, AT_GT);
    float Mg = dfM;
    for (int s2 = 0; s2 < n_other; ++s2) Mg = fmaxf(Mg, ml[2 * s2]);
    float Lg = 0.f, og = 0.f;
    for (int s0 = 0; s0 < n_other; s0 += 8) {
      unsigned long long w[8];
      bool ok;
      unsigned long long t0 = 0;
      do {                                                                // eight loads in flight, retried until all valid
        ok = true;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          w[k] = 1ull << 32;
          if (s0 + k < n_other)
            asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w[k]) : "l"(wb + (size_t)(s0 + k) * A5_REC + tg) : "memory");
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) ok = ok && (w[k] >> 32) != 0;
        if (!ok) {
          if (t0 == 0) t0 = global_timer_ns();
          else if (global_timer_ns() - t0 > 4000000000ull) {
            printf("attn v5: hand-off record timeout (item %d, cta %d, thread %d)\n", df_it, (int)blockIdx.x, (int)threadIdx.x);
            __trap();
          }
        }
      } while (!ok);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (s0 + k < n_other) {
          const float ms = ml[2 * (s0 + k)];
          const float f = (ms == -INFINITY) ? 0.f : exp2f(ms - Mg);
          Lg += ml[2 * (s0 + k) + 1] * f;
          og += __uint_as_float((unsigned)w[k]) * f;
          wb[(size_t)(s0 + k) * A5_REC + tg] = 0ull;
        }
      }
    }
    const float f = (dfM == -INFINITY) ? 0.f : exp2f(dfM - Mg);
    Lg += dfL * f;
    og += dfacc * f;
    out[(size_t)df_it * HEAD_DIM + tg] = __float2bfloat16_rn(og / Lg);
  }
}

__global__ void __launch_bounds__(AT_THREADS, 1)
attn_decode_v5_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ cosT,
                      const float* __restrict__ sinT, bf16* __restrict__ kcache, bf16* __restrict__ vcache,
                      const int32_t* __restrict__ kv_start, bf16* __restrict__ out, float* __restrict__ ws_ll_f,
                      int R, int H, int Tmax, int pos_base,
                      const int* __restrict__ step_ptr, float scale, int bf16_trig, int early_trigger, Prof prof,
                      unsigned long long* dbg, const int32_t* __restrict__ src_row, int alias_P) {
  extern __shared__ uint8_t smem_raw[];
  unsigned long long* ws_ll = reinterpret_cast<unsigned long long*>(ws_ll_f);   // zero-initialised {flag, value} words
  uint8_t* ring = (uint8_t*)(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  __shared__ uint64_t full_bar[A5_STAGES], empty_bar[A5_STAGES];
  __shared__ int row_units[AT_MAX_ROWS + 1], row_start[AT_MAX_ROWS], u_max;
  __shared__ A5GroupSmem gsm[AT_NG];
  __shared__ int stage_tab[AT_NG * A5_SPG];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < AT_NG) at_stamp(dbg, tid, 0);
  if (early_trigger & 1) pdl_launch_dependents();
  prof_begin(prof);
  // The step counter is only written by the last kernel of a decode step; graph replays are fully ordered, and
  // with plain launches the host passes the position explicitly (step_ptr == nullptr), so reading it before the
  // PDL wait is safe.
  const int pos = pos_base + (step_ptr ? *step_ptr : 0);

  if (tid == 0) {
    for (int i = 0; i < A5_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], AT_GW); }
    mbar_fence_init();
  }
  if (tid < A5_STAGES) stage_tab[(tid % AT_NG) * A5_SPG + tid / AT_NG] = tid;   // group g owns stages g, g+4, ..
  // the producers copy only the valid tokens of a tile (attn_produce_group): every slot must hold a finite value before
  // the first copy lands, because a masked slot still enters o += 0 * v
  for (int i = tid; i < A5_STAGES * 2 * AT_TILE_BYTES / 16; i += AT_THREADS)
    asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(smem_u32(ring) + (uint32_t)i * 16u), "r"(0u) : "memory");
  fence_proxy_async();
  if (warp == 0) build_row_units(row_units, kv_start, R, pos, lane, row_start, &u_max);
  __syncthreads();
  if (tid < AT_NG) at_stamp(dbg, tid, 1);
  AttnCut cut;
  cut.init(row_units[R] * H, (int)gridDim.x, u_max);
  const int c = blockIdx.x;
  const int g = (warp >= AT_NW) ? warp - AT_NW : warp / AT_GW;
  int gb, ge;
  cut.group_range(c, g, gb, ge);
  const int r0 = a5_row_of(row_units, R, H, gb, lane);

  if (warp >= AT_NW) {
    // ============================== producers: one warp (lane 0) per group stream ==============================
    if (lane == 0) {
      int kload = 0;
      attn_produce_group<A5_SPG>(gb, ge, row_units, R, H, Tmax, pos, row_start, kcache, vcache, ring, 2 * AT_TILE_BYTES,
                                 stage_tab + g * A5_SPG, full_bar, empty_bar, kload, policy_evict_first(), r0, src_row, alias_P,
                                 policy_evict_last());
      at_stamp(dbg, g, 7);
    }
    pdl_wait();
    return;
  }
  // ============================== consumers: 4 independent groups ==============================
  pdl_wait();                                             // QKV partials of this step are now visible
  const int tg = tid - g * AT_GT;
  a5_group_stream<A5_SPG>(tg, gb, ge, r0, cut, row_units, row_start, H, Tmax, pos, part, S, split_stride, cosT, sinT,
                          kcache, vcache, out, ws_ll, scale, bf16_trig, ring, 2 * AT_TILE_BYTES,
                          stage_tab + g * A5_SPG, full_bar, empty_bar, gsm[g], c * AT_NG + g, 1 + g, early_trigger & 2, dbg);
  if (tg == 0) at_stamp(dbg, g, 5);
  prof_end(prof);
}

}  // namespace pg
