// Fused CFG combine -> /temperature -> softmax -> torch.multinomial(1)-compatible Philox sampling
// -> teacher-forcing override -> token duplication -> prepare_gen_img_embeds (table gather).
// Replaces plangen_base.py:580-604.  One CTA per image (cond row 2b, uncond row 2b+1).
//
// Bit-compatibility with torch.multinomial on a CUDA generator (see oracle/philox.py for the
// restated algorithm and its sources): next = argmax_v( p[v] / q[v] ),  q = -log(u),
// u = curand_uniform4(Philox4x32-10(seed, subsequence = thread idx, offset)) where element
// li = b*V + v of the (B,V) tensor is produced by thread idx = li % (grid*256), component
// (li / (grid*256)) % 4, loop iteration li / (4*grid*256), grid = min(SMs * (maxThreadsPerSM/256),
// ceil(B*V/256)) — i.e. the mapping depends on the SM count of the device, as in torch.
#pragma once
#include "common.cuh"

namespace pg {

struct PhiloxOut { uint32_t v[4]; };

PG_DEVINL PhiloxOut philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  PhiloxOut o; o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}

// q for element li, exactly as torch's exponential_ kernel computes it
PG_DEVINL float torch_exponential_at(uint64_t li, uint64_t stride, uint64_t seed, uint64_t offset) {
  uint64_t idx, slot;
  if ((li | stride) >> 32) { idx = li % stride; slot = li / stride; }
  else { const uint32_t l32 = (uint32_t)li, s32 = (uint32_t)stride; slot = l32 / s32; idx = l32 - (uint32_t)slot * s32; }   // 64-bit division is ~10x the cost
  const uint32_t comp = (uint32_t)(slot & 3);
  const uint64_t ctr = offset / 4 + (slot >> 2);
  const PhiloxOut r = philox4x32_10((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)idx, (uint32_t)(idx >> 32),
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
  const uint32_t x = comp == 0 ? r.v[0] : comp == 1 ? r.v[1] : comp == 2 ? r.v[2] : r.v[3];
  const float u = fmaf((float)x, 2.3283064365386963e-10f, 1.1641532182693481e-10f);   // curand_uniform: (0, 1]
  // transformation::exponential (CUDA branch): u >= 1 - eps/2 -> eps/2, else -log(u)
  const float lg = (u >= 1.0f - 5.9604644775390625e-08f) ? -5.9604644775390625e-08f : logf(u);
  return -lg;
}

// logits: fp32 split partials [S][2B][V] of gen_head's second Linear (+ bias added here), or, when
// bias == nullptr and S == 1, final logits handed in through the drop-in API.
__device__ unsigned long long* g_sample_dbg = nullptr;   // debug timeline (tools/sample_timeline.py); nullptr in production
#define SAMPLE_STAMP(k) do { if (g_sample_dbg && threadIdx.x == 0) g_sample_dbg[blockIdx.x * 16 + (k)] = global_timer_ns(); } while (0)

// ---------------------------------------------------------------------------------------------------
// A thread-block CLUSTER per image: 8 CTAs, each owning an eighth of the vocabulary (and of the embedding row).
// One CTA per image kept a single SM busy for ~40 us per decode step (16 Philox evaluations + logf + two IEEE
// divisions per thread, behind 16 dependent logit loads); the cluster spreads the arithmetic over 128 SMs and
// combines max / sum / arg-max / sum of squares through distributed shared memory in rank order (deterministic).
// The arg-max is order independent (value, then lowest index).
//
// top_k > 0 (north_star (4); the reference has none, so 0 = off is the default): only logits >= the k-th largest
// CFG logit of the image survive (`logits[logits < topk(logits, k).values[..., -1:]] = -inf`, ties at the threshold
// kept), the rest get probability 0; softmax and the Philox draw still run over the full (B, V) tensor, so the
// result equals torch.multinomial on the masked distribution with the same generator.  The threshold is found by
// a 4-pass radix select (8 bits per pass) over an order-preserving integer key, histograms summed across the
// cluster through distributed shared memory.
//
// top_p < 1 (HF TopPLogitsWarper after TopKLogitsWarper, min_tokens_to_keep = 1; 1 = off is the default): in the
// ascending order of (t, index), the longest prefix whose cumulative probability is <= thr = fp32(1 - top_p) leaves
// the distribution, except the largest element.  The boundary key is the same radix select weighted by probability
// mass p_v = e_v / sum (the softmax's own numbers) in 2^62 fixed point, so the result does not depend on the order of
// the shared-memory atomics.  The tie group at the boundary key all has the same p; its members leave in index order
// while mass_below + j * p <= thr.  The removed e_v are zeroed and the sum recomputed over the kept set.  Greedy
// sampling skips it (the arg-max is always kept).
constexpr int SAMPLE_CLUSTER = 8;
// order-preserving map float -> uint32 (larger value, larger key; -0 < +0 is harmless here)
PG_DEVINL uint32_t sample_order_key(float t) {
  const uint32_t u = __float_as_uint(t);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
PG_DEVINL float sample_key_value(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
#ifndef PG_SAMPLE_CL_THREADS
#define PG_SAMPLE_CL_THREADS 256
#endif
constexpr int SAMPLE_CL_THREADS = PG_SAMPLE_CL_THREADS;   // light CTAs: a cluster needs 8 co-scheduled SMs of one GPC
constexpr float SAMPLE_MASS_ONE = 4611686018427387904.f;  // 2^62: fixed-point scale of the top-p probability masses

struct SampleXchg {
  float mx, sum, bv, ss;
  int bi, ties;
};

PG_DEVINL void sample_hist_add(uint32_t* h, uint32_t w) { atomicAdd(h, w); }
// a 64-bit shared-memory atomicAdd is a compare-and-swap loop, slow under the contention of the first passes: add the
// two halves with native 32-bit atomics and carry into the high word (the histograms are read only after a barrier)
PG_DEVINL void sample_hist_add(unsigned long long* h, unsigned long long w) {
  uint32_t* h32 = reinterpret_cast<uint32_t*>(h);
  const uint32_t lo = (uint32_t)w, old = atomicAdd(h32, lo);
  atomicAdd(h32 + 1, (uint32_t)(w >> 32) + (old + lo < old ? 1u : 0u));
}

// Cluster-wide radix select: the largest 32-bit key K with W(key < K) <= thr, where W sums weight(i) over the image's
// elements (each CTA contributes i in [0, n) of its slice).  Count weights with thr = V - k give the k-th largest key;
// probability-mass weights give the top-p boundary.  thr is first clamped to W(all) - 1, so K is always a present key.
// Returns K, *below = W(key < K) and, if total != nullptr, *total = W(all).  hist: [4][256], one histogram per pass, read by the other CTAs through DSMEM (so
// no pass overwrites what a peer may still be reading).  Called by the whole CTA of every CTA of the cluster.
template <typename W, typename KeyF, typename WeightF>
PG_DEVINL uint32_t cluster_radix_select(W (*hist)[256], W* hsum, W* sel_w, uint32_t* sel_d, int n, KeyF key,
                                        WeightF weight, W thr, W* below_out, W* total = nullptr) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 4 * 256; i += SAMPLE_CL_THREADS) (&hist[0][0])[i] = 0;
  __syncthreads();
  uint32_t prefix = 0;
  W below = 0;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    const uint32_t himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
    for (int i = tid; i < n; i += SAMPLE_CL_THREADS) {
      const uint32_t k = key(i);
      if ((k & himask) == prefix) sample_hist_add(&hist[pass][(k >> shift) & 255u], weight(i));
    }
    cluster_sync_all();                                  // every CTA's histogram of this pass is complete
    for (int d = tid; d < 256; d += SAMPLE_CL_THREADS) {
      W c = 0;
#pragma unroll
      for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) {
        if constexpr (sizeof(W) == 8) c += dsmem_ld_u64(&hist[pass][d], r);
        else c += dsmem_ld_u32(&hist[pass][d], r);
      }
      hsum[d] = c;
    }
    __syncthreads();
    if (tid < 32) {
      // lane l owns digits 8l .. 8l+7; prefix weights from the lowest digit up
      W mine = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) mine += hsum[tid * 8 + j];
      W run = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const W t = __shfl_up_sync(0xffffffffu, run, o);
        if (tid >= o) run += t;
      }
      if (pass == 0) {
        const W all = __shfl_sync(0xffffffffu, run, 31);
        thr = min(thr, (W)(all - 1));
        if (total && tid == 0) *total = all;
      }
      W lo = below + (run - mine);                       // weight of the keys below this lane's first digit
      const uint32_t ok = __ballot_sync(0xffffffffu, lo <= thr);   // lane 0 always: below <= thr
      if (tid == 31 - __clz(ok)) {
        uint32_t d = (uint32_t)tid * 8;
        for (int j = 1; j < 8; ++j) {
          const W nx = lo + hsum[tid * 8 + j - 1];
          if (nx > thr) break;
          lo = nx; d = (uint32_t)(tid * 8 + j);
        }
        *sel_d = d; *sel_w = lo;
      }
    }
    __syncthreads();
    prefix |= *sel_d << shift;
    below = *sel_w;
    __syncthreads();
  }
  *below_out = below;
  return prefix;
}

template <typename T>
__global__ void __cluster_dims__(SAMPLE_CLUSTER, 1, 1) __launch_bounds__(SAMPLE_CL_THREADS)
cfg_sample_embed_cluster_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ bias,
                                int B, int V, float cfg_weight, float temperature, uint64_t seed, uint64_t offset_base,
                                uint64_t offset_per_step, uint64_t philox_stride, int greedy, int top_k,
                                float top_p_thr, const int32_t* __restrict__ edit_region, const int32_t* __restrict__ gt_labels,
                                int step_base, const int* __restrict__ step_ptr, int n_steps,
                                int32_t* __restrict__ tokens_out, const T* __restrict__ embed_table, int D,
                                float* __restrict__ x_next, const float* __restrict__ next_norm_w, T* __restrict__ xn_next,
                                float eps, int round_resid, float* __restrict__ dbg_logits) {
  extern __shared__ __align__(16) float sh[];   // this CTA's slice of the CFG logits -> unnormalised probabilities
  // top_p_thr >= 0 (top-p on): sh is followed by the slice's logits t and the mass histograms of its radix select
  __shared__ uint32_t hist[4][256];  // top-k radix select: one histogram per pass (read by the other CTAs)
  __shared__ uint32_t hsum[256];
  __shared__ uint32_t sel_d, sel_c;  // digit and count below of the current pass
  __shared__ unsigned long long sel_m, mass_all;
  __shared__ float red[32];
  __shared__ float bestv[32];
  __shared__ int besti[32];
  __shared__ SampleXchg xc;          // read by the other CTAs of the cluster
  pdl_launch_dependents();
  SAMPLE_STAMP(0);
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_ctarank();
  const int b = blockIdx.x / SAMPLE_CLUSTER;
  const int chunk = (V + SAMPLE_CLUSTER - 1) / SAMPLE_CLUSTER;
  const int v_lo = (int)rank * chunk, v_hi = min(V, v_lo + chunk);
  // The step counter is only written by the last kernel of a decode step; graph replays are fully ordered, and with plain
  // launches the host passes the step explicitly (step_ptr == nullptr), so reading it before the PDL wait is safe.
  const int step = step_base + (step_ptr ? *step_ptr : 0);
  const uint64_t offset = offset_base + offset_per_step * (uint64_t)(step - step_base);
  // The exponential variates of torch.multinomial depend on (seed, offset, element index) only - not on the logits: they
  // are drawn while the head contraction is still streaming its weights (this kernel is launched ahead of its dependency).
  constexpr int QPRE = 8;
  float qpre[QPRE];
  const bool pre = !greedy && (v_hi - v_lo) <= QPRE * SAMPLE_CL_THREADS;
  if (pre) {
#pragma unroll
    for (int j = 0; j < QPRE; ++j) {
      const int v = v_lo + tid + j * SAMPLE_CL_THREADS;
      qpre[j] = v < v_hi ? torch_exponential_at((uint64_t)b * V + v, philox_stride, seed, offset) : 1.f;
    }
  }
  float bias_r[QPRE];
  const bool bias_pre = bias != nullptr && (v_hi - v_lo) <= QPRE * SAMPLE_CL_THREADS;     // the bias is a weight: before the wait too
  if (bias_pre) {
#pragma unroll
    for (int j = 0; j < QPRE; ++j) {
      const int v = v_lo + tid + j * SAMPLE_CL_THREADS;
      bias_r[j] = v < v_hi ? bias[v] : 0.f;
    }
  }
  pdl_wait();
  SAMPLE_STAMP(1);
  const size_t rc = (size_t)(2 * b) * V, ru = (size_t)(2 * b + 1) * V;
  float mx = -INFINITY;
  for (int v0 = v_lo + tid, it = 0; v0 < v_hi; v0 += QPRE * SAMPLE_CL_THREADS, ++it) {
    float cs[QPRE], us[QPRE];
#pragma unroll
    for (int j = 0; j < QPRE; ++j) {         // all of a thread's loads in flight at once
      const int v = v0 + j * SAMPLE_CL_THREADS;
      cs[j] = us[j] = 0.f;
      if (v < v_hi) {
        if (S == 1) { cs[j] = __ldcg(part + rc + v); us[j] = __ldcg(part + ru + v); }
        else { cs[j] = reduce_splits(part, S, split_stride, rc + v); us[j] = reduce_splits(part, S, split_stride, ru + v); }
      }
    }
#pragma unroll
    for (int j = 0; j < QPRE; ++j) {
      const int v = v0 + j * SAMPLE_CL_THREADS;
      if (v < v_hi) {
        float c = cs[j], u = us[j];
        if (bias) { const float bb = (bias_pre && it == 0) ? bias_r[j] : bias[v]; c += bb; u += bb; }
        c = Act<T>::rnd(c); u = Act<T>::rnd(u);
        float t = Act<T>::rnd(__fsub_rn(c, u));           // plangen_base.py:587-588, one rounded op each
        t = Act<T>::rnd(__fmul_rn(cfg_weight, t));
        t = Act<T>::rnd(__fadd_rn(u, t));
        t = Act<T>::rnd(__fdiv_rn(t, temperature));
        sh[v - v_lo] = t;
        if (dbg_logits) dbg_logits[((size_t)step * B + b) * V + v] = t;
        mx = fmaxf(mx, t);
      }
    }
  }
  SAMPLE_STAMP(2);
  if (top_k > 0 && top_k < V) {
    // k-th largest CFG logit of the image = the largest key with at most V - k keys below it
    uint32_t below;
    const uint32_t kth = cluster_radix_select<uint32_t>(
        hist, hsum, &sel_c, &sel_d, v_hi - v_lo, [&](int i) { return sample_order_key(sh[i]); }, [](int) { return 1u; },
        (uint32_t)(V - top_k), &below);
    // everything below the k-th largest leaves the distribution
    mx = -INFINITY;
    for (int v = v_lo + tid; v < v_hi; v += SAMPLE_CL_THREADS) {
      float t = sh[v - v_lo];
      if (sample_order_key(t) < kth) { t = -INFINITY; sh[v - v_lo] = t; }
      mx = fmaxf(mx, t);
    }
  }
  mx = block_max(mx, red);
  if (tid == 0) xc.mx = mx;
  cluster_sync_all();
#pragma unroll
  for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) mx = fmaxf(mx, __uint_as_float(dsmem_ld_u32(&xc.mx, r)));
  const bool top_p = top_p_thr >= 0.f && !greedy;
  float* const tsh = sh + chunk;                            // top-p: the logits t, ordering key of the select
  float sum = 0.f;
  for (int v = v_lo + tid; v < v_hi; v += SAMPLE_CL_THREADS) {
    const float t = sh[v - v_lo];
    if (top_p) tsh[v - v_lo] = t;
    const float e = expf(t - mx);
    sh[v - v_lo] = e;
    sum += e;
  }
  SAMPLE_STAMP(3);
  sum = block_sum(sum, red);
  if (tid == 0) xc.sum = sum;
  cluster_sync_all();
  sum = 0.f;
#pragma unroll
  for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) sum += __uint_as_float(dsmem_ld_u32(&xc.sum, r));   // rank order
  if (top_p) {
    typedef unsigned long long u64;
    u64(*mhist)[256] = reinterpret_cast<u64(*)[256]>(sh + 2 * ((chunk + 1) & ~1));
    u64* mhsum = &mhist[4][0];
    const u64 thr = __float2ull_rn(top_p_thr * SAMPLE_MASS_ONE);
    u64 below;
    const uint32_t kb = cluster_radix_select<u64>(
        mhist, mhsum, &sel_m, &sel_d, v_hi - v_lo, [&](int i) { return sample_order_key(tsh[i]); },
        [&](int i) { return __float2ull_rn(__fdiv_rn(sh[i], sum) * SAMPLE_MASS_ONE); }, thr, &below, &mass_all);
    // the tie group at kb: members per CTA (ranks own ascending index ranges), then how many of them leave
    const u64 pk = __float2ull_rn(__fdiv_rn(expf(sample_key_value(kb) - mx), sum) * SAMPLE_MASS_ONE);
    int mine = 0;
    for (int v0 = v_lo; v0 < v_hi; v0 += SAMPLE_CL_THREADS) {
      const int v = v0 + tid;
      mine += __syncthreads_count(v < v_hi && sample_order_key(tsh[v - v_lo]) == kb);
    }
    if (tid == 0) xc.ties = mine;
    cluster_sync_all();
    int first = 0, ties = 0;                                 // group members in lower ranks, in the whole image
#pragma unroll
    for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) {
      const int c = (int)dsmem_ld_u32(&xc.ties, r);
      if (r < rank) first += c;
      ties += c;
    }
    // member j = 1, 2, ... (index order) leaves while below + j * pk <= thr; the group of the largest key keeps one
    u64 drop = pk ? (thr - below) / pk : (u64)ties;
    if (below + (u64)ties * pk == mass_all) drop = min(drop, (u64)(ties - 1));
    drop = min(drop, (u64)ties);
    // zero the removed e_v and sum the kept set as the softmax of the masked logits does (same per-thread order)
    __shared__ int wcnt[SAMPLE_CL_THREADS / 32];
    const int lane = tid & 31, warp = tid >> 5;
    int seen = first;                                        // group members before this iteration's elements
    float kept = 0.f;
    for (int v0 = v_lo; v0 < v_hi; v0 += SAMPLE_CL_THREADS) {
      const int v = v0 + tid;
      const uint32_t k = v < v_hi ? sample_order_key(tsh[v - v_lo]) : 0u;
      const bool tie = v < v_hi && k == kb;
      const uint32_t bal = __ballot_sync(0xffffffffu, tie);
      if (lane == 0) wcnt[warp] = __popc(bal);
      __syncthreads();
      int before = seen + __popc(bal & ((1u << lane) - 1u)), all = 0;
#pragma unroll
      for (int w = 0; w < SAMPLE_CL_THREADS / 32; ++w) {
        if (w < warp) before += wcnt[w];
        all += wcnt[w];
      }
      __syncthreads();
      seen += all;
      if (v < v_hi) {
        float e = sh[v - v_lo];
        if (k < kb || (tie && (u64)before < drop)) { e = 0.f; sh[v - v_lo] = e; }
        kept += e;
      }
    }
    kept = block_sum(kept, red);
    if (tid == 0) xc.sum = kept;
    cluster_sync_all();
    sum = 0.f;
#pragma unroll
    for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) sum += __uint_as_float(dsmem_ld_u32(&xc.sum, r));
  }
  // argmax over p/q (first index wins ties, like torch.argmax)
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  if (pre) {
#pragma unroll
    for (int j = 0; j < QPRE; ++j) {
      const int v = v_lo + tid + j * SAMPLE_CL_THREADS;
      if (v < v_hi) {
        const float score = __fdiv_rn(__fdiv_rn(sh[v - v_lo], sum), qpre[j]);
        if (score > bv || (score == bv && v < bi)) { bv = score; bi = v; }
      }
    }
  } else {
    for (int v = v_lo + tid; v < v_hi; v += SAMPLE_CL_THREADS) {
      const float p = __fdiv_rn(sh[v - v_lo], sum);
      float score = p;
      if (!greedy) {
        const float q = torch_exponential_at((uint64_t)b * V + v, philox_stride, seed, offset);
        score = __fdiv_rn(p, q);
      }
      if (score > bv || (score == bv && v < bi)) { bv = score; bi = v; }
    }
  }
  SAMPLE_STAMP(4);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  if ((tid & 31) == 0) { bestv[tid >> 5] = bv; besti[tid >> 5] = bi; }
  __syncthreads();
  if (tid < 32) {
    const bool have = tid < SAMPLE_CL_THREADS / 32;          // one entry per warp of this CTA
    bv = have ? bestv[tid] : -INFINITY; bi = have ? besti[tid] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if (tid == 0) { xc.bv = bv; xc.bi = bi; }
  }
  cluster_sync_all();
  bv = -INFINITY; bi = 0x7fffffff;
#pragma unroll
  for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) {
    const float ov = __uint_as_float(dsmem_ld_u32(&xc.bv, r));
    const int oi = (int)dsmem_ld_u32(&xc.bi, r);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  int tok = bi;
  // teacher forcing (plangen_base.py:593-598): outside the edit region keep the ground truth
  if (edit_region != nullptr && edit_region[(size_t)b * n_steps + step] == 0) tok = gt_labels[(size_t)b * n_steps + step];
  tok = min(max(tok, 0), V - 1);
  if (rank == 0 && tid == 0) tokens_out[(size_t)b * n_steps + step] = tok;
  SAMPLE_STAMP(5);
  if (x_next == nullptr) { cluster_sync_all(); return; }   // nobody may exit while its xc can still be read
  // next input = gen_aligner(gen_embed(tok)) duplicated to the cond and uncond rows (:602-604), plus
  // (optionally) the first decoder layer's input RMSNorm of those rows; each CTA handles an eighth of the row
  const T* erow = embed_table + (size_t)tok * D;
  const int dchunk = (D + SAMPLE_CLUSTER - 1) / SAMPLE_CLUSTER;
  const int d_lo = (int)rank * dchunk, d_hi = min(D, d_lo + dchunk);
  float ss = 0.f;
  for (int d = d_lo + tid; d < d_hi; d += SAMPLE_CL_THREADS) {
    const float v = Act<T>::ld(erow + d);
    x_next[(size_t)(2 * b) * D + d] = v;
    x_next[(size_t)(2 * b + 1) * D + d] = v;
    ss += v * v;
  }
  SAMPLE_STAMP(6);
  ss = block_sum(ss, red);
  if (tid == 0) xc.ss = ss;
  cluster_sync_all();
  if (xn_next != nullptr) {
    ss = 0.f;
#pragma unroll
    for (uint32_t r = 0; r < SAMPLE_CLUSTER; ++r) ss += __uint_as_float(dsmem_ld_u32(&xc.ss, r));
    const float rs = rsqrtf(ss / (float)D + eps);
    for (int d = d_lo + tid; d < d_hi; d += SAMPLE_CL_THREADS) {
      float hn = Act<T>::ld(erow + d) * rs;
      if (round_resid) hn = Act<T>::rnd(hn);
      const float y = next_norm_w[d] * hn;
      Act<T>::st(xn_next + (size_t)(2 * b) * D + d, y);
      Act<T>::st(xn_next + (size_t)(2 * b + 1) * D + d, y);
    }
  }
  cluster_sync_all();                                       // keep xc alive until every peer has read it
  SAMPLE_STAMP(7);
}

// prepare_gen_img_embeds through the precomputed table (modeling_vlm.py:270-271)
template <typename T>
__global__ void gen_embed_gather_kernel(const int32_t* __restrict__ ids, const T* __restrict__ table,
                                        float* __restrict__ out, int D, int V) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x;
  const int id = min(max(ids[i], 0), V - 1);
  for (int d = threadIdx.x; d < D; d += blockDim.x) out[(size_t)i * D + d] = Act<T>::ld(table + (size_t)id * D + d);
}

// first Linear of gen_aligner on the 8-wide codes: h[v][n] = gelu(rnd(sum_k rnd(E[v][k]) * W0[n][k] + b0[n]))
template <typename T>
__global__ void aligner_l0_kernel(const float* __restrict__ gen_embed, const T* __restrict__ w0,
                                  const float* __restrict__ b0, T* __restrict__ h, int code_dim, int D, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t v = i / D, n = i % D;
    float acc = 0.f;
    for (int k = 0; k < code_dim; ++k)
      acc = fmaf(Act<T>::rnd(gen_embed[v * code_dim + k]), Act<T>::ld(w0 + n * code_dim + k), acc);
    acc = Act<T>::rnd(acc + b0[n]);
    Act<T>::st(h + i, acc * 0.5f * (1.0f + erff(acc * 0.70710678118654752440f)));
  }
}

}  // namespace pg
