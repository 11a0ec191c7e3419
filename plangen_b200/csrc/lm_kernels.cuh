// Row-wise kernels around the LM contractions: embedding gather, residual + RMSNorm, RoPE +
// KV-cache append, SwiGLU, bias + GELU, prefill attention and KV-cache decode attention.
// All of them consume the fp32 split-K partials written by gemm.cuh, reduce the splits in a fixed
// order, and reproduce the rounding points of the reference's regime (fp32 master weights under
// torch.autocast(bf16), plangen_base.py:360) when T = bf16; T = float is the fp32 check mode.
//
// Every kernel calls pdl_wait() before touching data produced by the previous kernel and
// pdl_launch_dependents() at its top, so a chain of them can be launched with programmatic
// dependent launch (the next GEMM prefetches its weight tiles while these run).
#pragma once
#include "common.cuh"

namespace pg {

constexpr int HEAD_DIM = 128;

// flags for resid_rmsnorm_kernel
constexpr int RN_ROUND_RESID = 1;   // keep the residual stream bf16-rounded (decode steps in the autocast regime:
                                    // inputs_embeds there is the bf16 output of gen_aligner, so HF's residual adds are bf16)
constexpr int RN_INC_STEP = 2;
// bit 1 of the decode-attention kernels' `bf16_trig` argument: RoPE position of the new token = column - kv_start[row]
// (HF generate() derives position_ids from the attention mask; the image loop passes none => absolute columns)
constexpr int ROPE_REL = 2;      // block 0 increments *step_ptr at the end (last kernel of a decode-step graph)

// Fixed-order (left to right) sum over the split-K slabs.  ALL slab loads are issued before the first add:
// a load-add-load-add loop serialises one L2 round trip (~0.45 us) per split on the in-order pipe.
constexpr int MAX_SPLITS = 16;
template <int MAXS>
PG_DEVINL void load_splits(const float* __restrict__ p, int S, size_t split_stride, float (&b)[MAXS]) {
#pragma unroll
  for (int s = 0; s < MAXS; ++s) b[s] = (s < S) ? __ldcg(p + (size_t)s * split_stride) : 0.f;
}
template <int MAXS>
PG_DEVINL float sum_loaded(const float (&b)[MAXS], int S) {
  float a = b[0];
#pragma unroll
  for (int s = 1; s < MAXS; ++s) if (s < S) a += b[s];
  return a;
}
// single element: slabs in chunks of 8 loads in flight (same left-to-right order)
PG_DEVINL float reduce_splits(const float* __restrict__ part, int S, size_t split_stride, size_t idx) {
  const float* p = part + idx;
  float b[8];
  load_splits(p, S, split_stride, b);
  float a = sum_loaded(b, S);
  if (S > 8) {
    load_splits(p + (size_t)8 * split_stride, S - 8, split_stride, b);
    a += b[0];
#pragma unroll
    for (int s = 1; s < 8; ++s) if (s < S - 8) a += b[s];
  }
  return a;
}

// ------------------------------------------------------------------- a9: embed_tokens
// replaces language_model.get_input_embeddings()(ids)  (plangen_base.py:548)
__global__ void embed_gather_kernel(const int32_t* __restrict__ ids, const float* __restrict__ table,
                                    float* __restrict__ x, int D, int vocab) {
  pdl_launch_dependents();
  pdl_wait();
  const int tok = blockIdx.x;
  int id = ids[tok];
  id = min(max(id, 0), vocab - 1);
  const float4* src = reinterpret_cast<const float4*>(table + (size_t)id * D);
  float4* dst = reinterpret_cast<float4*>(x + (size_t)tok * D);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = src[i];
}

// ------------------------------------------------- a4.1: residual add + LlamaRMSNorm
// x[tok] += rnd(sum_s part[s][tok]);  xn = w * (x * rsqrt(mean(x^2) + eps))   (HF modeling_llama.py:60-65)
// One CTA per output row.  Input row index = blockIdx.x * in_stride + in_off (lets the final norm of
// a prefill pick only the last position of every prompt row).
// debug timeline (tools/norm_timeline.py): 8 %globaltimer stamps per CTA of the decode-step norm kernels of the
// step g_norm_dbg_step, indexed by the kernel's timeline slot; nullptr in production
__device__ unsigned long long* g_norm_dbg = nullptr;
__device__ int g_norm_dbg_step = -1;
PG_DEVINL void norm_stamp(unsigned long long* d, int slot, int k) {
  if (d && threadIdx.x == 0) d[((size_t)slot * 64 + blockIdx.x) * 8 + k] = global_timer_ns();
}

constexpr int RN_THREADS = 1024;            // upper bound; launched with 256..1024 threads
constexpr int RN_MAX_PER_THREAD = 8;        // D <= 8 * blockDim.x
template <typename T>
__global__ void __launch_bounds__(RN_THREADS)
resid_rmsnorm_kernel(float* __restrict__ x, const float* __restrict__ part, int S, size_t split_stride,
                     const float* __restrict__ w, T* __restrict__ xn_out, float* __restrict__ y_out, int D,
                     float eps, int in_stride, int in_off, int flags, int* step_ptr, Prof prof) {
  __shared__ float red[32];
  pdl_launch_dependents();
  prof_begin(prof);
  unsigned long long* nd = (prof.buf && g_norm_dbg && step_ptr && *step_ptr == g_norm_dbg_step && blockIdx.x < 64) ? g_norm_dbg : nullptr;
  norm_stamp(nd, prof.slot, 0);
  // the norm weight is a constant: fetch it before the dependency wait instead of after the reduction
  float wv[RN_MAX_PER_THREAD];
#pragma unroll
  for (int k = 0; k < RN_MAX_PER_THREAD; ++k) {
    const int d = threadIdx.x + k * blockDim.x;
    wv[k] = (d < D) ? w[d] : 0.f;
  }
  pdl_wait();
  norm_stamp(nd, prof.slot, 1);
  const size_t row_in = (size_t)blockIdx.x * in_stride + in_off;
  const size_t row_out = blockIdx.x;
  float* xr = x + row_in * D;
  float v[RN_MAX_PER_THREAD];
  float ss = 0.f;
  // residual update + sum of squares; the row stays in registers (all split loads of a thread are
  // independent, so they are in flight together)
#pragma unroll
  for (int k0 = 0; k0 < RN_MAX_PER_THREAD; k0 += 2) {       // two elements (<= 34 loads) in flight at a time
    float b[2][MAX_SPLITS];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int d = threadIdx.x + (k0 + j) * blockDim.x;
      v[k0 + j] = 0.f;
      if (d < D) {
        v[k0 + j] = xr[d];
        if (part != nullptr) load_splits(part + row_in * D + d, S, split_stride, b[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int d = threadIdx.x + (k0 + j) * blockDim.x;
      if (d < D) {
        float t = v[k0 + j];
        if (part != nullptr) {
          t = t + Act<T>::rnd(sum_loaded(b[j], S));
          if (flags & RN_ROUND_RESID) t = Act<T>::rnd(t);
          xr[d] = t;
        }
        v[k0 + j] = t;
        ss += t * t;
      }
    }
  }
  norm_stamp(nd, prof.slot, 2);
  ss = block_sum(ss, red);
  norm_stamp(nd, prof.slot, 3);
  const float r = rsqrtf(ss / (float)D + eps);
#pragma unroll
  for (int k = 0; k < RN_MAX_PER_THREAD; ++k) {
    const int d = threadIdx.x + k * blockDim.x;
    if (d < D) {
      float hn = v[k] * r;
      if (flags & RN_ROUND_RESID) hn = Act<T>::rnd(hn);      // `.to(input_dtype)` with a bf16 residual stream
      const float y = wv[k] * hn;
      if (xn_out) Act<T>::st(xn_out + row_out * D + d, y);   // autocast cast at the next Linear
      if (y_out) y_out[row_out * D + d] = y;
    }
  }
  norm_stamp(nd, prof.slot, 4);
  if ((flags & RN_INC_STEP) && blockIdx.x == 0 && threadIdx.x == 0) *step_ptr += 1;
  prof_end(prof);
}

// Prefill variant (fused epilogues: the residual is already in x, bf16 output only, thousands of rows): ONE WARP PER ROW,
// the row in registers as float4 (NV per lane; NV = 0: two passes over the row, the second from L1 / L2), no shared
// memory, no block barrier.  The one-CTA-per-row kernel above moved 76 MB in 44.7 us (1.7 TB/s) at configs[1]'s prefill.
// Same expression per element (w * (x * r), r from the row's sum of squares); the sum is taken lane-sequentially and then
// over the lanes, so r can differ from the block-tree version in the last bit.
template <int NV>
__global__ void __launch_bounds__(256)
rmsnorm_rows_warp_kernel(const float* __restrict__ x, const float* __restrict__ w, bf16* __restrict__ xn, int rows, int D, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * D);
  const float4* w4 = reinterpret_cast<const float4*>(w);
  uint2* out = reinterpret_cast<uint2*>(xn + (size_t)row * D);
  const int n4 = D / 128;                         // float4 per lane
  float ss = 0.f;
  float4 v[NV > 0 ? NV : 1];
  if (NV > 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) v[k] = xr[lane + 32 * k];
#pragma unroll
    for (int k = 0; k < NV; ++k) ss += v[k].x * v[k].x + v[k].y * v[k].y + v[k].z * v[k].z + v[k].w * v[k].w;
  } else {
    for (int k = 0; k < n4; ++k) {
      const float4 t = xr[lane + 32 * k];
      ss += t.x * t.x + t.y * t.y + t.z * t.z + t.w * t.w;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float r = rsqrtf(ss / (float)D + eps);
  auto emit = [&](int k, const float4& t) {
    const float4 ww = w4[lane + 32 * k];
    const __nv_bfloat162 a = __floats2bfloat162_rn(ww.x * (t.x * r), ww.y * (t.y * r));
    const __nv_bfloat162 b = __floats2bfloat162_rn(ww.z * (t.z * r), ww.w * (t.w * r));
    out[lane + 32 * k] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
  };
  if (NV > 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) emit(k, v[k]);
  } else {
    for (int k = 0; k < n4; ++k) emit(k, xr[lane + 32 * k]);
  }
}

// Decode-step variant: the S split-K slabs of the row and the residual row are brought into shared memory by
// S + 1 TMA bulk copies issued by one thread, instead of 18-34 scalar loads per thread.  In-kernel stamps
// (tools/norm_timeline.py) showed the scalar version spending 3.3-3.7 us in its single round of L2 loads whether
// or not the neighbouring contractions were prefetching: with one CTA per row only 32 SMs take part and each is
// bound by its own load-miss parallelism (74 KB per SM); the copy engine keeps the whole 74 KB in flight.
// Same left-to-right summation order and rounding points as resid_rmsnorm_kernel => bit-identical results.
PG_DEVINL float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}
template <typename T>
__global__ void __launch_bounds__(RN_THREADS)
resid_rmsnorm_tma_kernel(float* __restrict__ x, const float* __restrict__ part, int S, size_t split_stride,
                         const float* __restrict__ w, T* __restrict__ xn_out, float* __restrict__ y_out, int D,
                         float eps, int flags, int* step_ptr, Prof prof) {
  extern __shared__ uint8_t rn_smem_raw[];
  __shared__ float red[32];
  __shared__ uint64_t bar;
  const uint32_t slab_s = (smem_u32(rn_smem_raw) + 127u) & ~127u;          // [S + 1][D] fp32, shared-space address
  pdl_launch_dependents();
  prof_begin(prof);
  unsigned long long* nd = (prof.buf && g_norm_dbg && step_ptr && *step_ptr == g_norm_dbg_step && blockIdx.x < 64) ? g_norm_dbg : nullptr;
  norm_stamp(nd, prof.slot, 0);
  const int tid = threadIdx.x;
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  // thread t owns the element quads 4 (t + k blockDim); the norm weight is a constant: fetched before the wait
  constexpr int NQ = RN_MAX_PER_THREAD / 4;
  float4 wv[NQ];
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    const int d = 4 * (tid + k * blockDim.x);
    wv[k] = (d < D) ? *reinterpret_cast<const float4*>(w + d) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncthreads();
  pdl_wait();
  norm_stamp(nd, prof.slot, 1);
  const size_t row = blockIdx.x;
  float* xr = x + row * D;
  const uint32_t row_bytes = (uint32_t)D * 4;
  if (tid == 0) {
    const uint64_t pol = policy_evict_first();
    mbar_expect_tx(&bar, (uint32_t)(S + 1) * row_bytes);
    uint32_t dst = slab_s;
    const float* src = part + row * D;
    for (int s = 0; s < S; ++s, dst += row_bytes, src += split_stride)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                   ::"r"(dst), "l"(src), "r"(row_bytes), "r"(smem_u32(&bar)), "l"(pol) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(xr), "r"(row_bytes), "r"(smem_u32(&bar)), "l"(pol) : "memory");
  }
  if (tid < 32) mbar_wait(&bar, 0, 40);          // one warp polls the barrier; bar.sync releases the rest
  __syncthreads();
  norm_stamp(nd, prof.slot, 2);
  float4 v[NQ];
  float ss = 0.f;
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    const int d = 4 * (tid + k * blockDim.x);
    v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d < D) {
      uint32_t a_s = slab_s + (uint32_t)d * 4;
      float4 a = lds_f4(a_s);
      int s = 1;
      for (; s + 4 <= S; s += 4) {               // four independent loads in flight, adds stay left to right
        const float4 b0 = lds_f4(a_s + (uint32_t)(s + 0) * row_bytes), b1 = lds_f4(a_s + (uint32_t)(s + 1) * row_bytes);
        const float4 b2 = lds_f4(a_s + (uint32_t)(s + 2) * row_bytes), b3 = lds_f4(a_s + (uint32_t)(s + 3) * row_bytes);
        a.x += b0.x; a.y += b0.y; a.z += b0.z; a.w += b0.w;
        a.x += b1.x; a.y += b1.y; a.z += b1.z; a.w += b1.w;
        a.x += b2.x; a.y += b2.y; a.z += b2.z; a.w += b2.w;
        a.x += b3.x; a.y += b3.y; a.z += b3.z; a.w += b3.w;
      }
      for (; s < S; ++s) {
        const float4 b = lds_f4(a_s + (uint32_t)s * row_bytes);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      const float4 xv = lds_f4(a_s + (uint32_t)S * row_bytes);
      float4 t;
      t.x = xv.x + Act<T>::rnd(a.x); t.y = xv.y + Act<T>::rnd(a.y); t.z = xv.z + Act<T>::rnd(a.z); t.w = xv.w + Act<T>::rnd(a.w);
      if (flags & RN_ROUND_RESID) { t.x = Act<T>::rnd(t.x); t.y = Act<T>::rnd(t.y); t.z = Act<T>::rnd(t.z); t.w = Act<T>::rnd(t.w); }
      *reinterpret_cast<float4*>(xr + d) = t;
      v[k] = t;
      ss += t.x * t.x; ss += t.y * t.y; ss += t.z * t.z; ss += t.w * t.w;
    }
  }
  ss = block_sum(ss, red);
  norm_stamp(nd, prof.slot, 3);
  const float r = rsqrtf(ss / (float)D + eps);
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    const int d = 4 * (tid + k * blockDim.x);
    if (d < D) {
      float h[4] = {v[k].x * r, v[k].y * r, v[k].z * r, v[k].w * r};
      if (flags & RN_ROUND_RESID) {
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = Act<T>::rnd(h[j]);
      }
      const float y[4] = {wv[k].x * h[0], wv[k].y * h[1], wv[k].z * h[2], wv[k].w * h[3]};
      if (xn_out) {
        if constexpr (sizeof(T) == 2) {
          const __nv_bfloat162 lo = __floats2bfloat162_rn(y[0], y[1]), hi = __floats2bfloat162_rn(y[2], y[3]);
          uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
          *reinterpret_cast<uint2*>(xn_out + row * D + d) = pk;
        } else {
          *reinterpret_cast<float4*>(xn_out + row * D + d) = make_float4(y[0], y[1], y[2], y[3]);
        }
      }
      if (y_out) *reinterpret_cast<float4*>(y_out + row * D + d) = make_float4(y[0], y[1], y[2], y[3]);
    }
  }
  norm_stamp(nd, prof.slot, 4);
  if ((flags & RN_INC_STEP) && blockIdx.x == 0 && tid == 0) *step_ptr += 1;
  prof_end(prof);
}

// plain RMSNorm of externally supplied rows (used for the first layer of a decode step when the
// caller hands in inputs_embeds through the drop-in API)
// -> same kernel with part == nullptr.

// ------------------------------------------------------ a4.2: RoPE (HF :138-168)
// q_embed = q * cos + rotate_half(q) * sin, rotate_half = [-x2, x1] over the two halves of head_dim.
// bf16_trig: decode steps in the autocast regime get cos/sin cast to bf16 and bf16 arithmetic
// (cos.to(x.dtype) with x = bf16 hidden states); prefill keeps fp32 trig (x = fp32 embeddings).
template <typename T>
PG_DEVINL void rope_pair(float x1, float x2, float c, float s, bool bf16_trig, float& o1, float& o2) {
  if (bf16_trig) {
    c = Act<T>::rnd(c); s = Act<T>::rnd(s);
    o1 = Act<T>::rnd(Act<T>::rnd(__fmul_rn(x1, c)) + Act<T>::rnd(__fmul_rn(-x2, s)));
    o2 = Act<T>::rnd(Act<T>::rnd(__fmul_rn(x2, c)) + Act<T>::rnd(__fmul_rn(x1, s)));
  } else {
    o1 = Act<T>::rnd(__fadd_rn(__fmul_rn(x1, c), __fmul_rn(-x2, s)));
    o2 = Act<T>::rnd(__fadd_rn(__fmul_rn(x2, c), __fmul_rn(x1, s)));
  }
}

// Prefill: reduce QKV partials, RoPE, write q [tok][H*128] and K/V into the cache
// cache layout per layer: [2 (k,v)][R][H][Tmax][128]
template <typename T>
__global__ void __launch_bounds__(256)
qkv_rope_store_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ cosT,
                      const float* __restrict__ sinT, T* __restrict__ q_out, T* __restrict__ kcache,
                      T* __restrict__ vcache, int P, int H, int Tmax, const int32_t* __restrict__ rope_start) {
  pdl_launch_dependents();
  pdl_wait();
  const int tok = blockIdx.x;
  const int r = tok / P, p = tok % P;
  const int HD = H * HEAD_DIM;
  const float* row = part + (size_t)tok * 3 * HD;
  // rope_start != nullptr: HF generate() positions, cumsum(attention_mask) - 1 = column - left-pad count
  // (GenerationMixin.prepare_inputs_for_generation); nullptr: absolute columns (LlamaModel.forward without
  // position_ids, the image loop, plangen_base.py:571-576).  Pad columns are never attended; their position is moot.
  const int pr = rope_start ? max(p - rope_start[r], 0) : p;
  if (S == 1) {
    // prefill (one split): four rotary pairs per thread, 16-byte loads / 8-byte stores
    for (int i = threadIdx.x; i < H * 16; i += blockDim.x) {
      const int h = i >> 4, j = (i & 15) * 4;
      const float4 c4 = *reinterpret_cast<const float4*>(cosT + pr * 64 + j), s4 = *reinterpret_cast<const float4*>(sinT + pr * 64 + j);
      const float cs[4] = {c4.x, c4.y, c4.z, c4.w}, sn[4] = {s4.x, s4.y, s4.z, s4.w};
      const size_t o1 = (size_t)h * HEAD_DIM + j, o2 = o1 + 64;
      const size_t cidx = (((size_t)r * H + h) * Tmax + p) * HEAD_DIM + j;
      float lo[4], hi[4], a[4], b[4];
      auto ld4 = [&](size_t off, float (&dst)[4]) {
        const float4 t = __ldcs(reinterpret_cast<const float4*>(row + off));
        dst[0] = t.x; dst[1] = t.y; dst[2] = t.z; dst[3] = t.w;
      };
      auto st4 = [&](T* dst, const float (&src)[4]) {
        if constexpr (sizeof(T) == 2) {
          const __nv_bfloat162 x0 = __floats2bfloat162_rn(src[0], src[1]), x1 = __floats2bfloat162_rn(src[2], src[3]);
          uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&x0); pk.y = *reinterpret_cast<const uint32_t*>(&x1);
          *reinterpret_cast<uint2*>(dst) = pk;
        } else {
          *reinterpret_cast<float4*>(dst) = make_float4(src[0], src[1], src[2], src[3]);
        }
      };
      ld4(o1, lo); ld4(o2, hi);
#pragma unroll
      for (int u = 0; u < 4; ++u) rope_pair<T>(Act<T>::rnd(lo[u]), Act<T>::rnd(hi[u]), cs[u], sn[u], false, a[u], b[u]);
      st4(q_out + (size_t)tok * HD + o1, a); st4(q_out + (size_t)tok * HD + o2, b);
      ld4(HD + o1, lo); ld4(HD + o2, hi);
#pragma unroll
      for (int u = 0; u < 4; ++u) rope_pair<T>(Act<T>::rnd(lo[u]), Act<T>::rnd(hi[u]), cs[u], sn[u], false, a[u], b[u]);
      st4(kcache + cidx, a); st4(kcache + cidx + 64, b);
      ld4(2 * HD + o1, lo); ld4(2 * HD + o2, hi);
      st4(vcache + cidx, lo); st4(vcache + cidx + 64, hi);
    }
    return;
  }
  for (int i = threadIdx.x; i < H * 64; i += blockDim.x) {
    const int h = i >> 6, j = i & 63;
    const float c = cosT[pr * 64 + j], s = sinT[pr * 64 + j];
    const size_t o1 = (size_t)h * HEAD_DIM + j, o2 = o1 + 64;
    float q1 = Act<T>::rnd(reduce_splits(row, S, split_stride, o1));
    float q2 = Act<T>::rnd(reduce_splits(row, S, split_stride, o2));
    float k1 = Act<T>::rnd(reduce_splits(row, S, split_stride, HD + o1));
    float k2 = Act<T>::rnd(reduce_splits(row, S, split_stride, HD + o2));
    const float v1 = reduce_splits(row, S, split_stride, 2 * HD + o1);
    const float v2 = reduce_splits(row, S, split_stride, 2 * HD + o2);
    float a, b;
    rope_pair<T>(q1, q2, c, s, false, a, b);
    Act<T>::st(q_out + (size_t)tok * HD + o1, a);
    Act<T>::st(q_out + (size_t)tok * HD + o2, b);
    rope_pair<T>(k1, k2, c, s, false, a, b);
    const size_t cidx = (((size_t)r * H + h) * Tmax + p) * HEAD_DIM + j;
    Act<T>::st(kcache + cidx, a);
    Act<T>::st(kcache + cidx + 64, b);
    Act<T>::st(vcache + cidx, v1);
    Act<T>::st(vcache + cidx + 64, v2);
  }
}

// ---------------------------------------------------------------- packed (ragged) prefill
// The reference pads every prompt row on the LEFT to the batch maximum P and runs the padded (R, P) block through the
// model (the 16 unconditional rows of configs[1] are ~110 tokens padded to ~350: 40 % of the positions are pads).  Pad
// positions never influence a real position (they are masked as keys and their own outputs are discarded), so the
// fused loops run the prefill on the REAL tokens only, packed row after row: token t of the packed stream belongs to
// row r with row_off[r] <= t < row_off[r+1] and sits at column kv_start[r] + (t - row_off[r]).
PG_DEVINL int packed_row_of(const int32_t* __restrict__ row_off, int R, int t) {
  int lo = 0, hi = R - 1;                       // largest r with row_off[r] <= t
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (row_off[mid] <= t) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// Rows that repeat an EARLIER row (PlanGen's unconditional rows all carry the same negative prompt, cfg/base.py:129) are
// prefilled ONCE: row r with dup_of[r] != r contributes no tokens to the packed stream (row_off[r+1] == row_off[r]); its
// K / V strips and its final hidden state are copied from row dup_of[r] afterwards (identical inputs through deterministic
// kernels give identical bits, so the copy equals the recomputation).
// Finding the repeats takes two passes.  (1) a 64-bit content hash per row (sum over the real columns of a mixed
// (word, position) pair: order-independent, so blocks just atomicAdd their share); the host groups rows by (left padding,
// hash) and proposes the FIRST row of each group as the source of the others.  (2) every proposal is verified word for word
// (a hash collision only costs the row its shortcut).  Repeats may sit anywhere in the batch: the unconditional rows of one
// negative prompt (distance 2), the copies of `parallel_size` > 1 (distance 2 * bs), repeated captions.
PG_DEVINL unsigned long long mix64(unsigned long long z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
// grid (P, R)
__global__ void __launch_bounds__(256)
prefill_row_hash_kernel(const float* __restrict__ x, const int32_t* __restrict__ kv_start, unsigned long long* __restrict__ hash, int P, int D) {
  const int p = blockIdx.x, r = blockIdx.y;
  if (p < kv_start[r]) return;
  const uint32_t* a = reinterpret_cast<const uint32_t*>(x + ((size_t)r * P + p) * D);
  unsigned long long h = 0;
  for (int i = threadIdx.x; i < D; i += blockDim.x)
    h += mix64(((unsigned long long)a[i] << 32) | (unsigned long long)(uint32_t)(p * D + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  __shared__ unsigned long long wsum[8];
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = h;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += wsum[w];
    atomicAdd(hash + r, t);
  }
}
// differs[r] = 1 when row r is not bitwise the row cand[r] over the real columns (same left padding by construction): grid (P, R)
__global__ void __launch_bounds__(256)
prefill_row_verify_kernel(const float* __restrict__ x, const int32_t* __restrict__ kv_start, const int32_t* __restrict__ cand,
                          int32_t* __restrict__ differs, int P, int D) {
  const int p = blockIdx.x, r = blockIdx.y, c = cand[r];
  if (c == r || p < kv_start[r]) return;
  const uint4* a = reinterpret_cast<const uint4*>(x + ((size_t)r * P + p) * D);
  const uint4* b = reinterpret_cast<const uint4*>(x + ((size_t)c * P + p) * D);
  bool diff = false;
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) {
    const uint4 u = a[i], v = b[i];
    diff |= (u.x != v.x) | (u.y != v.y) | (u.z != v.z) | (u.w != v.w);
  }
  if (diff) differs[r] = 1;                               // benign race: every writer stores 1
}
__global__ void iota_i32_kernel(int32_t* __restrict__ p, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i;
}
// K / V strips of the prompt columns of duplicate rows: grid (L * 2 * H, R), cache [L][2][R][H][Tmax][128] bf16
__global__ void __launch_bounds__(256)
kv_broadcast_rows_kernel(bf16* __restrict__ kv, const int32_t* __restrict__ dup_of, const int32_t* __restrict__ kv_start, int R, int H,
                         int Tmax, int P) {
  pdl_launch_dependents();
  pdl_wait();
  const int r = blockIdx.y, src = dup_of[r];
  if (src == r) return;
  const int lkh = blockIdx.x, h = lkh % H, lk = lkh / H;
  const int start = kv_start[r];
  const size_t strip = (size_t)Tmax * HEAD_DIM;
  const uint4* s4 = reinterpret_cast<const uint4*>(kv + (((size_t)lk * R + src) * H + h) * strip + (size_t)start * HEAD_DIM);
  uint4* d4 = reinterpret_cast<uint4*>(kv + (((size_t)lk * R + r) * H + h) * strip + (size_t)start * HEAD_DIM);
  const int n16 = (P - start) * HEAD_DIM * 2 / 16;
  for (int i = threadIdx.x; i < n16; i += blockDim.x) d4[i] = s4[i];
}

// x [R][P][D] -> xp [sum len][D]: grid (P, R)
__global__ void __launch_bounds__(256)
prefill_pack_kernel(const float* __restrict__ x, float* __restrict__ xp, const int32_t* __restrict__ kv_start,
                    const int32_t* __restrict__ row_off, int P, int D) {
  pdl_launch_dependents();
  pdl_wait();
  const int p = blockIdx.x, r = blockIdx.y;
  const int start = kv_start[r];
  if (p < start || row_off[r + 1] == row_off[r]) return;       // pad column, or a duplicate row (no tokens of its own)
  const float4* src = reinterpret_cast<const float4*>(x + ((size_t)r * P + p) * D);
  float4* dst = reinterpret_cast<float4*>(xp + (size_t)(row_off[r] + p - start) * D);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = src[i];
}
// last real token of every row (of the row it duplicates): xp[row_off[dup_of[r] + 1] - 1] -> out[r]
__global__ void __launch_bounds__(256)
gather_last_rows_kernel(const float* __restrict__ xp, float* __restrict__ out, const int32_t* __restrict__ row_off,
                        const int32_t* __restrict__ dup_of, int D) {
  pdl_launch_dependents();
  pdl_wait();
  const int r = blockIdx.x;
  const float4* src = reinterpret_cast<const float4*>(xp + (size_t)(row_off[dup_of[r] + 1] - 1) * D);
  float4* dst = reinterpret_cast<float4*>(out + (size_t)r * D);
  for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = src[i];
}

// teacher-forced scoring: the hidden states of the last `ncols` columns of every row (of the row it duplicates when
// packed), pair-major: column P - ncols + i of row r -> out[((r / 2) * ncols + i) * 2 + r % 2].  grid (ncols, R)
template <typename T>
__global__ void __launch_bounds__(256)
gather_tail_rows_kernel(const T* __restrict__ src, T* __restrict__ out, const int32_t* __restrict__ row_off,
                        const int32_t* __restrict__ dup_of, const int32_t* __restrict__ kv_start, int P, int ncols, int D) {
  pdl_launch_dependents();
  pdl_wait();
  const int i = blockIdx.x, r = blockIdx.y, col = P - ncols + i;
  const size_t pos = row_off ? (size_t)row_off[dup_of[r]] + max(col - kv_start[r], 0) : (size_t)r * P + col;
  const T* s = src + pos * D;
  T* o = out + ((size_t)((r / 2) * ncols + i) * 2 + (r & 1)) * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) o[d] = s[d];
}

// Prefill variant behind the contraction's fused bf16 epilogue (gemm.cuh EpiFuse): the projections arrive already
// rounded to bf16 ([tok][3*H*128], q | k | v), so this kernel only rotates and scatters - same values as
// qkv_rope_store_kernel<bf16> on the fp32 partials (it rounds them first), half the bytes.
__global__ void __launch_bounds__(256)
qkv_rope_store_bf16_kernel(const bf16* __restrict__ qkv, const float* __restrict__ cosT, const float* __restrict__ sinT,
                           bf16* __restrict__ q_out, bf16* __restrict__ kcache, bf16* __restrict__ vcache, int P, int H, int Tmax,
                           const int32_t* __restrict__ rope_start, const int32_t* __restrict__ row_off,
                           const int32_t* __restrict__ kv_start, int R) {
  pdl_launch_dependents();
  pdl_wait();
  const int tok = blockIdx.x;
  int r, p;
  if (row_off != nullptr) {                      // packed stream (see packed_row_of)
    r = packed_row_of(row_off, R, tok);
    p = kv_start[r] + (tok - row_off[r]);
  } else {
    r = tok / P; p = tok % P;
  }
  const int HD = H * HEAD_DIM;
  const bf16* row = qkv + (size_t)tok * 3 * HD;
  const int pr = rope_start ? max(p - rope_start[r], 0) : p;
  for (int i = threadIdx.x; i < H * 16; i += blockDim.x) {
    const int h = i >> 4, j = (i & 15) * 4;
    const float4 c4 = *reinterpret_cast<const float4*>(cosT + pr * 64 + j), s4 = *reinterpret_cast<const float4*>(sinT + pr * 64 + j);
    const float cs[4] = {c4.x, c4.y, c4.z, c4.w}, sn[4] = {s4.x, s4.y, s4.z, s4.w};
    const size_t o1 = (size_t)h * HEAD_DIM + j, o2 = o1 + 64;
    const size_t cidx = (((size_t)r * H + h) * Tmax + p) * HEAD_DIM + j;
    auto ld4 = [&](size_t off, float (&dst)[4]) {
      const uint2 t = *reinterpret_cast<const uint2*>(row + off);
      dst[0] = bf16lo(t.x); dst[1] = bf16hi(t.x); dst[2] = bf16lo(t.y); dst[3] = bf16hi(t.y);
    };
    auto st4 = [&](bf16* dst, const float (&src)[4]) {
      const __nv_bfloat162 x0 = __floats2bfloat162_rn(src[0], src[1]), x1 = __floats2bfloat162_rn(src[2], src[3]);
      uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&x0); pk.y = *reinterpret_cast<const uint32_t*>(&x1);
      *reinterpret_cast<uint2*>(dst) = pk;
    };
    float lo[4], hi[4], a[4], b[4];
    ld4(o1, lo); ld4(o2, hi);
#pragma unroll
    for (int u = 0; u < 4; ++u) rope_pair<bf16>(lo[u], hi[u], cs[u], sn[u], false, a[u], b[u]);
    st4(q_out + (size_t)tok * HD + o1, a); st4(q_out + (size_t)tok * HD + o2, b);
    ld4(HD + o1, lo); ld4(HD + o2, hi);
#pragma unroll
    for (int u = 0; u < 4; ++u) rope_pair<bf16>(lo[u], hi[u], cs[u], sn[u], false, a[u], b[u]);
    st4(kcache + cidx, a); st4(kcache + cidx + 64, b);
    *reinterpret_cast<uint2*>(vcache + cidx) = *reinterpret_cast<const uint2*>(row + 2 * HD + o1);
    *reinterpret_cast<uint2*>(vcache + cidx + 64) = *reinterpret_cast<const uint2*>(row + 2 * HD + o2);
  }
}

// ---------------------------------------------------------------- a4.3: SwiGLU
// h = silu(gate) * up   (HF LlamaMLP :182-184); partial layout [S][tok][2F]: [gate | up], or - when the
// weight rows were packed for the fused tcgen05 epilogue - interleaved in blocks of 64 (g0-63, u0-63, g64-127, ...)
template <typename T>
__global__ void __launch_bounds__(256)
swiglu_kernel(const float* __restrict__ part, int S, size_t split_stride, T* __restrict__ h, int F, size_t total,
              int interleaved, Prof prof) {
  pdl_launch_dependents();
  prof_begin(prof);
  pdl_wait();
  if (S == 1 && F % 64 == 0 && total < (size_t)1 << 31) {
    // prefill-sized inputs: 4 outputs per thread, 16-byte loads, 32-bit index arithmetic
    const int F4 = F / 4, n4 = (int)(total / 4);
    for (int i4 = blockIdx.x * blockDim.x + threadIdx.x; i4 < n4; i4 += gridDim.x * blockDim.x) {
      const int tok = i4 / F4, f = (i4 - tok * F4) * 4;
      const int gi = interleaved ? (f >> 6) * 128 + (f & 63) : f;
      const int ui = interleaved ? gi + 64 : F + f;
      const float* row = part + (size_t)tok * 2 * F;
      const float4 g4 = __ldcs(reinterpret_cast<const float4*>(row + gi));
      const float4 u4 = __ldcs(reinterpret_cast<const float4*>(row + ui));
      const float gs[4] = {g4.x, g4.y, g4.z, g4.w}, us[4] = {u4.x, u4.y, u4.z, u4.w};
      float o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float g = Act<T>::rnd(gs[j]), u = Act<T>::rnd(us[j]);
        o[j] = Act<T>::rnd(g / (1.0f + expf(-g))) * u;
      }
      T* dst = h + (size_t)tok * F + f;
      if constexpr (sizeof(T) == 2) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(o[0], o[1]), hi = __floats2bfloat162_rn(o[2], o[3]);
        uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(dst) = pk;
      } else {
        *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
      }
    }
    prof_end(prof);
    return;
  }
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t tok = i / F, f = i % F;
    const size_t gi = interleaved ? (f / 64) * 128 + f % 64 : f;
    const size_t ui = interleaved ? gi + 64 : F + f;
    const float g = Act<T>::rnd(reduce_splits(part, S, split_stride, tok * 2 * F + gi));
    const float u = Act<T>::rnd(reduce_splits(part, S, split_stride, tok * 2 * F + ui));
    const float sg = Act<T>::rnd(g / (1.0f + expf(-g)));
    Act<T>::st(h + i, sg * u);
  }
  prof_end(prof);
}

// ------------------------------------------------------- bias (+ exact GELU) epilogue
// out = act(rnd(sum_s part + bias)); GELU is the erf form (nn.GELU() default, modeling_vlm.py:43)
template <typename T>
__global__ void __launch_bounds__(256)
bias_act_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ bias,
                T* __restrict__ out_t, float* __restrict__ out_f, int N, size_t total, int gelu) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    float v = reduce_splits(part, S, split_stride, i);
    if (bias) v += bias[i % N];
    v = Act<T>::rnd(v);
    if (gelu) v = Act<T>::rnd(v * 0.5f * (1.0f + erff(v * 0.70710678118654752440f)));
    if (out_t) Act<T>::st(out_t + i, v);
    if (out_f) out_f[i] = v;
  }
}

// --------------------------------------------------------- a3: prefill attention
// Causal attention with LEFT padding: key j is visible to the query at column p iff
// kv_start[r] <= j <= p (the reference's (R, P+576) 0/1 mask + HF create_causal_mask).
// CUDA-core flash-style kernel: CTA = 64 queries x one head x one row, 256 threads;
// S = Q K^T in 4x4 register tiles, online softmax in fp32, O += P V in 4x8 register tiles.
// Masked cache columns in [(kv_start / 64) * 64, P) must hold finite values: they enter O += P V with weight 0.
template <typename T>
__global__ void __launch_bounds__(256)
attn_prefill_kernel(const T* __restrict__ q, const T* __restrict__ kcache, const T* __restrict__ vcache,
                    const int32_t* __restrict__ kv_start, T* __restrict__ out, int P, int H, int Tmax, float scale) {
  extern __shared__ float sm[];
  constexpr int LDQ = HEAD_DIM + 1;
  float* Qs = sm;                       // [64][129]
  float* Ks = Qs + 64 * LDQ;            // [64][129]
  float* Vs = Ks + 64 * LDQ;            // [64][128]
  float* Ss = Vs + 64 * HEAD_DIM;       // [64][65]
  float* row_m = Ss + 64 * 65;          // [64]
  float* row_l = row_m + 64;            // [64]
  float* row_c = row_l + 64;            // [64] correction factor of the current tile
  pdl_launch_dependents();
  pdl_wait();
  const int tid = threadIdx.x;
  const int q0 = blockIdx.x * 64, h = blockIdx.y, r = blockIdx.z;
  const int HD = H * HEAD_DIM;
  const int start = kv_start[r];
  const T* kbase = kcache + ((size_t)r * H + h) * Tmax * HEAD_DIM;
  const T* vbase = vcache + ((size_t)r * H + h) * Tmax * HEAD_DIM;
  for (int i = tid; i < 64 * HEAD_DIM; i += 256) {
    const int qi = i >> 7, d = i & 127;
    const int p = q0 + qi;
    Qs[qi * LDQ + d] = (p < P) ? Act<T>::ld(q + ((size_t)r * P + p) * HD + h * HEAD_DIM + d) * scale : 0.f;
  }
  if (tid < 64) { row_m[tid] = -INFINITY; row_l[tid] = 0.f; }
  const int ty = tid >> 4, tx = tid & 15;
  float o[4][8] = {};
  const int q_hi = min(q0 + 63, P - 1);
  const int j_begin = (start / 64) * 64;
  for (int j0 = j_begin; j0 <= q_hi; j0 += 64) {
    __syncthreads();
    for (int i = tid; i < 64 * HEAD_DIM; i += 256) {
      const int kj = i >> 7, d = i & 127;
      const int j = j0 + kj;
      const bool ok = j < P;
      Ks[kj * LDQ + d] = ok ? Act<T>::ld(kbase + (size_t)j * HEAD_DIM + d) : 0.f;
      Vs[kj * HEAD_DIM + d] = ok ? Act<T>::ld(vbase + (size_t)j * HEAD_DIM + d) : 0.f;
    }
    __syncthreads();
    float s[4][4] = {};
    for (int d = 0; d < HEAD_DIM; ++d) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = Qs[(ty * 4 + i) * LDQ + d]; b[i] = Ks[(tx * 4 + i) * LDQ + d]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(a[i], b[j], s[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int p = q0 + ty * 4 + i, kj = j0 + tx * 4 + j;
        const bool vis = (kj >= start) && (kj <= p) && (p < P);
        Ss[(ty * 4 + i) * 65 + tx * 4 + j] = vis ? s[i][j] : -INFINITY;
      }
    __syncthreads();
    {   // online softmax: 4 threads per query row, 16 columns each
      const int row = tid >> 2, part4 = tid & 3;
      float mx = -INFINITY;
      for (int c = part4 * 16; c < part4 * 16 + 16; ++c) mx = fmaxf(mx, Ss[row * 65 + c]);
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      const float m_old = row_m[row];
      const float m_new = fmaxf(m_old, mx);
      float sum = 0.f;
      for (int c = part4 * 16; c < part4 * 16 + 16; ++c) {
        const float sv = Ss[row * 65 + c];
        const float pv = (sv == -INFINITY) ? 0.f : expf(sv - m_new);
        Ss[row * 65 + c] = pv;
        sum += pv;
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      if (part4 == 0) {
        const float corr = (m_new == -INFINITY) ? 1.f : expf(m_old - m_new);   // expf(-inf) = 0 on the first tile
        row_c[row] = corr;
        row_l[row] = row_l[row] * corr + sum;
        row_m[row] = m_new;
      }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float c = row_c[ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[i][j] *= c;
    }
    for (int kj = 0; kj < 64; ++kj) {
      float pv[4], vv[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) pv[i] = Ss[(ty * 4 + i) * 65 + kj];
#pragma unroll
      for (int j = 0; j < 8; ++j) vv[j] = Vs[kj * HEAD_DIM + tx * 8 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) o[i][j] = fmaf(pv[i], vv[j], o[i][j]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int p = q0 + ty * 4 + i;
    if (p >= P) continue;
    const float l = row_l[ty * 4 + i];
    const float inv = l > 0.f ? 1.f / l : 0.f;      // pad queries (nothing visible) produce zeros
#pragma unroll
    for (int j = 0; j < 8; ++j)
      Act<T>::st(out + ((size_t)r * P + p) * HD + h * HEAD_DIM + tx * 8 + j, o[i][j] * inv);
  }
}
constexpr int ATTN_PREFILL_SMEM = (64 * 129 * 2 + 64 * 128 + 64 * 65 + 3 * 64) * 4;

// ------------------------------------------------- a4: KV-cache decode attention (paired CFG batch)
// One launch covers every (row, head) of the interleaved cond/uncond batch.  grid = (H, R, n_split);
// each CTA: reduces its head's q (and, for the last split, k/v) from the QKV partials, applies RoPE at
// column `pos`, the last split appends k/v to the cache, then every CTA streams its slice of the cached
// keys/values [kv_start[r], pos) with coalesced 256/512-byte row loads, 4 rows in flight per warp,
// online softmax in fp32.  Split results are merged by the last CTA to finish (threadfence + counter).
template <typename T> struct Row4;
template <> struct Row4<float> {
  static PG_DEVINL void ld(const float* p, float (&v)[4]) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
};
template <> struct Row4<bf16> {
  static PG_DEVINL void ld(const bf16* p, float (&v)[4]) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    v[0] = bf16lo(t.x); v[1] = bf16hi(t.x); v[2] = bf16lo(t.y); v[3] = bf16hi(t.y);
  }
};

template <typename T>
__global__ void __launch_bounds__(128)
attn_decode_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ cosT,
                   const float* __restrict__ sinT, T* __restrict__ kcache, T* __restrict__ vcache,
                   const int32_t* __restrict__ kv_start, T* __restrict__ out, float* __restrict__ ws_part,
                   int* __restrict__ ws_count, int H, int Tmax, int pos_base, const int* __restrict__ step_ptr,
                   float scale, int bf16_trig) {
  __shared__ float q_s[HEAD_DIM], k_s[HEAD_DIM], v_s[HEAD_DIM];
  __shared__ float m_s[4], l_s[4], o_s[4][HEAD_DIM];
  __shared__ int is_last;
  pdl_launch_dependents();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int h = blockIdx.x, r = blockIdx.y, sp = blockIdx.z, nsp = gridDim.z;
  const int HD = H * HEAD_DIM;
  pdl_wait();
  const int pos = pos_base + (step_ptr ? *step_ptr : 0);
  const int start = kv_start[r];
  // ---- q (all CTAs) and k, v (last split) of the current token
  {
    const float* row = part + (size_t)r * 3 * HD;
    const int j = tid & 63;
    const int pr = (bf16_trig & ROPE_REL) ? max(pos - start, 0) : pos;
    const float c = cosT[pr * 64 + j], s = sinT[pr * 64 + j];
    if (tid < 64) {
      const float x1 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)h * HEAD_DIM + j));
      const float x2 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)h * HEAD_DIM + j + 64));
      float a, b;
      rope_pair<T>(x1, x2, c, s, (bf16_trig & 1) != 0, a, b);
      q_s[j] = a * scale; q_s[j + 64] = b * scale;
    } else if (sp == nsp - 1) {
      const float x1 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)HD + h * HEAD_DIM + j));
      const float x2 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)HD + h * HEAD_DIM + j + 64));
      float a, b;
      rope_pair<T>(x1, x2, c, s, (bf16_trig & 1) != 0, a, b);
      const float v1 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)2 * HD + h * HEAD_DIM + j));
      const float v2 = Act<T>::rnd(reduce_splits(row, S, split_stride, (size_t)2 * HD + h * HEAD_DIM + j + 64));
      k_s[j] = a; k_s[j + 64] = b; v_s[j] = v1; v_s[j + 64] = v2;
      const size_t cidx = (((size_t)r * H + h) * Tmax + pos) * HEAD_DIM + j;
      Act<T>::st(kcache + cidx, a); Act<T>::st(kcache + cidx + 64, b);
      Act<T>::st(vcache + cidx, v1); Act<T>::st(vcache + cidx + 64, v2);
    }
  }
  __syncthreads();
  // ---- this CTA's slice of the cached tokens [start, pos)
  const int n_old = max(pos - start, 0);
  const int per = (n_old + nsp - 1) / nsp;
  const int t_lo = start + sp * per;
  const int t_hi = min(start + (sp + 1) * per, pos);
  const T* kb = kcache + ((size_t)r * H + h) * Tmax * HEAD_DIM + lane * 4;
  const T* vb = vcache + ((size_t)r * H + h) * Tmax * HEAD_DIM + lane * 4;
  float qv[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) qv[i] = q_s[lane * 4 + i];
  float m = -INFINITY, l = 0.f, o[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t0 = t_lo + warp * 4; t0 < t_hi; t0 += 16) {
    float kv[4][4], vv[4][4], sc[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int t = min(t0 + u, t_hi - 1);                  // clamp: duplicates are masked below
      Row4<T>::ld(kb + (size_t)t * HEAD_DIM, kv[u]);
      Row4<T>::ld(vb + (size_t)t * HEAD_DIM, vv[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float d = kv[u][0] * qv[0];
      d = fmaf(kv[u][1], qv[1], d); d = fmaf(kv[u][2], qv[2], d); d = fmaf(kv[u][3], qv[3], d);
      sc[u] = d;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u) sc[u] += __shfl_xor_sync(0xffffffffu, sc[u], off);
    }
    float mx = m;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (t0 + u >= t_hi) sc[u] = -INFINITY;
      mx = fmaxf(mx, sc[u]);
    }
    const float corr = (mx == -INFINITY) ? 1.f : expf(m - mx);
    l *= corr;
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] *= corr;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float p = (sc[u] == -INFINITY) ? 0.f : expf(sc[u] - mx);
      l += p;
#pragma unroll
      for (int i = 0; i < 4; ++i) o[i] = fmaf(p, vv[u][i], o[i]);
    }
    m = mx;
  }
  // ---- the current token itself (last split, warp 0), from shared memory
  if (sp == nsp - 1 && warp == 0) {
    float d = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) d = fmaf(k_s[lane * 4 + i], qv[i], d);
    d = warp_sum(d);
    const float mx = fmaxf(m, d);
    const float corr = (m == -INFINITY) ? 0.f : expf(m - mx);
    const float p = expf(d - mx);
    l = l * corr + p;
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = fmaf(p, v_s[lane * 4 + i], o[i] * corr);
    m = mx;
  }
  // ---- merge the 4 warps
  if (lane == 0) { m_s[warp] = m; l_s[warp] = l; }
#pragma unroll
  for (int i = 0; i < 4; ++i) o_s[warp][lane * 4 + i] = o[i];
  __syncthreads();
  float M = fmaxf(fmaxf(m_s[0], m_s[1]), fmaxf(m_s[2], m_s[3]));
  float Ltot = 0.f, acc = 0.f;
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    const float f = (m_s[w] == -INFINITY) ? 0.f : expf(m_s[w] - M);
    Ltot += l_s[w] * f;
    acc += o_s[w][tid] * f;
  }
  const size_t oidx = (size_t)r * HD + h * HEAD_DIM + tid;
  if (nsp == 1) {
    Act<T>::st(out + oidx, acc / Ltot);
    return;
  }
  // ---- split-T merge: last CTA of this (row, head) to arrive reduces all partials
  float* wp = ws_part + (((size_t)r * H + h) * nsp + sp) * (HEAD_DIM + 2);
  wp[tid] = acc;
  if (tid == 0) { wp[HEAD_DIM] = M; wp[HEAD_DIM + 1] = Ltot; }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const int prev = atomicAdd(ws_count + r * H + h, 1);
    is_last = (prev == nsp - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  const float* wb = ws_part + ((size_t)r * H + h) * nsp * (HEAD_DIM + 2);
  float Mg = -INFINITY;
  for (int s2 = 0; s2 < nsp; ++s2) Mg = fmaxf(Mg, __ldcg(wb + (size_t)s2 * (HEAD_DIM + 2) + HEAD_DIM));
  float Lg = 0.f, og = 0.f;
  for (int s2 = 0; s2 < nsp; ++s2) {
    const float ms = __ldcg(wb + (size_t)s2 * (HEAD_DIM + 2) + HEAD_DIM);
    const float f = (ms == -INFINITY) ? 0.f : expf(ms - Mg);
    Lg += __ldcg(wb + (size_t)s2 * (HEAD_DIM + 2) + HEAD_DIM + 1) * f;
    og += __ldcg(wb + (size_t)s2 * (HEAD_DIM + 2) + tid) * f;
  }
  Act<T>::st(out + oidx, og / Lg);
  if (tid == 0) ws_count[r * H + h] = 0;        // re-arm for the next launch / graph replay
}

}  // namespace pg
