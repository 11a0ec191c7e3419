// mmu front-end (SURVEY.md 8f rank 2): SigLIP vision tower + understanding aligner + embedding scatter.
//   CLIPVisionTower.forward (three_party/Janus/janus/models/clip_encoder.py:107-122) ->
//   VisionTransformer.forward_features / forward (siglip_vit.py:562-591): PatchEmbed (conv p/p) + learned pos-emb,
//   `layers` x Block (:209-256) [x += proj(SDPA(qkv(LN1 x))) (Attention :136-191); x += fc2(GELU(fc1(LN2 x)))],
//   final LayerNorm; aligner = MlpProjector mlp_gelu (projector.py:39-45);
//   MultiModalityCausalLM.prepare_inputs_embeds (modeling_vlm.py:221-268): scatter into the text embeddings.
// Row kernels around the contractions of gemm.cuh; T = bf16 reproduces the reference's autocast regime
// (`images.bfloat16()` :249, Linear / conv / SDPA in bf16, LayerNorm and residual stream in fp32), T = float is the
// fp32 check mode.  The attention of the bf16 regime runs on tcgen05 (vit_attn_tc_kernel).
#pragma once
#include "lm_kernels.cuh"

namespace pg {

// ---------------------------------------------------------------- PatchEmbed: im2col of non-overlapping patches
// pixel fp32 [n_img][3][S][S] -> col T [n_img * (S/p)^2][3*p*p], k = c*p*p + ky*p + kx  (= the flattened conv weight
// [width][3][p][p]); `images.bfloat16()` is the rounding to T.
template <typename T>
__global__ void __launch_bounds__(256)
vit_patchify_kernel(const float* __restrict__ pix, T* __restrict__ col, int S, int p, size_t total4) {
  pdl_launch_dependents();
  pdl_wait();
  const int g = S / p, K = 3 * p * p;
  for (size_t i4 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i4 < total4; i4 += (size_t)gridDim.x * blockDim.x) {
    const size_t i = i4 * 4;
    const size_t m = i / K;
    const int k = (int)(i - m * K);
    const int c = k / (p * p), ky = (k - c * p * p) / p, kx = k % p;
    const size_t img = m / (g * g);
    const int pi = (int)(m - img * g * g), py = pi / g, px = pi % g;
    const float4 v = *reinterpret_cast<const float4*>(pix + ((img * 3 + c) * S + (size_t)(py * p + ky)) * S + px * p + kx);
    T* dst = col + i;
    Act<T>::st(dst, v.x); Act<T>::st(dst + 1, v.y); Act<T>::st(dst + 2, v.z); Act<T>::st(dst + 3, v.w);
  }
}

// x[m][n] = rnd(sum_s part + bias[n]) + pos[m % NP][n]      (conv output in T, position embedding added in fp32)
template <typename T>
__global__ void __launch_bounds__(256)
vit_patch_epilogue_kernel(const float* __restrict__ part, int S, size_t split_stride, const float* __restrict__ bias,
                          const float* __restrict__ pos, float* __restrict__ x, int C, int NP, size_t total) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t m = i / C;
    const int n = (int)(i - m * C);
    const float v = Act<T>::rnd(reduce_splits(part, S, split_stride, i) + bias[n]);
    x[i] = v + pos[(m % NP) * C + n];
  }
}

// ---------------------------------------------------------------- residual add + LayerNorm (eps 1e-6, affine)
// x[m] += rnd(sum_s part[m] + bias)   (part == nullptr: no update);   xn[m] = T(LN(x[m]) * w + b)
// One CTA per row, values in registers (C <= 4 * 4 * blockDim), two-pass mean / variance in fp32 like torch.
constexpr int LN_THREADS = 256;
constexpr int LN_MAXQ = 4;         // float4 per thread
template <typename T>
__global__ void __launch_bounds__(LN_THREADS)
vit_resid_ln_kernel(float* __restrict__ x, const float* __restrict__ part, int S, size_t split_stride,
                    const float* __restrict__ bias, const float* __restrict__ w, const float* __restrict__ b,
                    T* __restrict__ xn_out, int C, float eps) {
  __shared__ float red[32];
  pdl_launch_dependents();
  pdl_wait();
  const size_t row = blockIdx.x;
  float* xr = x + row * C;
  float4 v[LN_MAXQ];
  float sum = 0.f;
#pragma unroll
  for (int q = 0; q < LN_MAXQ; ++q) {
    const int d = 4 * (threadIdx.x + q * LN_THREADS);
    v[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d < C) {
      v[q] = *reinterpret_cast<const float4*>(xr + d);
      if (part != nullptr) {
        float a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = Act<T>::rnd(reduce_splits(part, S, split_stride, row * C + d + j) + bias[d + j]);
        v[q].x += a[0]; v[q].y += a[1]; v[q].z += a[2]; v[q].w += a[3];
        *reinterpret_cast<float4*>(xr + d) = v[q];
      }
      sum += (v[q].x + v[q].y) + (v[q].z + v[q].w);
    }
  }
  const float mean = block_sum(sum, red) / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int q = 0; q < LN_MAXQ; ++q) {
    const int d = 4 * (threadIdx.x + q * LN_THREADS);
    if (d < C) {
      const float a = v[q].x - mean, bq = v[q].y - mean, c = v[q].z - mean, e = v[q].w - mean;
      sq += (a * a + bq * bq) + (c * c + e * e);
    }
  }
  const float rstd = rsqrtf(block_sum(sq, red) / (float)C + eps);
  if (xn_out == nullptr) return;
#pragma unroll
  for (int q = 0; q < LN_MAXQ; ++q) {
    const int d = 4 * (threadIdx.x + q * LN_THREADS);
    if (d < C) {
      const float4 wv = *reinterpret_cast<const float4*>(w + d), bv = *reinterpret_cast<const float4*>(b + d);
      T* dst = xn_out + row * C + d;
      Act<T>::st(dst, (v[q].x - mean) * rstd * wv.x + bv.x);
      Act<T>::st(dst + 1, (v[q].y - mean) * rstd * wv.y + bv.y);
      Act<T>::st(dst + 2, (v[q].z - mean) * rstd * wv.z + bv.z);
      Act<T>::st(dst + 3, (v[q].w - mean) * rstd * wv.w + bv.w);
    }
  }
}

// Warp-per-row variant for C <= 1024 (SigLIP-L: C = 1024): eight rows per CTA, the row in 8 float4 per lane, reductions by
// shuffles only - no block barrier.  The one-CTA-per-row kernel above moved 113 MB in 78 us (1.45 TB/s: latency of two
// block reductions per tiny CTA); same arithmetic (two-pass mean / variance), different summation tree.
constexpr int LNW_MAXQ = 8;
template <typename T>
__global__ void __launch_bounds__(256)
vit_resid_ln_warp_kernel(float* __restrict__ x, const float* __restrict__ part, int S, size_t split_stride,
                         const float* __restrict__ bias, const float* __restrict__ w, const float* __restrict__ b,
                         T* __restrict__ xn_out, int C, float eps, int rows) {
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31;
  const size_t row = (size_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  // the affine parameters are constants: fetched before the dependency wait, all loads of the row in flight together
  float4 wv[LNW_MAXQ], bv[LNW_MAXQ];
#pragma unroll
  for (int q = 0; q < LNW_MAXQ; ++q) {
    const int d = 4 * (lane + 32 * q);
    wv[q] = bv[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (d < C && xn_out != nullptr) { wv[q] = *reinterpret_cast<const float4*>(w + d); bv[q] = *reinterpret_cast<const float4*>(b + d); }
  }
  pdl_wait();
  if (row >= (size_t)rows) return;
  float* xr = x + row * C;
  float4 v[LNW_MAXQ];
#pragma unroll
  for (int q = 0; q < LNW_MAXQ; ++q) {
    const int d = 4 * (lane + 32 * q);
    v[q] = (d < C) ? __ldcs(reinterpret_cast<const float4*>(xr + d)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float sum = 0.f;
#pragma unroll
  for (int q = 0; q < LNW_MAXQ; ++q) {
    const int d = 4 * (lane + 32 * q);
    if (d < C) {
      if (part != nullptr) {
        float a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = Act<T>::rnd(reduce_splits(part, S, split_stride, row * C + d + j) + bias[d + j]);
        v[q].x += a[0]; v[q].y += a[1]; v[q].z += a[2]; v[q].w += a[3];
        *reinterpret_cast<float4*>(xr + d) = v[q];
      }
      sum += (v[q].x + v[q].y) + (v[q].z + v[q].w);
    }
  }
  const float mean = warp_sum(sum) / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int q = 0; q < LNW_MAXQ; ++q) {
    const int d = 4 * (lane + 32 * q);
    if (d < C) {
      const float a = v[q].x - mean, bq = v[q].y - mean, c = v[q].z - mean, e = v[q].w - mean;
      sq += (a * a + bq * bq) + (c * c + e * e);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)C + eps);
  if (xn_out == nullptr) return;
#pragma unroll
  for (int q = 0; q < LNW_MAXQ; ++q) {
    const int d = 4 * (lane + 32 * q);
    if (d < C) {
      T* dst = xn_out + row * C + d;
      const float y0 = (v[q].x - mean) * rstd * wv[q].x + bv[q].x, y1 = (v[q].y - mean) * rstd * wv[q].y + bv[q].y;
      const float y2 = (v[q].z - mean) * rstd * wv[q].z + bv[q].z, y3 = (v[q].w - mean) * rstd * wv[q].w + bv[q].w;
      if constexpr (sizeof(T) == 2) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(y0, y1), hi = __floats2bfloat162_rn(y2, y3);
        uint2 pk; pk.x = *reinterpret_cast<const uint32_t*>(&lo); pk.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(dst) = pk;
      } else {
        *reinterpret_cast<float4*>(dst) = make_float4(y0, y1, y2, y3);
      }
    }
  }
}

// ---------------------------------------------------------------- attention, CUDA cores (fp32 check mode / fallback)
// F.scaled_dot_product_attention(q, k, v) without mask (siglip_vit.py:176): one warp per query, the whole score row
// in registers (NP <= 32 * VA_MAXI keys), exact two-pass softmax in fp32.
constexpr int VA_MAXI = 32;
template <typename T>
__global__ void __launch_bounds__(128)
vit_attn_kernel(const T* __restrict__ qkv, T* __restrict__ out, int NP, int W, int heads, int hd, float scale) {
  __shared__ float qs[4][128];
  pdl_launch_dependents();
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 4 + warp, h = blockIdx.y, img = blockIdx.z;
  if (qi >= NP) return;
  const T* base = qkv + (size_t)img * NP * 3 * W;
  for (int d = lane; d < hd; d += 32) qs[warp][d] = Act<T>::ld(base + (size_t)qi * 3 * W + h * hd + d);
  __syncwarp();
  float s[VA_MAXI];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < VA_MAXI; ++i) {
    const int j = lane + 32 * i;
    s[i] = -INFINITY;
    if (j < NP) {
      const T* kr = base + (size_t)j * 3 * W + W + h * hd;
      float a = 0.f;
      for (int d = 0; d < hd; ++d) a = fmaf(qs[warp][d], Act<T>::ld(kr + d), a);
      s[i] = Act<T>::rnd(a) * scale;
      mx = fmaxf(mx, s[i]);
    }
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < VA_MAXI; ++i) {
    s[i] = (lane + 32 * i < NP) ? expf(s[i] - mx) : 0.f;
    sum += s[i];
  }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  float o[4] = {0.f, 0.f, 0.f, 0.f};                          // dims lane, lane + 32, ... (hd <= 128)
#pragma unroll
  for (int i = 0; i < VA_MAXI; ++i) {
    if (32 * i >= NP) break;
    for (int l = 0; l < 32; ++l) {
      const int j = l + 32 * i;
      if (j >= NP) break;
      const float p = Act<T>::rnd(__shfl_sync(0xffffffffu, s[i], l) * inv);
      const T* vr = base + (size_t)j * 3 * W + 2 * W + h * hd;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int d = lane + 32 * u;
        if (d < hd) o[u] = fmaf(p, Act<T>::ld(vr + d), o[u]);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int d = lane + 32 * u;
    if (d < hd) Act<T>::st(out + ((size_t)img * NP + qi) * W + h * hd + d, o[u]);
  }
}

// ---------------------------------------------------------------- attention on tcgen05 (bf16 regime, head_dim 64)
// One CTA = one (image, head, 128-query tile); it walks the key blocks of VT_BK keys:
//   S   = Q K_blk^T      tcgen05.mma 128 x VT_BK x 64, fp32 in TMEM columns 0 .. VT_BK-1    (operands by TMA, SWIZZLE_128B)
//   P   = online softmax of S, one thread per query row (= TMEM lane), two tcgen05.ld passes (row maximum, then
//         exp2 + running sum), written as bf16 into shared memory in the K-major swizzled image the second MMA
//         reads as its A operand - over the K tile, which is dead once S is complete
//   O_b = P V_blk        tcgen05.mma 128 x 64 x VT_BK into TMEM columns VT_BK .. VT_BK+63; V is taken straight from
//         the qkv rows ([key][64 dims], one TMA box) as an MN-major B operand
//   O   = O * exp(m_old - m_new) + O_b   in registers (64 fp32 per thread)
// Scores stay fp32 (fused SDPA kernels do not round them), probabilities enter the second product as bf16.
// 88 KB of shared memory and 256 TMEM columns per CTA: two CTAs per SM overlap each other's load / MMA / softmax phases.
constexpr int VT_BQ = 128;
constexpr int VT_BK = 192;
constexpr int VT_HD = 64;
constexpr int VT_QTILE = VT_BQ * 64 * 2;        // 16 KB
constexpr int VT_KTILE = VT_BK * 64 * 2;        // 24 KB
constexpr int VT_PTILE = VT_BQ * 64 * 2;        // one [128][64] tile of P, VT_BK / 64 of them
constexpr int VT_VTILE = VT_BK * 64 * 2;        // V tile [VT_BK keys][64 dims] (24 KB)
constexpr int VT_KP_BYTES = (VT_BK / 64) * VT_PTILE;          // K tile, later the P tiles (48 KB)
constexpr int VT_SMEM = VT_QTILE + VT_KP_BYTES + VT_VTILE + 1024 + 64;

__global__ void __launch_bounds__(128, 2)
vit_attn_tc_kernel(const __grid_constant__ CUtensorMap map_qk, const __grid_constant__ CUtensorMap map_k,
                   bf16* __restrict__ out, int NP, int W, float scale) {
  extern __shared__ uint8_t vt_smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)vt_smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;
  uint8_t* sK = smem + VT_QTILE;                 // K tile [VT_BK][64]; overwritten by P [128][VT_BK] (3 tiles)
  uint8_t* sP = sK;
  uint8_t* sV = sK + VT_KP_BYTES;                // V tile [VT_BK keys][64 dims]
  uint64_t* bars = (uint64_t*)(sV + VT_VTILE);
  uint64_t* bar_load = bars;
  uint64_t* bar_mma = bars + 1;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q0 = blockIdx.x * VT_BQ, h = blockIdx.y, img = blockIdx.z;
  pdl_launch_dependents();
  if (tid == 0) {
    tma_prefetch_desc(&map_qk); tma_prefetch_desc(&map_k);
    mbar_init(bar_load, 1); mbar_init(bar_mma, 1);
    mbar_fence_init();
  }
  if (warp == 0) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  const int row = warp * 32 + lane;                 // query row within the tile = TMEM lane
  const int q = q0 + row;
  float o[VT_HD];
#pragma unroll
  for (int j = 0; j < VT_HD; ++j) o[j] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;
  const float sl2 = scale * 1.4426950408889634f;     // scores in log2 units
  const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16);
  const uint32_t idesc_s = umma_idesc_bf16(VT_BQ, VT_BK);
  const uint32_t idesc_o = umma_idesc_bf16_bmn(VT_BQ, VT_HD);
  const int nkb = (NP + VT_BK - 1) / VT_BK;
  for (int kb = 0; kb < nkb; ++kb) {
    const int key0 = kb * VT_BK;
    if (tid == 0) {
      const uint64_t pol = policy_evict_first();
      mbar_expect_tx(bar_load, (kb == 0 ? VT_QTILE : 0) + VT_KTILE + VT_VTILE);
      if (kb == 0) tma_load_2d(sQ, &map_qk, bar_load, h * VT_HD, img * NP + q0, pol);
      tma_load_2d(sK, &map_k, bar_load, W + h * VT_HD, img * NP + key0, pol);
      tma_load_2d(sV, &map_k, bar_load, 2 * W + h * VT_HD, img * NP + key0, pol);
      mbar_wait(bar_load, (uint32_t)(kb & 1), 60);
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < VT_HD / 16; ++kk)
        umma_bf16(tmem_base, umma_desc_k_sw128(smem_u32(sQ)) + (uint64_t)(2 * kk), umma_desc_k_sw128(smem_u32(sK)) + (uint64_t)(2 * kk),
                  idesc_s, kk != 0);
      umma_commit(bar_mma);
    }
    mbar_wait(bar_mma, 0u, 61);
    tc_fence_after();
    // ---- pass 1: row maximum over the valid keys of the block
    float bm = -INFINITY;
#pragma unroll 1
    for (int c0 = 0; c0 < VT_BK; c0 += 64) {             // 64 columns per TMEM round trip (see tmem_ld_32x32b_x64)
      uint32_t v[64];
      tmem_ld_32x32b_x64(t_lane + (uint32_t)c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 64; ++j)
        if (key0 + c0 + j < NP) bm = fmaxf(bm, __uint_as_float(v[j]));
    }
    bm *= sl2;
    const float m_new = fmaxf(m_run, bm);
    const float alpha = exp2f(m_run - m_new);          // first block: exp2(-inf) = 0
    // ---- pass 2: probabilities -> bf16 -> shared memory (A operand of the second product), over the K tile
    float psum = 0.f;
    const uint32_t p_row = smem_u32(sP) + (uint32_t)row * 128;
#pragma unroll 1
    for (int c0 = 0; c0 < VT_BK; c0 += 64) {             // one P tile ([128][64 keys]) per TMEM round trip
      uint32_t v[64];
      tmem_ld_32x32b_x64(t_lane + (uint32_t)c0, v);
      tmem_ld_wait();
      const uint32_t tile = p_row + (uint32_t)(c0 >> 6) * VT_PTILE;
#pragma unroll
      for (int cc = 0; cc < 8; ++cc) {                     // 16-byte chunk (8 keys) of the 128-byte row
        uint32_t pk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = cc * 8 + 2 * u;
          const float p0 = (key0 + c0 + j < NP) ? exp2f(fmaf(__uint_as_float(v[j]), sl2, -m_new)) : 0.f;
          const float p1 = (key0 + c0 + j + 1 < NP) ? exp2f(fmaf(__uint_as_float(v[j + 1]), sl2, -m_new)) : 0.f;
          psum += p0; psum += p1;
          const __nv_bfloat162 b = __floats2bfloat162_rn(p0, p1);
          pk[u] = *reinterpret_cast<const uint32_t*>(&b);
        }
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(tile + (uint32_t)((cc ^ (row & 7)) << 4)),
                     "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
      }
    }
    l_run = l_run * alpha + psum;
    m_run = m_new;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < VT_BK / 16; ++kk)
        umma_bf16(tmem_base + (uint32_t)VT_BK, umma_desc_k_sw128(smem_u32(sP + (kk >> 2) * VT_PTILE)) + (uint64_t)(2 * (kk & 3)),
                  umma_desc_mn_sw128(smem_u32(sV) + (uint32_t)kk * 2048u, 1024u),
                  idesc_o, kk != 0);
      umma_commit(bar_mma);
    }
    mbar_wait(bar_mma, 1u, 62);
    tc_fence_after();
    {
      uint32_t v[64];
      tmem_ld_32x32b_x64(t_lane + (uint32_t)VT_BK, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < VT_HD; ++j) o[j] = o[j] * alpha + __uint_as_float(v[j]);
    }
    tc_fence_before();
    __syncthreads();          // next block: TMA overwrites K (= P) / V, the first MMA overwrites S
  }
  if (q < NP) {
    const float inv = 1.f / l_run;
    bf16* orow = out + ((size_t)img * NP + q) * W + h * VT_HD;
#pragma unroll
    for (int j = 0; j < VT_HD; j += 8) {
      uint32_t pk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(o[j + 2 * u] * inv, o[j + 2 * u + 1] * inv);
        pk[u] = *reinterpret_cast<const uint32_t*>(&b);
      }
      *reinterpret_cast<uint4*>(orow + j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 256);
}

// ---------------------------------------------------------------- scatter into the text embeddings
// inputs_embeds[images_seq_mask] = images_embeds[images_emb_mask]   (modeling_vlm.py:266): the k-th set position of
// the sequence mask (row-major over [b][T]) receives the k-th selected image token (row-major over [b][n * t]).
// One CTA: exclusive ranks of a 0/1 byte mask; rank[i] = -1 where the mask is 0; inv[rank] = i (optional); *count.
__global__ void __launch_bounds__(1024)
mask_rank_kernel(const uint8_t* __restrict__ mask, int n, int32_t* __restrict__ rank, int32_t* __restrict__ inv,
                 int32_t* __restrict__ count) {
  __shared__ int wsum[32];
  __shared__ int carry_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + tid;
    const int f = (i < n && mask[i] != 0) ? 1 : 0;
    int incl = f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const int w = wsum[lane];
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
      }
      wsum[lane] = wi - w;                                 // exclusive prefix over the 32 warps
    }
    __syncthreads();
    const int r = carry_s + wsum[warp] + incl - f;         // exclusive rank of element i
    if (i < n) {
      if (rank) rank[i] = f ? r : -1;
      if (f && inv) inv[r] = i;
    }
    __syncthreads();
    if (tid == 1023) carry_s = r + f;                       // set elements up to the end of this chunk
    __syncthreads();
  }
  if (tid == 0) *count = carry_s;
}

// out[p] = seq-masked ? feat[inv_src[rank_dst[p]]] (T -> fp32) : embed_tokens[max(id, 0)]
template <typename T>
__global__ void __launch_bounds__(256)
embed_scatter_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ rank_dst, const int32_t* __restrict__ inv_src,
                     const int32_t* __restrict__ n_src, const T* __restrict__ feat, const float* __restrict__ table,
                     float* __restrict__ out, int D, int vocab) {
  pdl_launch_dependents();
  pdl_wait();
  const int p = blockIdx.x;
  const int r = rank_dst[p];
  float4* dst = reinterpret_cast<float4*>(out + (size_t)p * D);
  if (r >= 0 && r < *n_src) {
    const T* src = feat + (size_t)inv_src[r] * D;
    for (int i = threadIdx.x; i < D / 4; i += blockDim.x)
      dst[i] = make_float4(Act<T>::ld(src + 4 * i), Act<T>::ld(src + 4 * i + 1), Act<T>::ld(src + 4 * i + 2), Act<T>::ld(src + 4 * i + 3));
  } else {
    const int id = min(max(ids[p], 0), vocab - 1);          // `input_ids[input_ids < 0] = 0` (:260)
    const float4* src = reinterpret_cast<const float4*>(table + (size_t)id * D);
    for (int i = threadIdx.x; i < D / 4; i += blockDim.x) dst[i] = src[i];
  }
}

template <typename T>
__global__ void __launch_bounds__(256) to_f32_kernel(const T* __restrict__ in, float* __restrict__ out, size_t n) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) out[i] = Act<T>::ld(in + i);
}

}  // namespace pg
