// a3: prompt-prefill attention on the 5th-gen tensor cores (bf16 regime).
// Causal attention with LEFT padding: key j is visible to the query at column p iff kv_start[r] <= j <= p
// (the reference's (R, P+576) 0/1 mask + HF create_causal_mask; eager_attention_forward, HF modeling_llama.py:199-221).
//
// Masked cache columns inside the key blocks a tile walks must hold finite values: they enter P V with weight 0, and
// 0 * NaN or 0 * Inf would poison the tile.  The engine zero-fills the cache at bind and writes only bf16 results; packed
// prefill leaves pad columns holding stale (finite) K / V.
//
// One CTA = one (row, head, 128-query tile); it walks the 128-key blocks from kv_start / 128 to the tile's last query
// (up to ceil(P / 128); a scorer or x2t prompt with 576 image tokens has P of about 600-1100, so 5-9 blocks):
//   S   = Q K_blk^T      tcgen05.mma 128x128x128, fp32 in TMEM columns 0..127      (operands by TMA, SWIZZLE_128B)
//   P   = online softmax of S, one thread per query row (= TMEM lane): two passes over the row with tcgen05.ld
//         (masked max, then exp2 + running sum), written as bf16 into shared memory in the K-major swizzled
//         image the second MMA reads as its A operand
//   O_b = P V_blk        tcgen05.mma 128x128x128 into TMEM columns 128..255; V is read straight from the cache rows
//         ([key][dim], dims contiguous) as an MN-major B operand
//   O   = O * exp(m_old - m_new) + O_b   in registers (128 fp32 per thread)
// Rounding points of the reference under autocast: scores are a bf16 matmul output, scaled in bf16; softmax in
// fp32; probabilities enter the second matmul as bf16.  (The probabilities here are rounded before the final
// division by the row sum instead of after it - inside the 2e-2 tolerance of the bf16 regime.)
#pragma once
#include "lm_kernels.cuh"

namespace pg {

constexpr int PA_BQ = 128;                     // queries per CTA (MMA M)
constexpr int PA_BK = 128;                     // keys per block (MMA N of the first product, K of the second)
constexpr int PA_TILE = 128 * 64 * 2;          // one [128 rows][64 bf16] swizzled tile = 16 KB
constexpr int PA_SMEM = 6 * PA_TILE + 1024 + 64;   // Q, K (later P), V: two tiles each; 97 KB -> two CTAs per SM

__global__ void __launch_bounds__(128, 2)
attn_prefill_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                       const __grid_constant__ CUtensorMap map_v, const int32_t* __restrict__ kv_start,
                       bf16* __restrict__ out, int P, int H, int Tmax, float scale, const int32_t* __restrict__ row_off) {
  extern __shared__ uint8_t pa_smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)pa_smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;                      // 2 tiles: dims 0-63 | 64-127 of the 128 queries
  uint8_t* sK = smem + 2 * PA_TILE;        // 2 tiles: dims 0-63 | 64-127 of the 128 keys
  uint8_t* sV = smem + 4 * PA_TILE;        // 2 tiles: dims 0-63 | 64-127 of the 128 keys
  uint8_t* sP = sK;                        // probabilities (2 tiles: keys 0-63 | 64-127 of the 128 queries) overwrite the K tiles:
                                           // every thread has waited for S = Q K^T before it writes P, and the next K load is
                                           // issued only after O_b = P V has completed
  uint64_t* bars = (uint64_t*)(smem + 6 * PA_TILE);
  uint64_t* bar_load = bars;
  uint64_t* bar_mma = bars + 1;
  uint32_t* tmem_slot = (uint32_t*)(bars + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q0 = blockIdx.x * PA_BQ, h = blockIdx.y, r = blockIdx.z;
  const int HD = H * HEAD_DIM;
  pdl_launch_dependents();
  // packed stream: a duplicate row has no tokens of its own (its K / V are copied from the row it repeats).  row_off is
  // written before the first prefill kernel is launched, so reading it ahead of the dependency wait is safe.
  if (row_off != nullptr && row_off[r + 1] == row_off[r]) return;
  if (tid == 0) {
    tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_k); tma_prefetch_desc(&map_v);
    mbar_init(bar_load, 1); mbar_init(bar_mma, 1);
    mbar_fence_init();
  }
  if (warp == 0) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  const int start = kv_start[r];
  const int row = warp * 32 + lane;                 // query row within the tile = TMEM lane
  const int q = q0 + row;
  const int q_hi = min(q0 + PA_BQ - 1, P - 1);
  // row_off != nullptr: q and out hold the real tokens only, packed row after row (lm_kernels.cuh packed_row_of): column
  // q of row r is packed row row_off[r] + q - start; the (pad) columns before `start` do not exist - a tile that
  // straddles `start` loads whatever precedes the row (finite, or zeros below row 0) for them and never stores them
  const int qbase = row_off != nullptr ? row_off[r] - start : r * P;
  bf16* orow = out + (ptrdiff_t)(qbase + q) * HD + h * HEAD_DIM;
  float o[HEAD_DIM];
#pragma unroll
  for (int j = 0; j < HEAD_DIM; ++j) o[j] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;
  const float LOG2E = 1.4426950408889634f;
  const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16);

  if (q_hi >= start) {                              // otherwise every query of the tile is a pad: zeros
    const int kb_lo = start / PA_BK, kb_hi = q_hi / PA_BK;
    const uint32_t idesc = umma_idesc_bf16(PA_BQ, PA_BK);
    int it = 0;
    for (int kb = kb_lo; kb <= kb_hi; ++kb, ++it) {
      const int key0 = kb * PA_BK;
      if (tid == 0) {
        const uint64_t pol = policy_evict_first();
        mbar_expect_tx(bar_load, (it == 0 ? 2 * PA_TILE : 0) + 4 * PA_TILE);
        if (it == 0) {
          tma_load_2d(sQ, &map_q, bar_load, h * HEAD_DIM, qbase + q0, pol);
          tma_load_2d(sQ + PA_TILE, &map_q, bar_load, h * HEAD_DIM + 64, qbase + q0, pol);
        }
        const int krow = (r * H + h) * Tmax + key0;
        tma_load_2d(sK, &map_k, bar_load, 0, krow, pol);
        tma_load_2d(sK + PA_TILE, &map_k, bar_load, 64, krow, pol);
        // V rows of the cache, [128 keys][64 dims] per tile: dims 0-63 | 64-127 (MN-major B operand)
        tma_load_2d(sV, &map_v, bar_load, 0, krow, pol);
        tma_load_2d(sV + PA_TILE, &map_v, bar_load, 64, krow, pol);
        mbar_wait(bar_load, (uint32_t)(it & 1), 50);
        tc_fence_after();
        // S = Q K^T : 8 K-steps of 16 dims over the two dim tiles
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          const uint64_t da = umma_desc_k_sw128(smem_u32(sQ + (kk >> 2) * PA_TILE)) + (uint64_t)(2 * (kk & 3));
          const uint64_t db = umma_desc_k_sw128(smem_u32(sK + (kk >> 2) * PA_TILE)) + (uint64_t)(2 * (kk & 3));
          umma_bf16(tmem_base, da, db, idesc, kk != 0);
        }
        umma_commit(bar_mma);
      }
      mbar_wait(bar_mma, 0u, 51);
      tc_fence_after();
      // ---- pass 1: masked row maximum (scores as the bf16 matmul output, scaled in bf16)
      float bm = -INFINITY;
#pragma unroll 1
      for (int c0 = 0; c0 < PA_BK; c0 += 64) {            // 64 columns per TMEM round trip (common.cuh tmem_ld_32x32b_x64)
        uint32_t v[64];
        tmem_ld_32x32b_x64(t_lane + (uint32_t)c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const int key = key0 + c0 + j;
          const bool vis = key >= start && key <= q && q < P;
          const float s = bf16_round(bf16_round(__uint_as_float(v[j])) * scale);
          if (vis) bm = fmaxf(bm, s);
        }
      }
      const float m_new = fmaxf(m_run, bm);
      const float alpha = (m_new == -INFINITY) ? 1.f : exp2f((m_run - m_new) * LOG2E);
      // ---- pass 2: probabilities -> bf16 -> shared memory (A operand of the second product)
      float psum = 0.f;
      const uint32_t p_row = smem_u32(sP) + (uint32_t)row * 128;
#pragma unroll 1
      for (int c0 = 0; c0 < PA_BK; c0 += 64) {            // one P tile ([128][64 keys]) per TMEM round trip
        uint32_t v[64];
        tmem_ld_32x32b_x64(t_lane + (uint32_t)c0, v);
        tmem_ld_wait();
        const uint32_t tile = p_row + (uint32_t)(c0 >> 6) * PA_TILE;
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {                     // 16-byte chunk (8 keys) of the 128-byte row
          uint32_t pk[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float p2[2];
#pragma unroll
            for (int w = 0; w < 2; ++w) {
              const int j = cc * 8 + 2 * u + w, key = key0 + c0 + j;
              const bool vis = key >= start && key <= q && q < P;
              const float s = bf16_round(bf16_round(__uint_as_float(v[j])) * scale);
              p2[w] = vis ? exp2f((s - m_new) * LOG2E) : 0.f;
              psum += p2[w];
            }
            const __nv_bfloat162 b = __floats2bfloat162_rn(p2[0], p2[1]);
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
        // O_b = P V : 8 K-steps of 16 keys over the two key tiles
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
          const uint64_t da = umma_desc_k_sw128(smem_u32(sP + (kk >> 2) * PA_TILE)) + (uint64_t)(2 * (kk & 3));
          // MN-major V: 16 keys = 2048 bytes down each [keys][64 dims] tile, the second 64 dims one tile further
          const uint64_t db = umma_desc_mn_sw128(smem_u32(sV) + (uint32_t)kk * 2048u, (uint32_t)PA_TILE);
          umma_bf16(tmem_base + 128u, da, db, umma_idesc_bf16_bmn(PA_BQ, HEAD_DIM), kk != 0);
        }
        umma_commit(bar_mma);
      }
      mbar_wait(bar_mma, 1u, 52);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < HEAD_DIM; c0 += 64) {
        uint32_t v[64];
        tmem_ld_32x32b_x64(t_lane + 128u + (uint32_t)c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 64; ++j) o[c0 + j] = o[c0 + j] * alpha + __uint_as_float(v[j]);
      }
      tc_fence_before();
      __syncthreads();          // next block: TMA overwrites K / V, the first MMA overwrites S
    }
  }
  if (q < P && (row_off == nullptr || q >= start)) {
    const float inv = l_run > 0.f ? 1.f / l_run : 0.f;      // pad queries (nothing visible) produce zeros
#pragma unroll
    for (int j = 0; j < HEAD_DIM; j += 8) {
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

}  // namespace pg
