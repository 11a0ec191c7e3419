// Wide-tile contraction on a CTA PAIR (tcgen05 cta_group::2):  C[m][n] = sum_k X[m][k] * W[n][k]  for the tensor-bound
// shapes (prompt prefill, SigLIP tower, aligner, VQ 1x1 convolutions): token tiles of 256 rows, no split-K.
//
// Why: gemm_tc_kernel<256> tops out at 52-56 % of the tensor pipe (profiles/r02_gemm_prefill.full.txt).  At full rate one
// SM's MMAs read their A (128 x 16) and B (256 x 16) operand slices from shared memory at 96 B/clk while TMA refills the
// ring at another 96 B/clk - against a 128 B/clk shared-memory port.  Two SMs of a TPC issuing ONE 256 x 256 x 16 MMA
// between them (swap-AB: 256 weight rows x 256 tokens) each hold their own 128 weight rows (A) and only HALF of the
// token tile (B; the tensor cores fetch the other half from the peer's shared memory): per SM 32 KB instead of 48 KB per
// k-block land in shared memory, and B is read once per pair instead of once per SM.
//
// Structure per CTA (cluster of 2 along the weight-tile axis, rank 0 = leader):
//   warp 0 (one thread)  TMA producer: its A tile + its half of the token tile, 2-SM loads whose completion bytes are
//                        counted on the LEADER's full barrier (the leader alone posts the expected byte count);
//   warp 1 (one thread)  leader only: tcgen05.mma.cta_group::2, commits multicast to both CTAs' empty / accumulator
//                        barriers; both CTAs: cta_group::2 TMEM allocation;
//   warps 2-5            epilogue of the CTA's own 128 weight rows x 256 tokens (accumulator in its own TMEM): fp32
//                        partial store, or the fused row epilogues of gemm.cuh (EpiFuse); after draining a TMEM set
//                        they arrive (remotely, for the peer) on the leader's accumulator-empty barrier.
#pragma once
#include "gemm.cuh"
#include "lm_kernels.cuh"

namespace pg {

constexpr int TC2_NT = 256;                        // tokens per pair tile (MMA N)
constexpr int TC2_BHALF = (TC2_NT / 2) * TC_BK * 2;  // one CTA's half of the token tile: 16 KB
constexpr int TC2_STAGE_BYTES = TC_A_BYTES + TC2_BHALF;
constexpr uint32_t TC2_PEER_MASK = 0xFEFFFFFFu;    // clears the CTA-rank bit of a shared::cluster address: CTA 0's copy

PG_DEVINL void tma2_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & TC2_PEER_MASK), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
PG_DEVINL void umma2_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once all previously issued MMAs of this thread completed) on the barrier at this offset in BOTH CTAs of the pair
PG_DEVINL void umma2_commit_mc(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
PG_DEVINL void tmem2_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
PG_DEVINL void tmem2_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
PG_DEVINL void tmem2_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// remote arrive on the barrier at this offset in the LEADER CTA (rank 0) of the pair
PG_DEVINL void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & TC2_PEER_MASK) : "memory");
}

// Persistent: one CTA per SM, 74 pairs walk the (token tile, weight-tile pair) space; TWO accumulator sets in TMEM (2 x 256
// columns) so the epilogue of tile i (TMEM -> bias / GELU -> bf16 staging -> 256-byte row stores) overlaps the main loop of
// tile i+1, and the operand ring never drains between tiles.
constexpr int TC2_STG_BYTES = TC2_NT * 256;        // bf16 staging tile [256 tokens][128 n]
static constexpr int tc2p_smem_bytes(int stages) { return stages * TC2_STAGE_BYTES + TC2_STG_BYTES + 1024 + 256; }

constexpr int TC2_THREADS = 320;                   // producer warp, MMA warp, eight epilogue warps
constexpr int TC2_EPI = 256;                       // epilogue threads: two warps per TMEM lane quarter, 128 columns each

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC2_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x, float* __restrict__ C, int M, int N,
                int K, int num_stages, int use_pdl, Prof prof, EpiFuse ep, QkvEpi qe) {
  extern __shared__ uint8_t smem_raw2[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw2 + 1023) & ~(uintptr_t)1023);
  uint8_t* stg_buf = smem + num_stages * TC2_STAGE_BYTES;
  uint64_t* bars = (uint64_t*)(stg_buf + TC2_STG_BYTES);
  uint64_t* full_bar = bars;                       // used in the leader only
  uint64_t* empty_bar = bars + num_stages;
  uint64_t* acc_full = bars + 2 * num_stages;      // [2] both CTAs (multicast commit)
  uint64_t* acc_empty = bars + 2 * num_stages + 2; // [2] leader only: 16 arrivals (8 epilogue warps x 2 CTAs)
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * num_stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int nkb = (K + TC_BK - 1) / TC_BK;
  // tile space: weight-tile pairs vary fastest, so the pairs running at the same time share their token tile in L2
  const int pairs_x = ((N + TC_BM - 1) / TC_BM + 1) / 2, tiles_m = (M + TC2_NT - 1) / TC2_NT;
  const int n_tiles = pairs_x * tiles_m;
  const int pair_id = (int)blockIdx.x >> 1, n_pairs = (int)gridDim.x >> 1;

  if (use_pdl) pdl_launch_dependents();
  prof_begin(prof);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_w);
    tma_prefetch_desc(&map_x);
    for (int i = 0; i < num_stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], 16); mbar_init(&acc_empty[1], 16);
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem2_alloc(tmem_slot, 512);
    tmem2_relinquish();
  }
  tc_fence_before();
  cluster_sync_all();                               // barriers of both CTAs initialised before any remote completion / commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (one thread per CTA) =====================
    if (lane == 0) {
      const uint64_t pol = policy_evict_last();      // both operands are re-read by other tiles
      if (use_pdl) pdl_wait();
      int it = 0;                                    // k-blocks issued so far (ring position)
      for (int t = pair_id; t < n_tiles; t += n_pairs) {
        const int n0 = ((t % pairs_x) * 2 + (int)rank) * TC_BM, m0 = (t / pairs_x) * TC2_NT + (int)rank * (TC2_NT / 2);
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % num_stages;
          mbar_wait(&empty_bar[s], (((uint32_t)(it / num_stages)) & 1u) ^ 1u, 81);
          // the leader posts the bytes of BOTH CTAs' loads of this stage; the peer's loads count on the same barrier
          if (leader) mbar_expect_tx(&full_bar[s], 2 * TC2_STAGE_BYTES);
          tma2_load_2d(smem + s * TC2_STAGE_BYTES, &map_w, &full_bar[s], i * TC_BK, n0, pol);
          tma2_load_2d(smem + s * TC2_STAGE_BYTES + TC_A_BYTES, &map_x, &full_bar[s], i * TC_BK, m0, pol);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader only, one thread) =====================
    if (leader && lane == 0) {
      const uint32_t idesc = umma_idesc_bf16(2 * TC_BM, TC2_NT);
      int it = 0, j = 0;
      for (int t = pair_id; t < n_tiles; t += n_pairs, ++j) {
        const int set = j & 1;
        mbar_wait(&acc_empty[set], (((uint32_t)(j >> 1)) & 1u) ^ 1u, 84);   // both CTAs' epilogues drained this set (tile j - 2)
        tc_fence_after();
        for (int i = 0; i < nkb; ++i, ++it) {
          const int s = it % num_stages;
          mbar_wait(&full_bar[s], ((uint32_t)(it / num_stages)) & 1u, 82);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * TC2_STAGE_BYTES);
          const uint64_t da = umma_desc_k_sw128(a_addr);
          const uint64_t db = umma_desc_k_sw128(a_addr + TC_A_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            umma2_bf16(tmem_base + (uint32_t)(set * TC2_NT), da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (uint32_t)((i | k) != 0));
          umma2_commit_mc(&empty_bar[s]);           // frees the stage in both CTAs once these MMAs retire
        }
        umma2_commit_mc(&acc_full[set]);            // this tile's accumulators (both CTAs) complete
      }
    }
  } else {
    // ===================== epilogue: own 128 weight rows x 256 tokens per tile =====================
    const int quarter = warp & 3;                     // TMEM lanes 32 * quarter ..
    const int chalf = (warp - 2) >> 2;                // columns chalf * 128 .. + 127 of the tile
    const int tE = threadIdx.x - 64;                  // 0 .. 255 over the epilogue warps
    if (use_pdl) pdl_wait();
    int j = 0;
    for (int t = pair_id; t < n_tiles; t += n_pairs, ++j) {
      const int set = j & 1;
      const int n0 = ((t % pairs_x) * 2 + (int)rank) * TC_BM, m0 = (t / pairs_x) * TC2_NT;
      const int n = n0 + quarter * 32 + lane;
      mbar_wait(&acc_full[set], ((uint32_t)(j >> 1)) & 1u, 83);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(set * TC2_NT);
      if (ep.out != nullptr) {
        const float bias_n = (ep.bias && n < N) ? ep.bias[n] : 0.f;
        const uint32_t stg = smem_u32(stg_buf);
        const int nl = quarter * 32 + lane;
        asm volatile("bar.sync 2, 256;" ::: "memory");       // the previous tile's row stores have read the staging tile
#pragma unroll 1
        for (int c0 = chalf * 128; c0 < chalf * 128 + 128; c0 += 32) {
          uint32_t v[2][16];
          tmem_ld_32x32b_x16(taddr + (uint32_t)c0, v[0]);
          tmem_ld_32x32b_x16(taddr + (uint32_t)c0 + 16u, v[1]);
          tmem_ld_wait();
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              float x = bf16_round(__uint_as_float(v[h2][q]) + bias_n);
              if (ep.gelu == 1) x = x * 0.5f * (1.0f + erf_fast(x * 0.70710678118654752440f));
              const unsigned short hb = __bfloat16_as_ushort(__float2bfloat16_rn(x));
              asm volatile("st.shared.u16 [%0], %1;" ::"r"(stg + (uint32_t)((c0 + h2 * 16 + q) * 256 + nl * 2)), "h"(hb) : "memory");
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&acc_empty[set]);   // TMEM set drained: the issuer may start tile j + 2 into it
        asm volatile("bar.sync 2, 256;" ::: "memory");
        if (ep.gelu == 3) {
          // prefill QKV (QkvEpi, gemm.cuh): this tile is head h of q (which = 0), k (1) or v (2) for 256 tokens
          const int c8 = tE & 7, rr0 = tE >> 3, tile = n0 / TC_BM, which = tile / qe.H, h = tile % qe.H;
          if (n0 < N) {
#pragma unroll 1
            for (int r = rr0; r < TC2_NT; r += 32) {
              const int m = m0 + r;
              if (m >= M) continue;
              int rw, p;
              if (qe.row_off != nullptr) {
                rw = packed_row_of(qe.row_off, qe.R, m);
                p = qe.kv_start[rw] + (m - qe.row_off[rw]);
              } else {
                rw = m / qe.P; p = m % qe.P;
              }
              uint32_t lo[4], hi[4];
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo[0]), "=r"(lo[1]), "=r"(lo[2]), "=r"(lo[3])
                           : "r"(stg + (uint32_t)(r * 256 + c8 * 16)));
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(hi[0]), "=r"(hi[1]), "=r"(hi[2]), "=r"(hi[3])
                           : "r"(stg + (uint32_t)(r * 256 + 128 + c8 * 16)));
              const size_t cidx = (((size_t)rw * qe.H + h) * qe.Tmax + p) * HEAD_DIM + c8 * 8;
              if (which == 2) {
                *reinterpret_cast<uint4*>(qe.vcache + cidx) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                *reinterpret_cast<uint4*>(qe.vcache + cidx + 64) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
              } else {
                const int pr = qe.rope_start ? max(p - qe.rope_start[rw], 0) : p;
                const float4* c4 = reinterpret_cast<const float4*>(qe.cosT + (size_t)pr * 64 + c8 * 8);
                const float4* s4 = reinterpret_cast<const float4*>(qe.sinT + (size_t)pr * 64 + c8 * 8);
                const float4 ca = c4[0], cb = c4[1], sa = s4[0], sb = s4[1];
                const float cs[8] = {ca.x, ca.y, ca.z, ca.w, cb.x, cb.y, cb.z, cb.w};
                const float sn[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
                uint32_t oa[4], ob[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  float a0, b0, a1, b1;
                  rope_pair<bf16>(bf16lo(lo[u]), bf16lo(hi[u]), cs[2 * u], sn[2 * u], false, a0, b0);
                  rope_pair<bf16>(bf16hi(lo[u]), bf16hi(hi[u]), cs[2 * u + 1], sn[2 * u + 1], false, a1, b1);
                  const __nv_bfloat162 xa = __floats2bfloat162_rn(a0, a1), xb = __floats2bfloat162_rn(b0, b1);
                  oa[u] = *reinterpret_cast<const uint32_t*>(&xa); ob[u] = *reinterpret_cast<const uint32_t*>(&xb);
                }
                bf16* dst = which == 0 ? qe.q_out + (size_t)m * (qe.H * HEAD_DIM) + h * HEAD_DIM + c8 * 8 : qe.kcache + cidx;
                *reinterpret_cast<uint4*>(dst) = make_uint4(oa[0], oa[1], oa[2], oa[3]);
                *reinterpret_cast<uint4*>(dst + 64) = make_uint4(ob[0], ob[1], ob[2], ob[3]);
              }
            }
          }
          continue;
        }
        if (ep.gelu == 2) {
          // SwiGLU (prefill gate|up): the tile's 128 weight rows are gate(f0 .. f0+63) | up(f0 .. f0+63) (rows interleaved in
          // blocks of 64, weights.py), so a staged token row holds g in bytes 0-127 and u in bytes 128-255:
          // h = rnd(rnd(silu(g)) * u), 64 values = 128 bytes per token into out [M][N / 2]  (values identical to swiglu_kernel<bf16>)
          const int c8 = tE & 7, rr0 = tE >> 3, F = N >> 1, f0 = (n0 / TC_BM) * 64;
          if (n0 < N) {
#pragma unroll 2
            for (int r = rr0; r < TC2_NT; r += 32) {
              const size_t m = (size_t)m0 + r;
              if (m < (size_t)M) {
                uint32_t gw[4], uw[4], ow[4];
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(gw[0]), "=r"(gw[1]), "=r"(gw[2]), "=r"(gw[3])
                             : "r"(stg + (uint32_t)(r * 256 + c8 * 16)));
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(uw[0]), "=r"(uw[1]), "=r"(uw[2]), "=r"(uw[3])
                             : "r"(stg + (uint32_t)(r * 256 + 128 + c8 * 16)));
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const float g0 = bf16lo(gw[u]), g1 = bf16hi(gw[u]), u0 = bf16lo(uw[u]), u1 = bf16hi(uw[u]);
                  const float h0 = bf16_round(g0 / (1.0f + expf(-g0))) * u0, h1 = bf16_round(g1 / (1.0f + expf(-g1))) * u1;
                  const __nv_bfloat162 o = __floats2bfloat162_rn(h0, h1);
                  ow[u] = *reinterpret_cast<const uint32_t*>(&o);
                }
                *reinterpret_cast<uint4*>(ep.out + m * F + f0 + c8 * 8) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
              }
            }
          }
          continue;
        }
        const int ch = tE & 15, r0 = tE >> 4;
        if (n0 + ch * 8 < N) {
#pragma unroll 4
          for (int r = r0; r < TC2_NT; r += 16) {
            const size_t m = (size_t)m0 + r;
            if (m < (size_t)M) {
              uint4 q;
              asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w)
                           : "r"(stg + (uint32_t)(r * 256 + ch * 16)));
              if (ep.add16 != nullptr) {
                const uint4 a = *reinterpret_cast<const uint4*>(ep.add16 + m * N + n0 + ch * 8);
                uint32_t qs[4] = {q.x, q.y, q.z, q.w};
                const uint32_t as[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const __nv_bfloat162 o = __floats2bfloat162_rn(bf16lo(qs[u]) + bf16lo(as[u]), bf16hi(qs[u]) + bf16hi(as[u]));
                  qs[u] = *reinterpret_cast<const uint32_t*>(&o);
                }
                q = make_uint4(qs[0], qs[1], qs[2], qs[3]);
              }
              *reinterpret_cast<uint4*>(ep.out + m * N + n0 + ch * 8) = q;
            }
          }
        }
      } else {
        const float bias_n = (ep.bias && n < N) ? ep.bias[n] : 0.f;
#pragma unroll 1
        for (int c0 = chalf * 128; c0 < chalf * 128 + 128; c0 += 16) {
          uint32_t v[16];
          tmem_ld_32x32b_x16(taddr + (uint32_t)c0, v);
          tmem_ld_wait();
          if (c0 + 16 >= chalf * 128 + 128) {                    // this warp's last TMEM read of the tile
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(&acc_empty[set]);
          }
          if (n < N) {
            if (ep.resid != nullptr) {
              float xo[16];
#pragma unroll
              for (int q = 0; q < 16; ++q) {
                const int m = m0 + c0 + q;
                xo[q] = (m < M) ? ep.resid[(size_t)m * N + n] : 0.f;
              }
#pragma unroll
              for (int q = 0; q < 16; ++q) {
                const int m = m0 + c0 + q;
                if (m < M) ep.resid[(size_t)m * N + n] = xo[q] + bf16_round(__uint_as_float(v[q]) + bias_n);
              }
            } else {
#pragma unroll
              for (int q = 0; q < 16; ++q) {
                const int m = m0 + c0 + q;
                if (m < M) C[(size_t)m * N + n] = __uint_as_float(v[q]);
              }
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();                               // nobody leaves (or frees TMEM) while the pair can still touch it
  prof_end(prof);
  if (warp == 1) tmem2_dealloc(tmem_base, 512);
}

}  // namespace pg
