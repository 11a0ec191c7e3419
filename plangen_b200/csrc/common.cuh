// Common device helpers for the sm_100a kernels: mbarrier / TMA / tcgen05 / PDL PTX
// wrappers, bf16 conversion and small reductions.  No torch, no CUTLASS.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define PG_DEVINL __device__ __forceinline__

namespace pg {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------- type helpers
template <typename T> struct Act;
template <> struct Act<float> {
  static PG_DEVINL float ld(const float* p) { return *p; }
  static PG_DEVINL void st(float* p, float v) { *p = v; }
  static PG_DEVINL float rnd(float v) { return v; }          // rounding to the activation type
};
template <> struct Act<bf16> {
  static PG_DEVINL float ld(const bf16* p) { return __bfloat162float(*p); }
  static PG_DEVINL void st(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
  static PG_DEVINL float rnd(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

PG_DEVINL float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
PG_DEVINL float bf16lo(uint32_t u) { return __uint_as_float(u << 16); }
PG_DEVINL float bf16hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

PG_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
PG_DEVINL float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum; `red` is >= 32 floats of shared memory; all threads get the result
PG_DEVINL float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}
PG_DEVINL float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : -INFINITY;
  r = warp_max(r);
  return r;
}

// ------------------------------------------------------ programmatic dependent launch
// griddepcontrol.wait: block until every prerequisite grid has completed and its
// memory is visible.  launch_dependents: allow the next kernel in the stream to start
// its prologue (weight prefetch) while this one is still running.
PG_DEVINL void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
PG_DEVINL void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------- mbarrier
PG_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

PG_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
PG_DEVINL void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
PG_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
PG_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
PG_DEVINL bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
PG_DEVINL uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Bounded spin: a protocol bug must surface as a trapped kernel (an error the host sees), never as a
// hung GPU.  `tag` identifies the wait site in the diagnostic.
PG_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity, int tag = 0, int info = 0) {
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3FFFu) == 0) {                       // look at the clock only every 16K failed polls
      const uint64_t now = global_timer_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) {
        if ((threadIdx.x & 31) == 0)
          printf("plangen_b200: mbarrier wait timed out (site %d, block %d,%d,%d thread %d parity %u info %d)\n", tag,
                 blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, parity, info);
        __trap();
      }
    }
  }
}

// Optional in-situ timeline: every CTA stamps kernel begin (min) into buf[slot] and end (max) into
// buf[PROF_SLOTS + slot]; buf[2*PROF_SLOTS ..] receives a snapshot after the profiled step.
constexpr int PROF_SLOTS = 256;
struct Prof { unsigned long long* buf; int slot; };
PG_DEVINL void prof_begin(const Prof& p) {
  if (p.buf && threadIdx.x == 0) atomicMin(&p.buf[p.slot], (unsigned long long)global_timer_ns());
}
PG_DEVINL void prof_end(const Prof& p) {
  if (p.buf && threadIdx.x == 0) atomicMax(&p.buf[PROF_SLOTS + p.slot], (unsigned long long)global_timer_ns());
}

// ------------------------------------------------------------------------------ thread-block clusters
PG_DEVINL uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
PG_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// read a 32-bit word of CTA `rank`'s copy of a shared-memory variable
PG_DEVINL uint32_t dsmem_ld_u32(const void* my_smem_ptr, uint32_t rank) {
  uint32_t remote, v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(my_smem_ptr)), "r"(rank));
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(remote) : "memory");
  return v;
}
PG_DEVINL uint64_t dsmem_ld_u64(const void* my_smem_ptr, uint32_t rank) {
  uint32_t remote;
  uint64_t v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(my_smem_ptr)), "r"(rank));
  asm volatile("ld.shared::cluster.u64 %0, [%1];" : "=l"(v) : "r"(remote) : "memory");
  return v;
}


// generic-proxy writes (st.shared) made visible to the async proxy (TMA / tcgen05)
PG_DEVINL void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------ TMA
PG_DEVINL void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// L2 cache policies
PG_DEVINL uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
PG_DEVINL uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
PG_DEVINL void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
PG_DEVINL void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                           uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
PG_DEVINL void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3,
                           uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(policy)
      : "memory");
}

// contiguous global -> shared bulk copy (TMA, no tensor map), completion on an mbarrier
PG_DEVINL void bulk_copy_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

// --------------------------------------------------------------------------- tcgen05
PG_DEVINL bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
PG_DEVINL void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
PG_DEVINL void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory"); }
PG_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // one full warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
PG_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
PG_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> fp32, issued by ONE thread
PG_DEVINL void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread completed
PG_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
PG_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp gets lane (base_lane + i)
PG_DEVINL void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 64 consecutive fp32 columns in ONE instruction: a tcgen05.ld round trip costs ~150 ns whatever its width, so
// row-wise passes over an accumulator (softmax) should use few wide loads rather than many x16 loads with a wait each
PG_DEVINL void tmem_ld_32x32b_x64(uint32_t taddr, uint32_t (&v)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,"
      "%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]),
        "=r"(v[30]), "=r"(v[31]), "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]),
        "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]),
        "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]),
        "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
      : "r"(taddr)
      : "memory");
}

// Shared-memory matrix descriptor for a K-major bf16 operand tile written by TMA with
// SWIZZLE_128B: rows of 64 bf16 (128 B), 8-row groups 1024 B apart.
//   start address >> 4 | LBO (ignored for swizzled K-major; 1) << 16 | SBO (1024 B >> 4) << 32
//   | version 1 << 46 | layout SWIZZLE_128B (2) << 61
PG_DEVINL uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major operand tile, SWIZZLE_128B: rows are K indices, 128 bytes (64 bf16 along M / N) each, eight rows per 1024-byte
// swizzle atom - exactly what a TMA box of [k rows][64 elements] leaves in shared memory.  Stride byte offset = the next
// eight K rows (1024 B), leading byte offset = the next 64 elements along M / N (a second box).  One K = 16 step is 2048 B.
PG_DEVINL uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor, kind::f16: D fp32 (1<<4), A bf16 (1<<7), B bf16 (1<<10),
// A and B K-major (bits 15,16 = 0), N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ inline uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// the same with B MN-major (bit 16): B is read as [k][n] rows, n contiguous
__host__ __device__ inline uint32_t umma_idesc_bf16_bmn(int M, int N) { return umma_idesc_bf16(M, N) | (1u << 16); }

}  // namespace pg
