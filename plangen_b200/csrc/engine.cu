// plangen_b200 engine: host-side orchestration of the sm_100a kernels behind the C-ABI declared in
// include/plangen_b200.h.  No torch, no CPU fallback: every entry point launches CUDA kernels or fails.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/plangen_b200.h"
#include "common.cuh"
#include "gemm.cuh"
#include "gemm_sk.cuh"
#include "gemm_tc2.cuh"
#include "lm_kernels.cuh"
#include "attn_tma.cuh"
#include "attn_v5.cuh"
#include "sample.cuh"
#include "text_decode.cuh"
#include "attn_prefill_tc.cuh"
#include "vq_kernels.cuh"
#include "vit_kernels.cuh"

using namespace pg;

// ------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) return fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
  } while (0)
#define TRY(call)                 \
  do {                            \
    int _r = (call);              \
    if (_r) return _r;            \
  } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------ engine
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct Carve {
  uint8_t* base = nullptr;
  size_t off = 0;
  void* take(size_t bytes) {
    off = align_up(off, 1024);
    void* p = base ? base + off : nullptr;
    off += bytes;
    return p;
  }
};

struct pg_engine {
  pg_dims d;
  int device = 0, num_sms = 0, max_threads_per_sm = 2048;
  bool bf16 = true;
  size_t esz = 2;                 // bytes per activation / weight element
  int Tmax = 0, HD = 0;
  std::unordered_map<std::string, std::pair<const void*, size_t>> tensors;
  struct Tiled { const uint8_t* ptr; int N, K; };
  std::unordered_map<const void*, Tiled> tiled;      // row-major weight -> engine-owned tile-major copy (bf16 mode)
  uint8_t* tiled_buf = nullptr;
  int prefill_attn_tc = 1;                   // prompt-prefill attention on tcgen05 (attn_prefill_tc.cuh); 0 = CUDA-core kernel
  int tc_wide_stages = 2, fuse_conv_epilogue = 1;   // conv bias / residual / bf16 store in the contraction epilogue
  EncodeTiledFn encode = nullptr;
  // options
  uint64_t attn_dbg_ptr = 0;
  int64_t attn_test_flags = 0;
  int use_tc = 1, use_pdl = 1, use_graph = 1, attn_impl = 3, attn_ctas = 0, tc_stages = 0, tc_stages_gu = 0, vq_chunk = 0, attn_splits = 0, gemm_splits = 0;
  float* dbg_logits = nullptr;
  float* dbg_text_logits = nullptr;
  unsigned long long* prof_buf = nullptr;   // per-kernel timeline of ONE decode step (plain-launch mode)
  int prof_step = -1, prof_slot = 0;
  bool prof_active = false;
  int64_t launches = 0;
  int64_t graph_captures = 0;                // decode-step graphs captured (graph_for misses)
  bool finalized = false;
  // bound buffers
  void* kv = nullptr; size_t kv_bytes = 0;
  void* ws = nullptr; size_t ws_bytes = 0;
  // workspace carve-outs
  void *xn = nullptr, *qbuf = nullptr, *attn_out = nullptr, *hbuf = nullptr, *hidden_t = nullptr, *head_h = nullptr;
  float *part = nullptr, *x_dec = nullptr, *hidden_f = nullptr, *attn_ws = nullptr, *attn_ll = nullptr;
  // engine-owned staging of the per-call inputs / outputs of the fused loops, so captured graphs depend on shapes
  // and scalars only (the caller's tensors are fresh allocations on every call)
  int32_t *st_kv_start = nullptr, *st_edit = nullptr, *st_gt = nullptr, *st_tokens = nullptr;
  ImageSampling* st_sampling = nullptr;               // sampling settings of every image: [B] (sample.cuh)
  float* st_logprobs = nullptr;                       // image loop log-probs: [B][n_steps]
  float* st_cfg = nullptr;                            // guidance schedule: [B][n_steps] (loop) or [B][n] (scorer)
  // mmu front-end (SigLIP tower + aligner + scatter, vit_kernels.cuh); carved only when dims.sig_layers > 0
  int sig_chunk = 0, sig_np = 0;                      // images per pass, patches per image
  float *sig_x = nullptr, *sig_part = nullptr;
  void *sig_xn = nullptr, *sig_qkv = nullptr, *sig_attn = nullptr, *sig_h = nullptr, *sig_feat = nullptr;
  size_t sig_part_bytes = 0;
  int32_t *sig_rank_dst = nullptr, *sig_inv_src = nullptr, *sig_counts = nullptr;
  int tc2_stages = 4;                                 // wide-tile contractions on CTA pairs (gemm_tc2.cuh, tcgen05 cta_group::2)
  int stage_cap_once = 0, down_stages = 4;            // ring cap of the next launch_tc; decode down projection (see decode_layers)
  int tc_stages_k = 0;
  int tc_stages_n = 0;                                // tc_stages applies to contractions with this N only (0 = all)
  int attn_test_alias_p = 0;                          // pg_test_attn_decode: prompt length of the batch whose dup_of is current
  int attn_alias = 1;                                 // decode attention reads a duplicate row's prompt K / V from its source row (attn_tma.cuh)
  int prefill_dedup = 1;                              // packed prefill: rows repeating an earlier row are prefilled once (lm_kernels.cuh)
  int32_t* dup_of = nullptr; int32_t* row_differs = nullptr;
  unsigned long long* row_hash = nullptr; unsigned long long* row_hash_host = nullptr;   // content hash per prompt row (device / pinned)
  int prefill_pack = 1;                               // fused loops prefill the real tokens only (lm_kernels.cuh packed_row_of)
  float* xpack = nullptr; float* x_last = nullptr; int32_t* row_off = nullptr; int32_t* row_off_host = nullptr;
  int gu_streamk = 1;                                 // decode gate|up + SwiGLU as a stream-K launch over all SMs (gemm_sk.cuh)
  int* sk_counters = nullptr;
  int last_path = PG_PATH_NONE, last_nt = 0;          // kernel the last run_gemm / run_conv_gemm launched (pg_test_contraction_run)
  int prefill_qkv_fuse = 1;                           // prefill QKV: RoPE + q / cache stores in the CTA-pair contraction's epilogue
  QkvEpi qkv_epi_next = {};                           // consumed (and cleared) by the next CTA-pair launch
  int sig_attn_tc = 1;                                // tcgen05 attention (bf16, head_dim 64); 0 = CUDA-core kernel
  size_t part_bytes = 0;
  int *attn_cnt = nullptr, *attn_flag = nullptr, *step_ctr = nullptr, *greedy_state = nullptr;
  int* poll_host = nullptr;                          // pinned: early-exit poll of the greedy loop
  void *embed_table = nullptr, *align_tmp = nullptr;
  void *vq_act[3] = {nullptr, nullptr, nullptr};
  void* vq_col = nullptr; float* vq_part = nullptr; float *gn_partial = nullptr, *gn_stats = nullptr;
  size_t vq_act_elems = 0, vq_col_elems = 0, vq_part_elems = 0;
  int gn_chunks_max = 0;
  // graph cache: one instantiated decode-step graph per (kind, shape, scalars) key; a handful of shapes alternate in
  // practice (x2t and t2i of the two-stage flow, edit / non-edit calls), so a small map, flushed when it outgrows its cap
  struct GraphEntry { cudaGraphExec_t exec = nullptr; int64_t launches = 0; };   // launches: kernels per replay
  std::unordered_map<std::string, GraphEntry> graphs;
  // the decode loop runs on the engine's own stream (the caller's may be the legacy default stream,
  // which cannot be captured); ordered against the caller's stream with events
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr;
};

static const void* T_(pg_engine* e, const std::string& name, size_t* nbytes = nullptr) {
  auto it = e->tensors.find(name);
  if (it == e->tensors.end()) return nullptr;
  if (nbytes) *nbytes = it->second.second;
  return it->second.first;
}
#define NEED(var, type, name)                                        \
  const type* var = (const type*)T_(e, (name));                      \
  if (!var) return fail("tensor '%s' was not registered", std::string(name).c_str());

static Prof next_prof(pg_engine* e) {
  Prof p;
  p.buf = (e->prof_active && e->prof_buf) ? e->prof_buf : nullptr;
  p.slot = p.buf ? std::min(e->prof_slot++, PROF_SLOTS - 1) : 0;
  return p;
}

// ------------------------------------------------------------------------------ launch helper
template <typename... KArgs, typename... Args>
static int launch(pg_engine* e, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                  Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  int na = 0;
  if (e->use_pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  e->launches++;
  cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  if (le != cudaSuccess)
    return fail("kernel launch #%lld failed (grid %u,%u,%u block %u smem %zu): %s", (long long)e->launches, grid.x, grid.y,
                grid.z, block.x, smem, cudaGetErrorString(le));
  return 0;
}

// ------------------------------------------------------------------------------ GEMM dispatch
static int make_map_2d(pg_engine* e, CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t K, uint32_t box_rows) {
  cuuint64_t gdim[2] = {K, rows};
  cuuint64_t gstr[1] = {K * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = e->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d) rows=%llu K=%llu ptr=%p", (int)r,
                                     (unsigned long long)rows, (unsigned long long)K, ptr);
  return 0;
}

template <int NT>
static int launch_tc(pg_engine* e, const CUtensorMap& mw, const CUtensorMap& mx, float* C, int M, int N, int K,
                     int splits, int kb_per_split, bool w_const, const void* w_tiled, void* swiglu_out, cudaStream_t st,
                     const ConvGeom* conv = nullptr, int grid_y = 0, const EpiFuse* epi = nullptr) {
  using Cfg = TcCfg<NT>;
  // wide token tiles (prefill, VQ convolutions) are tensor-bound: a shallow ring leaves room for two CTAs per SM,
  // whose epilogues overlap each other's main loops (measured: prefill 75.6 -> 68 ms); the weight-streaming decode
  // shapes want the deepest ring (1.64 ms/step at 8-10 stages, 1.76 at 4)
  int stages = NT >= 192 ? e->tc_wide_stages : (200 * 1024) / Cfg::STAGE_BYTES;
  // options: cap the ring depth of the split-K contractions / of the (unsplit, long-stream) gate|up contraction
  if (e->tc_stages > 0 && !swiglu_out && (e->tc_stages_n == 0 || e->tc_stages_n == N) && (e->tc_stages_k == 0 || e->tc_stages_k == K)) stages = std::min(stages, e->tc_stages);
  if (e->stage_cap_once > 0) stages = std::min(stages, e->stage_cap_once);
  e->stage_cap_once = 0;
  if (e->tc_stages_gu > 0 && swiglu_out) stages = std::min(stages, e->tc_stages_gu);
  stages = std::max(2, std::min(stages, 12));
  stages = std::min(stages, std::max(2, kb_per_split));
  if (stages < kb_per_split && (stages & 1)) --stages;   // reused rings must be even (see the invariant in gemm_tc_kernel)
  const size_t smem = Cfg::smem_bytes(stages);
  dim3 grid((N + TC_BM - 1) / TC_BM, conv ? grid_y : (M + NT - 1) / NT, splits);
  ConvGeom cg = {};
  if (conv) cg = *conv;
  EpiFuse ep = {};
  if (epi) ep = *epi;
  if (ep.out && (size_t)stages * Cfg::STAGE_BYTES < (size_t)NT * 256) return fail("internal: operand ring too small to stage the output tile");
  return launch(e, gemm_tc_kernel<NT>, grid, dim3(192), smem, st, mw, mx, C, M, N, K, kb_per_split, stages,
                e->use_pdl ? (w_const ? 3 : 1) : 0, (const uint8_t*)w_tiled, next_prof(e), (bf16*)swiglu_out, cg,
                ep);
}

// 3x3 convolution (pad 1) as an implicit GEMM on the tcgen05 path: act bf16 NHWC [B][H][W][Cin], Wc bf16
// [Cout][9*Cin] (k = tap*Cin + cin), C fp32 [B*H*W][Cout].  Returns 1 through *taken when the shape qualifies
// (bf16, Cin % 64 == 0, W or a 192-pixel part of it tiles a 192-pixel block), 0 -> caller uses im2col.
constexpr int CONV_NT = 192;
static int run_conv_gemm(pg_engine* e, const void* act, const void* Wc, int B, int H, int W, int Cin, int Cout, float* C,
                         size_t c_bytes, cudaStream_t st, int* taken, const EpiFuse* epi = nullptr) {
  *taken = 0;
  e->last_path = PG_PATH_IM2COL; e->last_nt = 0;
  if (!e->bf16 || !e->use_tc || Cin % TC_BK != 0) return 0;
  if ((((uintptr_t)act) & 15) || (((uintptr_t)Wc) & 15)) return 0;
  int bw = 0;
  if (W <= CONV_NT && CONV_NT % W == 0) bw = W;
  else if (W % CONV_NT == 0) bw = CONV_NT;
  if (!bw) return 0;
  const int bh = CONV_NT / bw;
  const size_t pixels = (size_t)B * H * W;
  if (pixels * Cout * 4 > c_bytes) return fail("conv partial buffer too small");
  ConvGeom cg;
  cg.enabled = 1; cg.H = H; cg.W = W; cg.Cin = Cin; cg.bw = bw; cg.bh = bh;
  cg.tiles_x = W / bw; cg.tiles_y = (H + bh - 1) / bh;
  CUtensorMap mw, mx;
  TRY(make_map_2d(e, &mw, Wc, (uint64_t)Cout, (uint64_t)9 * Cin, TC_BM));
  cuuint64_t gdim[4] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2};
  cuuint32_t box[4] = {(cuuint32_t)TC_BK, (cuuint32_t)bw, (cuuint32_t)bh, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = e->encode(&mx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(act), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (conv activation) failed (%d) B=%d H=%d W=%d C=%d", (int)r, B, H, W, Cin);
  const int num_kb = 9 * Cin / TC_BK;
  TRY(launch_tc<CONV_NT>(e, mw, mx, C, (int)pixels, Cout, 9 * Cin, 1, num_kb, true, nullptr, nullptr, st, &cg,
                         B * cg.tiles_x * cg.tiles_y, epi));
  e->last_path = PG_PATH_CONV; e->last_nt = CONV_NT;
  *taken = 1;
  return 0;
}

// the tcgen05 contraction runs on CTA pairs (gemm_tc2.cuh) for 256-token tiles without split-K, SwiGLU-to-hbuf or a lone
// weight tile
static bool tc_pair_taken(int M, int N, int splits, bool swiglu_out) { return M > 128 && splits == 1 && !swiglu_out && N > TC_BM; }

// C[splits][M][N] fp32 = X[M][K] * W[N][K]^T.  Returns the number of splits used through *splits_out.
static int run_gemm(pg_engine* e, const void* X, const void* W, int M, int N, int K, float* C, size_t c_bytes,
                    int* splits_out, cudaStream_t st, int force_impl = -1, int force_splits = 0, bool w_const = true,
                    const void* w_tiled = nullptr, void* swiglu_out = nullptr, const EpiFuse* epi = nullptr) {
  const bool tc = e->bf16 && ((force_impl == 1) || (force_impl < 0 && e->use_tc)) && (K % 8 == 0) &&
                  (((uintptr_t)X & 15) == 0) && (((uintptr_t)W & 15) == 0);
  if (force_impl == 1 && !tc) return fail("tcgen05 GEMM needs bf16 operands, K %% 8 == 0 and 16-byte aligned pointers");
  int splits = 1;
  if (tc) {
    const int NT = M <= 16 ? 16 : M <= 32 ? 32 : M <= 64 ? 64 : M <= 128 ? 128 : 256;
    const int tiles = ((N + TC_BM - 1) / TC_BM) * ((M + NT - 1) / NT);
    const int num_kb = (K + TC_BK - 1) / TC_BK;
    const bool opt_splits = e->gemm_splits > 0 && (e->tc_stages_n == 0 || e->tc_stages_n == N) && (e->tc_stages_k == 0 || e->tc_stages_k == K);
    int want = force_splits > 0 ? force_splits : (opt_splits ? e->gemm_splits : 0);
    if (want == 0) {
      // split-K count: every CTA pays a fixed fill / drain cost (~3 us, about 9 k-blocks of streaming) on top of its
      // k-blocks, CTAs run one per SM in waves.  Minimise waves x (9 + k-blocks per split); e.g. the 7B QKV projection
      // (96 tiles x 64 k-blocks) takes 3 splits = 288 CTAs = two full waves of 22 k-blocks instead of one wave of 64
      // on 96 of the 148 SMs.
      long best = -1;
      for (int sp = 1; sp <= std::min(16, num_kb); ++sp) {
        const int kbp = (num_kb + sp - 1) / sp, real = (num_kb + kbp - 1) / kbp;
        const long waves = ((long)tiles * real + e->num_sms - 1) / e->num_sms;
        const long cost = waves * (9 + kbp);
        if (best < 0 || cost < best) { best = cost; want = real; }
      }
    }
    if (swiglu_out || epi) want = 1;                        // fused epilogues need the whole K in one CTA
    if (epi && (N % 8 != 0)) return fail("fused epilogue needs N %% 8 == 0 (N=%d)", N);
    want = std::min(std::min(want, 16), num_kb);
    while (want > 1 && (size_t)want * M * N * 4 > c_bytes) --want;
    const int kb_per_split = (num_kb + want - 1) / want;
    splits = (num_kb + kb_per_split - 1) / kb_per_split;
    if ((size_t)splits * M * N * 4 > c_bytes) return fail("GEMM partial buffer too small (%d x %d x %d)", splits, M, N);
    if (!w_tiled && w_const) {                             // stream the tile-major copy when the weight has one
      auto it = e->tiled.find(W);
      if (it != e->tiled.end() && it->second.N == N && it->second.K == K) w_tiled = it->second.ptr;
    }
    CUtensorMap mw, mx;
    TRY(make_map_2d(e, &mw, W, (uint64_t)N, (uint64_t)K, TC_BM));
    if (tc_pair_taken(M, N, splits, swiglu_out != nullptr)) {
      // tensor-bound shape: CTA pairs, one 256 x 256 x 16 MMA per pair and k-step (gemm_tc2.cuh)
      TRY(make_map_2d(e, &mx, X, (uint64_t)M, (uint64_t)K, (uint32_t)(TC2_NT / 2)));
      EpiFuse ep2 = {};
      if (epi) ep2 = *epi;
      const int n_tiles = (((N + TC_BM - 1) / TC_BM + 1) / 2) * ((M + TC2_NT - 1) / TC2_NT);
      const int pairs = std::max(1, std::min(n_tiles, e->num_sms / 2));       // persistent: one CTA per SM
      const QkvEpi qe = e->qkv_epi_next;
      e->qkv_epi_next = QkvEpi{};
      if (ep2.gelu == 3 && (qe.q_out == nullptr || N != 3 * qe.H * HEAD_DIM)) return fail("internal: QKV epilogue without its destinations");
      TRY(launch(e, gemm_tc2_kernel, dim3(2 * pairs, 1, 1), dim3(TC2_THREADS), (size_t)tc2p_smem_bytes(e->tc2_stages), st, mw, mx, C, M,
                 N, K, e->tc2_stages, e->use_pdl, next_prof(e), ep2, qe));
      e->last_path = PG_PATH_TC2; e->last_nt = TC2_NT;
      *splits_out = 1;
      return 0;
    }
    if (epi && epi->gelu >= 2) return fail("internal: the SwiGLU / QKV epilogues exist in the CTA-pair contraction only (M=%d N=%d)", M, N);
    TRY(make_map_2d(e, &mx, X, (uint64_t)M, (uint64_t)K, (uint32_t)NT));
    switch (NT) {
      case 16: TRY(launch_tc<16>(e, mw, mx, C, M, N, K, splits, kb_per_split, w_const, w_tiled, swiglu_out, st, nullptr, 0, epi)); break;
      case 32: TRY(launch_tc<32>(e, mw, mx, C, M, N, K, splits, kb_per_split, w_const, w_tiled, swiglu_out, st, nullptr, 0, epi)); break;
      case 64: TRY(launch_tc<64>(e, mw, mx, C, M, N, K, splits, kb_per_split, w_const, w_tiled, swiglu_out, st, nullptr, 0, epi)); break;
      case 128: TRY(launch_tc<128>(e, mw, mx, C, M, N, K, splits, kb_per_split, w_const, w_tiled, swiglu_out, st, nullptr, 0, epi)); break;
      default: TRY(launch_tc<256>(e, mw, mx, C, M, N, K, splits, kb_per_split, w_const, w_tiled, swiglu_out, st, nullptr, 0, epi)); break;
    }
    e->last_path = PG_PATH_TC; e->last_nt = NT;
  } else {
    if (swiglu_out || epi) return fail("internal: fused epilogues need the tcgen05 path");
    if (K % 4 != 0) return fail("SIMT GEMM needs K %% 4 == 0 (K=%d)", K);
    const int tiles = ((N + 63) / 64) * ((M + 63) / 64);
    int want = force_splits > 0 ? force_splits : (e->gemm_splits > 0 ? e->gemm_splits : std::max(1, (2 * e->num_sms) / tiles));
    want = std::min(std::min(want, 16), (K + 15) / 16);
    while (want > 1 && (size_t)want * M * N * 4 > c_bytes) --want;
    int k_per_split = ((K + want - 1) / want + 15) / 16 * 16;
    splits = (K + k_per_split - 1) / k_per_split;
    if ((size_t)splits * M * N * 4 > c_bytes) return fail("GEMM partial buffer too small (%d x %d x %d)", splits, M, N);
    dim3 grid((N + 63) / 64, (M + 63) / 64, splits);
    if (e->bf16)
      TRY(launch(e, gemm_simt_kernel<bf16>, grid, dim3(256), 0, st, (const bf16*)X, (const bf16*)W, C, M, N, K, k_per_split));
    else
      TRY(launch(e, gemm_simt_kernel<float>, grid, dim3(256), 0, st, (const float*)X, (const float*)W, C, M, N, K, k_per_split));
    e->last_path = PG_PATH_SIMT; e->last_nt = 0;
  }
  *splits_out = splits;
  return 0;
}

// Tile-major, pre-swizzled copy of a row-major bf16 weight [N][K] (tile_weight_kernel): ceil(N/128) x ceil(K/64) tiles of
// 16 KB, zero-padded at the edges.
static size_t tile_major_bytes(int N, int K) { return (size_t)((N + TC_BM - 1) / TC_BM) * ((K + TC_BK - 1) / TC_BK) * TC_A_BYTES; }
static int build_tile_major(pg_engine* e, const void* W, int N, int K, uint8_t* dst, cudaStream_t st) {
  const size_t n_chunks = tile_major_bytes(N, K) / 16;
  const int blocks = (int)std::min<size_t>((n_chunks + 255) / 256, (size_t)e->num_sms * 16);
  tile_weight_kernel<<<blocks, 256, 0, st>>>((const bf16*)W, dst, N, K, (K + TC_BK - 1) / TC_BK, n_chunks);
  CK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------ sizes
// images per VQ pass: the whole batch up to 16 in the bf16 regime (16 x 530 MB of scratch; measured 46.2 / 41.1 / 38.8 ms
// per 16 images at 4 / 8 / 16 - fewer, larger launches), one image at a time in fp32 check mode
static int vq_chunk_of(const pg_engine* e) {
  if (e->vq_chunk > 0) return e->vq_chunk;
  return e->bf16 ? std::max(1, std::min(16, e->d.max_rows / 2)) : 1;
}

static void layout_workspace(pg_engine* e, Carve& c) {
  const pg_dims& d = e->d;
  const size_t es = e->esz;
  const size_t max_tok = (size_t)d.max_rows * std::max(d.max_prompt, 1);
  const size_t R = d.max_rows;
  const size_t wide = std::max<size_t>(std::max(3 * e->HD, 2 * d.F), std::max(d.D, d.img_embed));
  e->xpack = (float*)c.take(max_tok * d.D * 4);
  e->x_last = (float*)c.take(R * d.D * 4);
  e->row_off = (int32_t*)c.take((R + 1) * 4);
  e->dup_of = (int32_t*)c.take(R * 4);
  e->row_differs = (int32_t*)c.take(R * 4);
  e->row_hash = (unsigned long long*)c.take(R * 8);
  e->xn = c.take(max_tok * d.D * es);
  e->qbuf = c.take(max_tok * e->HD * es);
  e->attn_out = c.take(max_tok * e->HD * es);
  e->hbuf = c.take(max_tok * d.F * es);
  size_t pb = max_tok * wide * 4;                                         // prefill, 1 split
  pb = std::max(pb, (size_t)16 * R * std::max<size_t>(wide, d.img_vocab) * 4);   // decode, <= 16 splits
  pb = std::max(pb, (size_t)d.img_vocab * d.D * 4);                       // gen_aligner table build
  e->part_bytes = pb;
  e->part = (float*)c.take(pb);
  e->x_dec = (float*)c.take(R * d.D * 4);
  e->hidden_f = (float*)c.take(R * d.D * 4);
  e->hidden_t = c.take(R * d.D * es);
  e->head_h = c.take(R * d.img_embed * es);
  e->attn_ws = (float*)c.take(R * d.H * 64 * (HEAD_DIM + 2) * 4);
  e->attn_cnt = (int*)c.take(R * d.H * 4);
  e->attn_flag = (int*)c.take(R * d.H * 64 * 4);
  e->attn_ll = (float*)c.take(R * d.H * 64 * (HEAD_DIM + 2) * 8);
  e->step_ctr = (int*)c.take(256);
  e->sk_counters = (int*)c.take((size_t)((2 * d.F + TC_BM - 1) / TC_BM) * 4);
  e->greedy_state = (int*)c.take(256 + R * 4);      // [0] rows unfinished, [1] steps generated, [64..] per-row flags
  e->embed_table = c.take((size_t)d.img_vocab * d.D * es);
  e->align_tmp = c.take((size_t)d.img_vocab * d.D * es);
  {
    const size_t B = (R + 1) / 2;
    e->st_kv_start = (int32_t*)c.take(R * 4);
    e->st_edit = (int32_t*)c.take(B * std::max(d.max_steps, 1) * 4);
    e->st_gt = (int32_t*)c.take(B * std::max(d.max_steps, 1) * 4);
    e->st_tokens = (int32_t*)c.take(R * (size_t)e->Tmax * 4);      // image loop: [B][n_steps]; text loop: [R][max_new]
    e->st_sampling = (ImageSampling*)c.take(B * sizeof(ImageSampling));
    e->st_logprobs = (float*)c.take(B * std::max(d.max_steps, 1) * 4);
    e->st_cfg = (float*)c.take(B * std::max(d.max_steps, 1) * 4);
  }
  if (d.sig_layers > 0 && d.max_images > 0) {
    // SigLIP tower scratch for one pass of sig_chunk images; features of ALL images stay (the scatter needs them)
    e->sig_np = (d.sig_image / d.sig_patch) * (d.sig_image / d.sig_patch);
    e->sig_chunk = std::min(d.max_images, 32);
    const size_t Mc = (size_t)e->sig_chunk * e->sig_np, W = d.sig_width, Kp = (size_t)3 * d.sig_patch * d.sig_patch;
    const size_t widest = std::max<size_t>(std::max<size_t>(3 * W, d.sig_mlp), d.D);
    e->sig_x = (float*)c.take(Mc * W * 4);
    e->sig_xn = c.take(Mc * std::max(W, Kp) * es);
    e->sig_qkv = c.take(Mc * 3 * W * es);
    e->sig_attn = c.take(Mc * W * es);
    e->sig_h = c.take(Mc * std::max<size_t>(d.sig_mlp, d.D) * es);
    e->sig_part_bytes = Mc * widest * 4;
    e->sig_part = (float*)c.take(e->sig_part_bytes);
    e->sig_feat = c.take((size_t)d.max_images * e->sig_np * d.D * es);
    e->sig_rank_dst = (int32_t*)c.take(max_tok * 4);
    e->sig_inv_src = (int32_t*)c.take((size_t)d.max_images * e->sig_np * 4);
    e->sig_counts = (int32_t*)c.take(256);
  }
  // VQ decoder scratch, per chunk of images
  const int Bc = vq_chunk_of(e);
  size_t act = 0, col = 0, part = 0;
  {
    int res = d.grid;
    const int nres = d.vq_nres;
    int ch = d.vq_ch * d.vq_ch_mult[nres - 1];
    act = std::max(act, (size_t)res * res * std::max(ch, d.vq_z));
    col = std::max(col, (size_t)res * res * 9 * std::max(ch, d.vq_z));
    col = std::max(col, (size_t)res * res * ch * 6 + (size_t)res * res * res * res);   // attention scratch
    part = std::max(part, (size_t)res * res * std::max<size_t>(ch, (size_t)res * res));
    for (int idx = 0; idx < nres; ++idx) {
      const int i_level = nres - 1 - idx;
      const int cout = d.vq_ch * d.vq_ch_mult[i_level];
      act = std::max(act, (size_t)res * res * std::max(ch, cout));
      col = std::max(col, (size_t)res * res * 9 * std::max(ch, cout));
      part = std::max(part, (size_t)res * res * std::max(ch, cout));
      ch = cout;
      if (idx != nres - 1) {
        res *= 2;
        act = std::max(act, (size_t)res * res * ch);
        col = std::max(col, (size_t)res * res * 9 * ch);
        part = std::max(part, (size_t)res * res * ch);
      }
    }
  }
  e->vq_act_elems = act * Bc; e->vq_col_elems = col * Bc; e->vq_part_elems = part * Bc;
  e->vq_part_elems = std::max(e->vq_part_elems, (size_t)d.img_vocab * (d.code_dim + 1));   // normalised codebook + norms (pg_vq_encode)
  for (int i = 0; i < 3; ++i) e->vq_act[i] = c.take(e->vq_act_elems * es);
  e->vq_col = c.take(e->vq_col_elems * es);
  e->vq_part = (float*)c.take(e->vq_part_elems * 4);
  e->gn_chunks_max = 1024;
  e->gn_partial = (float*)c.take((size_t)Bc * e->gn_chunks_max * 32 * 2 * 4);
  e->gn_stats = (float*)c.take((size_t)Bc * 32 * 2 * 4);
}

static void drop_graphs(pg_engine* e) {
  for (auto& kv : e->graphs) if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  e->graphs.clear();
}

// ------------------------------------------------------------------------------ C-ABI: lifetime
extern "C" const char* pg_last_error(void) { return g_err; }
extern "C" int pg_abi_version(void) { return PG_ABI_VERSION; }

extern "C" int pg_engine_create(const pg_dims* dims, int device, pg_engine** out) {
  if (!dims || !out) return fail("null argument");
  if (dims->head_dim != HEAD_DIM) return fail("head_dim must be %d", HEAD_DIM);
  if (dims->D % 8 || dims->F % 8 || dims->img_embed % 8) return fail("D, F, img_embed must be multiples of 8");
  if (dims->D > RN_THREADS * RN_MAX_PER_THREAD) return fail("D > %d is not supported by the RMSNorm kernel", RN_THREADS * RN_MAX_PER_THREAD);
  if (dims->vq_nres < 1 || dims->vq_nres > 8) return fail("bad vq_nres");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail("no CUDA device %d (have %d): plangen_b200 has no CPU path", device, ndev);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail("plangen_b200 kernels are built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
  pg_engine* e = new pg_engine();
  e->d = *dims;
  e->device = device;
  e->num_sms = prop.multiProcessorCount;
  e->max_threads_per_sm = prop.maxThreadsPerMultiProcessor;
  e->bf16 = dims->mode == PG_MODE_BF16;
  e->esz = e->bf16 ? 2 : 4;
  e->HD = dims->H * dims->head_dim;
  e->Tmax = (int)align_up((size_t)dims->max_prompt + dims->max_steps, 64);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) { delete e; return fail("cuTensorMapEncodeTiled not available"); }
  e->encode = (EncodeTiledFn)fn;
  CK(cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_tc_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(resid_rmsnorm_tma_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(resid_rmsnorm_tma_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(resid_rmsnorm_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(resid_rmsnorm_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  CK(cudaFuncSetAttribute(attn_prefill_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PA_SMEM));
  CK(cudaFuncSetAttribute(vit_attn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, VT_SMEM));
  CK(cudaFuncSetAttribute(gemm_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_swiglu_sk_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_swiglu_sk_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CK(cudaFuncSetAttribute(gemm_swiglu_sk_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  if (dims->sig_layers > 0) {
    if (dims->sig_width % 8 || dims->sig_mlp % 8 || dims->sig_patch % 4 || dims->sig_heads < 1 || dims->sig_width % dims->sig_heads ||
        dims->sig_image % dims->sig_patch || dims->sig_width > 4 * LN_MAXQ * LN_THREADS)
      return fail("unsupported SigLIP dims (width %d, heads %d, patch %d, image %d, mlp %d)", dims->sig_width, dims->sig_heads,
                  dims->sig_patch, dims->sig_image, dims->sig_mlp);
    const int np = (dims->sig_image / dims->sig_patch) * (dims->sig_image / dims->sig_patch);
    if (np > 32 * VA_MAXI || (np & 1) || dims->sig_width / dims->sig_heads > 128) return fail("unsupported SigLIP patch count %d / head_dim", np);
  }
  CK(cudaFuncSetAttribute(attn_decode_v5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, A5_SMEM));
  CK(cudaFuncSetAttribute(attn_prefill_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTN_PREFILL_SMEM));
  CK(cudaFuncSetAttribute(attn_prefill_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTN_PREFILL_SMEM));
  *out = e;
  return 0;
}

extern "C" int pg_engine_destroy(pg_engine* e) {
  if (!e) return 0;
  drop_graphs(e);
  if (e->poll_host) cudaFreeHost(e->poll_host);
  if (e->row_off_host) cudaFreeHost(e->row_off_host);
  if (e->row_hash_host) cudaFreeHost(e->row_hash_host);
  if (e->tiled_buf) cudaFree(e->tiled_buf);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_out) cudaEventDestroy(e->ev_out);
  delete e;
  return 0;
}

extern "C" int pg_engine_query_bytes(const pg_engine* e_, size_t* kv_bytes, size_t* ws_bytes) {
  if (!e_) return fail("null engine");
  pg_engine tmp = *e_;
  Carve c;
  layout_workspace(&tmp, c);
  if (kv_bytes) *kv_bytes = (size_t)tmp.d.L * 2 * tmp.d.max_rows * tmp.d.H * tmp.Tmax * HEAD_DIM * tmp.esz;
  if (ws_bytes) *ws_bytes = align_up(c.off, 1024) + 1024;
  tmp.graphs.clear();
  return 0;
}

extern "C" int pg_engine_bind_buffers(pg_engine* e, void* kv, size_t kv_bytes, void* ws, size_t ws_bytes) {
  if (!e) return fail("null engine");
  size_t need_kv, need_ws;
  TRY(pg_engine_query_bytes(e, &need_kv, &need_ws));
  if (kv_bytes < need_kv) return fail("kv buffer too small: %zu < %zu", kv_bytes, need_kv);
  if (ws_bytes < need_ws) return fail("workspace too small: %zu < %zu", ws_bytes, need_ws);
  if (((uintptr_t)kv & 255) || ((uintptr_t)ws & 255)) return fail("buffers must be 256-byte aligned");
  e->kv = kv; e->kv_bytes = kv_bytes; e->ws = ws; e->ws_bytes = ws_bytes;
  // TMA tiles of the attention kernels read cache slots past the newest token (and pad slots): they are masked, but a masked
  // probability of 0 times a NaN bit pattern is NaN, so the cache must hold finite values from the start
  CK(cudaMemset(kv, 0, kv_bytes));
  Carve c;
  c.base = (uint8_t*)align_up((uintptr_t)ws, 1024);
  layout_workspace(e, c);
  return 0;
}

extern "C" int pg_engine_set_tensor(pg_engine* e, const char* name, const void* dev_ptr, size_t nbytes) {
  if (!e || !name || !dev_ptr) return fail("null argument");
  if ((uintptr_t)dev_ptr & 15) return fail("tensor '%s' is not 16-byte aligned", name);
  e->tensors[name] = {dev_ptr, nbytes};
  return 0;
}

extern "C" int pg_engine_set_option(pg_engine* e, const char* key, int64_t value) {
  if (!e || !key) return fail("null argument");
  const std::string k(key);
  if (k == "use_tc") e->use_tc = (int)value;
  else if (k == "use_pdl") e->use_pdl = (int)value;
  else if (k == "use_graph") e->use_graph = (int)value;
  else if (k == "tc_stages") e->tc_stages = (int)value;
  else if (k == "tc_stages_gu") e->tc_stages_gu = (int)value;
  else if (k == "tc_stages_n") e->tc_stages_n = (int)value;
  else if (k == "tc_stages_k") e->tc_stages_k = (int)value;
  else if (k == "down_stages") e->down_stages = (int)value;
  else if (k == "vq_chunk") e->vq_chunk = (int)value;
  else if (k == "attn_splits") e->attn_splits = (int)value;
  else if (k == "attn_impl") e->attn_impl = (int)value;
  else if (k == "prefill_attn_tc") e->prefill_attn_tc = (int)value;
  else if (k == "sig_attn_tc") e->sig_attn_tc = (int)value;
  else if (k == "prefill_qkv_fuse") e->prefill_qkv_fuse = (int)value;
  else if (k == "gu_streamk") e->gu_streamk = (int)value;
  else if (k == "prefill_pack") e->prefill_pack = (int)value;
  else if (k == "prefill_dedup") e->prefill_dedup = (int)value;
  else if (k == "attn_alias") e->attn_alias = (int)value;
  else if (k == "attn_test_alias_p") e->attn_test_alias_p = (int)value;
  else if (k == "tc2_stages") e->tc2_stages = std::max(2, std::min(4, (int)value));
  else if (k == "fuse_conv_epilogue") e->fuse_conv_epilogue = (int)value;
  else if (k == "tc_wide_stages") e->tc_wide_stages = std::max(2, (int)value);
  else if (k == "attn_dbg_ptr") e->attn_dbg_ptr = (uint64_t)value;
  else if (k == "gemm_dbg_ptr") { unsigned long long* p = (unsigned long long*)value; CK(cudaMemcpyToSymbol(g_gemm_dbg, &p, sizeof(p))); }
  else if (k == "sample_dbg_ptr") { unsigned long long* p = (unsigned long long*)value; CK(cudaMemcpyToSymbol(g_sample_dbg, &p, sizeof(p))); }
  else if (k == "norm_dbg_ptr") { unsigned long long* p = (unsigned long long*)value; CK(cudaMemcpyToSymbol(g_norm_dbg, &p, sizeof(p))); }
  else if (k == "norm_dbg_step") { int n = (int)value; CK(cudaMemcpyToSymbol(g_norm_dbg_step, &n, sizeof(n))); }
  else if (k == "gemm_dbg_n") { int n = (int)value; CK(cudaMemcpyToSymbol(g_gemm_dbg_n, &n, sizeof(n))); }
  else if (k == "attn_test_flags") e->attn_test_flags = value;
  else if (k == "attn_ctas") e->attn_ctas = (int)value;
  else if (k == "gemm_splits") e->gemm_splits = (int)value;
  else if (k == "dbg_logits_ptr") e->dbg_logits = (float*)(uintptr_t)value;
  else if (k == "dbg_text_logits_ptr") e->dbg_text_logits = (float*)(uintptr_t)value;   // [max_new][R][vocab] fp32
  else if (k == "prof_ptr") e->prof_buf = (unsigned long long*)(uintptr_t)value;
  else if (k == "prof_step") e->prof_step = (int)value;
  else if (k == "reset_launches") e->launches = 0;
  else return fail("unknown option '%s'", key);
  drop_graphs(e);          // options are baked into captured launches
  return 0;
}

extern "C" int pg_engine_get_counter(const pg_engine* e, const char* key, int64_t* value) {
  if (!e || !key || !value) return fail("null argument");
  const std::string k(key);
  if (k == "launches") *value = e->launches;
  else if (k == "num_sms") *value = e->num_sms;
  else if (k == "max_threads_per_sm") *value = e->max_threads_per_sm;
  else if (k == "tmax") *value = e->Tmax;
  else if (k == "graph_captures") *value = e->graph_captures;
  else if (k == "philox_offset_per_step") *value = 0;
  else return fail("unknown counter '%s'", key);
  return 0;
}

// ------------------------------------------------------------------------------ typed dispatch helpers
#define DISPATCH_T(e, expr_bf16, expr_f32) \
  do {                                     \
    if ((e)->bf16) { TRY(expr_bf16); }     \
    else { TRY(expr_f32); }                \
  } while (0)

static int k_resid_norm(pg_engine* e, float* x, const float* part, int S, size_t sstride, const float* w, void* xn,
                        float* y, int rows, int in_stride, int in_off, int flags, cudaStream_t st) {
  const int D = e->d.D;
  // split-K slabs + residual row through TMA bulk copies into shared memory (bit-identical, see lm_kernels.cuh)
  const size_t tma_smem = (size_t)(S + 1) * D * 4 + 128;
  const int tma_threads = std::min(RN_THREADS, std::max(128, (D / 4 + 31) / 32 * 32));   // one element quad per thread
  if (part != nullptr && in_stride == 1 && in_off == 0 && D % 4 == 0 &&
      D <= RN_MAX_PER_THREAD * tma_threads && tma_smem <= 200 * 1024 && (sstride * 4) % 16 == 0 &&
      (((uintptr_t)part | (uintptr_t)x) & 15) == 0) {
    DISPATCH_T(e,
               launch(e, resid_rmsnorm_tma_kernel<bf16>, dim3(rows), dim3(tma_threads), tma_smem, st, x, part, S, sstride, w, (bf16*)xn, y, D,
                      e->d.rms_eps, flags, e->step_ctr, next_prof(e)),
               launch(e, resid_rmsnorm_tma_kernel<float>, dim3(rows), dim3(tma_threads), tma_smem, st, x, part, S, sstride, w, (float*)xn, y, D,
                      e->d.rms_eps, flags, e->step_ctr, next_prof(e)));
    return 0;
  }
  // prefill with fused epilogues: plain RMSNorm of thousands of rows to bf16 - one warp per row (lm_kernels.cuh)
  if (e->bf16 && part == nullptr && y == nullptr && xn != nullptr && in_stride == 1 && in_off == 0 && flags == 0 &&
      rows > 256 && D % 128 == 0 && (((uintptr_t)x | (uintptr_t)xn | (uintptr_t)w) & 15) == 0) {
    const dim3 grid((rows + 7) / 8);
    if (D == 2048) return launch(e, rmsnorm_rows_warp_kernel<16>, grid, dim3(256), 0, st, (const float*)x, w, (bf16*)xn, rows, D, e->d.rms_eps);
    if (D == 4096) return launch(e, rmsnorm_rows_warp_kernel<32>, grid, dim3(256), 0, st, (const float*)x, w, (bf16*)xn, rows, D, e->d.rms_eps);
    return launch(e, rmsnorm_rows_warp_kernel<0>, grid, dim3(256), 0, st, (const float*)x, w, (bf16*)xn, rows, D, e->d.rms_eps);
  }
  // few rows (decode): 1024 threads so one row's split-K loads are all in flight; many rows (prefill): 256+
  int threads = rows <= 256 ? RN_THREADS : 256;
  while (threads * RN_MAX_PER_THREAD < D) threads *= 2;
  DISPATCH_T(e,
             launch(e, resid_rmsnorm_kernel<bf16>, dim3(rows), dim3(threads), 0, st, x, part, S, sstride, w, (bf16*)xn, y, D,
                    e->d.rms_eps, in_stride, in_off, flags, e->step_ctr, next_prof(e)),
             launch(e, resid_rmsnorm_kernel<float>, dim3(rows), dim3(threads), 0, st, x, part, S, sstride, w, (float*)xn, y,
                    D, e->d.rms_eps, in_stride, in_off, flags, e->step_ctr, next_prof(e)));
  return 0;
}

static void* kv_ptr(pg_engine* e, int layer, int which, int R) {
  // [L][2][R][H][Tmax][128]; R here is the row count of the CURRENT batch (cache is re-laid per batch)
  const size_t per = (size_t)R * e->d.H * e->Tmax * HEAD_DIM * e->esz;
  return (uint8_t*)e->kv + ((size_t)layer * 2 + which) * per;
}

static int check_ready(pg_engine* e) {
  if (!e) return fail("null engine");
  if (!e->ws || !e->kv) return fail("buffers not bound (pg_engine_bind_buffers)");
  if (!e->finalized) return fail("engine not finalized (pg_engine_finalize)");
  return 0;
}

// ------------------------------------------------------------------------------ LM layer weights
struct LayerW { const float *ln1, *ln2; const void *wqkv, *wo, *wgu, *wd; };
static int layer_weights(pg_engine* e, int l, LayerW* w) {
  const std::string p = "l" + std::to_string(l) + ".";
  w->ln1 = (const float*)T_(e, p + "ln1"); w->ln2 = (const float*)T_(e, p + "ln2");
  w->wqkv = T_(e, p + "wqkv"); w->wo = T_(e, p + "wo"); w->wgu = T_(e, p + "wgu"); w->wd = T_(e, p + "wd");
  if (!w->ln1 || !w->ln2 || !w->wqkv || !w->wo || !w->wgu || !w->wd) return fail("layer %d weights missing", l);
  return 0;
}

// ------------------------------------------------------------------------------ finalize
extern "C" int pg_engine_finalize(pg_engine* e, void* stream) {
  if (!e) return fail("null engine");
  if (!e->ws) return fail("bind buffers before finalize");
  cudaStream_t st = (cudaStream_t)stream;
  const pg_dims& d = e->d;
  // gen_aligner(gen_embed(v)) for every v: the next-input embedding is a pure function of the id
  NEED(gen_embed, float, "gen_embed");
  NEED(w0, void, "align.w0");
  NEED(b0, float, "align.b0");
  NEED(w1, void, "align.w1");
  NEED(b1, float, "align.b1");
  const size_t total = (size_t)d.img_vocab * d.D;
  void* htmp = e->align_tmp;   // scratch: V x D activations
  const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
  const int saved_pdl = e->use_pdl;
  e->use_pdl = 0;
  int rc = 0;
  do {
    if (e->bf16) rc = launch(e, aligner_l0_kernel<bf16>, dim3(blocks), dim3(256), 0, st, gen_embed, (const bf16*)w0, b0, (bf16*)htmp, d.code_dim, d.D, total);
    else rc = launch(e, aligner_l0_kernel<float>, dim3(blocks), dim3(256), 0, st, gen_embed, (const float*)w0, b0, (float*)htmp, d.code_dim, d.D, total);
    if (rc) break;
    int S = 1;
    rc = run_gemm(e, htmp, w1, d.img_vocab, d.D, d.D, e->part, e->part_bytes, &S, st, -1, 1);
    if (rc) break;
    if (e->bf16) rc = launch(e, bias_act_kernel<bf16>, dim3(blocks), dim3(256), 0, st, e->part, S, total, b1, (bf16*)e->embed_table, (float*)nullptr, d.D, total, 0);
    else rc = launch(e, bias_act_kernel<float>, dim3(blocks), dim3(256), 0, st, e->part, S, total, b1, (float*)e->embed_table, (float*)nullptr, d.D, total, 0);
  } while (0);
  e->use_pdl = saved_pdl;
  if (rc) return rc;
  CK(cudaMemsetAsync(e->attn_cnt, 0, (size_t)d.max_rows * d.H * 4, st));
  CK(cudaMemsetAsync(e->attn_flag, 0, (size_t)d.max_rows * d.H * 64 * 4, st));
  CK(cudaMemsetAsync(e->attn_ll, 0, (size_t)d.max_rows * d.H * 64 * (HEAD_DIM + 2) * 8, st));
  CK(cudaMemsetAsync(e->step_ctr, 0, 256, st));
  CK(cudaMemsetAsync(e->sk_counters, 0, (size_t)((2 * d.F + TC_BM - 1) / TC_BM) * 4, st));
  if (e->bf16 && !e->tiled_buf) {
    // tile-major copies of the weights that are streamed once per step (see tile_weight_kernel)
    struct Item { const void* w; int N, K; };
    std::vector<Item> items;
    for (int l = 0; l < d.L; ++l) {
      LayerW w;
      TRY(layer_weights(e, l, &w));
      items.push_back({w.wqkv, 3 * e->HD, d.D});
      items.push_back({w.wo, d.D, e->HD});
      items.push_back({w.wgu, 2 * d.F, d.D});
      items.push_back({w.wd, d.D, d.F});
    }
    if (const void* hw0 = T_(e, "head.w0")) items.push_back({hw0, d.img_embed, d.D});
    if (const void* hw1 = T_(e, "head.w1")) items.push_back({hw1, d.img_vocab, d.img_embed});
    if (const void* lmh = T_(e, "lm_head")) items.push_back({lmh, d.vocab, d.D});      // stage-1 text decode (optional)
    size_t total_bytes = 0;
    for (const Item& it : items) if (it.K % 8 == 0) total_bytes += tile_major_bytes(it.N, it.K);
    CK(cudaMalloc(&e->tiled_buf, std::max<size_t>(total_bytes, 16)));
    size_t off = 0;
    for (const Item& it : items) {
      if (it.K % 8 != 0 || (((uintptr_t)it.w) & 15) != 0) continue;
      TRY(build_tile_major(e, it.w, it.N, it.K, e->tiled_buf + off, st));
      e->tiled[it.w] = {e->tiled_buf + off, it.N, it.K};
      off += tile_major_bytes(it.N, it.K);
    }
  }
  CK(cudaStreamSynchronize(st));
  e->finalized = true;
  return 0;
}

// ------------------------------------------------------------------------------ a9
extern "C" int pg_embed_tokens(pg_engine* e, const int32_t* ids, int n_tokens, float* x_out, void* stream) {
  TRY(check_ready(e));
  NEED(table, float, "embed_tokens");
  return launch(e, embed_gather_kernel, dim3(n_tokens), dim3(256), 0, (cudaStream_t)stream, ids, table, x_out, e->d.D,
                e->d.vocab);
}

// ------------------------------------------------------------------------------ LM layers
static int elementwise_blocks(pg_engine* e, size_t total) {
  return (int)std::max<size_t>(1, std::min<size_t>((total + 255) / 256, (size_t)e->num_sms * 16));
}

// gate|up projection + SwiGLU -> hbuf.  bf16 + tcgen05: one kernel (fused epilogue, interleaved weight rows);
// otherwise the contraction followed by swiglu_kernel.
// (decode-sized token counts only: with 256-token tiles the two gate warps' expf work would outlast the MMAs)
static bool fused_swiglu_ok(const pg_engine* e, int tok) { return e->bf16 && e->use_tc && e->d.F % 64 == 0 && tok <= 128; }

// Stream-K gate|up + SwiGLU (gemm_sk.cuh) of X [tok][D] (tok <= 64) against the tile-major gate|up weight [2F][D] into
// h [tok][F].  ctas: the grid, 0 = one CTA per SM (at most one per unit).  scratch holds n_tiles x max_contrib partial
// tiles; counters[n_tiles] are zero on entry and zero again once the launch completes.
static int launch_swiglu_sk(pg_engine* e, const void* X, const uint8_t* w_tiled, int tok, int F, int D, int ctas, float* scratch,
                            size_t scratch_bytes, int* counters, int n_counters, bf16* h_out, cudaStream_t st) {
  if (tok < 1 || tok > 64) return fail("stream-K SwiGLU: M=%d must be in [1, 64]", tok);
  if (F % 64 != 0 || D % TC_BK != 0) return fail("stream-K SwiGLU: F=%d must be a multiple of 64 and D=%d of %d", F, D, TC_BK);
  const int NT = tok <= 16 ? 16 : tok <= 32 ? 32 : 64;
  const int n_tiles = 2 * F / TC_BM, num_kb = D / TC_BK;
  const long U = (long)n_tiles * num_kb;
  if (ctas < 0 || ctas > e->num_sms) return fail("stream-K SwiGLU: ctas=%d must be in [0, num_sms=%d]", ctas, e->num_sms);
  const int G = (int)std::min<long>(ctas > 0 ? ctas : e->num_sms, U);
  const int per_min = (int)std::max<long>(1, U / G);
  const int max_contrib = (num_kb + per_min - 1) / per_min + 1;
  // a CTA keeps at most SKG_MAX_FRAGS fragments; one whose range touched more tiles would drop the rest, and their
  // finishers would wait for partials nobody publishes
  for (int c = 0; c < G; ++c) {
    const long u0 = ((long)c * U) / G, u1 = ((long)(c + 1) * U) / G;
    if (u1 > u0 && (u1 - 1) / num_kb - u0 / num_kb + 1 > SKG_MAX_FRAGS)
      return fail("stream-K SwiGLU: CTA %d of %d spans %ld tiles (at most %d fragments per CTA; %ld units of %d k-blocks)", c, G,
                  (u1 - 1) / num_kb - u0 / num_kb + 1, SKG_MAX_FRAGS, U, num_kb);
  }
  if ((size_t)n_tiles * max_contrib * NT * TC_BM * 4 > scratch_bytes)
    return fail("stream-K SwiGLU: scratch of %zu bytes holds fewer than %d tiles x %d contributors x %d x %d fp32", scratch_bytes, n_tiles,
                max_contrib, NT, TC_BM);
  if (n_counters < n_tiles) return fail("stream-K SwiGLU: %d counters for %d tiles", n_counters, n_tiles);
  CUtensorMap mx;
  TRY(make_map_2d(e, &mx, X, (uint64_t)tok, (uint64_t)D, (uint32_t)NT));
  const int stage_bytes = TC_A_BYTES + NT * TC_BK * 2;
  int stages = std::min(12, (200 * 1024) / stage_bytes) & ~1;
  const size_t smem = (size_t)stages * stage_bytes + SKG_XCH_BYTES + 1024 + 512;
  e->last_path = PG_PATH_SK; e->last_nt = NT;
  if (NT == 64)
    return launch(e, gemm_swiglu_sk_kernel<64>, dim3(G), dim3(SKG_THREADS), smem, st, mx, w_tiled, tok, F, n_tiles, num_kb, stages,
                  e->use_pdl, scratch, max_contrib, counters, h_out, next_prof(e));
  if (NT == 16)
    return launch(e, gemm_swiglu_sk_kernel<16>, dim3(G), dim3(SKG_THREADS), smem, st, mx, w_tiled, tok, F, n_tiles, num_kb, stages,
                  e->use_pdl, scratch, max_contrib, counters, h_out, next_prof(e));
  return launch(e, gemm_swiglu_sk_kernel<32>, dim3(G), dim3(SKG_THREADS), smem, st, mx, w_tiled, tok, F, n_tiles, num_kb, stages,
                e->use_pdl, scratch, max_contrib, counters, h_out, next_prof(e));
}

static int k_gate_up(pg_engine* e, const LayerW& w, int tok, cudaStream_t st) {
  const pg_dims& d = e->d;
  const int F = d.F, D = d.D;
  int S = 1;
  // Stream-K over all SMs (gemm_sk.cuh) when the one-CTA-per-tile launch would need more than one wave (Janus-Pro-7B:
  // 172 tiles on 148 SMs; measured 4.17 -> 3.98 ms per step at B=16).  With fewer tiles than SMs (Janus-1.3B: 88) the
  // plain launch is faster (1.49 vs 1.58 ms per step): the SMs it leaves free are not idle, they host the early-launched
  // CTAs of the down projection prefetching their weights.  gu_streamk = 2 forces it.
  if (fused_swiglu_ok(e, tok) && tok <= 64 && D % TC_BK == 0 &&
      (e->gu_streamk == 2 || (e->gu_streamk == 1 && 2 * F / TC_BM > e->num_sms))) {
    auto it = e->tiled.find(w.wgu);
    if (it != e->tiled.end() && it->second.N == 2 * F && it->second.K == D)
      return launch_swiglu_sk(e, e->xn, it->second.ptr, tok, F, D, 0, e->part, e->part_bytes, e->sk_counters, 2 * F / TC_BM,
                              (bf16*)e->hbuf, st);
  }
  if (fused_swiglu_ok(e, tok)) return run_gemm(e, e->xn, w.wgu, tok, 2 * F, D, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, e->hbuf);
  TRY(run_gemm(e, e->xn, w.wgu, tok, 2 * F, D, e->part, e->part_bytes, &S, st));
  const size_t total = (size_t)tok * F;
  const int il = (e->bf16 && F % 64 == 0) ? 1 : 0;         // bf16 weights are packed interleaved when F % 64 == 0 (weights.py)
  DISPATCH_T(e,
             launch(e, swiglu_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, (size_t)tok * 2 * F, (bf16*)e->hbuf, F, total, il, next_prof(e)),
             launch(e, swiglu_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, (size_t)tok * 2 * F, (float*)e->hbuf, F, total, il, next_prof(e)));
  return 0;
}

extern "C" int pg_host_group_rows(const int32_t* start, const uint64_t* hash, int R, int32_t* source_row) {
  if (!start || !hash || !source_row || R < 0) return -1;
  std::map<std::pair<int32_t, uint64_t>, int> first;
  int proposals = 0;
  for (int r = 0; r < R; ++r) {
    auto ins = first.emplace(std::make_pair(start[r], hash[r]), r);
    source_row[r] = ins.first->second;
    if (!ins.second) ++proposals;
  }
  return proposals;
}

// One prefill-attention launch (prefill_impl and pg_test_attn_prefill_io).  q / out: [tok][H*128] in the engine's dtype,
// tok = R*P (padded) or row_off[R] (packed stream, tcgen05 only); kcache / vcache: [R][H][Tmax][128].
static int launch_prefill_attn(pg_engine* e, bool tc, const void* q, int tok, const void* kcache, const void* vcache,
                               const int32_t* kv_start, const int32_t* row_off, void* out, int R, int P, int H, int Tmax,
                               cudaStream_t st) {
  const float scale = 1.0f / sqrtf((float)HEAD_DIM);
  if (tc) {
    // tensor-core path: one CTA per (row, head, 128-query tile); V is read from the cache rows as an MN-major operand
    CUtensorMap mq, mk, mv;
    TRY(make_map_2d(e, &mq, q, (uint64_t)tok, (uint64_t)H * HEAD_DIM, PA_BQ));
    TRY(make_map_2d(e, &mk, kcache, (uint64_t)R * H * Tmax, (uint64_t)HEAD_DIM, PA_BK));
    TRY(make_map_2d(e, &mv, vcache, (uint64_t)R * H * Tmax, (uint64_t)HEAD_DIM, PA_BK));
    return launch(e, attn_prefill_tc_kernel, dim3((P + PA_BQ - 1) / PA_BQ, H, R), dim3(128), PA_SMEM, st, mq, mk, mv, kv_start,
                  (bf16*)out, P, H, Tmax, scale, row_off);
  }
  DISPATCH_T(e,
             launch(e, attn_prefill_kernel<bf16>, dim3((P + 63) / 64, H, R), dim3(256), ATTN_PREFILL_SMEM, st, (const bf16*)q,
                    (const bf16*)kcache, (const bf16*)vcache, kv_start, (bf16*)out, P, H, Tmax, scale),
             launch(e, attn_prefill_kernel<float>, dim3((P + 63) / 64, H, R), dim3(256), ATTN_PREFILL_SMEM, st, (const float*)q,
                    (const float*)kcache, (const float*)vcache, kv_start, (float*)out, P, H, Tmax, scale));
  return 0;
}

// One SigLIP attention launch (the vision tower and pg_test_vit_attn_io).  qkv: [qkv_rows][3W] in the engine's dtype,
// image i in rows [i*NP, (i+1)*NP); out: [n*NP][W].  The tcgen05 kernel's maps cover all qkv_rows.
static int launch_vit_attn(pg_engine* e, bool tc, const void* qkv, int qkv_rows, void* out, int n, int NP, int W, int heads,
                           cudaStream_t st) {
  const int hd = W / heads;
  const float scale = 1.0f / sqrtf((float)hd);
  if (tc) {
    CUtensorMap mq, mk;      // K and V rows both through mk (V read in place as an MN-major operand)
    TRY(make_map_2d(e, &mq, qkv, (uint64_t)qkv_rows, (uint64_t)3 * W, VT_BQ));
    TRY(make_map_2d(e, &mk, qkv, (uint64_t)qkv_rows, (uint64_t)3 * W, VT_BK));
    return launch(e, vit_attn_tc_kernel, dim3((NP + VT_BQ - 1) / VT_BQ, heads, n), dim3(128), VT_SMEM, st, mq, mk, (bf16*)out,
                  NP, W, scale);
  }
  DISPATCH_T(e,
             launch(e, vit_attn_kernel<bf16>, dim3((NP + 3) / 4, heads, n), dim3(128), 0, st, (const bf16*)qkv, (bf16*)out, NP, W, heads, hd, scale),
             launch(e, vit_attn_kernel<float>, dim3((NP + 3) / 4, heads, n), dim3(128), 0, st, (const float*)qkv, (float*)out, NP, W, heads, hd, scale));
  return 0;
}

// a3: prompt prefill.  x fp32 [R*P, D] in place.
static int prefill_impl(pg_engine* e, float* x, const int32_t* kv_start, int R, int P, float* hidden_out, int all_positions,
                        bool rope_rel, void* stream, int tail = 0);
extern "C" int pg_prefill(pg_engine* e, float* x, const int32_t* kv_start, int R, int P, float* hidden_out,
                          int all_positions, void* stream) {
  return prefill_impl(e, x, kv_start, R, P, hidden_out, all_positions, false, stream);
}
// rope_rel: RoPE positions = column - kv_start[row] (what HF generate() derives from the attention mask, x2t);
// otherwise absolute columns (the image loop calls LlamaModel.forward without position_ids).
// tail > 0 (pg_score_image_tokens): no last-row output; instead the final-norm'ed hidden states of the last `tail` columns
// of every row go to hbuf in the activation type, pair-major (row ((r / 2) * tail + i) * 2 + r % 2).
static int prefill_impl(pg_engine* e, float* x, const int32_t* kv_start, int R, int P, float* hidden_out, int all_positions,
                        bool rope_rel, void* stream, int tail) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (R < 1 || R > d.max_rows || P < 1 || P > d.max_prompt) return fail("prefill shape R=%d P=%d exceeds engine limits", R, P);
  cudaStream_t st = (cudaStream_t)stream;
  NEED(cosT, float, "rope_cos");
  NEED(sinT, float, "rope_sin");
  NEED(normw, float, "norm");
  const int D = d.D, HD = e->HD, F = d.F;
  int tok = R * P;
  int S = 1;
  // ---- packed prefill (fused loops only: the drop-in call returns every position, pads included)
  const int32_t* row_off = nullptr;
  int packed_dups = 0;
  if (!all_positions && e->bf16 && e->use_tc && e->prefill_attn_tc && e->prefill_pack && D % 8 == 0 && HD % 8 == 0 &&
      F % 64 == 0) {
    if (!e->row_off_host) CK(cudaMallocHost(&e->row_off_host, (size_t)(3 * d.max_rows + 2) * 4));
    if (!e->row_hash_host) CK(cudaMallocHost(&e->row_hash_host, (size_t)d.max_rows * 8));
    int32_t* differs_host = e->row_off_host + d.max_rows + 1;
    int32_t* dup_host = e->row_off_host + 2 * d.max_rows + 1;
    const bool dedup = e->prefill_dedup && R > 1 && D % 4 == 0;
    if (dedup) {
      CK(cudaMemsetAsync(e->row_hash, 0, (size_t)R * 8, st));
      prefill_row_hash_kernel<<<dim3(P, R), 256, 0, st>>>((const float*)x, kv_start, e->row_hash, P, D);
      CK(cudaGetLastError());
      e->launches++;
      CK(cudaMemcpyAsync(e->row_hash_host, e->row_hash, (size_t)R * 8, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaMemcpyAsync(e->row_off_host, kv_start, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::vector<int32_t> off((size_t)R + 1, 0), dup((size_t)R, 0), start((size_t)R, 0);
    for (int r = 0; r < R; ++r) { start[r] = e->row_off_host[r]; dup[r] = r; }
    if (dedup) {
      // proposal: the first row with the same left padding and content hash; verified word for word on the device
      const int proposals = pg_host_group_rows(start.data(), (const uint64_t*)e->row_hash_host, R, dup.data());
      if (proposals > 0) {
        memcpy(dup_host, dup.data(), (size_t)R * 4);
        CK(cudaMemcpyAsync(e->dup_of, dup_host, (size_t)R * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemsetAsync(e->row_differs, 0, (size_t)R * 4, st));
        prefill_row_verify_kernel<<<dim3(P, R), 256, 0, st>>>((const float*)x, kv_start, (const int32_t*)e->dup_of, e->row_differs, P, D);
        CK(cudaGetLastError());
        e->launches++;
        CK(cudaMemcpyAsync(differs_host, e->row_differs, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int r = 0; r < R; ++r) if (dup[r] != r && differs_host[r] != 0) dup[r] = r;
      }
    }
    bool ok = true;
    int n_dup = 0;
    for (int r = 0; r < R; ++r) {
      const int len = P - start[r];
      if (len < 1 || len > P) ok = false;                  // an empty row: leave it to the padded path
      if (dup[r] != r) ++n_dup;
      off[r + 1] = off[r] + (dup[r] == r ? std::max(len, 0) : 0);
    }
    if (ok && off[R] < R * P) {
      memcpy(e->row_off_host, off.data(), (size_t)(R + 1) * 4);
      CK(cudaMemcpyAsync(e->row_off, e->row_off_host, (size_t)(R + 1) * 4, cudaMemcpyHostToDevice, st));
      memcpy(dup_host, dup.data(), (size_t)R * 4);
      CK(cudaMemcpyAsync(e->dup_of, dup_host, (size_t)R * 4, cudaMemcpyHostToDevice, st));
      packed_dups = n_dup;
      TRY(launch(e, prefill_pack_kernel, dim3(P, R), dim3(256), 0, st, (const float*)x, e->xpack, kv_start, (const int32_t*)e->row_off, P, D));
      x = e->xpack;
      tok = off[R];
      row_off = e->row_off;
    }
  }
  if (row_off == nullptr) {     // no packed prefill, no de-duplication: every row owns its prompt K / V (decode attention's src_row)
    iota_i32_kernel<<<(R + 255) / 256, 256, 0, st>>>(e->dup_of, R);
    CK(cudaGetLastError());
    e->launches++;
  }
  // fused epilogues (bf16 regime on tcgen05): QKV and gate|up leave the contraction as bf16 rows, O and down add straight
  // into the fp32 residual stream - no fp32 partial round trip (same values: the row kernels rounded the partials first)
  const bool fuse = e->bf16 && e->use_tc && D % 8 == 0 && HD % 8 == 0 && F % 64 == 0 &&
                    (size_t)tok * std::max(3 * HD, 2 * F) * 2 <= e->part_bytes;
  bf16* stage16 = (bf16*)e->part;
  for (int l = 0; l < d.L; ++l) {
    LayerW w;
    TRY(layer_weights(e, l, &w));
    if (l == 0) TRY(k_resid_norm(e, x, nullptr, 0, 0, w.ln1, e->xn, nullptr, tok, 1, 0, 0, st));
    if (fuse && e->prefill_qkv_fuse && tok > 128) {
      // RoPE + q / K / V stores in the contraction's epilogue (gemm.cuh QkvEpi)
      EpiFuse ep = {nullptr, (bf16*)e->qbuf, nullptr, 3};
      e->qkv_epi_next = QkvEpi{cosT, sinT, (bf16*)e->qbuf, (bf16*)kv_ptr(e, l, 0, R), (bf16*)kv_ptr(e, l, 1, R), row_off, kv_start,
                               rope_rel ? kv_start : (const int32_t*)nullptr, R, P, d.H, e->Tmax};
      TRY(run_gemm(e, e->xn, w.wqkv, tok, 3 * HD, D, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, nullptr, &ep));
      e->qkv_epi_next = QkvEpi{};
    } else if (fuse) {
      EpiFuse ep = {nullptr, stage16, nullptr, 0};
      TRY(run_gemm(e, e->xn, w.wqkv, tok, 3 * HD, D, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, nullptr, &ep));
      TRY(launch(e, qkv_rope_store_bf16_kernel, dim3(tok), dim3(256), 0, st, (const bf16*)stage16, cosT, sinT, (bf16*)e->qbuf,
                 (bf16*)kv_ptr(e, l, 0, R), (bf16*)kv_ptr(e, l, 1, R), P, d.H, e->Tmax, rope_rel ? kv_start : (const int32_t*)nullptr,
                 row_off, kv_start, R));
    } else {
    TRY(run_gemm(e, e->xn, w.wqkv, tok, 3 * HD, D, e->part, e->part_bytes, &S, st));
    DISPATCH_T(e,
               launch(e, qkv_rope_store_kernel<bf16>, dim3(tok), dim3(256), 0, st, e->part, S, (size_t)tok * 3 * HD, cosT, sinT,
                      (bf16*)e->qbuf, (bf16*)kv_ptr(e, l, 0, R), (bf16*)kv_ptr(e, l, 1, R), P, d.H, e->Tmax,
                      rope_rel ? kv_start : (const int32_t*)nullptr),
               launch(e, qkv_rope_store_kernel<float>, dim3(tok), dim3(256), 0, st, e->part, S, (size_t)tok * 3 * HD, cosT, sinT,
                      (float*)e->qbuf, (float*)kv_ptr(e, l, 0, R), (float*)kv_ptr(e, l, 1, R), P, d.H, e->Tmax,
                      rope_rel ? kv_start : (const int32_t*)nullptr));
    }
    TRY(launch_prefill_attn(e, e->bf16 && e->use_tc && e->prefill_attn_tc, e->qbuf, tok, kv_ptr(e, l, 0, R), kv_ptr(e, l, 1, R),
                            kv_start, row_off, e->attn_out, R, P, d.H, e->Tmax, st));
    if (fuse) {
      EpiFuse er = {nullptr, nullptr, x, 0};
      TRY(run_gemm(e, e->attn_out, w.wo, tok, D, HD, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, nullptr, &er));
      TRY(k_resid_norm(e, x, nullptr, 0, 0, w.ln2, e->xn, nullptr, tok, 1, 0, 0, st));
      if (fused_swiglu_ok(e, tok)) {
        TRY(k_gate_up(e, w, tok, st));
      } else {
        // SwiGLU in the CTA-pair contraction's epilogue (gemm_tc2.cuh, EpiFuse::gelu == 2): h leaves the kernel directly
        EpiFuse eg = {nullptr, (bf16*)e->hbuf, nullptr, 2};
        TRY(run_gemm(e, e->xn, w.wgu, tok, 2 * F, D, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, nullptr, &eg));
      }
      TRY(run_gemm(e, e->hbuf, w.wd, tok, D, F, e->part, e->part_bytes, &S, st, -1, 0, true, nullptr, nullptr, &er));
      if (l + 1 < d.L) {
        LayerW wn;
        TRY(layer_weights(e, l + 1, &wn));
        TRY(k_resid_norm(e, x, nullptr, 0, 0, wn.ln1, e->xn, nullptr, tok, 1, 0, 0, st));
      }
      continue;
    }
    TRY(run_gemm(e, e->attn_out, w.wo, tok, D, HD, e->part, e->part_bytes, &S, st));
    TRY(k_resid_norm(e, x, e->part, S, (size_t)tok * D, w.ln2, e->xn, nullptr, tok, 1, 0, 0, st));
    TRY(k_gate_up(e, w, tok, st));
    TRY(run_gemm(e, e->hbuf, w.wd, tok, D, F, e->part, e->part_bytes, &S, st));
    if (l + 1 < d.L) {
      LayerW wn;
      TRY(layer_weights(e, l + 1, &wn));
      TRY(k_resid_norm(e, x, e->part, S, (size_t)tok * D, wn.ln1, e->xn, nullptr, tok, 1, 0, 0, st));
    }
  }
  // final norm: all positions -> caller's buffer; last position of every row -> hidden_t for gen_head
  const float* last_part = fuse ? nullptr : e->part;      // fused: the last down projection is already in the stream
  if (tail > 0) {
    TRY(k_resid_norm(e, x, last_part, S, (size_t)tok * D, normw, e->xn, nullptr, tok, 1, 0, 0, st));
    DISPATCH_T(e,
               launch(e, gather_tail_rows_kernel<bf16>, dim3(tail, R), dim3(256), 0, st, (const bf16*)e->xn, (bf16*)e->hbuf, row_off,
                      (const int32_t*)e->dup_of, kv_start, P, tail, D),
               launch(e, gather_tail_rows_kernel<float>, dim3(tail, R), dim3(256), 0, st, (const float*)e->xn, (float*)e->hbuf, row_off,
                      (const int32_t*)e->dup_of, kv_start, P, tail, D));
    return 0;
  }
  if (row_off != nullptr) {
    // packed: the last real token of every row
    if (packed_dups > 0)     // rows that repeat an earlier row: their K / V strips are copies
      TRY(launch(e, kv_broadcast_rows_kernel, dim3(d.L * 2 * d.H, R), dim3(256), 0, st, (bf16*)e->kv, (const int32_t*)e->dup_of, kv_start, R, d.H,
                 e->Tmax, P));
    TRY(launch(e, gather_last_rows_kernel, dim3(R), dim3(256), 0, st, (const float*)x, e->x_last, row_off, (const int32_t*)e->dup_of, D));
    TRY(k_resid_norm(e, e->x_last, nullptr, 0, 0, normw, e->hidden_t, e->hidden_f, R, 1, 0, 0, st));
    if (hidden_out) CK(cudaMemcpyAsync(hidden_out, e->hidden_f, (size_t)R * D * 4, cudaMemcpyDeviceToDevice, st));
  } else if (all_positions) {
    TRY(k_resid_norm(e, x, last_part, S, (size_t)tok * D, normw, nullptr, hidden_out, tok, 1, 0, 0, st));
    TRY(k_resid_norm(e, x, nullptr, 0, 0, normw, e->hidden_t, e->hidden_f, R, P, P - 1, 0, st));
  } else {
    TRY(k_resid_norm(e, x, last_part, S, (size_t)tok * D, normw, e->hidden_t, e->hidden_f, R, P, P - 1, 0, st));
    if (hidden_out) CK(cudaMemcpyAsync(hidden_out, e->hidden_f, (size_t)R * D * 4, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

static int attn_split_count(pg_engine* e, int R, int T) {
  if (e->attn_splits > 0) return std::min(e->attn_splits, 64);
  const int ctas = R * e->d.H;
  int s = (4 * e->num_sms + ctas - 1) / ctas;
  s = std::min(s, std::max(1, T / 64));
  return std::max(1, std::min(s, 64));
}

// one decode step over e->x_dec (fp32 [R, D]); xn for layer 0 already in e->xn when first_norm_done
// regime 0: image-token decode (inputs_embeds = bf16 gen_aligner output => bf16 residual stream, bf16 trig, absolute
// positions); regime 1: text decode inside generate() (fp32 embed_tokens rows => fp32 residual stream, fp32 trig,
// mask-aware positions) - the rounding points HF's autocast produces for each input dtype
static int decode_layers(pg_engine* e, const int32_t* kv_start, int R, int pos_base, const int* step_ptr,
                         bool first_norm_done, bool inc_step, int T_hint, cudaStream_t st, int regime = 0, int alias_P = 0) {
  const pg_dims& d = e->d;
  NEED(cosT, float, "rope_cos");
  NEED(sinT, float, "rope_sin");
  NEED(normw, float, "norm");
  const int D = d.D, HD = e->HD, F = d.F;
  const float scale = 1.0f / sqrtf((float)HEAD_DIM);
  const int rflag = (e->bf16 && regime == 0) ? RN_ROUND_RESID : 0;
  const int trig = regime == 0 ? (e->bf16 ? 1 : 0) : ROPE_REL;
  const int nsp = attn_split_count(e, R, T_hint);
  int S = 1;
  for (int l = 0; l < d.L; ++l) {
    LayerW w;
    TRY(layer_weights(e, l, &w));
    if (l == 0 && !first_norm_done) TRY(k_resid_norm(e, e->x_dec, nullptr, 0, 0, w.ln1, e->xn, nullptr, R, 1, 0, rflag, st));
    TRY(run_gemm(e, e->xn, w.wqkv, R, 3 * HD, D, e->part, e->part_bytes, &S, st));
    if (e->bf16 && e->attn_impl >= 1 && R <= AT_MAX_ROWS) {
      const int ctas = e->attn_ctas > 0 ? e->attn_ctas : e->num_sms;
      TRY(launch(e, attn_decode_v5_kernel, dim3(ctas), dim3(AT_THREADS), A5_SMEM, st, e->part, S, (size_t)R * 3 * HD, cosT, sinT,
                 (bf16*)kv_ptr(e, l, 0, R), (bf16*)kv_ptr(e, l, 1, R), kv_start, (bf16*)e->attn_out, e->attn_ll,
                 R, d.H, e->Tmax, pos_base, step_ptr, scale, trig, 1, next_prof(e), (unsigned long long*)nullptr,
                 (const int32_t*)((alias_P > 0 && e->attn_alias) ? e->dup_of : nullptr), alias_P));
    } else {
    DISPATCH_T(e,
                 launch(e, attn_decode_kernel<bf16>, dim3(d.H, R, nsp), dim3(128), 0, st, e->part, S, (size_t)R * 3 * HD, cosT, sinT,
                        (bf16*)kv_ptr(e, l, 0, R), (bf16*)kv_ptr(e, l, 1, R), kv_start, (bf16*)e->attn_out, e->attn_ws,
                        e->attn_cnt, d.H, e->Tmax, pos_base, step_ptr, scale, trig),
                 launch(e, attn_decode_kernel<float>, dim3(d.H, R, nsp), dim3(128), 0, st, e->part, S, (size_t)R * 3 * HD, cosT, sinT,
                        (float*)kv_ptr(e, l, 0, R), (float*)kv_ptr(e, l, 1, R), kv_start, (float*)e->attn_out, e->attn_ws,
                        e->attn_cnt, d.H, e->Tmax, pos_base, step_ptr, scale, trig));
    }
    TRY(run_gemm(e, e->attn_out, w.wo, R, D, HD, e->part, e->part_bytes, &S, st));
    TRY(k_resid_norm(e, e->x_dec, e->part, S, (size_t)R * D, w.ln2, e->xn, nullptr, R, 1, 0, rflag, st));
    TRY(k_gate_up(e, w, R, st));
    // gate|up runs one CTA per weight tile; when that leaves SMs free (Janus-1.3B: 88 tiles on 148 SMs) the early-launched
    // CTAs of the down projection start on them and have their weight share in flight before gate|up ends.  With an 80 KB
    // ring (4 stages) instead of 200 KB TWO of them fit on a free SM: 120 of the 144 CTAs prefetch early instead of 60
    // (measured at R = 32: 1.469 -> 1.453 ms per step; 6 or 8 stages are slower than either).  Only there: with 16 or fewer
    // rows (1.212 -> 1.241 ms at R = 16) and with 64 (1.651 -> 1.673) the deep ring wins, and without free SMs (stream-K) too.
    if (e->bf16 && e->use_tc && e->down_stages > 0 && 2 * F / TC_BM < e->num_sms && R > 16 && R <= 32) e->stage_cap_once = e->down_stages;
    TRY(run_gemm(e, e->hbuf, w.wd, R, D, F, e->part, e->part_bytes, &S, st));
    e->stage_cap_once = 0;
    if (l + 1 < d.L) {
      LayerW wn;
      TRY(layer_weights(e, l + 1, &wn));
      TRY(k_resid_norm(e, e->x_dec, e->part, S, (size_t)R * D, wn.ln1, e->xn, nullptr, R, 1, 0, rflag, st));
    }
  }
  TRY(k_resid_norm(e, e->x_dec, e->part, S, (size_t)R * D, normw, e->hidden_t, e->hidden_f, R, 1, 0,
                   rflag | (inc_step ? RN_INC_STEP : 0), st));
  return 0;
}

// a4
extern "C" int pg_decode_step(pg_engine* e, const float* x, const int32_t* kv_start, int R, int pos, float* hidden_out,
                              void* stream) {
  TRY(check_ready(e));
  if (R < 1 || R > e->d.max_rows || pos < 0 || pos >= e->Tmax) return fail("decode shape R=%d pos=%d exceeds engine limits", R, pos);
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(e->x_dec, x, (size_t)R * e->d.D * 4, cudaMemcpyDeviceToDevice, st));
  TRY(decode_layers(e, kv_start, R, pos, nullptr, false, false, pos + 1, st));
  if (hidden_out) CK(cudaMemcpyAsync(hidden_out, e->hidden_f, (size_t)R * e->d.D * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// gen_head GEMMs: X (hidden_t, activation type) -> H (head_h) -> logits partials in e->part.  Returns split count / stride.
static int head_gemms(pg_engine* e, const void* X, void* H, int R, int* S_out, cudaStream_t st) {
  const pg_dims& d = e->d;
  NEED(w0, void, "head.w0");
  NEED(b0, float, "head.b0");
  NEED(w1, void, "head.w1");
  int S = 1;
  TRY(run_gemm(e, X, w0, R, d.img_embed, d.D, e->part, e->part_bytes, &S, st));
  const size_t total = (size_t)R * d.img_embed;
  DISPATCH_T(e,
             launch(e, bias_act_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, total, b0, (bf16*)H, (float*)nullptr, d.img_embed, total, 1),
             launch(e, bias_act_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, total, b0, (float*)H, (float*)nullptr, d.img_embed, total, 1));
  TRY(run_gemm(e, H, w1, R, d.img_vocab, d.img_embed, e->part, e->part_bytes, &S, st));
  *S_out = S;
  return 0;
}

// a5
extern "C" int pg_gen_head(pg_engine* e, const float* hidden, int R, float* logits_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (R < 1 || R > d.max_rows) return fail("gen_head R=%d exceeds engine limits", R);
  cudaStream_t st = (cudaStream_t)stream;
  NEED(b1, float, "head.b1");
  // cast the caller's fp32 hidden states to the activation type (autocast cast at the Linear)
  const size_t n = (size_t)R * d.D;
  DISPATCH_T(e,
             launch(e, bias_act_kernel<bf16>, dim3(elementwise_blocks(e, n)), dim3(256), 0, st, hidden, 1, n, (const float*)nullptr, (bf16*)e->hidden_t, (float*)nullptr, d.D, n, 0),
             launch(e, bias_act_kernel<float>, dim3(elementwise_blocks(e, n)), dim3(256), 0, st, hidden, 1, n, (const float*)nullptr, (float*)e->hidden_t, (float*)nullptr, d.D, n, 0));
  int S = 1;
  TRY(head_gemms(e, e->hidden_t, e->head_h, R, &S, st));
  const size_t total = (size_t)R * d.img_vocab;
  DISPATCH_T(e,
             launch(e, bias_act_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, total, b1, (bf16*)nullptr, logits_out, d.img_vocab, total, 0),
             launch(e, bias_act_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->part, S, total, b1, (float*)nullptr, logits_out, d.img_vocab, total, 0));
  return 0;
}

static void philox_policy(pg_engine* e, size_t numel, uint64_t* counter_offset, uint64_t* stride) {
  // torch calc_execution_policy (ATen/native/cuda/DistributionTemplates.h:50-62), unroll 4, block 256
  const uint64_t block = 256;
  uint64_t grid = (numel + block - 1) / block;
  const uint64_t cap = (uint64_t)e->num_sms * (e->max_threads_per_sm / block);
  grid = std::min(grid, cap);
  *counter_offset = ((numel - 1) / (block * grid * 4) + 1) * 4;
  *stride = grid * block;
}

// The sampling settings of one sampler launch or decode loop, staged in engine memory (stage_per_image):
// `dev` = st_sampling [B], cfg_sched = st_cfg [B][n] or nullptr (dev's cfg_weight).  any_top_p: some image has top_p < 1.
struct PerImage {
  const ImageSampling* dev;
  int rng_per_image;
  bool any_top_p;
  const float* cfg_sched;
};

// Philox element count of one draw: the whole (B, V) tensor, or one image's (1, V) row with per-image generators
static size_t philox_numel(const pg_engine* e, int B, const PerImage& pi) {
  return (pi.rng_per_image ? 1 : (size_t)B) * e->d.img_vocab;
}

// top-p threshold: what torch compares the fp32 cumulative sum with, fp32(1 - top_p) with 1 - top_p in double; -1 = off
static float top_p_threshold(double top_p) { return top_p < 1.0 ? (float)(1.0 - top_p) : -1.f; }

static int k_sample(pg_engine* e, const float* part, int S, size_t sstride, const float* bias, int B, uint64_t offset_base,
                    int greedy, const int32_t* edit_region, const int32_t* gt_labels, int step_base, const int* step_ptr,
                    int n_steps, int32_t* tokens_out, float* x_next, const float* next_norm_w, void* xn_next, cudaStream_t st,
                    const PerImage& pi, float* logprobs = nullptr, int score_n = 0) {
  const pg_dims& d = e->d;
  uint64_t per_step, stride;
  philox_policy(e, philox_numel(e, B, pi), &per_step, &stride);
  const size_t chunk = (size_t)((d.img_vocab + SAMPLE_CLUSTER - 1) / SAMPLE_CLUSTER);
  size_t csm = chunk * 4;
  // top-p: the kernel keeps the logits and the select's 5 x 256 fixed-point mass histograms in dynamic shared memory
  // (per image: sized when any image uses it; the others skip the select)
  if (pi.any_top_p) {
    csm = ((chunk + 1) & ~(size_t)1) * 8 + 5 * 256 * 8;
    if (csm > 48 * 1024) return fail("top_p needs %zu B of shared memory per CTA at img_vocab %d (48 KB available)", csm, d.img_vocab);
  }
  DISPATCH_T(e,
             launch(e, cfg_sample_embed_cluster_kernel<bf16>, dim3(B * SAMPLE_CLUSTER), dim3(SAMPLE_CL_THREADS), csm, st, part, S, sstride, bias, B, d.img_vocab,
                    offset_base, per_step, stride, greedy, edit_region, gt_labels, step_base, step_ptr, n_steps, tokens_out,
                    (const bf16*)e->embed_table, d.D, x_next, next_norm_w, (bf16*)xn_next, d.rms_eps, 1,
                    score_n ? nullptr : e->dbg_logits, pi.dev, pi.rng_per_image, logprobs, score_n, pi.cfg_sched),
             launch(e, cfg_sample_embed_cluster_kernel<float>, dim3(B * SAMPLE_CLUSTER), dim3(SAMPLE_CL_THREADS), csm, st, part, S, sstride, bias, B, d.img_vocab,
                    offset_base, per_step, stride, greedy, edit_region, gt_labels, step_base, step_ptr, n_steps, tokens_out,
                    (const float*)e->embed_table, d.D, x_next, next_norm_w, (float*)xn_next, d.rms_eps, 0,
                    score_n ? nullptr : e->dbg_logits, pi.dev, pi.rng_per_image, logprobs, score_n, pi.cfg_sched));
  return 0;
}

// The caller's sampling settings, validated (naming the image) and converted to the kernel's entries on the host, the
// only place they are checked.  Batch-wide RNG: every entry takes image 0's seed and offset.  cfg_sched: the guidance
// schedule [B][n] (empty: none).
struct StagedSampling {
  std::vector<ImageSampling> dev;
  int rng_per_image = 0;
  bool any_top_p = false;
  std::vector<float> cfg_sched;
};

static int convert_per_image(const pg_image_sampling* h, int B, int rng_per_image, StagedSampling* out) {
  if (!h) return fail("null argument");
  out->dev.resize((size_t)B);
  out->rng_per_image = rng_per_image ? 1 : 0;
  out->any_top_p = false;
  for (int b = 0; b < B; ++b) {
    if (h[b].top_k < 0) return fail("image %d: top_k must be >= 0, got %d", b, h[b].top_k);
    if (!(h[b].top_p >= 0.0 && h[b].top_p <= 1.0)) return fail("image %d: top_p must be in [0, 1], got %g", b, h[b].top_p);
    const pg_image_sampling& rng = h[rng_per_image ? b : 0];
    out->dev[b] = {rng.seed, rng.offset, h[b].cfg_weight, h[b].temperature, h[b].top_k, top_p_threshold(h[b].top_p)};
    out->any_top_p |= h[b].top_p < 1.0;
  }
  return 0;
}

// The caller's guidance schedule (HOST [B][n]), checked on the host (no device sync; a failure names the entry) and kept
// in `out` for stage_per_image.
static int convert_schedule(const float* h, int B, int n, StagedSampling* out) {
  if (!h) return fail("null argument");
  for (int b = 0; b < B; ++b)
    for (int i = 0; i < n; ++i)
      if (!std::isfinite(h[(size_t)b * n + i]))
        return fail("image %d, step %d: cfg_schedule must be finite, got %g", b, i, h[(size_t)b * n + i]);
  out->cfg_sched.assign(h, h + (size_t)B * n);
  return 0;
}

// copy into st_sampling (and st_cfg) on `st` (plain copies from pageable memory: `ss` may go when it returns)
static int stage_per_image(pg_engine* e, const StagedSampling& ss, cudaStream_t st, PerImage* out) {
  CK(cudaMemcpyAsync(e->st_sampling, ss.dev.data(), ss.dev.size() * sizeof(ImageSampling), cudaMemcpyHostToDevice, st));
  const bool sched = !ss.cfg_sched.empty();
  if (sched)
    CK(cudaMemcpyAsync(e->st_cfg, ss.cfg_sched.data(), ss.cfg_sched.size() * 4, cudaMemcpyHostToDevice, st));
  *out = {e->st_sampling, ss.rng_per_image, ss.any_top_p, sched ? e->st_cfg : nullptr};
  return 0;
}

// a6-a8
extern "C" int pg_cfg_sample_embed(pg_engine* e, const float* logits, int B, const pg_image_sampling* per_image,
                                   int rng_per_image, int greedy, const int32_t* edit_region, const int32_t* gt_labels,
                                   int step, int n_steps, int32_t* tokens_out, float* x_next, float* logprobs_out,
                                   void* stream) {
  TRY(check_ready(e));
  if (B < 1 || 2 * B > e->d.max_rows) return fail("sample B=%d exceeds engine limits", B);
  if (step < 0 || step >= n_steps) return fail("step %d out of range", step);
  if ((edit_region == nullptr) != (gt_labels == nullptr)) return fail("edit_region and gt_labels go together");
  StagedSampling ss;
  TRY(convert_per_image(per_image, B, rng_per_image, &ss));
  cudaStream_t st = (cudaStream_t)stream;
  PerImage pi;
  TRY(stage_per_image(e, ss, st, &pi));
  return k_sample(e, logits, 1, 0, nullptr, B, 0, greedy, edit_region, gt_labels, step, nullptr, n_steps, tokens_out, x_next,
                  nullptr, nullptr, st, pi, logprobs_out);
}

extern "C" int pg_prepare_gen_img_embeds(pg_engine* e, const int32_t* ids, int n, float* out, void* stream) {
  TRY(check_ready(e));
  cudaStream_t st = (cudaStream_t)stream;
  DISPATCH_T(e,
             launch(e, gen_embed_gather_kernel<bf16>, dim3(n), dim3(256), 0, st, ids, (const bf16*)e->embed_table, out, e->d.D, e->d.img_vocab),
             launch(e, gen_embed_gather_kernel<float>, dim3(n), dim3(256), 0, st, ids, (const float*)e->embed_table, out, e->d.D, e->d.img_vocab));
  return 0;
}

// ------------------------------------------------------------------------------ a2: the whole loop
// step_host >= 0: the host supplies the step index (plain launches); < 0: read the device-side counter
// (graph replays; consecutive graph launches are fully ordered, so kernels may read it before their
// PDL wait).
static int one_step(pg_engine* e, const int32_t* kv_start, int R, int P, int n_steps, int greedy, const int32_t* edit_region,
                    const int32_t* gt_labels, int32_t* tokens_out, bool with_lm, int step_host, cudaStream_t st,
                    const PerImage& pi, float* logprobs) {
  NEED(b1, float, "head.b1");
  LayerW w0;
  TRY(layer_weights(e, 0, &w0));
  int S = 1;
  TRY(head_gemms(e, e->hidden_t, e->head_h, R, &S, st));
  const bool host = step_host >= 0;
  uint64_t per_step, stride;
  philox_policy(e, philox_numel(e, R / 2, pi), &per_step, &stride);
  TRY(k_sample(e, e->part, S, (size_t)R * e->d.img_vocab, b1, R / 2, host ? per_step * (uint64_t)step_host : 0, greedy,
               edit_region, gt_labels, host ? step_host : 0, host ? nullptr : e->step_ctr, n_steps, tokens_out,
               with_lm ? e->x_dec : nullptr, w0.ln1, with_lm ? e->xn : nullptr, st, pi, logprobs));
  if (with_lm)
    TRY(decode_layers(e, kv_start, R, host ? P + step_host : P, host ? nullptr : e->step_ctr, true, !host,
                      P + n_steps / 2, st, 0, P));
  return 0;
}

// Captured decode-step graphs, keyed by shape and scalars only: the per-call tensors live in engine-owned staging
// buffers (pg_engine::st_*), so a second call with the same shape replays the instantiated graph whatever addresses
// the caller's allocator hands out.  `capture` records one step on `st`.
template <typename F>
static int graph_for(pg_engine* e, const std::string& key, cudaStream_t st, F&& capture, pg_engine::GraphEntry** out) {
  auto it = e->graphs.find(key);
  if (it != e->graphs.end()) { *out = &it->second; return 0; }
  if (e->graphs.size() >= 8) drop_graphs(e);
  cudaGraph_t graph = nullptr;
  CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  const int64_t before = e->launches;
  int rc = capture();
  cudaError_t ce = cudaStreamEndCapture(st, &graph);
  const int64_t per_replay = e->launches - before;
  e->launches = before;
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (ce != cudaSuccess) return fail("stream capture failed: %s", cudaGetErrorString(ce));
  cudaGraphExec_t exec = nullptr;
  ce = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) return fail("graph instantiate failed: %s", cudaGetErrorString(ce));
  pg_engine::GraphEntry& ge = e->graphs[key];
  ge.exec = exec; ge.launches = per_replay;
  ++e->graph_captures;
  *out = &ge;
  return 0;
}

extern "C" int pg_sample_image(pg_engine* e, float* x_prompt, const int32_t* kv_start, int R, int P, int n_steps,
                               const pg_image_sampling* per_image, int rng_per_image, int greedy, const int32_t* edit_region,
                               const int32_t* gt_labels, const float* cfg_schedule_host, int32_t* tokens_out,
                               float* logprobs_out, void* stream) {
  TRY(check_ready(e));
  if (R % 2) return fail("R must be even (interleaved cond/uncond rows)");
  if (R < 2 || R > e->d.max_rows) return fail("sample_image R=%d exceeds engine limits", R);
  if (n_steps < 1 || n_steps > e->d.max_steps) return fail("n_steps %d exceeds engine limit %d", n_steps, e->d.max_steps);
  if ((edit_region == nullptr) != (gt_labels == nullptr)) return fail("edit_region and gt_labels go together ([R/2][n_steps] each)");
  if (!kv_start || !tokens_out) return fail("null argument");
  const int B = R / 2;
  StagedSampling ss;
  TRY(convert_per_image(per_image, B, rng_per_image, &ss));
  if (cfg_schedule_host) TRY(convert_schedule(cfg_schedule_host, B, n_steps, &ss));
  cudaStream_t user = (cudaStream_t)stream;
  cudaStream_t st = e->own_stream;
  const size_t tok_bytes = (size_t)B * n_steps * 4;
  CK(cudaEventRecord(e->ev_in, user));
  CK(cudaStreamWaitEvent(st, e->ev_in, 0));
  CK(cudaMemcpyAsync(e->st_kv_start, kv_start, (size_t)R * 4, cudaMemcpyDeviceToDevice, st));
  if (edit_region) {
    CK(cudaMemcpyAsync(e->st_edit, edit_region, tok_bytes, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(e->st_gt, gt_labels, tok_bytes, cudaMemcpyDeviceToDevice, st));
  }
  PerImage pi;
  TRY(stage_per_image(e, ss, st, &pi));
  const int32_t* kvs = e->st_kv_start;
  const int32_t* er = edit_region ? e->st_edit : nullptr;
  const int32_t* gl = edit_region ? e->st_gt : nullptr;
  int32_t* toks = e->st_tokens;
  float* lps = logprobs_out ? e->st_logprobs : nullptr;
  TRY(pg_prefill(e, x_prompt, kvs, R, P, nullptr, 0, (void*)st));
  CK(cudaMemsetAsync(e->step_ctr, 0, 4, st));
  if (n_steps > 1) {
    if (e->use_graph) {
      // settings and schedule are read from st_sampling / st_cfg: one graph serves every value of this shape
      char key[256];
      const int prof = (e->prof_buf && e->prof_step >= 0) ? 1 : 0;
      snprintf(key, sizeof(key), "imgpi/%d/%d/%d/%d/%d/%d/%d/%d/%d/%d", R, P, n_steps, greedy, edit_region ? 1 : 0,
               pi.rng_per_image, pi.any_top_p ? 1 : 0, lps ? 1 : 0, pi.cfg_sched ? 1 : 0, prof);
      pg_engine::GraphEntry* ge = nullptr;
      TRY(graph_for(e, key, st, [&]() {
        e->prof_active = (e->prof_buf != nullptr && e->prof_step >= 0);
        e->prof_slot = 0;
        int rc = one_step(e, kvs, R, P, n_steps, greedy, er, gl, toks, true, -1, st, pi, lps);
        e->prof_active = false;
        return rc;
      }, &ge));
      for (int i = 0; i < n_steps - 1; ++i) {
        const bool prof_now = e->prof_buf && i == e->prof_step;
        if (prof_now) {
          CK(cudaMemsetAsync(e->prof_buf, 0xFF, PROF_SLOTS * 8, st));
          CK(cudaMemsetAsync(e->prof_buf + PROF_SLOTS, 0, PROF_SLOTS * 8, st));
        }
        CK(cudaGraphLaunch(ge->exec, st));
        if (prof_now)
          CK(cudaMemcpyAsync(e->prof_buf + 2 * PROF_SLOTS, e->prof_buf, 2 * PROF_SLOTS * 8, cudaMemcpyDeviceToDevice, st));
      }
      e->launches += ge->launches * (n_steps - 1);
    } else {
      for (int i = 0; i < n_steps - 1; ++i) {
        e->prof_active = (e->prof_buf && i == e->prof_step);
        e->prof_slot = 0;
        if (e->prof_active) {
          CK(cudaMemsetAsync(e->prof_buf, 0xFF, PROF_SLOTS * 8, st));
          CK(cudaMemsetAsync(e->prof_buf + PROF_SLOTS, 0, PROF_SLOTS * 8, st));
        }
        int rc = one_step(e, kvs, R, P, n_steps, greedy, er, gl, toks, true, i, st, pi, lps);
        if (e->prof_active)
          CK(cudaMemcpyAsync(e->prof_buf + 2 * PROF_SLOTS, e->prof_buf, 2 * PROF_SLOTS * 8, cudaMemcpyDeviceToDevice, st));
        e->prof_active = false;
        TRY(rc);
      }
    }
  }
  // last token: head + sample only (the reference computes and drops one more embed, SURVEY appendix A.12)
  TRY(one_step(e, kvs, R, P, n_steps, greedy, er, gl, toks, false, n_steps - 1, st, pi, lps));
  CK(cudaMemcpyAsync(tokens_out, toks, tok_bytes, cudaMemcpyDeviceToDevice, st));
  if (lps) CK(cudaMemcpyAsync(logprobs_out, lps, tok_bytes, cudaMemcpyDeviceToDevice, st));
  CK(cudaEventRecord(e->ev_out, st));
  CK(cudaStreamWaitEvent(user, e->ev_out, 0));
  return 0;
}

// ------------------------------------------------------------------------------ teacher-forced scoring
// One prefill over prompt + image tokens, the hidden states of columns P-1 .. P+n-2 pair-major in hbuf (prefill_impl's
// `tail`), gen_head over those R * n rows in as few wide contractions as the idle prefill scratch allows (part holds one
// chunk's logits, qbuf its first-layer activations), and the sampler kernel in score mode per chunk.
extern "C" int pg_score_image_tokens(pg_engine* e, float* x_seq, const int32_t* kv_start, int R, int P, int n,
                                     const int32_t* image_tokens, const pg_image_sampling* per_image,
                                     const float* cfg_schedule_host, float* logprobs_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (!x_seq || !kv_start || !image_tokens || !logprobs_out) return fail("null argument");
  if (R < 2 || R % 2) return fail("score R=%d: R must be even (interleaved cond/uncond rows) and >= 2", R);
  if (R > d.max_rows) return fail("score R=%d exceeds the engine's max_rows %d", R, d.max_rows);
  if (P < 1) return fail("score P=%d: the prompt needs at least one column", P);
  if (n < 1 || n > d.max_steps) return fail("score n=%d exceeds the engine's max_steps %d", n, d.max_steps);
  const int T = P + n - 1;
  if (T > d.max_prompt)
    return fail("score: prompt + image tokens - 1 = %d columns exceed the engine's max_prompt %d (the prefill limit)", T,
                d.max_prompt);
  if (d.F < d.D) return fail("score needs F >= D (the gathered hidden states live in the prefill's MLP scratch)");
  NEED(b1, float, "head.b1");
  StagedSampling ss;
  TRY(convert_per_image(per_image, R / 2, 0, &ss));
  if (cfg_schedule_host) TRY(convert_schedule(cfg_schedule_host, R / 2, n, &ss));
  cudaStream_t st = (cudaStream_t)stream;
  PerImage pi;
  TRY(stage_per_image(e, ss, st, &pi));
  if (n > 1)
    DISPATCH_T(e,
               launch(e, score_embed_kernel<bf16>, dim3(n - 1, R), dim3(256), 0, st, image_tokens, (const bf16*)e->embed_table,
                      x_seq, P, T, n, d.D, d.img_vocab),
               launch(e, score_embed_kernel<float>, dim3(n - 1, R), dim3(256), 0, st, image_tokens, (const float*)e->embed_table,
                      x_seq, P, T, n, d.D, d.img_vocab));
  TRY(prefill_impl(e, x_seq, kv_start, R, T, nullptr, 0, false, stream, n));
  const size_t rows = (size_t)R * n;
  size_t cap = e->part_bytes / ((size_t)std::max(d.img_vocab, d.img_embed) * 4);          // one split of logits
  cap = std::min(cap, (size_t)d.max_rows * d.max_prompt * e->HD / d.img_embed);          // first-layer rows in qbuf
  cap &= ~(size_t)1;
  if (cap < 2) return fail("score: the prefill scratch holds no pair of logit rows");
  for (size_t r0 = 0; r0 < rows; r0 += cap) {
    const int M = (int)std::min(cap, rows - r0);
    int S = 1;
    TRY(head_gemms(e, (const char*)e->hbuf + r0 * d.D * e->esz, e->qbuf, M, &S, st));
    TRY(k_sample(e, e->part, S, (size_t)M * d.img_vocab, b1, M / 2, 0, 0, nullptr, image_tokens, (int)(r0 / 2), nullptr, n,
                 nullptr, nullptr, nullptr, nullptr, st, pi, logprobs_out, n));
  }
  return 0;
}

// ------------------------------------------------------------------------------ f1: stage-1 text decode (x2t)
// One greedy step: lm_head contraction -> argmax / eos bookkeeping / embed_tokens / first RMSNorm -> decoder layers.
static int text_step(pg_engine* e, const int32_t* kv_start, int R, int P, int max_new, int eos_id, int pad_id,
                     int32_t* tokens_out, bool with_lm, int step_host, cudaStream_t st) {
  const pg_dims& d = e->d;
  NEED(lm_head, void, "lm_head");
  NEED(table, float, "embed_tokens");
  LayerW w0;
  TRY(layer_weights(e, 0, &w0));
  int S = 1;
  TRY(run_gemm(e, e->hidden_t, lm_head, R, d.vocab, d.D, e->part, e->part_bytes, &S, st));
  const bool host = step_host >= 0;
  GreedyState gs = {e->greedy_state + 64, e->greedy_state, e->greedy_state + 1};
  DISPATCH_T(e,
             launch(e, lm_argmax_embed_kernel<bf16>, dim3(R), dim3(TXT_THREADS), 0, st, e->part, S, (size_t)R * d.vocab, d.vocab, eos_id, pad_id, gs,
                    host ? step_host : 0, host ? (const int*)nullptr : e->step_ctr, max_new, tokens_out, table, d.vocab, d.D,
                    with_lm ? e->x_dec : (float*)nullptr, w0.ln1, with_lm ? (bf16*)e->xn : (bf16*)nullptr, d.rms_eps, e->dbg_text_logits),
             launch(e, lm_argmax_embed_kernel<float>, dim3(R), dim3(TXT_THREADS), 0, st, e->part, S, (size_t)R * d.vocab, d.vocab, eos_id, pad_id, gs,
                    host ? step_host : 0, host ? (const int*)nullptr : e->step_ctr, max_new, tokens_out, table, d.vocab, d.D,
                    with_lm ? e->x_dec : (float*)nullptr, w0.ln1, with_lm ? (float*)e->xn : (float*)nullptr, d.rms_eps, e->dbg_text_logits));
  if (with_lm)
    TRY(decode_layers(e, kv_start, R, host ? P + step_host : P, host ? nullptr : e->step_ctr, true, !host, P + max_new / 2, st, 1));
  return 0;
}

// language_model.generate(inputs_embeds=, attention_mask=, pad_token_id=, eos_token_id=, max_new_tokens=, do_sample=False,
// use_cache=True)  (plangen_base.py:513-523; HF GenerationMixin greedy search).  x_prompt fp32 [R][P][D] (overwritten),
// tokens_out int32 [R][max_new_tokens] on the device; *n_generated (host) = number of columns that are valid = the
// step after which every row had produced eos (HF stops there), or max_new_tokens.  Synchronises the stream.
extern "C" int pg_generate_greedy(pg_engine* e, float* x_prompt, const int32_t* kv_start, int R, int P, int max_new_tokens,
                                  int eos_id, int pad_id, int32_t* tokens_out, int* n_generated, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (!n_generated || !tokens_out) return fail("null argument");
  if (R < 1 || R > d.max_rows) return fail("generate R=%d exceeds engine limits", R);
  if (max_new_tokens < 1 || P + max_new_tokens > e->Tmax) return fail("P + max_new_tokens = %d exceeds the KV capacity %d", P + max_new_tokens, e->Tmax);
  if (d.D > TXT_MAX_PER_THREAD * TXT_THREADS) return fail("hidden size %d too large for the greedy-step kernel", d.D);
  if (!T_(e, "lm_head")) return fail("tensor 'lm_head' not set: the engine was built without language_model.lm_head.weight");
  if (!e->poll_host) CK(cudaMallocHost(&e->poll_host, 64));
  cudaStream_t user = (cudaStream_t)stream;
  cudaStream_t st = e->own_stream;
  CK(cudaEventRecord(e->ev_in, user));
  CK(cudaStreamWaitEvent(st, e->ev_in, 0));
  CK(cudaMemcpyAsync(e->st_kv_start, kv_start, (size_t)R * 4, cudaMemcpyDeviceToDevice, st));
  const int32_t* kvs = e->st_kv_start;
  int32_t* toks = e->st_tokens;                      // [R][max_new_tokens]
  TRY(prefill_impl(e, x_prompt, kvs, R, P, nullptr, 0, true, (void*)st));
  CK(cudaMemsetAsync(e->step_ctr, 0, 4, st));
  GreedyState gs = {e->greedy_state + 64, e->greedy_state, e->greedy_state + 1};
  greedy_state_init_kernel<<<(R + 127) / 128, 128, 0, st>>>(gs, R, max_new_tokens);
  CK(cudaGetLastError());
  const int poll_every = 16;
  bool stopped = false;
  pg_engine::GraphEntry* ge = nullptr;
  if (max_new_tokens > 1 && e->use_graph) {
    char key[256];
    snprintf(key, sizeof(key), "txt/%d/%d/%d/%d/%d/%d", R, P, max_new_tokens, eos_id, pad_id, e->dbg_text_logits ? 1 : 0);
    TRY(graph_for(e, key, st, [&]() { return text_step(e, kvs, R, P, max_new_tokens, eos_id, pad_id, toks, true, -1, st); }, &ge));
  }
  for (int i = 0; i < max_new_tokens - 1 && !stopped; ++i) {
    if (ge) { CK(cudaGraphLaunch(ge->exec, st)); e->launches += ge->launches; }
    else TRY(text_step(e, kvs, R, P, max_new_tokens, eos_id, pad_id, toks, true, i, st));
    if ((i + 1) % poll_every == 0) {            // every row done?  (HF checks after every token, with a host sync each)
      CK(cudaMemcpyAsync(e->poll_host, e->greedy_state, 8, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      if (e->poll_host[0] == 0) stopped = true;
    }
  }
  if (!stopped) TRY(text_step(e, kvs, R, P, max_new_tokens, eos_id, pad_id, toks, false, max_new_tokens - 1, st));
  CK(cudaMemcpyAsync(tokens_out, toks, (size_t)R * max_new_tokens * 4, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemcpyAsync(e->poll_host, e->greedy_state, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  *n_generated = e->poll_host[1];
  CK(cudaEventRecord(e->ev_out, st));
  CK(cudaStreamWaitEvent(user, e->ev_out, 0));
  return 0;
}

// ------------------------------------------------------------------------------ f2: mmu front-end
// replaces: vl_gpt.prepare_inputs_embeds(input_ids, pixel_values, images_seq_mask, images_emb_mask)
//           (plangen_base.py:289,366,855; modeling_vlm.py:221-268)
static int sig_tensor(pg_engine* e, const std::string& name, const void** out) {
  *out = T_(e, name);
  if (!*out) return fail("tensor '%s' was not registered (the engine was built without the vision tower / aligner)", name.c_str());
  return 0;
}
#define SIGT(var, type, name) const type* var = nullptr; TRY(sig_tensor(e, (name), (const void**)&var))

// vision tower + aligner for images [i0, i0 + n): pixel fp32 [n][3][S][S] -> feat T [n * NP][D]
static int sig_tower(pg_engine* e, const float* pixel, int n, void* feat, cudaStream_t st) {
  const pg_dims& d = e->d;
  const int W = d.sig_width, NP = e->sig_np, heads = d.sig_heads, hd = W / heads, Kp = 3 * d.sig_patch * d.sig_patch;
  const int M = n * NP;
  const float eps = 1e-6f;
  int S = 1;
  SIGT(pw, void, "sig.patch.w"); SIGT(pb, float, "sig.patch.b"); SIGT(pos, float, "sig.pos");
  {
    const size_t total4 = (size_t)M * Kp / 4;
    DISPATCH_T(e,
               launch(e, vit_patchify_kernel<bf16>, dim3(elementwise_blocks(e, total4)), dim3(256), 0, st, pixel, (bf16*)e->sig_xn, d.sig_image, d.sig_patch, total4),
               launch(e, vit_patchify_kernel<float>, dim3(elementwise_blocks(e, total4)), dim3(256), 0, st, pixel, (float*)e->sig_xn, d.sig_image, d.sig_patch, total4));
    TRY(run_gemm(e, e->sig_xn, pw, M, W, Kp, e->sig_part, e->sig_part_bytes, &S, st, -1, 1));
    const size_t total = (size_t)M * W;
    DISPATCH_T(e,
               launch(e, vit_patch_epilogue_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->sig_part, S, total, pb, pos, e->sig_x, W, NP, total),
               launch(e, vit_patch_epilogue_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->sig_part, S, total, pb, pos, e->sig_x, W, NP, total));
  }
  auto resid_ln = [&](const float* part, const float* bias, const float* w, const float* b) {
    const size_t stride = (size_t)M * W;
    if (W <= 4 * 32 * LNW_MAXQ) {          // a warp per row
      DISPATCH_T(e,
                 launch(e, vit_resid_ln_warp_kernel<bf16>, dim3((M + 7) / 8), dim3(256), 0, st, e->sig_x, part, S, stride, bias, w, b, (bf16*)e->sig_xn, W, eps, M),
                 launch(e, vit_resid_ln_warp_kernel<float>, dim3((M + 7) / 8), dim3(256), 0, st, e->sig_x, part, S, stride, bias, w, b, (float*)e->sig_xn, W, eps, M));
      return 0;
    }
    DISPATCH_T(e,
               launch(e, vit_resid_ln_kernel<bf16>, dim3(M), dim3(LN_THREADS), 0, st, e->sig_x, part, S, stride, bias, w, b, (bf16*)e->sig_xn, W, eps),
               launch(e, vit_resid_ln_kernel<float>, dim3(M), dim3(LN_THREADS), 0, st, e->sig_x, part, S, stride, bias, w, b, (float*)e->sig_xn, W, eps));
    return 0;
  };
  auto bias_act = [&](const float* bias, void* out, int N, int gelu) {
    const size_t total = (size_t)M * N;
    DISPATCH_T(e,
               launch(e, bias_act_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->sig_part, S, total, bias, (bf16*)out, (float*)nullptr, N, total, gelu),
               launch(e, bias_act_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, e->sig_part, S, total, bias, (float*)out, (float*)nullptr, N, total, gelu));
    return 0;
  };
  const bool tc_attn = e->bf16 && e->use_tc && e->sig_attn_tc && hd == VT_HD;
  const bool fuse = e->bf16 && e->use_tc;
  // contraction + bias (+ GELU) -> T, or contraction + bias + residual add; fused into the tcgen05 epilogue when possible
  auto linear_out = [&](const void* X, const void* Wt, const float* bias, void* out, int N, int K, int gelu) {
    if (fuse) {
      EpiFuse ep = {bias, (bf16*)out, nullptr, gelu};
      return run_gemm(e, X, Wt, M, N, K, e->sig_part, e->sig_part_bytes, &S, st, -1, 1, true, nullptr, nullptr, &ep);
    }
    TRY(run_gemm(e, X, Wt, M, N, K, e->sig_part, e->sig_part_bytes, &S, st, -1, 1));
    return bias_act(bias, out, N, gelu);
  };
  auto linear_resid_ln = [&](const void* X, const void* Wt, const float* bias, int K, const float* lw, const float* lb) {
    if (fuse) {
      EpiFuse ep = {bias, nullptr, e->sig_x, 0};
      TRY(run_gemm(e, X, Wt, M, W, K, e->sig_part, e->sig_part_bytes, &S, st, -1, 1, true, nullptr, nullptr, &ep));
      return resid_ln(nullptr, nullptr, lw, lb);
    }
    TRY(run_gemm(e, X, Wt, M, W, K, e->sig_part, e->sig_part_bytes, &S, st, -1, 1));
    return resid_ln(e->sig_part, bias, lw, lb);
  };
  for (int l = 0; l < d.sig_layers; ++l) {
    const std::string p = "sig." + std::to_string(l) + ".";
    SIGT(ln1w, float, p + "ln1.w"); SIGT(ln1b, float, p + "ln1.b"); SIGT(ln2w, float, p + "ln2.w"); SIGT(ln2b, float, p + "ln2.b");
    SIGT(wqkv, void, p + "qkv.w"); SIGT(bqkv, float, p + "qkv.b"); SIGT(wproj, void, p + "proj.w"); SIGT(bproj, float, p + "proj.b");
    SIGT(wfc1, void, p + "fc1.w"); SIGT(bfc1, float, p + "fc1.b"); SIGT(wfc2, void, p + "fc2.w"); SIGT(bfc2, float, p + "fc2.b");
    if (l == 0) TRY(resid_ln(nullptr, nullptr, ln1w, ln1b));
    TRY(linear_out(e->sig_xn, wqkv, bqkv, e->sig_qkv, 3 * W, W, 0));
    TRY(launch_vit_attn(e, tc_attn, e->sig_qkv, M, e->sig_attn, n, NP, W, heads, st));
    TRY(linear_resid_ln(e->sig_attn, wproj, bproj, W, ln2w, ln2b));
    TRY(linear_out(e->sig_xn, wfc1, bfc1, e->sig_h, d.sig_mlp, W, 1));
    if (l + 1 < d.sig_layers) {
      const std::string pn = "sig." + std::to_string(l + 1) + ".";
      SIGT(nw, float, pn + "ln1.w"); SIGT(nb, float, pn + "ln1.b");
      TRY(linear_resid_ln(e->sig_h, wfc2, bfc2, d.sig_mlp, nw, nb));
    } else {
      SIGT(nw, float, "sig.norm.w"); SIGT(nb, float, "sig.norm.b");
      TRY(linear_resid_ln(e->sig_h, wfc2, bfc2, d.sig_mlp, nw, nb));
    }
  }
  // aligner: Linear(W, D) -> GELU -> Linear(D, D)   (projector.py:39-45)
  SIGT(aw0, void, "ualign.w0"); SIGT(ab0, float, "ualign.b0"); SIGT(aw1, void, "ualign.w1"); SIGT(ab1, float, "ualign.b1");
  TRY(linear_out(e->sig_xn, aw0, ab0, e->sig_h, d.D, W, 1));
  TRY(linear_out(e->sig_h, aw1, ab1, feat, d.D, d.D, 0));
  return 0;
}

extern "C" int pg_prepare_inputs_embeds(pg_engine* e, const float* pixel_values, int n_images, const int32_t* input_ids,
                                        const uint8_t* images_seq_mask, const uint8_t* images_emb_mask, int B, int T,
                                        float* embeds_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (d.sig_layers <= 0 || !e->sig_x) return fail("the engine was created without the vision tower (pg_dims.sig_layers / max_images = 0)");
  if (!input_ids || !images_seq_mask || !embeds_out || B < 1 || T < 1) return fail("bad argument");
  if ((size_t)B * T > (size_t)d.max_rows * std::max(d.max_prompt, 1)) return fail("B*T = %d x %d exceeds max_rows x max_prompt", B, T);
  if (n_images < 0 || n_images > d.max_images) return fail("n_images %d exceeds max_images %d", n_images, d.max_images);
  if (n_images > 0 && (!pixel_values || !images_emb_mask)) return fail("pixel_values / images_emb_mask missing");
  cudaStream_t st = (cudaStream_t)stream;
  NEED(table, float, "embed_tokens");
  if (!e->poll_host) CK(cudaMallocHost(&e->poll_host, 64));
  const int NP = e->sig_np;
  const int saved_pdl = e->use_pdl;
  for (int i0 = 0; i0 < n_images; i0 += e->sig_chunk) {
    const int n = std::min(e->sig_chunk, n_images - i0);
    const size_t img_elems = (size_t)3 * d.sig_image * d.sig_image;
    TRY(sig_tower(e, pixel_values + (size_t)i0 * img_elems, n, (uint8_t*)e->sig_feat + (size_t)i0 * NP * d.D * e->esz, st));
  }
  e->use_pdl = saved_pdl;
  // scatter: k-th set position of images_seq_mask <- k-th selected image token
  CK(cudaMemsetAsync(e->sig_counts, 0, 8, st));
  if (n_images > 0) mask_rank_kernel<<<1, 1024, 0, st>>>(images_emb_mask, n_images * NP, (int32_t*)nullptr, e->sig_inv_src, e->sig_counts + 1);
  mask_rank_kernel<<<1, 1024, 0, st>>>(images_seq_mask, B * T, e->sig_rank_dst, (int32_t*)nullptr, e->sig_counts);
  CK(cudaGetLastError());
  e->launches += 2;
  CK(cudaMemcpyAsync(e->poll_host, e->sig_counts, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (e->poll_host[0] != e->poll_host[1])
    return fail("images_seq_mask selects %d positions but images_emb_mask selects %d image tokens (modeling_vlm.py:236 asserts they are equal)",
                e->poll_host[0], e->poll_host[1]);
  DISPATCH_T(e,
             launch(e, embed_scatter_kernel<bf16>, dim3(B * T), dim3(256), 0, st, input_ids, (const int32_t*)e->sig_rank_dst, (const int32_t*)e->sig_inv_src,
                    (const int32_t*)(e->sig_counts + 1), (const bf16*)e->sig_feat, table, embeds_out, d.D, d.vocab),
             launch(e, embed_scatter_kernel<float>, dim3(B * T), dim3(256), 0, st, input_ids, (const int32_t*)e->sig_rank_dst, (const int32_t*)e->sig_inv_src,
                    (const int32_t*)(e->sig_counts + 1), (const float*)e->sig_feat, table, embeds_out, d.D, d.vocab));
  return 0;
}

// Vision tower + aligner alone (bench / tests): pixel fp32 [n][3][S][S] -> features fp32 [n * NP][D]
extern "C" int pg_vision_features(pg_engine* e, const float* pixel_values, int n_images, float* feat_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (d.sig_layers <= 0 || !e->sig_x) return fail("the engine was created without the vision tower");
  if (n_images < 1 || n_images > d.max_images || !pixel_values) return fail("bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int NP = e->sig_np;
  for (int i0 = 0; i0 < n_images; i0 += e->sig_chunk) {
    const int n = std::min(e->sig_chunk, n_images - i0);
    TRY(sig_tower(e, pixel_values + (size_t)i0 * 3 * d.sig_image * d.sig_image, n, (uint8_t*)e->sig_feat + (size_t)i0 * NP * d.D * e->esz, st));
  }
  if (feat_out) {
    const size_t total = (size_t)n_images * NP * d.D;
    DISPATCH_T(e,
               launch(e, to_f32_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, (const bf16*)e->sig_feat, feat_out, total),
               launch(e, to_f32_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, (const float*)e->sig_feat, feat_out, total));
  }
  return 0;
}

// ------------------------------------------------------------------------------ images -> uint8
// replaces: denorm_pt (src/utils/funcs.py:511-512: (x.clamp(-1,1)+1)/2) followed by `(x*255).astype(np.uint8)`
// (funcs.py:497-498 / pt2pil :507; truncation toward zero)
__global__ void __launch_bounds__(256) images_to_u8_kernel(const float* __restrict__ x, uint8_t* __restrict__ out, size_t n) {
  for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += (size_t)gridDim.x * blockDim.x * 4) {
    if (i + 4 <= n) {
      const float4 v = *reinterpret_cast<const float4*>(x + i);
      const float f[4] = {v.x, v.y, v.z, v.w};
      uint32_t pk = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float t = ((fminf(fmaxf(f[j], -1.f), 1.f) + 1.f) / 2.f) * 255.f;
        pk |= (uint32_t)(uint8_t)(int)t << (8 * j);
      }
      *reinterpret_cast<uint32_t*>(out + i) = pk;
    } else {
      for (size_t j = i; j < n; ++j) out[j] = (uint8_t)(int)(((fminf(fmaxf(x[j], -1.f), 1.f) + 1.f) / 2.f) * 255.f);
    }
  }
}
extern "C" int pg_images_to_u8(pg_engine* e, const float* image, size_t n, uint8_t* out, void* stream) {
  if (!e || !image || !out) return fail("null argument");
  if (((uintptr_t)image & 15) || ((uintptr_t)out & 3)) return fail("pg_images_to_u8: image must be 16-byte and out 4-byte aligned");
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((n / 4 + 255) / 256, (size_t)e->num_sms * 16));
  images_to_u8_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(image, out, n);
  CK(cudaGetLastError());
  e->launches++;
  return 0;
}

// ------------------------------------------------------------------------------ a10: VQ decode
struct VqCtx {
  pg_engine* e; cudaStream_t st; int Bc;
};

static int vq_gn_stats(VqCtx& c, const void* x, int HW, int C) {
  pg_engine* e = c.e;
  int chunk_pix = std::max(64, (HW + e->gn_chunks_max - 1) / e->gn_chunks_max);
  chunk_pix = std::max(chunk_pix, (HW + 255) / 256);
  const int nchunks = (HW + chunk_pix - 1) / chunk_pix;
  if (nchunks > e->gn_chunks_max) return fail("internal: gn chunks");
  if (C % 32 || C > 512) return fail("GroupNorm(32) needs C %% 32 == 0 and C <= 512 (C=%d)", C);
  const int gn_threads = C > 256 ? 512 : 256;
  if (e->bf16 && C % 128 == 0) {
    TRY(launch(e, gn_partial_vec_kernel, dim3(nchunks, c.Bc), dim3(256), 0, c.st, (const bf16*)x, e->gn_partial, HW, C, chunk_pix));
  } else
  DISPATCH_T(e,
             launch(e, gn_partial_kernel<bf16>, dim3(nchunks, c.Bc), dim3(gn_threads), 0, c.st, (const bf16*)x, e->gn_partial, HW, C, chunk_pix),
             launch(e, gn_partial_kernel<float>, dim3(nchunks, c.Bc), dim3(gn_threads), 0, c.st, (const float*)x, e->gn_partial, HW, C, chunk_pix));
  TRY(launch(e, gn_finalize_kernel, dim3(c.Bc), dim3(32), 0, c.st, (const float*)e->gn_partial, e->gn_stats, nchunks,
             1.0 / ((double)HW * (C / 32)), 1e-6f));
  return 0;
}

static int vq_im2col(VqCtx& c, const void* in, void* col, int Hi, int Wi, int C, int ks, int up, bool gn,
                     const std::string& gn_name, bool swish) {
  pg_engine* e = c.e;
  const float *gamma = nullptr, *beta = nullptr;
  if (gn) {
    gamma = (const float*)T_(e, "vq." + gn_name + ".weight");
    beta = (const float*)T_(e, "vq." + gn_name + ".bias");
    if (!gamma || !beta) return fail("missing GroupNorm tensors for %s", gn_name.c_str());
  }
  if (ks == 1 && e->bf16 && C % 8 == 0 && C <= 2048 && 256 % (C / 8) == 0) {   // activation only: vectorised apply
    const int Ho = Hi * up, Wo = Wi * up, PL = 256 / (C / 8);
    if ((size_t)c.Bc * Ho * Wo * C > e->vq_col_elems) return fail("internal: im2col scratch too small");
    const int blocks = std::max(1, std::min((Ho * Wo + PL - 1) / PL, (e->num_sms * 8 + c.Bc - 1) / c.Bc));
    return launch(e, gn_apply_kernel, dim3(blocks, c.Bc), dim3(256), 0, c.st, (const bf16*)in, (bf16*)col,
                  gn ? (const float*)e->gn_stats : (const float*)nullptr, gamma, beta, Hi, Wi, C, up, swish ? 1 : 0);
  }
  if (C % 4) return fail("im2col needs C %% 4 == 0");
  const size_t n_pix = (size_t)c.Bc * Hi * up * Wi * up;
  if (n_pix * ks * ks * C > e->vq_col_elems) return fail("internal: im2col scratch too small");
  const float* stats = gn ? e->gn_stats : nullptr;
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((n_pix + 7) / 8, (size_t)e->num_sms * 32));
  DISPATCH_T(e,
             launch(e, im2col_kernel<bf16>, dim3(blocks), dim3(256), 0, c.st, (const bf16*)in, (bf16*)col, stats, gamma, beta, Hi, Wi, C, ks, up, swish ? 1 : 0, n_pix),
             launch(e, im2col_kernel<float>, dim3(blocks), dim3(256), 0, c.st, (const float*)in, (float*)col, stats, gamma, beta, Hi, Wi, C, ks, up, swish ? 1 : 0, n_pix));
  return 0;
}

static int vq_epilogue(VqCtx& c, const float* part, const float* bias, const void* residual, void* out, float* out_nchw,
                       int Cout, int HW, size_t pixels, int bias_per_row) {
  pg_engine* e = c.e;
  const size_t total = pixels * Cout;
  DISPATCH_T(e,
             launch(e, conv_epilogue_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, c.st, part, bias, (const bf16*)residual, (bf16*)out, out_nchw, Cout, HW, total, bias_per_row),
             launch(e, conv_epilogue_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, c.st, part, bias, (const float*)residual, (float*)out, out_nchw, Cout, HW, total, bias_per_row));
  return 0;
}

// conv2d(ks x ks, pad ks/2) over NHWC `in` [Bc, Hi, Wi, Cin] (optionally GroupNorm+swish'ed and x2 upsampled first)
static int vq_conv(VqCtx& c, const void* in, int Hi, int Wi, int Cin, const std::string& name, int Cout, int ks, int up,
                   const char* gn_name, bool swish, const void* residual, void* out, float* out_nchw) {
  pg_engine* e = c.e;
  const void* W = T_(e, "vq." + name + ".weight");
  const float* bias = (const float*)T_(e, "vq." + name + ".bias");
  if (!W || !bias) return fail("missing conv tensors for %s", name.c_str());
  const int Ho = Hi * up, Wo = Wi * up;
  const size_t pixels = (size_t)c.Bc * Ho * Wo;
  const void* X = in;
  if (gn_name) TRY(vq_gn_stats(c, in, Hi * Wi, Cin));
  if (ks == 3) {
    // implicit GEMM: only the (normalised, activated, upsampled) activation is materialised, not its 9 taps
    const void* act = in;
    const bool qualifies = e->bf16 && e->use_tc && Cin % TC_BK == 0 &&
                           ((Wo <= CONV_NT && CONV_NT % Wo == 0) || Wo % CONV_NT == 0);
    if (qualifies) {
      if (gn_name || up != 1) {
        TRY(vq_im2col(c, in, e->vq_col, Hi, Wi, Cin, 1, up, gn_name != nullptr, gn_name ? gn_name : "", swish));
        act = e->vq_col;
      }
      if (pixels * Cout > e->vq_part_elems) return fail("internal: vq partial buffer too small");
      int taken = 0;
      // bias (+ residual) -> bf16 NHWC rows in the contraction's epilogue (gemm.cuh EpiFuse); the final conv_out (3 channels,
      // fp32 NCHW) keeps the row kernel
      const bool fuse = out != nullptr && out_nchw == nullptr && e->fuse_conv_epilogue && Cout % 8 == 0;
      EpiFuse ep = {bias, (bf16*)out, nullptr, 0, (const bf16*)residual};
      TRY(run_conv_gemm(e, act, W, c.Bc, Ho, Wo, Cin, Cout, e->vq_part, e->vq_part_elems * 4, c.st, &taken, fuse ? &ep : nullptr));
      if (taken) {
        if (!fuse) TRY(vq_epilogue(c, e->vq_part, bias, residual, out, out_nchw, Cout, Ho * Wo, pixels, 0));
        return 0;
      }
    }
  }
  if (ks != 1 || gn_name || up != 1) {
    TRY(vq_im2col(c, in, e->vq_col, Hi, Wi, Cin, ks, up, gn_name != nullptr, gn_name ? gn_name : "", swish));
    X = e->vq_col;
  }
  if (pixels * Cout > e->vq_part_elems) return fail("internal: vq partial buffer too small");
  int S = 1;
  TRY(run_gemm(e, X, W, (int)pixels, Cout, ks * ks * Cin, e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1));
  TRY(vq_epilogue(c, e->vq_part, bias, residual, out, out_nchw, Cout, Ho * Wo, pixels, 0));
  return 0;
}

// ResnetBlock (vq_model.py:337-352).  bufs: x (input), t (scratch), y (output)
static int vq_resblock(VqCtx& c, const std::string& name, const void* x, void* t, void* y, int H, int W, int Cin, int Cout) {
  const std::string n1 = name + ".norm1", n2 = name + ".norm2";
  TRY(vq_conv(c, x, H, W, Cin, name + ".conv1", Cout, 3, 1, n1.c_str(), true, nullptr, t, nullptr));
  const void* res = x;
  if (Cin != Cout) {
    TRY(vq_conv(c, x, H, W, Cin, name + ".nin_shortcut", Cout, 1, 1, nullptr, false, nullptr, y, nullptr));
    res = y;   // in-place residual: epilogue reads y[i] then writes y[i]
  }
  TRY(vq_conv(c, t, H, W, Cout, name + ".conv2", Cout, 3, 1, n2.c_str(), true, res, y, nullptr));
  return 0;
}

// AttnBlock (vq_model.py:366-390): single head over H*W tokens, head dim C
static int vq_attnblock(VqCtx& c, const std::string& name, const void* x, void* y, int H, int W, int C) {
  pg_engine* e = c.e;
  const size_t es = e->esz;
  const int HW = H * W;
  const size_t pix = (size_t)c.Bc * HW;
  uint8_t* scratch = (uint8_t*)e->vq_col;
  void* hn = scratch;                                   // [Bc*HW, C]
  void* qb = scratch + pix * C * es;                    // [Bc*HW, C]
  void* kb = scratch + 2 * pix * C * es;
  void* vT = scratch + 3 * pix * C * es;                // [Bc][C, HW]
  void* ha = scratch + 4 * pix * C * es;                // [Bc*HW, C]
  void* Pm = scratch + 5 * pix * C * es;                // [HW, HW] (one image at a time)
  if ((5 * pix * C + (size_t)HW * HW) > e->vq_col_elems) return fail("internal: attention scratch too small");
  const std::string nn = name + ".norm";
  TRY(vq_gn_stats(c, x, HW, C));
  TRY(vq_im2col(c, x, hn, H, W, C, 1, 1, true, nn, false));
  const char* names[2] = {".q", ".k"};
  void* outs[2] = {qb, kb};
  int S = 1;
  for (int i = 0; i < 2; ++i) {
    const void* Wt = T_(e, "vq." + name + names[i] + ".weight");
    const float* bias = (const float*)T_(e, "vq." + name + names[i] + ".bias");
    if (!Wt || !bias) return fail("missing attn tensors for %s", name.c_str());
    TRY(run_gemm(e, hn, Wt, (int)pix, C, C, e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1));
    TRY(vq_epilogue(c, e->vq_part, bias, nullptr, outs[i], nullptr, C, HW, pix, 0));
  }
  const void* Wv = T_(e, "vq." + name + ".v.weight");
  const float* bv = (const float*)T_(e, "vq." + name + ".v.bias");
  if (!Wv || !bv) return fail("missing attn v tensors for %s", name.c_str());
  const float scale = 1.0f / sqrtf((float)C);
  for (int b = 0; b < c.Bc; ++b) {
    const uint8_t* hn_b = (const uint8_t*)hn + (size_t)b * HW * C * es;
    uint8_t* vT_b = (uint8_t*)vT + (size_t)b * HW * C * es;
    // v^T[c][pix] = sum_k Wv[c][k] hn[pix][k] + bv[c]
    TRY(run_gemm(e, Wv, hn_b, C, HW, C, e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1, false));
    VqCtx one = c; one.Bc = 1;
    TRY(vq_epilogue(one, e->vq_part, bv, nullptr, vT_b, nullptr, HW, HW, (size_t)C, 1));
    // scores[i][j] = q_i . k_j
    TRY(run_gemm(e, (const uint8_t*)qb + (size_t)b * HW * C * es, (const uint8_t*)kb + (size_t)b * HW * C * es, HW, HW, C,
                 e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1, false));
    DISPATCH_T(e,
               launch(e, softmax_rows_kernel<bf16>, dim3(HW), dim3(256), 0, c.st, (const float*)e->vq_part, (bf16*)Pm, HW, scale),
               launch(e, softmax_rows_kernel<float>, dim3(HW), dim3(256), 0, c.st, (const float*)e->vq_part, (float*)Pm, HW, scale));
    // h[i][c] = sum_j P[i][j] v^T[c][j]
    TRY(run_gemm(e, Pm, vT_b, HW, C, HW, e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1, false));
    TRY(vq_epilogue(one, e->vq_part, nullptr, nullptr, (uint8_t*)ha + (size_t)b * HW * C * es, nullptr, C, HW, (size_t)HW, 0));
  }
  TRY(vq_conv(c, ha, H, W, C, name + ".proj_out", C, 1, 1, nullptr, false, x, y, nullptr));
  return 0;
}

extern "C" int pg_vq_decode_code(pg_engine* e, const int32_t* codes, int B, int gh, int gw, float* image_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  if (gh < 1 || gw < 1 || gh > d.grid || gw > d.grid) return fail("token grid %dx%d exceeds engine limit %d", gh, gw, d.grid);
  cudaStream_t st = (cudaStream_t)stream;
  NEED(codebook, float, "vq.codebook");
  NEED(pqc_w, void, "vq.pqc.w");
  NEED(pqc_b, float, "vq.pqc.b");
  const int nres = d.vq_nres;
  const int scale_up = 1 << (nres - 1);
  const int chunk = vq_chunk_of(e);
  const int saved_pdl = e->use_pdl;
  for (int b0 = 0; b0 < B; b0 += chunk) {
    VqCtx c{e, st, std::min(chunk, B - b0)};
    void *A = e->vq_act[0], *Bf = e->vq_act[1], *Cf = e->vq_act[2];
    const size_t n_pix = (size_t)c.Bc * gh * gw;
    const int32_t* cb = codes + (size_t)b0 * gh * gw;
    DISPATCH_T(e,
               launch(e, vq_codebook_pqc_kernel<bf16>, dim3((unsigned)n_pix), dim3(128), 0, st, cb, codebook, (const bf16*)pqc_w, pqc_b, (bf16*)A, d.code_dim, d.vq_z, d.img_vocab, n_pix),
               launch(e, vq_codebook_pqc_kernel<float>, dim3((unsigned)n_pix), dim3(128), 0, st, cb, codebook, (const float*)pqc_w, pqc_b, (float*)A, d.code_dim, d.vq_z, d.img_vocab, n_pix));
    int H = gh, W = gw;
    int ch = d.vq_ch * d.vq_ch_mult[nres - 1];
    TRY(vq_conv(c, A, H, W, d.vq_z, "decoder.conv_in", ch, 3, 1, nullptr, false, nullptr, Bf, nullptr));
    // cur = Bf
    void *cur = Bf, *t1 = A, *t2 = Cf;
    auto rot = [&](void* newcur) {   // newcur becomes cur; old cur becomes scratch
      void* old = cur;
      if (newcur == t1) t1 = old; else t2 = old;
      cur = newcur;
    };
    TRY(vq_resblock(c, "decoder.mid.0", cur, t1, t2, H, W, ch, ch)); rot(t2);
    TRY(vq_attnblock(c, "decoder.mid.1", cur, t1, H, W, ch)); rot(t1);
    TRY(vq_resblock(c, "decoder.mid.2", cur, t1, t2, H, W, ch, ch)); rot(t2);
    for (int idx = 0; idx < nres; ++idx) {
      const int i_level = nres - 1 - idx;
      const int cout = d.vq_ch * d.vq_ch_mult[i_level];
      for (int j = 0; j < d.vq_res_blocks + 1; ++j) {
        const std::string rn = "decoder.conv_blocks." + std::to_string(idx) + ".res." + std::to_string(j);
        TRY(vq_resblock(c, rn, cur, t1, t2, H, W, ch, cout)); rot(t2);
        ch = cout;
        if (idx == 0) {
          const std::string an = "decoder.conv_blocks." + std::to_string(idx) + ".attn." + std::to_string(j);
          TRY(vq_attnblock(c, an, cur, t1, H, W, ch)); rot(t1);
        }
      }
      if (idx != nres - 1) {
        const std::string un = "decoder.conv_blocks." + std::to_string(idx) + ".upsample.conv";
        TRY(vq_conv(c, cur, H, W, ch, un, ch, 3, 2, nullptr, false, nullptr, t1, nullptr)); rot(t1);
        H *= 2; W *= 2;
      }
    }
    float* img = image_out + (size_t)b0 * 3 * gh * scale_up * gw * scale_up;
    TRY(vq_conv(c, cur, H, W, ch, "decoder.conv_out", 3, 3, 1, "decoder.norm_out", true, nullptr, nullptr, img));
  }
  e->use_pdl = saved_pdl;
  return 0;
}

// ------------------------------------------------------------------------------ f3: VQ encode (editing path)
// Downsample: asymmetric zero pad + 3x3 stride-2 conv (vq_model.py:440-445) as im2col + contraction
static int vq_conv_down(VqCtx& c, const void* in, int Hi, int Wi, int C, const std::string& name, void* out) {
  pg_engine* e = c.e;
  const void* W = T_(e, "vq." + name + ".weight");
  const float* bias = (const float*)T_(e, "vq." + name + ".bias");
  if (!W || !bias) return fail("missing conv tensors for %s", name.c_str());
  if (C % 4 || (Hi & 1) || (Wi & 1)) return fail("downsample needs C %% 4 == 0 and even H, W");
  const int Ho = Hi / 2, Wo = Wi / 2;
  const size_t pixels = (size_t)c.Bc * Ho * Wo;
  if (pixels * 9 * C > e->vq_col_elems || pixels * C > e->vq_part_elems) return fail("internal: vq scratch too small (downsample)");
  const int blocks = (int)std::max<size_t>(1, std::min<size_t>((pixels + 7) / 8, (size_t)e->num_sms * 32));
  DISPATCH_T(e,
             launch(e, im2col_down_kernel<bf16>, dim3(blocks), dim3(256), 0, c.st, (const bf16*)in, (bf16*)e->vq_col, Hi, Wi, C, pixels),
             launch(e, im2col_down_kernel<float>, dim3(blocks), dim3(256), 0, c.st, (const float*)in, (float*)e->vq_col, Hi, Wi, C, pixels));
  int S = 1;
  TRY(run_gemm(e, e->vq_col, W, (int)pixels, C, 9 * C, e->vq_part, e->vq_part_elems * 4, &S, c.st, -1, 1));
  TRY(vq_epilogue(c, e->vq_part, bias, nullptr, out, nullptr, C, Ho * Wo, pixels, 0));
  return 0;
}

constexpr int VQ_IN_CPAD = 8;     // image channels padded 3 -> 8 (weights.py pads conv_in's taps with zeros)

// replaces: vl_gpt.gen_vision_model.encode(img)[-1][-1]   (plangen_base.py:532; VQModel.encode vq_model.py:494-498)
extern "C" int pg_vq_encode(pg_engine* e, const float* image, int B, int H, int W, int32_t* codes_out, void* stream) {
  TRY(check_ready(e));
  const pg_dims& d = e->d;
  const int nres = d.vq_nres;
  const int down = 1 << (nres - 1);
  if (H < down || W < down || H % down || W % down || H / down > d.grid || W / down > d.grid)
    return fail("image %dx%d: sides must be multiples of %d and at most %d", H, W, down, d.grid * down);
  if (d.code_dim > VQ_CD_MAX) return fail("code_dim %d exceeds %d", d.code_dim, VQ_CD_MAX);
  cudaStream_t st = (cudaStream_t)stream;
  NEED(codebook, float, "vq.codebook");
  if (!T_(e, "vq.encoder.conv_in.weight") || !T_(e, "vq.quant_conv.weight"))
    return fail("VQ encoder tensors not set: the engine was built without gen_vision_model.encoder.* / quant_conv.*");
  const int chunk = vq_chunk_of(e);
  const int saved_pdl = e->use_pdl;
  for (int b0 = 0; b0 < B; b0 += chunk) {
    VqCtx c{e, st, std::min(chunk, B - b0)};
    void *A = e->vq_act[0], *Bf = e->vq_act[1], *Cf = e->vq_act[2];
    int Hc = H, Wc = W;
    {
      const size_t total = (size_t)c.Bc * H * W * VQ_IN_CPAD;
      if (total > e->vq_act_elems) return fail("internal: vq activation buffer too small");
      const float* img = image + (size_t)b0 * 3 * H * W;
      DISPATCH_T(e,
                 launch(e, nchw_to_nhwc_pad_kernel<bf16>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, img, (bf16*)A, 3, VQ_IN_CPAD, H * W, total),
                 launch(e, nchw_to_nhwc_pad_kernel<float>, dim3(elementwise_blocks(e, total)), dim3(256), 0, st, img, (float*)A, 3, VQ_IN_CPAD, H * W, total));
    }
    int ch = d.vq_ch;
    TRY(vq_conv(c, A, Hc, Wc, VQ_IN_CPAD, "encoder.conv_in", ch, 3, 1, nullptr, false, nullptr, Bf, nullptr));
    void *cur = Bf, *t1 = A, *t2 = Cf;
    auto rot = [&](void* newcur) {
      void* old = cur;
      if (newcur == t1) t1 = old; else t2 = old;
      cur = newcur;
    };
    for (int lvl = 0; lvl < nres; ++lvl) {
      const int cout = d.vq_ch * d.vq_ch_mult[lvl];
      for (int j = 0; j < d.vq_res_blocks; ++j) {
        const std::string rn = "encoder.conv_blocks." + std::to_string(lvl) + ".res." + std::to_string(j);
        TRY(vq_resblock(c, rn, cur, t1, t2, Hc, Wc, ch, cout)); rot(t2);
        ch = cout;
        if (lvl == nres - 1) {
          const std::string an = "encoder.conv_blocks." + std::to_string(lvl) + ".attn." + std::to_string(j);
          TRY(vq_attnblock(c, an, cur, t1, Hc, Wc, ch)); rot(t1);
        }
      }
      if (lvl != nres - 1) {
        const std::string dn = "encoder.conv_blocks." + std::to_string(lvl) + ".downsample.conv";
        TRY(vq_conv_down(c, cur, Hc, Wc, ch, dn, t1)); rot(t1);
        Hc /= 2; Wc /= 2;
      }
    }
    TRY(vq_resblock(c, "encoder.mid.0", cur, t1, t2, Hc, Wc, ch, ch)); rot(t2);
    TRY(vq_attnblock(c, "encoder.mid.1", cur, t1, Hc, Wc, ch)); rot(t1);
    TRY(vq_resblock(c, "encoder.mid.2", cur, t1, t2, Hc, Wc, ch, ch)); rot(t2);
    TRY(vq_conv(c, cur, Hc, Wc, ch, "encoder.conv_out", d.vq_z, 3, 1, "encoder.norm_out", true, nullptr, t1, nullptr)); rot(t1);
    TRY(vq_conv(c, cur, Hc, Wc, d.vq_z, "quant_conv", d.code_dim, 1, 1, nullptr, false, nullptr, t1, nullptr)); rot(t1);
    // nearest code: normalised codebook + its squared norms in the (now idle) partial buffer
    const size_t n_pix = (size_t)c.Bc * Hc * Wc;
    float* en = e->vq_part;
    float* e2 = e->vq_part + (size_t)d.img_vocab * d.code_dim;
    if ((size_t)d.img_vocab * (d.code_dim + 1) > e->vq_part_elems) return fail("internal: vq partial buffer too small (codebook)");
    TRY(launch(e, vq_codebook_norm_kernel, dim3((d.img_vocab + 255) / 256), dim3(256), 0, st, codebook, en, e2, d.img_vocab, d.code_dim));
    int32_t* out = codes_out + (size_t)b0 * Hc * Wc;
    DISPATCH_T(e,
               launch(e, vq_quantize_kernel<bf16>, dim3((unsigned)n_pix), dim3(256), 0, st, (const bf16*)cur, (const float*)en, (const float*)e2, out, d.img_vocab, d.code_dim),
               launch(e, vq_quantize_kernel<float>, dim3((unsigned)n_pix), dim3(256), 0, st, (const float*)cur, (const float*)en, (const float*)e2, out, d.img_vocab, d.code_dim));
  }
  e->use_pdl = saved_pdl;
  return 0;
}


// ------------------------------------------------------------------------------ debug / test hooks
// Launch the decode-attention kernel of one layer alone on the current KV cache (bench roofline leg).
// The QKV partial buffer is zero-filled, so the arithmetic is a uniform softmax over the cached tokens;
// bytes moved and control flow are those of a real step at column `pos`.
extern "C" int pg_test_attn_decode(pg_engine* e, const int32_t* kv_start, int R, int pos, int layer, void* stream) {
  TRY(check_ready(e));
  if (!e->bf16) return fail("pg_test_attn_decode: bf16 mode only");
  if (R < 1 || R > e->d.max_rows || R > AT_MAX_ROWS || pos < 1 || pos >= e->Tmax || layer < 0 || layer >= e->d.L)
    return fail("pg_test_attn_decode: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  NEED(cosT, float, "rope_cos");
  NEED(sinT, float, "rope_sin");
  const int HD = e->HD;
  const int ctas = e->attn_ctas > 0 ? e->attn_ctas : e->num_sms;
  const int saved = e->use_pdl;
  e->use_pdl = 0;
  int rc = launch(e, attn_decode_v5_kernel, dim3(ctas), dim3(AT_THREADS), A5_SMEM, st, (const float*)e->part, 1, (size_t)R * 3 * HD,
                  cosT, sinT, (bf16*)kv_ptr(e, layer, 0, R), (bf16*)kv_ptr(e, layer, 1, R), kv_start, (bf16*)e->attn_out,
                  e->attn_ll, R, e->d.H, e->Tmax, pos, (const int*)nullptr, 1.0f / sqrtf((float)HEAD_DIM), 1,
                  (int)e->attn_test_flags, next_prof(e), (unsigned long long*)e->attn_dbg_ptr,
                  (const int32_t*)((e->attn_test_alias_p > 0 && e->attn_alias) ? e->dup_of : nullptr), e->attn_test_alias_p);
  e->use_pdl = saved;
  return rc;
}
// One decode-attention launch as decode_layers issues it (same kernel, block, shared memory and cut for a CTA count),
// on caller-owned operands and with PDL off, so a test can compare the kernel with a reference of its own operation.
extern "C" int pg_test_attn_decode_io(pg_engine* e, int impl, int splits, const float* part, int S, int R, int H,
                                      void* kcache, void* vcache, int Tmax, const int32_t* kv_start,
                                      const int32_t* src_row, int alias_P, int pos, const int32_t* step_ptr,
                                      int rope_flags, int ctas, void* out, uint64_t* ws, void* stream) {
  TRY(check_ready(e));
  cudaStream_t st = (cudaStream_t)stream;
  if (impl != 0 && impl != 3) return fail("pg_test_attn_decode_io: impl must be 0 (plain kernel) or 3 (v5)");
  if (impl == 3 && !e->bf16) return fail("pg_test_attn_decode_io: impl 3 needs a bf16 engine");
  if (!part || !kcache || !vcache || !kv_start || !out) return fail("pg_test_attn_decode_io: null operand");
  if (S < 1 || S > 64) return fail("pg_test_attn_decode_io: S=%d must be in [1, 64]", S);
  if (H < 1) return fail("pg_test_attn_decode_io: H=%d must be >= 1", H);
  if (R < 1 || (impl == 3 && R > AT_MAX_ROWS)) return fail("pg_test_attn_decode_io: R=%d must be in [1, %d]", R, AT_MAX_ROWS);
  if (Tmax < 1) return fail("pg_test_attn_decode_io: Tmax=%d must be >= 1", Tmax);
  if (rope_flags != 0 && rope_flags != 1 && rope_flags != ROPE_REL)
    return fail("pg_test_attn_decode_io: rope_flags=%d must be 0, 1 or %d", rope_flags, ROPE_REL);
  if (ctas < 0 || ctas > e->num_sms) return fail("pg_test_attn_decode_io: ctas=%d must be in [0, num_sms=%d]", ctas, e->num_sms);
  if (splits < 0 || splits > 64) return fail("pg_test_attn_decode_io: splits=%d must be in [0, 64]", splits);
  // the position the kernel will use: with step_ptr it is pos + *step_ptr, read here to check its bounds
  int pos_eff = pos;
  if (step_ptr) {
    int32_t step = 0;
    CK(cudaMemcpyAsync(&step, step_ptr, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    pos_eff = pos + step;
  }
  if (pos_eff < 0 || pos_eff >= Tmax) return fail("pg_test_attn_decode_io: pos=%d must be in [0, Tmax=%d)", pos_eff, Tmax);
  if (pos_eff >= e->Tmax) return fail("pg_test_attn_decode_io: pos=%d must be below the engine's Tmax=%d (RoPE tables)", pos_eff, e->Tmax);
  NEED(cosT, float, "rope_cos");
  NEED(sinT, float, "rope_sin");
  const float scale = 1.0f / sqrtf((float)HEAD_DIM);
  const size_t split_stride = (size_t)R * 3 * H * HEAD_DIM;
  const int saved = e->use_pdl;
  e->use_pdl = 0;
  int rc = 0;
  if (impl == 3) {
    if (!ws) rc = fail("pg_test_attn_decode_io: ws (R*H*%d*%d zeroed words) is required for impl 3", AT_MAX_SLOTS, A5_REC);
    if (!src_row && alias_P != 0) rc = fail("pg_test_attn_decode_io: alias_P=%d without src_row", alias_P);
    if (!rc)
      rc = launch(e, attn_decode_v5_kernel, dim3(ctas > 0 ? ctas : e->num_sms), dim3(AT_THREADS), A5_SMEM, st, part, S,
                  split_stride, cosT, sinT, (bf16*)kcache, (bf16*)vcache, kv_start, (bf16*)out, (float*)ws, R, H, Tmax, pos,
                  (const int*)step_ptr, scale, rope_flags, 1, next_prof(e), (unsigned long long*)nullptr, src_row, alias_P);
  } else {
    const int nsp = splits > 0 ? splits : attn_split_count(e, R, pos_eff + 1);
    if (src_row || alias_P != 0) rc = fail("pg_test_attn_decode_io: the plain kernel reads every row's own cache (src_row, alias_P)");
    else if ((size_t)R * H * nsp > (size_t)e->d.max_rows * e->d.H * 64)
      rc = fail("pg_test_attn_decode_io: R*H*splits=%zu exceeds the split workspace (%zu)", (size_t)R * H * nsp,
                (size_t)e->d.max_rows * e->d.H * 64);
    else if ((size_t)R * H > (size_t)e->d.max_rows * e->d.H)
      rc = fail("pg_test_attn_decode_io: R*H=%d exceeds the split counters (%d)", R * H, e->d.max_rows * e->d.H);
    else if (e->bf16)
      rc = launch(e, attn_decode_kernel<bf16>, dim3(H, R, nsp), dim3(128), 0, st, part, S, split_stride, cosT, sinT,
                  (bf16*)kcache, (bf16*)vcache, kv_start, (bf16*)out, e->attn_ws, e->attn_cnt, H, Tmax, pos,
                  (const int*)step_ptr, scale, rope_flags);
    else
      rc = launch(e, attn_decode_kernel<float>, dim3(H, R, nsp), dim3(128), 0, st, part, S, split_stride, cosT, sinT,
                  (float*)kcache, (float*)vcache, kv_start, (float*)out, e->attn_ws, e->attn_cnt, H, Tmax, pos,
                  (const int*)step_ptr, scale, rope_flags);
  }
  e->use_pdl = saved;
  return rc;
}

// One prefill-attention launch as prefill_impl issues it (launch_prefill_attn, PDL off) on caller-owned operands.
extern "C" int pg_test_attn_prefill_io(pg_engine* e, int impl, const void* q, const void* kcache, const void* vcache,
                                       const int32_t* kv_start, const int32_t* row_off, int R, int P, int H, int Tmax,
                                       void* out, void* stream) {
  TRY(check_ready(e));
  cudaStream_t st = (cudaStream_t)stream;
  if (impl != 0 && impl != 1) return fail("pg_test_attn_prefill_io: impl=%d must be 0 (CUDA-core kernel) or 1 (tcgen05)", impl);
  if (impl == 1 && !(e->bf16 && e->use_tc)) return fail("pg_test_attn_prefill_io: impl 1 (tcgen05) needs a bf16 engine with use_tc");
  if (row_off && impl != 1) return fail("pg_test_attn_prefill_io: row_off (packed stream) needs impl 1 (tcgen05)");
  if (!q || !kcache || !vcache || !kv_start || !out) return fail("pg_test_attn_prefill_io: null operand");
  if (R < 1 || H < 1 || P < 1) return fail("pg_test_attn_prefill_io: R=%d H=%d P=%d must be >= 1", R, H, P);
  if (P > Tmax) return fail("pg_test_attn_prefill_io: P=%d must be <= Tmax=%d", P, Tmax);
  std::vector<int32_t> ks(R), ro(R + 1);
  CK(cudaMemcpyAsync(ks.data(), kv_start, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
  if (row_off) CK(cudaMemcpyAsync(ro.data(), row_off, (size_t)(R + 1) * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int r = 0; r < R; ++r)
    if (ks[r] < 0 || ks[r] > P) return fail("pg_test_attn_prefill_io: kv_start[%d]=%d must be in [0, P=%d]", r, ks[r], P);
  int tok = R * P;
  if (row_off) {
    if (ro[0] < 0) return fail("pg_test_attn_prefill_io: row_off[0]=%d must be >= 0", ro[0]);
    for (int r = 0; r < R; ++r) {
      const int n = ro[r + 1] - ro[r];
      if (n != 0 && n != P - ks[r])
        return fail("pg_test_attn_prefill_io: row_off[%d]-row_off[%d]=%d must be 0 or P-kv_start=%d (row_off monotone)", r + 1, r, n,
                    P - ks[r]);
    }
    tok = ro[R];
    if (tok < 1) return fail("pg_test_attn_prefill_io: row_off[R]=%d: the packed stream has no token", tok);
  }
  const int saved = e->use_pdl;
  e->use_pdl = 0;
  const int rc = launch_prefill_attn(e, impl == 1, q, tok, kcache, vcache, kv_start, row_off, out, R, P, H, Tmax, st);
  e->use_pdl = saved;
  return rc;
}

// One SigLIP attention launch as the vision tower issues it (launch_vit_attn, PDL off) on a caller-owned qkv buffer.
extern "C" int pg_test_vit_attn_io(pg_engine* e, int impl, const void* qkv, int qkv_rows, int n, int NP, int W, int heads,
                                   void* out, void* stream) {
  TRY(check_ready(e));
  if (impl != 0 && impl != 1) return fail("pg_test_vit_attn_io: impl=%d must be 0 (CUDA-core kernel) or 1 (tcgen05)", impl);
  if (!qkv || !out) return fail("pg_test_vit_attn_io: null operand");
  if (n < 1 || NP < 1 || heads < 1 || W < heads || W % heads != 0)
    return fail("pg_test_vit_attn_io: n=%d NP=%d W=%d heads=%d: need n, NP >= 1 and W a multiple of heads", n, NP, W, heads);
  if ((int64_t)n * NP > qkv_rows) return fail("pg_test_vit_attn_io: n*NP=%lld must be <= qkv_rows=%d", (long long)n * NP, qkv_rows);
  const int hd = W / heads;
  if (impl == 1) {
    if (!(e->bf16 && e->use_tc)) return fail("pg_test_vit_attn_io: impl 1 (tcgen05) needs a bf16 engine with use_tc");
    if (hd != VT_HD) return fail("pg_test_vit_attn_io: impl 1 (tcgen05) needs hd == %d (hd=%d)", VT_HD, hd);
  } else {
    if (NP > 32 * VA_MAXI) return fail("pg_test_vit_attn_io: NP=%d must be <= 32 * VA_MAXI = %d for impl 0", NP, 32 * VA_MAXI);
    if (hd > 128) return fail("pg_test_vit_attn_io: hd=%d must be <= 128 for impl 0", hd);
  }
  const int saved = e->use_pdl;
  e->use_pdl = 0;
  const int rc = launch_vit_attn(e, impl == 1, qkv, qkv_rows, out, n, NP, W, heads, (cudaStream_t)stream);
  e->use_pdl = saved;
  return rc;
}

extern "C" int pg_debug_zero_part(pg_engine* e, size_t nbytes, void* stream) {
  if (!e || !e->part) return fail("null engine");
  CK(cudaMemsetAsync(e->part, 0, std::min(nbytes, e->part_bytes), (cudaStream_t)stream));
  return 0;
}

extern "C" int pg_debug_copy(pg_engine* e, const char* name, void* dst_dev, size_t nbytes, void* stream) {
  if (!e || !name || !dst_dev) return fail("null argument");
  const std::string k(name);
  const void* src = nullptr;
  if (k == "x_dec") src = e->x_dec;
  else if (k == "xn") src = e->xn;
  else if (k == "attn_out") src = e->attn_out;
  else if (k == "hbuf") src = e->hbuf;
  else if (k == "hidden_f") src = e->hidden_f;
  else if (k == "part") src = e->part;
  else if (k == "qbuf") src = e->qbuf;
  else return fail("unknown debug buffer '%s'", name);
  CK(cudaMemcpyAsync(dst_dev, src, nbytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}


extern "C" int pg_test_gemm(pg_engine* e, int impl, int is_bf16, const void* X, const void* W, int M, int N, int K,
                            int splits, float* C, void* stream) {
  if (!e) return fail("null engine");
  if ((is_bf16 != 0) != e->bf16) return fail("operand type does not match the engine mode");
  int S = 0;
  TRY(run_gemm(e, X, W, M, N, K, C, (size_t)std::max(splits, 1) * M * N * 4, &S, (cudaStream_t)stream, impl, std::max(splits, 1), false));
  if (S != std::max(splits, 1)) {
    // fewer splits were possible: zero the remainder so the caller can always sum `splits` slabs
    CK(cudaMemsetAsync(C + (size_t)S * M * N, 0, (size_t)(std::max(splits, 1) - S) * M * N * 4, (cudaStream_t)stream));
  }
  return 0;
}

// One contraction as the engine issues it (run_gemm / run_conv_gemm / launch_swiglu_sk, PDL off) on caller-owned operands,
// reporting the kernel that ran, so a test can compare each fused epilogue with a restatement of its rounding points.
extern "C" int pg_test_contraction_run(pg_engine* e, pg_test_contraction* p, void* stream) {
  TRY(check_ready(e));
  if (!p) return fail("pg_test_contraction_run: null parameters");
  p->path = PG_PATH_NONE; p->path_nt = 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (!e->bf16 || !e->use_tc) return fail("pg_test_contraction_run: needs a bf16 engine with use_tc");
  const int M = p->M, N = p->N, K = p->K, mode = p->mode;
  if (mode < PG_TC_PLAIN || mode > PG_TC_CONV) return fail("pg_test_contraction_run: mode=%d must be in [0, 6]", mode);
  if (M < 1 || N < 1 || K < 1) return fail("pg_test_contraction_run: M=%d N=%d K=%d must be >= 1", M, N, K);
  if (K % 8 != 0) return fail("pg_test_contraction_run: K=%d must be a multiple of 8", K);
  if (!p->X || !p->W) return fail("pg_test_contraction_run: null X or W");
  if ((((uintptr_t)p->X) | ((uintptr_t)p->W)) & 15) return fail("pg_test_contraction_run: X and W must be 16-byte aligned");
  if (p->weights != 0 && p->weights != 1) return fail("pg_test_contraction_run: weights=%d must be 0 (row-major) or 1 (tile-major)", p->weights);
  const bool out_mode = mode == PG_TC_ROWS || mode == PG_TC_SWIGLU || mode == PG_TC_SWIGLU_SK || (mode == PG_TC_CONV && p->out);
  if (out_mode && !p->out) return fail("pg_test_contraction_run: out is required for mode %d", mode);
  if ((mode == PG_TC_PLAIN || (mode == PG_TC_CONV && !p->out)) && !p->C) return fail("pg_test_contraction_run: C is required for mode %d", mode);
  if (mode == PG_TC_RESID && !p->resid) return fail("pg_test_contraction_run: resid is required for mode %d", mode);
  if ((p->gelu != 0 && p->gelu != 1) || (p->gelu && mode != PG_TC_ROWS)) return fail("pg_test_contraction_run: gelu=%d is 0, or 1 in PG_TC_ROWS", p->gelu);
  if (p->add16 && p->gelu) return fail("pg_test_contraction_run: add16 and gelu are exclusive");
  if (p->add16 && mode != PG_TC_ROWS && mode != PG_TC_CONV) return fail("pg_test_contraction_run: add16 needs PG_TC_ROWS or PG_TC_CONV");
  if (p->bias && mode != PG_TC_ROWS && mode != PG_TC_RESID && mode != PG_TC_CONV) return fail("pg_test_contraction_run: bias needs PG_TC_ROWS, PG_TC_RESID or PG_TC_CONV");
  if ((mode == PG_TC_SWIGLU || mode == PG_TC_SWIGLU_SK) && N % TC_BM != 0) return fail("pg_test_contraction_run: SwiGLU needs N %% 128 == 0 (N=%d)", N);
  if (mode == PG_TC_SWIGLU && M > 128 && N <= TC_BM) return fail("pg_test_contraction_run: SwiGLU with M=%d > 128 runs on the CTA pair, which needs N > 128", M);
  if ((mode == PG_TC_ROWS || mode == PG_TC_RESID) && N % 8 != 0) return fail("pg_test_contraction_run: fused epilogues need N %% 8 == 0 (N=%d)", N);
  if (mode != PG_TC_PLAIN && p->splits > 1) return fail("pg_test_contraction_run: splits=%d: only PG_TC_PLAIN splits K", p->splits);
  // weights: tile-major copy into the caller's buffer (the kernel pg_engine_finalize uses)
  const uint8_t* w_tiled = nullptr;
  if (p->weights == 1) {
    if (mode == PG_TC_CONV) return fail("pg_test_contraction_run: the implicit convolution reads row-major weights only");
    if (tc_pair_taken(M, N, mode == PG_TC_PLAIN ? std::max(p->splits, 1) : 1, mode == PG_TC_SWIGLU && M <= 128) && mode != PG_TC_SWIGLU_SK)
      return fail("pg_test_contraction_run: M=%d N=%d runs on the CTA pair, which streams row-major weights (weights=1)", M, N);
    if (!p->w_tiled || p->w_tiled_bytes < tile_major_bytes(N, K))
      return fail("pg_test_contraction_run: w_tiled needs %zu bytes (has %zu)", tile_major_bytes(N, K), p->w_tiled_bytes);
    TRY(build_tile_major(e, p->W, N, K, (uint8_t*)p->w_tiled, st));
    w_tiled = (const uint8_t*)p->w_tiled;
  } else if (mode == PG_TC_SWIGLU_SK) {
    return fail("pg_test_contraction_run: stream-K streams tile-major weights (weights=1)");
  }
  QkvEpi qe = {};
  if (mode == PG_TC_QKV) {
    const int R = p->R, P = p->P, H = p->H, Tmax = p->Tmax;
    if (H < 1 || N != 3 * H * HEAD_DIM) return fail("pg_test_contraction_run: QKV needs N == 3*H*128 (N=%d H=%d)", N, H);
    if (!tc_pair_taken(M, N, 1, false)) return fail("pg_test_contraction_run: the QKV epilogue runs on the CTA pair only (M=%d must be > 128)", M);
    if (!p->q_out || !p->kcache || !p->vcache || !p->kv_start) return fail("pg_test_contraction_run: QKV needs q_out, kcache, vcache and kv_start");
    if (R < 1 || Tmax < 1) return fail("pg_test_contraction_run: QKV needs R=%d >= 1 and Tmax=%d >= 1", R, Tmax);
    // every token's cache column and RoPE position, restated on the host for the bounds
    std::vector<int32_t> ks(R), ro(R), rs(R, 0);
    CK(cudaMemcpyAsync(ks.data(), p->kv_start, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
    if (p->row_off) CK(cudaMemcpyAsync(ro.data(), p->row_off, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
    if (p->rope_start) CK(cudaMemcpyAsync(rs.data(), p->rope_start, (size_t)R * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (!p->row_off && (P < 1 || (size_t)M > (size_t)R * P)) return fail("pg_test_contraction_run: QKV padded block needs M=%d <= R*P (R=%d P=%d)", M, R, P);
    for (int m = 0; m < M; ++m) {
      int rw = 0, col = 0;
      if (p->row_off) {
        int lo = 0, hi = R - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (ro[mid] <= m) lo = mid; else hi = mid - 1; }
        rw = lo; col = ks[rw] + (m - ro[rw]);
        if (m < ro[rw]) return fail("pg_test_contraction_run: QKV token %d lies before row_off[0]=%d", m, ro[0]);
      } else {
        rw = m / P; col = m % P;
      }
      const int pr = p->rope_start ? std::max(col - rs[rw], 0) : col;
      if (col < 0 || col >= Tmax) return fail("pg_test_contraction_run: QKV token %d: cache column %d must be in [0, Tmax=%d)", m, col, Tmax);
      if (pr >= e->Tmax) return fail("pg_test_contraction_run: QKV token %d: RoPE position %d must be below the engine's Tmax=%d", m, pr, e->Tmax);
    }
    NEED(cosT, float, "rope_cos");
    NEED(sinT, float, "rope_sin");
    qe = QkvEpi{cosT, sinT, (bf16*)p->q_out, (bf16*)p->kcache, (bf16*)p->vcache, p->row_off, p->kv_start, p->rope_start, R, P, H, Tmax};
  }
  const int saved_pdl = e->use_pdl;
  e->use_pdl = 0;
  int rc = 0;
  int S = 1;
  const size_t fused_bytes = (size_t)M * N * 4;   // the fused epilogues write no partials; run_gemm only checks the size
  EpiFuse ep = {p->bias, (bf16*)p->out, nullptr, p->gelu, (const bf16*)p->add16};
  switch (mode) {
    case PG_TC_PLAIN: {
      const int sp = std::max(p->splits, 1);
      if (!p->C || p->c_bytes < (size_t)sp * M * N * 4) { rc = fail("pg_test_contraction_run: C needs splits*M*N*4 = %zu bytes", (size_t)sp * M * N * 4); break; }
      rc = run_gemm(e, p->X, p->W, M, N, K, p->C, (size_t)sp * M * N * 4, &S, st, 1, sp, false, w_tiled);
      if (!rc && S != sp) rc = cudaMemsetAsync(p->C + (size_t)S * M * N, 0, (size_t)(sp - S) * M * N * 4, st) == cudaSuccess ? 0 : fail("memset of unused splits failed");
      break;
    }
    case PG_TC_ROWS:
      rc = run_gemm(e, p->X, p->W, M, N, K, nullptr, fused_bytes, &S, st, 1, 1, false, w_tiled, nullptr, &ep);
      break;
    case PG_TC_RESID: {
      const EpiFuse er = {p->bias, nullptr, p->resid, 0, nullptr};
      rc = run_gemm(e, p->X, p->W, M, N, K, nullptr, fused_bytes, &S, st, 1, 1, false, w_tiled, nullptr, &er);
      break;
    }
    case PG_TC_SWIGLU:
      if (M <= 128) {
        rc = run_gemm(e, p->X, p->W, M, N, K, nullptr, fused_bytes, &S, st, 1, 1, false, w_tiled, p->out);
      } else {
        const EpiFuse eg = {nullptr, (bf16*)p->out, nullptr, 2, nullptr};
        rc = run_gemm(e, p->X, p->W, M, N, K, nullptr, fused_bytes, &S, st, 1, 1, false, nullptr, nullptr, &eg);
      }
      break;
    case PG_TC_QKV: {
      const EpiFuse eq = {nullptr, (bf16*)p->q_out, nullptr, 3, nullptr};
      e->qkv_epi_next = qe;
      rc = run_gemm(e, p->X, p->W, M, N, K, nullptr, fused_bytes, &S, st, 1, 1, false, nullptr, nullptr, &eq);
      e->qkv_epi_next = QkvEpi{};
      break;
    }
    case PG_TC_SWIGLU_SK:
      if (!p->scratch || !p->counters) { rc = fail("pg_test_contraction_run: stream-K needs scratch and counters"); break; }
      rc = launch_swiglu_sk(e, p->X, w_tiled, M, N / 2, K, p->ctas, p->scratch, p->scratch_bytes, p->counters, p->n_counters, (bf16*)p->out, st);
      break;
    case PG_TC_CONV: {
      const int B = p->img_b, H = p->img_h, W = p->img_w, Cin = K / 9;
      if (K % 9 != 0 || B < 1 || H < 1 || W < 1 || (size_t)M != (size_t)B * H * W) {
        rc = fail("pg_test_contraction_run: conv needs K = 9*Cin and M = img_b*img_h*img_w (M=%d K=%d B=%d H=%d W=%d)", M, K, B, H, W);
        break;
      }
      if (p->out && N % 8 != 0) { rc = fail("pg_test_contraction_run: the fused conv epilogue needs N %% 8 == 0 (N=%d)", N); break; }
      int taken = 0;
      rc = run_conv_gemm(e, p->X, p->W, B, H, W, Cin, N, p->C, p->C ? p->c_bytes : (size_t)M * N * 4, st, &taken, p->out ? &ep : nullptr);
      break;
    }
  }
  e->use_pdl = saved_pdl;
  if (!rc) { p->path = e->last_path; p->path_nt = e->last_nt; }
  return rc;
}
