/* plangen_b200 C-ABI — the drop-in boundary for PlanGen's CFG image-token decode path (and the rows next to it:
 * stage-1 layout-text decode pg_generate_greedy, VQ encode of the editing path pg_vq_encode).
 *
 * The reference (360CVGroup/PlanGen) is pure Python: the seam is duck-typed attribute
 * access on `self.vl_gpt` from `System.t2i` / `System.sample_image`
 * (project/plangen/plangen_base.py:525-607).  Each entry point below names the
 * reference call it replaces.  All pointers are DEVICE pointers unless a name ends in
 * `_host`; sizes are explicit; `stream` is a `cudaStream_t` passed as `void*`.
 * Every function returns 0 on success and a non-zero status otherwise (never throws);
 * `pg_last_error()` gives the message.  The caller owns all memory; weights are
 * borrowed read-only for the engine's lifetime.  One host thread per engine.
 */
#ifndef PLANGEN_B200_H
#define PLANGEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_ABI_VERSION 10

/* arithmetic regimes */
#define PG_MODE_BF16 0 /* the reference's regime: fp32 master weights under autocast(bf16), plangen_base.py:360 */
#define PG_MODE_FP32 1 /* fp32 check mode (BASELINE config 1; north_star "fp32 check mode") */

typedef struct pg_engine pg_engine;

typedef struct pg_dims {
  int32_t D, L, H, head_dim, F;      /* LlamaConfig: hidden, layers, heads, head_dim, intermediate */
  int32_t vocab, img_vocab, code_dim, img_embed, grid;
  float rms_eps, rope_theta;
  int32_t vq_ch, vq_nres, vq_ch_mult[8], vq_z, vq_res_blocks;
  int32_t mode;                      /* PG_MODE_* */
  int32_t max_rows;                  /* R = 2 * B * parallel_size upper bound */
  int32_t max_prompt;                /* padded prompt length P upper bound */
  int32_t max_steps;                 /* image tokens per image (576) upper bound */
  /* mmu front-end (SigLIP vision tower, siglip_vit.py:628-637 SigLIP_MODEL_CONFIG); sig_layers = 0 or max_images = 0: not built */
  int32_t sig_width, sig_layers, sig_heads, sig_patch, sig_image, sig_mlp;
  int32_t max_images;                /* images per prepare_inputs_embeds call upper bound */
} pg_dims;

const char* pg_last_error(void);
int pg_abi_version(void);

/* Engine lifetime.  replaces: MultiModalityCausalLM.__init__ / from_pretrained
 * (three_party/Janus/janus/models/modeling_vlm.py:190-219; plangen_base.py:95-97). */
int pg_engine_create(const pg_dims* dims, int device, pg_engine** out);
int pg_engine_destroy(pg_engine* e);

/* Bytes of KV cache / scratch workspace the caller must allocate and bind.  pg_engine_bind_buffers zero-fills the KV
 * cache once (the attention kernels' TMA tiles read masked slots past the newest token: they must hold finite values). */
int pg_engine_query_bytes(const pg_engine* e, size_t* kv_bytes, size_t* ws_bytes);
int pg_engine_bind_buffers(pg_engine* e, void* kv, size_t kv_bytes, void* ws, size_t ws_bytes);

/* Register one weight tensor by its (packed) name; see plangen_b200/weights.py for the
 * packing of the reference state_dict names (SURVEY.md §8b) into these slots. */
int pg_engine_set_tensor(pg_engine* e, const char* name, const void* dev_ptr, size_t nbytes);

/* Build derived tables (gen_aligner(gen_embed(.)) table, L2-normalised codebook,
 * TMA descriptors).  Must be called once after all tensors are set. */
int pg_engine_finalize(pg_engine* e, void* stream);

/* replaces: language_model.get_input_embeddings()(ids)   plangen_base.py:548
 * ids int32 [R*P] -> x fp32 [R*P, D] */
int pg_embed_tokens(pg_engine* e, const int32_t* ids, int n_tokens, float* x_out, void* stream);

/* replaces: language_model.model(inputs_embeds=(R,P,D), attention_mask, use_cache=True,
 *           past_key_values=None)                           plangen_base.py:571-576 (i == 0)
 * x fp32 [R,P,D] is consumed in place (residual stream).  kv_start[r] = number of LEFT pad
 * columns of row r (lossless encoding of the 0/1 mask, SURVEY.md appendix A.2).
 * hidden_out: final-norm'ed last_hidden_state; all_positions=1 -> [R,P,D], 0 -> [R,D] (last). */
int pg_prefill(pg_engine* e, float* x, const int32_t* kv_start, int R, int P,
               float* hidden_out, int all_positions, void* stream);

/* replaces: language_model.model(inputs_embeds=(R,1,D), past_key_values=prev)  (i >= 1)
 * x fp32 [R,D]; pos = absolute column index of this token (P + i - 1). */
int pg_decode_step(pg_engine* e, const float* x, const int32_t* kv_start, int R, int pos,
                   float* hidden_out, void* stream);

/* replaces: vl_gpt.gen_head(h)          modeling_vlm.py:36-51 / plangen_base.py:579
 * hidden fp32 [R,D] -> logits fp32 [R,img_vocab] (bf16-rounded values in PG_MODE_BF16). */
int pg_gen_head(pg_engine* e, const float* hidden, int R, float* logits_out, void* stream);

/* Sampling settings of one image, passed to the three sampling entry points below as a HOST array of B entries (copied at
 * entry; the array may be reused when the call returns).  One batch can serve requests with different seeds, guidance
 * scales, temperatures, top-k and top-p; batch-wide settings are the same entry repeated.
 * Image b is sampled with its (cfg_weight, temperature, top_k, top_p): CFG rounded per op in the engine dtype, a
 * correctly rounded /temperature, top-k, top-p, softmax.
 *   top_k > 0: only CFG logits >= the k-th largest survive (`logits[logits < topk(logits,k)[..., -1:]] = -inf`) before
 *     the softmax; 0 = off = the reference (it has no top-k; north_star names the option).
 *   top_p in [0, 1) (after top-k): HF TopPLogitsWarper with min_tokens_to_keep = 1 - in ascending (logit, index) order
 *     the longest prefix whose cumulative probability is <= fp32(1 - top_p) is removed, the largest logit always stays;
 *     1 = off (the unfiltered path).  top_p is a double: the kernel compares against fp32(1 - top_p) with 1 - top_p in
 *     double, as torch does.  Ignored when greedy != 0.
 *   top_k >= 0 and top_p in [0, 1] (NaN fails) are checked per image, and a failure names the image.
 * seed / offset: torch.multinomial(1) with Philox4x32-10, bit-compatible with torch's CUDA generator at (seed, offset).
 *   rng_per_image != 0 - image b draws as torch.multinomial(probs[b:b+1], 1, generator=g_b) with g_b at (seed, offset):
 *   element v of a (1, V) tensor, so its tokens depend neither on b nor on B; each step advances its offset by torch's
 *   per-draw increment for numel = V (4 at V = 16384).  rng_per_image == 0 - entry 0's seed and offset serve the whole
 *   call as one generator drawing a (B, V) tensor (element b * V + v); the other entries' seed and offset are ignored. */
typedef struct pg_image_sampling {
  uint64_t seed, offset;
  float cfg_weight, temperature;
  int32_t top_k;
  double top_p;
} pg_image_sampling;

/* Image-token log-probabilities (logprobs_out; NULL: none).  For image b at step i the value is log p(tok) in fp32, p
 * being exactly the distribution the sampler draws from (CFG rounded per op in the engine dtype, /temperature, top-k,
 * top-p, softmax; in greedy mode top-k only) and tok the token emitted at that step, sampled or forced by teacher forcing:
 * (t_tok - max) - log(sum of the kept e), HF compute_transition_scores(..., normalize_logits=True) on the processed
 * scores.  A forced token a filter removed gets -inf; a kept one whose exp underflows still gets its finite value.
 * Log-probs change no token, no Philox draw and no offset.
 *
 * Guidance schedules (cfg_schedule_host; NULL: per_image[b].cfg_weight): a guidance weight per image AND per step
 * (LlamaGen's cfg_interval, MAR's linear ramp), a HOST fp32 array [R/2][n] (row-major; copied at entry, reusable when the
 * call returns).  At step i image b is sampled exactly as with per_image[b].cfg_weight = cfg_schedule[b][i] (same
 * rounding per op, /temperature, top-k, top-p, softmax, Philox draws and offsets); its log-probs are taken under that
 * distribution.  per_image[b].cfg_weight is then IGNORED (it may hold anything, NaN included); every other field keeps
 * its meaning.  Every entry must be finite: a failure names the image and the step ("image b, step i"), checked on the
 * host without a device sync.  A weight of 1 is u + 1 * (c - u) rounded per op, not the conditional logits alone: in
 * bf16 the two can differ by a rounding, so an interval schedule (w, then 1) reproduces "guidance off" in distribution,
 * not bit for bit.  The unconditional rows are computed on every step, also after the last step whose weight differs
 * from 1. */

/* replaces: plangen_base.py:580-604 — CFG combine, /temperature, softmax, torch.multinomial(1), teacher-forcing override
 * (:593-598), token duplication and prepare_gen_img_embeds.  logits fp32 [2B, V] (rows interleaved cond/uncond).
 * per_image HOST [B] (see pg_image_sampling; its offsets are the offsets of this draw).
 * edit_region / gt_labels: int32 [B, n_steps], both or neither (NULL = no teacher forcing; the caller gates them on
 * args.use_teacher_forcing as the reference does, :593).  greedy != 0 -> argmax.
 * tokens_out int32 [B, n_steps] (column `step` written); x_next fp32 [2B, D]; logprobs_out fp32 [B, n_steps] (column
 * `step` written) or NULL.  The settings are staged in engine memory on `stream`: like every entry point, calls on one
 * engine must be made in order. */
int pg_cfg_sample_embed(pg_engine* e, const float* logits, int B, const pg_image_sampling* per_image, int rng_per_image,
                        int greedy, const int32_t* edit_region, const int32_t* gt_labels, int step, int n_steps,
                        int32_t* tokens_out, float* x_next, float* logprobs_out, void* stream);

/* replaces: vl_gpt.prepare_gen_img_embeds(ids)     modeling_vlm.py:270-271
 * ids int32 [n] -> fp32 [n, D] */
int pg_prepare_gen_img_embeds(pg_engine* e, const int32_t* ids, int n, float* out, void* stream);

/* replaces: System.sample_image (plangen_base.py:567-607), whole loop on the device:
 * prefill + n_steps x (gen_head, CFG, sample, embed, decode step) with no host sync.
 * x_prompt fp32 [R,P,D] (consumed).  per_image HOST [R/2]; cfg_schedule_host HOST [R/2][n_steps] or NULL.
 * tokens_out int32 [R/2, n_steps]; logprobs_out fp32 [R/2, n_steps] or NULL.  kv_start / edit_region / gt_labels, the
 * settings and the schedule are copied into engine-owned buffers at entry and read on the device, so the captured
 * decode-step graph is keyed on the shape, greedy, teacher forcing, rng_per_image, whether any image uses top-p, whether
 * log-probs are asked for and whether there is a schedule - not on caller addresses nor on the values: new seeds,
 * settings and schedules replay the same graph.  The log-probs are staged in the engine inside the captured graph and
 * copied out with the tokens. */
int pg_sample_image(pg_engine* e, float* x_prompt, const int32_t* kv_start, int R, int P, int n_steps,
                    const pg_image_sampling* per_image, int rng_per_image, int greedy, const int32_t* edit_region,
                    const int32_t* gt_labels, const float* cfg_schedule_host, int32_t* tokens_out, float* logprobs_out,
                    void* stream);

/* Teacher-forced scoring of given image tokens in one pass: logprobs_out fp32 [R/2, n] = the log-probs (as above) the
 * image loop would report with every token forced, computed by ONE prefill over prompt + image tokens (the reference's
 * single full-sequence forward: fp32 residual stream, the prefill's rounding points - not the decode loop's bf16
 * residual regime, so in bf16 the two are different valid evaluations), one wide gen_head contraction over all R * n
 * positions (in chunks that fit the prefill scratch) and the sampler's reduction in score mode.
 * x_seq fp32 [R, P + n - 1, D] (consumed): columns < P hold the prompt embeddings (LEFT padded, kv_start as for
 * pg_prefill); columns P .. P + n - 2 are written here from the gen_aligner(gen_embed) table, token i at column P + i
 * on both rows of the pair.  image_tokens int32 [R/2, n] (ids clamped to [0, img_vocab)); per_image HOST [R/2]
 * (cfg_weight, temperature, top_k, top_p; seeds and offsets are unused); cfg_schedule_host HOST [R/2][n] or NULL:
 * position i of image b is scored with cfg_schedule[b][i].  R even, n <= max_steps and P + n - 1 <= max_prompt (build
 * the engine with a larger max_prompt to score long sequences).  Overwrites the KV cache.  No allocation; the prefill's
 * host syncs are the only ones. */
int pg_score_image_tokens(pg_engine* e, float* x_seq, const int32_t* kv_start, int R, int P, int n,
                          const int32_t* image_tokens, const pg_image_sampling* per_image,
                          const float* cfg_schedule_host, float* logprobs_out, void* stream);

/* replaces: System.x2t (plangen_base.py:513-523) = vl_gpt.language_model.generate(inputs_embeds=,
 *           attention_mask=, pad_token_id=, eos_token_id=, max_new_tokens=, do_sample=False, use_cache=True),
 *           HF GenerationMixin greedy search with position_ids derived from the attention mask.
 * Stage-1 layout-text decode (SURVEY.md 8f rank 1).  Needs the optional tensor "lm_head" [vocab, D].
 * x_prompt fp32 [R,P,D] (consumed); kv_start int32 [R] = leading pad columns per row.
 * tokens_out int32 [R, max_new_tokens] (device): rows that produced eos continue with pad_id, as in HF.
 * *n_generated (HOST int) = number of valid columns: HF stops after the step at which every row has finished.
 * Synchronises `stream` before returning (generate() is synchronous in the reference too). */
int pg_generate_greedy(pg_engine* e, float* x_prompt, const int32_t* kv_start, int R, int P,
                       int max_new_tokens, int eos_id, int pad_id, int32_t* tokens_out,
                       int* n_generated, void* stream);

/* replaces: gen_vision_model.decode_code(code_b, shape=[B,8,g,g], channel_first=True)
 *           three_party/Janus/janus/models/vq_model.py:505-508
 * codes int32 [B, gh*gw] -> image fp32 NCHW [B,3,16*gh,16*gw] (unclamped). */
int pg_vq_decode_code(pg_engine* e, const int32_t* codes, int B, int gh, int gw,
                      float* image_out, void* stream);

/* replaces: vl_gpt.gen_vision_model.encode(img)[-1][-1]   (plangen_base.py:532, editing path;
 *           three_party/Janus/janus/models/vq_model.py:494-498 -> Encoder.forward :108-124, quant_conv,
 *           VectorQuantizer.forward :236-262)
 * image fp32 NCHW [B,3,H,W] in [-1,1] (H, W multiples of 16) -> codes int32 [B, (H/16)*(W/16)]: index of the nearest
 * L2-normalised codebook entry per position (first index on ties).  Needs the optional encoder / quant_conv tensors. */
int pg_vq_encode(pg_engine* e, const float* image, int B, int H, int W, int32_t* codes_out, void* stream);

/* replaces: vl_gpt.prepare_inputs_embeds(input_ids, pixel_values, images_seq_mask, images_emb_mask)
 *           (plangen_base.py:289,366,855 -> three_party/Janus/janus/models/modeling_vlm.py:221-268): every image through the
 *           SigLIP vision tower (clip_encoder.py:107-122, siglip_vit.py:562-591) and the `aligner` MLP (projector.py:39-45),
 *           scattered into the text embeddings at the positions images_seq_mask selects; ids < 0 are embedded as id 0.
 * mmu front-end (SURVEY.md 8f rank 2).  pixel_values fp32 [n_images,3,S,S] ("b n c h w" flattened over (b n)); input_ids
 * int32 [B*T]; images_seq_mask uint8 [B*T]; images_emb_mask uint8 [n_images * n_patches]; embeds_out fp32 [B,T,D].
 * Fails if the two masks select different counts (the reference asserts it).  Synchronises `stream` once (that check).
 * Needs the optional tensors sig.* / ualign.* and pg_dims.sig_layers > 0, max_images > 0. */
int pg_prepare_inputs_embeds(pg_engine* e, const float* pixel_values, int n_images, const int32_t* input_ids,
                             const uint8_t* images_seq_mask, const uint8_t* images_emb_mask, int B, int T,
                             float* embeds_out, void* stream);

/* Vision tower + aligner alone: aligner(vision_model(images)) (modeling_vlm.py:250), pixel fp32 [n,3,S,S] ->
 * feat_out fp32 [n * n_patches, D] (NULL: features stay in the engine; bench). */
int pg_vision_features(pg_engine* e, const float* pixel_values, int n_images, float* feat_out, void* stream);

/* replaces: denorm_pt + `(x*255).astype(np.uint8)` of the image writers (src/utils/funcs.py:511-512, :497-498;
 *           plangen_base.py:444, :1168-1181): image fp32 [n] in about [-1,1] -> uint8 [n] = trunc(((clamp(x,-1,1)+1)/2)*255) */
int pg_images_to_u8(pg_engine* e, const float* image, size_t n, uint8_t* out, void* stream);

/* Bench / profiling helpers */
int pg_engine_set_option(pg_engine* e, const char* key, int64_t value);
int pg_engine_get_counter(const pg_engine* e, const char* key, int64_t* value);

/* Copy an internal workspace buffer (x_dec, xn, attn_out, hbuf, hidden_f, part, qbuf) for debugging. */
int pg_debug_copy(pg_engine* e, const char* name, void* dst_dev, size_t nbytes, void* stream);

/* Decode-attention kernel of one layer alone on the current KV cache (bench roofline leg); the QKV partial
 * buffer must have been zeroed with pg_debug_zero_part. */
int pg_test_attn_decode(pg_engine* e, const int32_t* kv_start, int R, int pos, int layer, void* stream);
int pg_debug_zero_part(pg_engine* e, size_t nbytes, void* stream);

/* One decode-attention launch exactly as the decode step issues it (same kernel, block, shared memory and cut for a
 * given CTA count; PDL off), on caller-owned operands, for unit tests of the kernel's own operation.
 *   impl 3: attn_decode_v5_kernel (bf16 engines); impl 0: the plain kernel in the engine's dtype with `splits`
 *           T-splits (0 = the engine's rule); it uses the engine's split workspace and takes no src_row.
 *   part: fp32 QKV split-K partials [S][R][3*H*128], S <= 64.
 *   kcache / vcache: [R][H][Tmax][128] in the engine's dtype; the kernel writes column pos (the new k / v).
 *   kv_start[R] (<= pos), src_row[R] or NULL, alias_P: cached columns below alias_P of row r are read from row
 *           src_row[r] (impl 3 only).
 *   pos, step_ptr: the position is pos + *step_ptr when step_ptr is not NULL (read once on the host for the
 *           bounds check, which synchronises `stream`); it must be below Tmax and the engine's Tmax (RoPE tables).
 *   rope_flags: 1 = bf16 trig with absolute positions (image decode), 0 = fp32 trig, 2 = fp32 trig with positions
 *           relative to kv_start (text decode).
 *   ctas: grid of impl 3, 0 = number of SMs, never more (a contributor waits for lower-numbered CTAs).
 *   H: any head count.  out: [R][H*128] in the engine's dtype.
 *   ws: impl 3's hand-off records, R*H*64*130 64-bit words, zero on entry and zero again on return. */
int pg_test_attn_decode_io(pg_engine* e, int impl, int splits, const float* part, int S, int R, int H, void* kcache,
                           void* vcache, int Tmax, const int32_t* kv_start, const int32_t* src_row, int alias_P, int pos,
                           const int32_t* step_ptr, int rope_flags, int ctas, void* out, uint64_t* ws, void* stream);

/* One prefill-attention launch exactly as the prefill issues it (same kernel, grid, shared memory and TMA maps; PDL off)
 * on caller-owned operands, for unit tests of the kernel's own operation.  Synchronises `stream` once (bounds checks).
 *   impl 1: attn_prefill_tc_kernel (bf16 engine with use_tc); impl 0: attn_prefill_kernel in the engine's dtype.
 *   kcache / vcache: [R][H][Tmax][128], P <= Tmax; kv_start[R] in [0, P] (left padding of each row).
 *   row_off: NULL - q and out are the padded block [R*P][H*128] (pad queries get zeros); otherwise (impl 1 only) the
 *           packed stream of the real tokens, row_off[R+1] monotone with row_off[r+1] - row_off[r] either 0 (a duplicate
 *           row: no tokens, nothing written) or P - kv_start[r]; q and out then hold row_off[R] rows.
 *   Masked cache columns inside the 128-key blocks a tile walks must be finite (they enter P.V with weight 0). */
int pg_test_attn_prefill_io(pg_engine* e, int impl, const void* q, const void* kcache, const void* vcache,
                            const int32_t* kv_start, const int32_t* row_off, int R, int P, int H, int Tmax, void* out,
                            void* stream);

/* One SigLIP attention launch exactly as the vision tower issues it (PDL off) on a caller qkv buffer [qkv_rows][3W] in the
 * engine's dtype: image i is rows [i*NP, (i+1)*NP), n*NP <= qkv_rows; the tcgen05 kernel's TMA maps cover all qkv_rows,
 * so rows after image n-1 hold data the kernel must not use.  out: [n*NP][W].
 *   impl 1: vit_attn_tc_kernel (bf16 engine with use_tc, W / heads == 64); impl 0: vit_attn_kernel in the engine's dtype
 *   (NP <= 1024, W / heads <= 128). */
int pg_test_vit_attn_io(pg_engine* e, int impl, const void* qkv, int qkv_rows, int n, int NP, int W, int heads, void* out,
                        void* stream);

/* Host-only helper of the prefill (no device work, callable without a GPU): proposes, for every prompt row, the FIRST
 * row of the batch with the same left padding `start[r]` and the same 64-bit content hash (itself when there is none).
 * The prefill verifies every proposal word for word on the device before using it (t2i's shared negative prompt,
 * cfg/base.py:129; the `parallel_size` copies of plangen_base.py:547-549).  Returns the number of proposals. */
int pg_host_group_rows(const int32_t* start, const uint64_t* hash, int R, int32_t* source_row);

/* Plain GEMM exposed for unit tests:  C[m,n] = sum_k X[m,k] * W[n,k]
 * impl 0 = SIMT (fp32 or bf16 inputs), 1 = tcgen05 (bf16 inputs).  C fp32 [splits][M][N]. */
int pg_test_gemm(pg_engine* e, int impl, int is_bf16, const void* X, const void* W, int M, int N,
                 int K, int splits, float* C, void* stream);

/* One tcgen05 contraction exactly as the engine issues it (run_gemm, run_conv_gemm, the stream-K gate|up launch; PDL
 * off) on caller-owned bf16 operands, for unit tests of the fused epilogues.  bf16 engines only.
 *   X [M][K] (conv: NHWC activation [img_b][img_h][img_w][K / 9]), W [N][K] row-major (conv: [Cout = N][9 * Cin]).
 *   weights 1: W is first copied tile-major (tile_weight_kernel, as pg_engine_finalize does) into w_tiled, which the
 *   contraction then streams; the copy stays there for inspection.  Read by gemm_tc and stream-K only.
 *   mode:
 *     PG_TC_PLAIN   C fp32 [splits][M][N] split-K partials (splits >= 1; fewer may be used, as pg_test_gemm);
 *     PG_TC_ROWS    out bf16 [M][N] = bf16(act(bf16(acc + bias))) or bf16(bf16(acc + bias) + add16) (add16 may be out),
 *                   act = GELU when gelu == 1; bias may be NULL;
 *     PG_TC_RESID   resid fp32 [M][N] += bf16(acc + bias);
 *     PG_TC_SWIGLU  out bf16 [M][N / 2]: W rows interleaved by 64 (weights.py), N % 128 == 0;
 *     PG_TC_QKV     q_out [M][H*128], kcache / vcache [R][H][Tmax][128]; N == 3*H*128, M > 128 (CTA pair); row_off[R]
 *                   (packed stream, positions kv_start[r] + t - row_off[r]) or NULL (padded [R][P] block, position t % P);
 *                   rope_start[R] or NULL.  Positions must be below Tmax and the engine's Tmax (RoPE tables);
 *     PG_TC_SWIGLU_SK  stream-K gate|up + SwiGLU (M <= 64, tile-major weights): out as PG_TC_SWIGLU, ctas (0 = the
 *                   production rule), scratch fp32 and counters (zero on entry, zero again on return) of the caller;
 *     PG_TC_CONV    3x3 implicit convolution, pad 1: C fp32 [pixels][N], or with out set the fused bias / add16 bf16 store.
 *   path / path_nt (out): the kernel that ran (PG_PATH_*), and its token-tile width. */
#define PG_TC_PLAIN 0
#define PG_TC_ROWS 1
#define PG_TC_RESID 2
#define PG_TC_SWIGLU 3
#define PG_TC_QKV 4
#define PG_TC_SWIGLU_SK 5
#define PG_TC_CONV 6
#define PG_PATH_NONE 0
#define PG_PATH_SIMT 1
#define PG_PATH_TC 2      /* gemm_tc_kernel<path_nt> */
#define PG_PATH_TC2 3     /* gemm_tc2_kernel (CTA pair) */
#define PG_PATH_SK 4      /* gemm_swiglu_sk_kernel<path_nt> */
#define PG_PATH_CONV 5    /* gemm_tc_kernel<192> as implicit convolution */
#define PG_PATH_IM2COL 6  /* the convolution does not qualify: the engine would use im2col (nothing launched) */
typedef struct pg_test_contraction {
  int mode, weights;
  int M, N, K, splits;
  const void* X;
  const void* W;
  void* w_tiled; size_t w_tiled_bytes;
  float* C; size_t c_bytes;
  void* out;
  const float* bias;
  int gelu;
  const void* add16;
  float* resid;
  void* q_out; void* kcache; void* vcache;
  const int32_t* row_off; const int32_t* kv_start; const int32_t* rope_start;
  int R, P, H, Tmax;
  int ctas;
  float* scratch; size_t scratch_bytes;
  int* counters; int n_counters;
  int img_b, img_h, img_w;
  int path, path_nt;
} pg_test_contraction;
int pg_test_contraction_run(pg_engine* e, pg_test_contraction* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PLANGEN_B200_H */
