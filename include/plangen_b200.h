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

#define PG_ABI_VERSION 3

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

/* replaces: plangen_base.py:580-604 — CFG combine, /temperature, softmax,
 * torch.multinomial(1) (Philox4x32-10, bit-compatible with torch's CUDA generator at
 * (seed, philox_offset)), teacher-forcing override (:593-598), token duplication and
 * prepare_gen_img_embeds.  logits fp32 [2B, V] (rows interleaved cond/uncond).
 * edit_region / gt_labels: int32 [B, n_steps], both or neither (NULL = no teacher forcing; the caller gates them on
 * args.use_teacher_forcing as the reference does, :593).  greedy != 0 -> argmax.
 * top_k > 0: only CFG logits >= the k-th largest survive (`logits[logits < topk(logits,k)[..., -1:]] = -inf`) before
 * the softmax; 0 = off = the reference (it has no top-k; north_star names the option).
 * top_p in [0, 1) (after top-k): HF TopPLogitsWarper with min_tokens_to_keep = 1 - in ascending (logit, index) order
 * the longest prefix whose cumulative probability is <= fp32(1 - top_p) is removed, the largest logit always stays;
 * 1 = off (the default, the unfiltered path).  Outside [0, 1] or NaN: failure.  Ignored when greedy != 0.
 * tokens_out int32 [B, n_steps] (column `step` written); x_next fp32 [2B, D]. */
int pg_cfg_sample_embed(pg_engine* e, const float* logits, int B, float cfg_weight,
                        float temperature, uint64_t seed, uint64_t philox_offset, int greedy, int top_k,
                        double top_p, const int32_t* edit_region, const int32_t* gt_labels, int step,
                        int n_steps, int32_t* tokens_out, float* x_next, void* stream);

/* replaces: vl_gpt.prepare_gen_img_embeds(ids)     modeling_vlm.py:270-271
 * ids int32 [n] -> fp32 [n, D] */
int pg_prepare_gen_img_embeds(pg_engine* e, const int32_t* ids, int n, float* out, void* stream);

/* replaces: System.sample_image (plangen_base.py:567-607), whole loop on the device:
 * prefill + n_steps x (gen_head, CFG, sample, embed, decode step) with no host sync.
 * x_prompt fp32 [R,P,D] (consumed).  tokens_out int32 [R/2, n_steps].  kv_start / edit_region / gt_labels are copied
 * into engine-owned buffers at entry (captured graphs are keyed on shapes and scalars, not on caller addresses).
 * top_k / top_p as for pg_cfg_sample_embed. */
int pg_sample_image(pg_engine* e, float* x_prompt, const int32_t* kv_start, int R, int P,
                    int n_steps, float cfg_weight, float temperature, uint64_t seed, int greedy, int top_k,
                    double top_p, const int32_t* edit_region, const int32_t* gt_labels,
                    int32_t* tokens_out, void* stream);

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

/* Host-only helper of the prefill (no device work, callable without a GPU): proposes, for every prompt row, the FIRST
 * row of the batch with the same left padding `start[r]` and the same 64-bit content hash (itself when there is none).
 * The prefill verifies every proposal word for word on the device before using it (t2i's shared negative prompt,
 * cfg/base.py:129; the `parallel_size` copies of plangen_base.py:547-549).  Returns the number of proposals. */
int pg_host_group_rows(const int32_t* start, const uint64_t* hash, int R, int32_t* source_row);

/* Plain GEMM exposed for unit tests:  C[m,n] = sum_k X[m,k] * W[n,k]
 * impl 0 = SIMT (fp32 or bf16 inputs), 1 = tcgen05 (bf16 inputs).  C fp32 [splits][M][N]. */
int pg_test_gemm(pg_engine* e, int impl, int is_bf16, const void* X, const void* W, int M, int N,
                 int K, int splits, float* C, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PLANGEN_B200_H */
