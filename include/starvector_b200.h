/*
 * starvector_b200 — C-ABI of the B200-native im2svg generation engine.
 *
 * The reference (joanrod/star-vector) has no FFI: its boundary for this path is the Python
 * method surface `StarVectorForCausalLM.generate_im2svg` / `.model.svg_transformer
 * .transformer.generate` (reference: starvector/model/starvector_arch.py:186-187,
 * starvector/model/models/starvector_base.py:203-259).  The Python facade in
 * `starvector_b200/modeling.py` keeps that surface and binds THESE entry points with ctypes
 * (see INTEGRATION.md).  Each entry point below names the reference code it replaces.
 *
 * Conventions: plain pointers and sizes only (no torch types); every pointer is a DEVICE
 * pointer unless the name ends in `_host` or the comment says "host or device"; `stream` is
 * a `cudaStream_t` passed as `void*` (NULL = legacy default stream); return 0 on success,
 * <0 on error with the message available from `sv_last_error`; no exceptions cross the
 * ABI; an engine is not re-entrant (the caller serialises; the Python shim holds a lock).
 * There is no CPU fallback: every call fails with SV_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef STARVECTOR_B200_H
#define STARVECTOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SV_ABI_VERSION 6
#if defined(__GNUC__)
#define SV_API __attribute__((visibility("default")))
#else
#define SV_API
#endif

enum {
  SV_OK = 0,
  SV_ERR_INVALID = -1,     /* bad argument / shape / name */
  SV_ERR_CUDA = -2,        /* CUDA runtime or driver error (message has the cudaError string) */
  SV_ERR_UNSUPPORTED = -3, /* valid request this build does not implement */
  SV_ERR_STATE = -4        /* call order violated (weights missing, no prefill before generate, ...) */
};

enum { SV_DTYPE_BF16 = 0, SV_DTYPE_F32 = 1, SV_DTYPE_F16 = 2 };

/* activation selectors of the fused linear epilogue */
enum {
  SV_ACT_NONE = 0,
  SV_ACT_QUICKGELU = 1, /* x*sigmoid(1.702x)  — clip_model.py:126-128 */
  SV_ACT_GELU_TANH = 2, /* gelu_pytorch_tanh  — GPTBigCodeMLP */
  SV_ACT_SILU = 3       /* x*sigmoid(x)       — adapters/adapter.py:5-10 */
};

/* implementation selector for sv_op_linear (tests cross-check the two kernels) */
enum { SV_LINEAR_AUTO = 0, SV_LINEAR_ROWGROUP = 1, SV_LINEAR_TCGEN05 = 2 };

typedef struct sv_engine sv_engine;

/* Dimensions of one StarVector model (SURVEY.md §8; reference: image_encoder.py:50-61,
 * starvector_base.py:87-104, adapters/adapter.py:13-31, bigcode/starcoderbase-1b config). */
typedef struct sv_model_desc {
  int32_t variant;      /* 0 = v1 (1B): CLIP ViT-L/14 + Adapter + GPTBigCode (MQA, learned positions).
                           1 = v2 (8B): SigLIP tower (no class token, LN eps 1e-6, gelu_tanh, patch bias, post_layernorm)
                               + StarCoder2 (GQA, RoPE, sliding-window attention, biased linears) — models/starvector_v2.py */
  int32_t image_size;   /* 224 */
  int32_t patch_size;   /* 14  */
  int32_t vit_width;    /* 1024 */
  int32_t vit_layers;   /* 23 (penultimate-layer CLIP ViT-L/14) */
  int32_t vit_heads;    /* 16 (head dim must be 64) */
  int32_t vit_mlp;      /* 4096 */
  int32_t adapter_norm; /* 0 = LayerNorm([Q,H]); 1 = BatchNorm1d(Q) in eval mode */
  int32_t hidden;       /* 2048 */
  int32_t n_layer;      /* 24 */
  int32_t n_head;       /* 16 */
  int32_t n_kv_head;    /* 1 (multi-query) */
  int32_t head_dim;     /* 128 */
  int32_t n_inner;      /* 8192 */
  int32_t n_positions;  /* 8192 learned absolute positions */
  int32_t vocab;        /* 49156 = 49152 + [PAD] + 3 added tokens (llm/starcoder.py:43-53) */
  float ln_eps;         /* 1e-5 */
  int32_t max_batch;    /* images per call on this GPU */
  int32_t max_len;      /* KV-cache capacity in tokens (prefix + generated) */
  /* v2 only (ignored for variant 0) */
  float rope_theta;       /* StarCoder2 rope_theta (hub config of bigcode/starcoder2-7b; default 10000 in transformers) */
  int32_t sliding_window; /* 4096 for starcoder2-7b; 0 = full causal attention */
  float vit_ln_eps;       /* 1e-6 for SigLIP (1e-5 is used for variant 0) */
} sv_model_desc;

/* Decoding parameters = the kwargs the reference forwards to HF generate()
 * (starvector_base.py:223-241, :289-295) after HF's own length fix-up (SURVEY.md App. B). */
typedef struct sv_gen_params {
  int32_t max_new_tokens;    /* = max_length - (Q + P)  (generation/utils.py:1629-1638) */
  int32_t do_sample;         /* use_nucleus_sampling; 0 = greedy argmax (lowest index wins ties) */
  float temperature;
  float top_p;
  float repetition_penalty;  /* applies to generated ids only (App. B.4) */
  int32_t eos_token_id;      /* -1 = none (throughput configs) */
  int32_t pad_token_id;
  int32_t n_stop_ids;        /* 0..8: ids of '</svg>' (StoppingCriteriaSub, starvector_base.py:9-20) */
  int32_t stop_ids[8];
  int32_t stop_row0_only;    /* 1 = reference behaviour D6 (row 0 matching ends the WHOLE batch);
                                0 = per-row: a matching row is finished/padded, batch ends when all rows are */
  uint64_t seed;             /* Philox seed for sampling */
  int32_t poll_interval;     /* host polls the device stop flag every this many steps (0 -> 16) */
} sv_gen_params;

/* Beam search / beam-sample parameters = what HF `generate(num_beams > 1)` receives from the reference
 * (starvector_base.py:231-241: num_beams=2, do_sample, top_p, temperature, repetition_penalty, length_penalty;
 * :289-295: early_stopping=True, pad_token_id; starvector_v2.py:53-57: nothing -> HF defaults). */
typedef struct sv_beam_params {
  int32_t num_beams;          /* >= 2; batch * num_beams <= 8 cache rows */
  int32_t max_new_tokens;
  int32_t do_sample;          /* 1 = beam-sample (candidates drawn without replacement, device Philox stream) */
  int32_t early_stopping;     /* 0 = False (HF default), 1 = True (v1), 2 = "never" */
  float temperature;
  float top_p;
  float repetition_penalty;   /* on the log-probs, over each running beam's own generated ids */
  float length_penalty;
  int32_t eos_token_id;       /* -1 = none */
  int32_t pad_token_id;       /* fill of the returned rectangle (HF: pad if given, else eos) */
  int32_t n_stop_ids;         /* 0..8: StoppingCriteriaSub, candidate 0 of image 0 matching ends every beam */
  int32_t stop_ids[8];
  int32_t poll_interval;      /* host polls the device done flag every this many steps (0 -> 16) */
  uint64_t seed;
} sv_beam_params;

/* ---- lifecycle ------------------------------------------------------------------------ */
SV_API int sv_abi_version(void);
/* Replaces module construction (starvector_base.py:22-48): allocates packed weights, KV cache
 * and workspaces on `device`. */
SV_API int sv_engine_create(const sv_model_desc* desc, int device, sv_engine** out);
SV_API void sv_engine_destroy(sv_engine* e);
/* Message for the last failing call on `e` (or the last failing create when e == NULL). */
SV_API const char* sv_last_error(const sv_engine* e);
/* Replaces load_state_dict/from_pretrained: copy one tensor by its reference state-dict name
 * (SURVEY.md §8b "Ownership"), e.g. "model.image_encoder.visual_encoder.conv1.weight".
 * `data` may be a host or device pointer (UVA); borrowed only during the call. */
SV_API int sv_engine_load_weight(sv_engine* e, const char* hf_name, const void* data, const int64_t* shape,
                          int32_t ndim, int32_t dtype);
/* Number of tensors still missing (0 = ready); names (newline separated) via sv_last_error. */
SV_API int sv_engine_missing_weights(sv_engine* e);

/* ---- the hot path --------------------------------------------------------------------- */
/* ImageEncoder.forward + Adapter.forward (image_encoder.py:91-94, adapter.py:33-39,
 * starvector_base.py:206-209).  pixels: bf16 [B,3,S,S].  Result stays resident as the visual
 * prefix; if out_embeds != NULL it is also copied there (bf16 [B,Q,H]).  If vit_out != NULL the
 * pre-adapter `ln_vision` output (bf16 [B,Q,W]) is copied there (parity tests). */
SV_API int sv_encode_images(sv_engine* e, const void* pixels, int32_t batch, void* out_embeds, void* vit_out,
                     void* stream);
/* Prompt embedding + concat (starvector_base.py:213-219) and the decoder prefill over the
 * Q+P prefix (the first forward inside generate(), SURVEY.md §3.1).  prompt_ids int32 [B,P].
 * last_logits (optional) float [B,V]: logits of the last prefix position. */
SV_API int sv_prefill(sv_engine* e, const int32_t* prompt_ids, int32_t batch, int32_t prompt_len,
               float* last_logits, void* stream);
/* The same prefill from caller-provided inputs_embeds bf16 [B,T,H] (the `.generate(inputs_embeds=...)`
 * form of starvector_base.py:255; wpe is added inside, as GPTBigCodeModel.forward does). */
SV_API int sv_prefill_embeds(sv_engine* e, const void* inputs_embeds, int32_t batch, int32_t seq_len,
                             float* last_logits, void* stream);
/* One teacher-forced decode step: feed ids int32 [B], append to the KV cache, return fp32 logits
 * [B,V] (optional).  The parity-test hook; also the body the generate loop replays. */
SV_API int sv_decode_step(sv_engine* e, const int32_t* ids, float* logits, void* stream);
/* Teacher forcing over a chunk (the scoring half of RL fine-tuning, reference StarVectorForCausalLM.forward,
 * starvector_arch.py:161-184): append T tokens per row to the cached sequence of every row.
 * Allowed after sv_prefill / sv_prefill_embeds / sv_expand_batch / sv_decode_step / sv_extend (not after sv_generate or
 * sv_beam_search: SV_ERR_STATE).  ids int32 [B,T] (device), B = current batch, 1 <= T <= max_len - cur_len - 1.
 * KV rows [cur_len, cur_len+T) are written and cur_len advances by T; the engine's last-position logits become those of
 * the chunk's last token, so sv_decode_step / sv_extend may follow.
 * logits (optional) float [B, keep, V]: logits of the last `keep` new positions (bf16-rounded, as HF's lm_head returns).
 * logps  (optional) float [B, T]: logps[b][t] = log_softmax(L[b][t-1] / temperature)[ids[b][t]], in fp32, where L[b][t-1] is
 * the bf16 logits row that predicts token t (for t = 0 the logits the engine held before the call).
 * Runs in chunks of 4096 / B tokens (one tcgen05 GEMM of ~4096 rows per linear layer); the lm_head never writes the
 * [B,T,V] logits for the log-probs.  Synchronises `stream`. */
SV_API int sv_extend(sv_engine* e, const int32_t* ids, int32_t T, float* logits, int32_t keep, float* logps,
                     float temperature, void* stream);
/* Beam search support (SURVEY.md §8f-1): permute the image rows of the KV cache, row r <- row src_rows[r]
 * (int32 [B] on the device) for the tokens cached so far = HF `_reorder_cache` (vendored modeling_gpt_bigcode.py:1282-1291). */
SV_API int sv_reorder_cache(sv_engine* e, const int32_t* src_rows, void* stream);
/* Prefix-KV sharing (SURVEY.md §8f-4; reference starvector_base.py:261-286 `num_return_sequences`, starvector_arch.py:161-184
 * `vision_embeds.repeat(num_generations, 1, 1)`): directly after sv_prefill / sv_prefill_embeds of b rows, make the engine hold
 * new_batch rows where row r is a copy of prefilled row src_rows_host[r] (HOST int32 [new_batch]): KV cache, last-position
 * logits and generation state are replicated, so the visual prefix is encoded and prefilled once per image, not once per
 * completion.  new_batch <= max_batch. */
SV_API int sv_expand_batch(sv_engine* e, const int32_t* src_rows_host, int32_t new_batch, void* stream);
/* `GenerationMixin._beam_search` after a prefill of batch * num_beams rows (every image repeated num_beams times,
 * adjacent: HF `_expand_inputs_for_generation`): the whole search runs on the device -- per decode step the candidate
 * selection, the beam bookkeeping and the cache permutation (as suffix copies between rows that diverged) follow the
 * lm_head inside the replayed CUDA graph; the host only polls a done flag.  out_ids int32 [batch, max_new_tokens] = the best
 * hypothesis per image (new tokens only, padded with pad_token_id), out_len int32 [batch] = rectangular length (HF's
 * max_generated).  SV_ERR_UNSUPPORTED when a logits row does not fit the SM's shared memory (vocab > ~55k): use the
 * host-stepped loop (sv_decode_step + sv_reorder_cache, starvector_b200/beam_search.py).  Synchronises `stream`. */
SV_API int sv_beam_search(sv_engine* e, const sv_beam_params* p, int32_t batch, int32_t* out_ids, int32_t* out_len,
                          void* stream);
/* Host replays of the device stages of sv_beam_search (no GPU needed; the same bookkeeping code, sv_beam_core.h):
 * parameter validation; size / initialisation / read-out of the opaque state blob; one logits row (fp32 values of the bf16
 * logits) -> its 2 * num_beams best continuations {ordering key, log-prob + running score, token}; one bookkeeping step
 * over row candidates [batch * num_beams][2 * num_beams] with the double-buffered sequence arrays
 * [2][batch * num_beams][seq_stride] -> next tokens, parent rows (= HF beam_idx), returns 1 while the search continues.
 * tests/test_beam_core.py runs whole searches with them against HF generate(num_beams > 1). */
SV_API int sv_beam_params_check(const sv_beam_params* p, int32_t batch);
SV_API int sv_beam_state_bytes(void);
SV_API int sv_beam_state_init_host(const sv_beam_params* p, int32_t batch, int32_t first_cache_pos, void* state);
SV_API int sv_beam_state_read_host(const void* state, int32_t* parity, int32_t* cur_len, int32_t* fin_len8,
                                   float* beam_scores8);
SV_API int sv_beam_row_candidates_host(const sv_beam_params* p, const float* logits, int32_t vocab, const int32_t* seq,
                                       int32_t seq_len, float running_score, int32_t step, int32_t row, float* cand_key,
                                       float* cand_val, int32_t* cand_tok);
SV_API int sv_beam_step_host(const sv_beam_params* p, int32_t batch, int32_t vocab, int32_t seq_stride, void* state,
                             const float* cand_key, const float* cand_val, const int32_t* cand_tok, int32_t* run_seq,
                             int32_t* fin_seq, int32_t cache_hi, int32_t* next_tokens, int32_t* src_rows, int32_t* plan_out);
/* GenerationMixin.generate() after the prefill (greedy / sampling loop, App. B): runs up to
 * max_new_tokens steps as a replayed CUDA graph.  out_ids int32 [B,max_new_tokens] (new tokens
 * only, padded with pad_token_id), out_len int32 [B] = rectangular generated length.
 * Synchronises `stream` before returning. */
SV_API int sv_generate(sv_engine* e, const sv_gen_params* p, int32_t* out_ids, int32_t* out_len, void* stream);
/* sv_generate with token streaming (SURVEY.md §8f-4: serve/model_worker.py:161-181 hands a `streamer` to generate(),
 * which the reference's kwarg whitelist drops, starvector_base.py:223-241).  Every `poll_interval` steps, and once at the
 * end, `on_tokens(user, ids_host, batch, first_step, n_steps)` is called on the calling thread with the new tokens of
 * every row, ids_host int32 [batch][n_steps] (valid during the call); the concatenation over calls is exactly the
 * rectangle sv_generate returns.  A non-zero return cancels the generation after the current poll. */
typedef int (*sv_token_callback)(void* user, const int32_t* ids_host, int32_t batch, int32_t first_step, int32_t n_steps);
SV_API int sv_generate_stream(sv_engine* e, const sv_gen_params* p, int32_t* out_ids, int32_t* out_len,
                              sv_token_callback on_tokens, void* user, void* stream);
/* Whole path with HOST buffers (copies inside): pixels_host bf16 [B,3,S,S], prompt_ids_host
 * int32 [B,P] -> out_ids_host int32 [B,max_new_tokens], out_len_host int32 [B]. */
SV_API int sv_generate_im2svg_host(sv_engine* e, const void* pixels_host, int32_t batch,
                            const int32_t* prompt_ids_host, int32_t prompt_len, const sv_gen_params* p,
                            int32_t* out_ids_host, int32_t* out_len_host, void* stream);

/* ---- introspection for bench/profiles ------------------------------------------------- */
/* Kernel launches issued by this engine since creation (graph replays count their nodes). */
SV_API int64_t sv_launch_count(const sv_engine* e);
/* Human-readable configuration of the engine (decode mode, PDL, kernel selection) for logs/bench JSON. */
SV_API const char* sv_engine_describe(sv_engine* e);
/* Debug (SV_MEGA_DEBUG=1): timeline records of CTA 0 for the first token of the last persistent-decode launch,
 * `id << 48 | SM clock` (ids: sv_decode_flow.cu); entries [0,4096) consumer thread 0, [4096,8192) producer warp;
 * unused entries are 0; n <= 8192. */
SV_API int sv_debug_read_timeline(sv_engine* e, long long* out_host, int32_t n);
/* Device time (ms) of the last sv_generate decode loop and its step count, from CUDA events
 * recorded on the launching stream. */
SV_API int sv_last_decode_timing(const sv_engine* e, float* ms, int32_t* steps);

/* ---- single-kernel entry points (unit parity tests; all bf16 unless noted) -------------- */
SV_API int sv_op_layernorm(const void* x, const void* w, const void* b, void* y, int32_t rows, int32_t cols,
                    float eps, void* stream);
/* y[M,N] = act(x[M,K] . w[N,K]^T + bias[N]) (+ residual[M,N]); rounding points follow the
 * reference's bf16 module boundaries (DESIGN.md §numerics). */
SV_API int sv_op_linear(int32_t impl, const void* x, const void* w, const void* bias, const void* residual, void* y,
                 int32_t M, int32_t N, int32_t K, int32_t act, void* stream);
/* ViT self-attention over packed qkv [B*L, 3*heads*64] -> out [B*L, heads*64]. */
SV_API int sv_op_attention_vit(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t heads, void* stream);
/* Causal multi-query attention over packed qkv [B*T, heads*D + 2*D] (D=128) -> out [B*T, heads*D]. */
SV_API int sv_op_attention_mqa(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t heads, void* stream);
/* Causal grouped-query attention of the decoder prefill over packed qkv [B*T, (n_head + 2*n_kv)*D] (D=128)
 * -> out [B*T, n_head*D]; window > 0 restricts token t to keys (t - window, t] (StarCoder2 sliding window). */
SV_API int sv_op_attention_prefill(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t n_head, int32_t n_kv,
                                   int32_t window, void* stream);

/* The decode-step kernels one at a time.  Each call validates its arguments before any launch (SV_ERR_INVALID),
 * allocates its own scratch (generation state, partial buffers, tiled weight copy) and synchronises `stream`. */
enum { SV_ATTN_DECODE_CLUSTER = 0, SV_ATTN_DECODE_SPLIT = 1 };
/* One decode token per row: q [B, n_head*D] against K [B][n_kv][tcap][D] and V^T [B][n_kv][D][tcap] -> out [B, n_head*D].
 * Keys [max(0, nkeys - window), nkeys) take part (window 0 = all); 1 <= nkeys <= tcap, tcap % 32 == 0, B <= 8, group <= 16.
 * nparts forces the cluster size (1..8) or the split count (1..128); 0 = what the engine picks for nkeys. */
SV_API int sv_op_attention_decode(int32_t impl, const void* q, const void* kcache, const void* vtcache, void* out,
                                  int32_t batch, int32_t n_head, int32_t n_kv, int32_t tcap, int32_t nkeys, int32_t window,
                                  int32_t nparts, void* stream);
enum { SV_GEMV_EPI_PLAIN = 0, SV_GEMV_EPI_QKV = 1, SV_GEMV_EPI_LMHEAD = 2 };
/* One weight-ring decode GEMV: y[B,N] = epilogue(LayerNorm?(x)[B,K] . w[N,K]^T), B <= 8, K % 32 == 0; LayerNorm when
 * ln_w / ln_b are given; bias, residual (may alias y) optional.  Epilogues: SV_GEMV_EPI_QKV also appends the K row and the
 * V^T column at `pos` of the caches (N == (n_head + 2*n_kv)*128, pos < tcap); SV_GEMV_EPI_LMHEAD also writes per-tile
 * argmax partials amax_val float / amax_idx int32 [tile][8] (capacity in tiles).  tiled = 1 streams a slab-tiled copy of
 * w made inside the call.  *ntiles_out (host, optional) = the number of partial tiles. */
SV_API int sv_op_gemv_ring(const void* x, const void* w, const void* bias, const void* residual, const void* ln_w,
                           const void* ln_b, void* y, int32_t batch, int32_t N, int32_t K, int32_t act, float ln_eps,
                           int32_t epi, int32_t tiled, void* kcache, void* vtcache, int32_t n_head, int32_t n_kv,
                           int32_t tcap, int32_t pos, float* amax_val, int32_t* amax_idx, int32_t amax_capacity,
                           int32_t* ntiles_out, void* stream);
/* The scoring lm_head (the hot kernel of sv_extend) on its own: x bf16 [M,K] (already final-LayerNormed), w bf16 [N,K],
 * ids int32 [M] -> logps float [M] = log_softmax(bf16(x.w^T) / temperature)[ids] (NaN where an id is outside [0,N));
 * logits (optional) float [M,N] = the bf16-rounded products.  Any N >= 1 (N % 8 != 0 included), K % 64 == 0. */
SV_API int sv_op_lm_head_logps(const void* x, const void* w, const int32_t* ids, float* logps, float* logits, int32_t M,
                               int32_t N, int32_t K, float temperature, void* stream);
enum { SV_SELECT_GREEDY = 0, SV_SELECT_FUSED = 1, SV_SELECT_FUSED_PARTIALS = 2, SV_SELECT_SAMPLE = 3 };
/* Token selection of one step from bf16 logits [B,V] and a seen bitmap uint8 [B,V] (host or device; not modified) at
 * generation step `step` with `cur_len` tokens in the cache -> tokens int32 [B] (host or device).  The fused kernels also
 * write x_out [B,h] = wte[token] + wpe[min(cur_len + 1, n_positions - 1)] (wpe may be NULL); SV_SELECT_FUSED_PARTIALS
 * reduces lm_head argmax partials [ntiles][8] instead of the logits. */
SV_API int sv_op_select(int32_t mode, const void* logits, const uint8_t* seen, const sv_gen_params* p, int32_t batch,
                        int32_t vocab, int32_t step, int32_t cur_len, const float* amax_val, const int32_t* amax_idx,
                        int32_t ntiles, const void* wte, const void* wpe, int32_t h, int32_t n_positions, void* x_out,
                        int32_t* tokens, void* stream);

/* ---- image preprocessing (SURVEY.md §8f-2) ------------------------------------------------ */
/* Replaces `ImageTrainProcessor.__call__` (reference starvector/data/util.py:40-66: RGBA pasted on white, pad to
 * square with 255, `transforms.Resize(size, BICUBIC)` on the PIL image, ToTensor, Normalize) and
 * `SimpleStarVectorProcessor.transform` (starvector_arch.py:39-45: the same with `convert("RGB")` for RGBA),
 * bit for bit with Pillow's 8-bit resample.  On-wire input = what PIL holds: uint8 HWC host buffers. */
enum { SV_ALPHA_WHITE = 0 /* data/util.py:63-66 */, SV_ALPHA_DROP = 1 /* starvector_arch.py:40 */ };

typedef struct sv_preproc sv_preproc;

typedef struct sv_preproc_desc {
  int32_t out_size;    /* S: output is [n,3,S,S] (224 for CLIP ViT-L/14, data/util.py:41) */
  int32_t alpha_mode;  /* SV_ALPHA_WHITE | SV_ALPHA_DROP: what happens to a 4th channel */
  int32_t pad_square;  /* 1: pad the shorter side with 255 to a centred square first (data/util.py:55-61); 0: resize (w,h)->(S,S) */
  int32_t out_dtype;   /* SV_DTYPE_BF16 (what sv_encode_images takes) | SV_DTYPE_F32 (the reference's tensor, for parity) */
  float mean[3];       /* Normalize(mean, std), data/util.py:33-38 */
  float std[3];
} sv_preproc_desc;

typedef struct sv_image_u8 {
  const uint8_t* data; /* HOST pointer, uint8 [height][width][channels]; pinned memory makes the upload asynchronous */
  int32_t width, height;
  int32_t channels;    /* 3 (RGB) or 4 (RGBA) */
  int32_t row_stride;  /* bytes between rows; 0 = width*channels */
} sv_image_u8;

SV_API int sv_preproc_create(const sv_preproc_desc* desc, int device, sv_preproc** out);
SV_API void sv_preproc_destroy(sv_preproc* p);
/* Message for the last failing call on `p` (or the last failing create when p == NULL). */
SV_API const char* sv_preproc_last_error(const sv_preproc* p);
/* `[processor(img) for img in images]` + stack: uploads the n images (ragged sizes), runs the horizontal and the
 * vertical resample pass, writes DEVICE out_pixels [n,3,S,S] (out_dtype).  Asynchronous on `stream`. */
SV_API int sv_preproc_run_host(sv_preproc* p, const sv_image_u8* images_host, int32_t n, void* out_pixels, void* stream);
/* Kernels launched by `p` so far. */
SV_API long long sv_preproc_launch_count(const sv_preproc* p);
/* Host-only pieces of the above, exported so that they can be checked against Pillow / torch without a GPU:
 * the fixed-point resample taps of one axis (Pillow Resample.c precompute_coeffs + normalize_coeffs_8bpc; call with
 * bounds == taps == NULL to query ksize; bounds int32 [out_size][2] = first tap, tap count; taps int32
 * [out_size][ksize]) and the 3x256 ToTensor+Normalize table (float [3][256]). */
SV_API int sv_resample_coeffs_host(int32_t in_size, int32_t out_size, int32_t* ksize, int32_t* bounds, int32_t* taps,
                                   int32_t taps_capacity);
SV_API int sv_preproc_lut_host(const sv_preproc_desc* desc, float* lut768);
/* The batch plan sv_preproc_run_host uploads: per-image metadata (padding, arena offsets) followed by the coefficient
 * arena.  sizes[5] = {blob bytes, metadata bytes, input-arena bytes, intermediate pixels, max input rows}; blob may be
 * NULL to query sizes.  Test hook: tests/test_preprocess_emul.py replays the kernels' index arithmetic from it. */
SV_API int sv_preproc_plan_host(const sv_preproc_desc* desc, const sv_image_u8* images_host, int32_t n, void* blob,
                                int64_t blob_capacity, int64_t sizes[5]);

#ifdef __cplusplus
}
#endif
#endif /* STARVECTOR_B200_H */
