// Launcher declarations shared by the kernel translation units and sv_engine.cu.
// All tensors are bf16 unless noted; `st` is the stream every launch goes to.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sv_beam_core.h"
#include "sv_common.cuh"

namespace sv {

// Counts kernel launches issued through the launchers (sv_launch_count()).
extern thread_local int64_t* g_launch_counter;
inline void count_launch(int n = 1) { if (g_launch_counter) *g_launch_counter += n; }

// Device-resident generation state, read/written by kernels so a captured graph can be replayed.
struct GenState {
  int32_t cur_len;      // tokens in the KV cache == position of the token fed next
  int32_t step;         // generated tokens so far == next free column of out_ids
  int32_t done;         // all rows finished (or row-0 stop fired)
  int32_t row0_stop;    // scratch: row 0 matched the stop sequence this step
  int32_t unfinished[64];
};

struct GenParamsDev {
  int32_t max_new, do_sample, eos_id, pad_id, n_stop, stop_ids[8], stop_row0_only, out_stride;
  float temperature, top_p, rep_penalty;
  unsigned long long seed;
};

// ---- sv_kernels_basic.cu
void launch_layernorm(const bf16* x, const bf16* w, const bf16* b, bf16* y, int rows, int cols, float eps,
                      int64_t x_row_stride, cudaStream_t st);
void launch_convert_to_bf16(const void* src, int dtype, bf16* dst, int64_t n, cudaStream_t st);
void launch_pad_rows(const bf16* src, bf16* dst, int rows, int src_cols, int dst_cols, cudaStream_t st);
void launch_im2col(const bf16* pixels, bf16* patches, int batch, int image, int patch, int kpad, cudaStream_t st);
void launch_vit_assemble(const bf16* pe, const bf16* cls, const bf16* pos, bf16* x, int batch, int np, int width,
                         cudaStream_t st);   // cls == nullptr: no class token (SigLIP): x = pe + pos
void launch_vit_transpose_v(const bf16* qkv, bf16* vt, int batch, int seq, int heads, int seq_pad, cudaStream_t st);
void launch_slab_layernorm(const bf16* z, const bf16* w, const bf16* b, bf16* y, float* partial, int batch,
                           int64_t slab, float eps, cudaStream_t st);
void launch_batchnorm_tokens(const bf16* z, const bf16* w, const bf16* b, const bf16* rmean, const bf16* rvar, bf16* y,
                             int batch, int q, int h, float eps, cudaStream_t st);
void launch_embed_prefix(const bf16* visual, const int32_t* prompt_ids, const bf16* wte, const bf16* wpe, bf16* x,
                         int batch, int q, int p, int h, int vocab, cudaStream_t st);
// teacher-forcing chunk: x[b*seq + t] = wte[ids[b*ids_ld + t]] + wpe[pos0 + t] (wpe may be nullptr)
void launch_embed_chunk(const int32_t* ids, int ids_ld, const bf16* wte, const bf16* wpe, bf16* x, int batch, int seq, int pos0,
                        int h, int vocab, int n_positions, cudaStream_t st);
// per-row maps of one scoring chunk (rows b*seq + t, t0 + t = position in the call's T tokens), see sv_extend
void launch_score_maps(const int32_t* ids, int T, int batch, int seq, int t0, int keep, int vocab, bool want_logps,
                       int32_t* tgt, int32_t* lg_row, int32_t* lp_idx, cudaStream_t st);
// logps[b*lp_ld] = log_softmax(logits[b] / T)[ids[b*ids_ld]] over bf16 rows [batch][vocab] (one block per row)
void launch_row_logp(const bf16* logits, int vocab, int batch, const int32_t* ids, int ids_ld, float inv_temp, float* logps,
                     int lp_ld, cudaStream_t st);
// dst bf16 [batch][n] = src fp32 rows (row b at src + b * src_ld), values already bf16-exact
void launch_float_rows_to_bf16(const float* src, int64_t src_ld, bf16* dst, int batch, int n, cudaStream_t st);
void launch_embed_tokens(const int32_t* ids, const bf16* wte, const bf16* wpe, const GenState* state, bf16* x,
                         int batch, int h, int vocab, int n_positions, cudaStream_t st);
// cache positions pos0 .. pos0 + seq - 1 of every row
void launch_kv_scatter(const bf16* qkv, bf16* kcache, bf16* vtcache, int batch, int seq, int q_cols, int n_kv, int d,
                       int tcap, int pos0, cudaStream_t st);
void launch_kv_append(const bf16* qkv, bf16* kcache, bf16* vtcache, const GenState* state, int batch, int q_cols,
                      int n_kv, int d, int tcap, cudaStream_t st);
void launch_kv_gather(const bf16* ksrc, const bf16* vsrc, bf16* kdst, bf16* vdst, const int32_t* idx, int rows, int n_kv,
                      int tcap, int d, int len, cudaStream_t st);
void launch_gather_rows(const bf16* x, bf16* y, int batch, int seq, int row, int h, cudaStream_t st);
void launch_logits_to_float(const bf16* logits, float* out, int64_t n, cudaStream_t st);
void launch_select_greedy(const bf16* logits, int vocab, int batch, GenState* state, const GenParamsDev* params,
                          uint8_t* seen, int32_t* next_ids, int32_t* out_ids, cudaStream_t st);
void launch_select_sample(const bf16* logits, int vocab, int batch, GenState* state, const GenParamsDev* params,
                          uint8_t* seen, int32_t* next_ids, int32_t* out_ids, float* probs, cudaStream_t st);
void launch_gen_finalize(GenState* state, const GenParamsDev* params, int batch, int advance_len, cudaStream_t st);
void launch_advance_len(GenState* state, cudaStream_t st);
void launch_fill_i32(int32_t* p, int32_t v, int n, cudaStream_t st);

// ---- sv_gemm_rowgroup.cu : y[M,N] = epi(x[M,K] . w[N,K]^T) with mma.sync, weight streaming
void launch_linear_rowgroup(const bf16* x, const bf16* w, const bf16* bias, const bf16* res, bf16* y, int M, int N,
                            int K, int act, cudaStream_t st);

// ---- sv_gemm_tc05.cu : same contract on tcgen05 + TMA + TMEM (M >= 1, N % 8 == 0, K % 64 == 0)
bool tc05_supported(int M, int N, int K);
// returns cudaSuccess or the error of tensor-map creation / launch
cudaError_t launch_linear_tc05(const bf16* x, const bf16* w, const bf16* bias, const bf16* res, bf16* y, int M, int N,
                               int K, int act, cudaStream_t st);
// Scoring lm_head: logits = bf16(x[M,K] . w[N,K]^T) (any N >= 1, K % 64 == 0) reduced on the fly to log-probs of one target
// per row, logp = logits[tgt] / T - logsumexp(logits / T), without writing the logits (unless `logits` is given).
struct LogpsEpilogue {
  const int32_t* tgt;     // [M] target column of each row; < 0: no target
  const int32_t* lg_row;  // [M] output row of the fp32 logits (< 0: not stored); nullptr = identity
  float* logits;          // fp32 [.., N] bf16-rounded unscaled logits, or nullptr
  float2* part;           // [M][lm_head_logps_ntiles(N)] per-tile (max, sum exp(x - max)) of the scaled row
  float* tlogit;          // [M] scaled target logit
  float inv_temp;
};
int lm_head_logps_ntiles(int N);
// GEMM + partials, then (logps != nullptr) the merge: logps[lp_idx ? lp_idx[r] : r] = logp of row r (lp_idx[r] < 0: skipped;
// a row without target gets NaN)
cudaError_t launch_lm_head_logps(const bf16* x, const bf16* w, int M, int N, int K, const LogpsEpilogue& lp,
                                 const int32_t* lp_idx, float* logps, cudaStream_t st);

// ---- sv_attention.cu
void launch_attention_vit(const bf16* qkv, const bf16* vt, bf16* out, int batch, int seq, int heads, int seq_pad,
                          cudaStream_t st);
// causal attention of `seq` new tokens per row against the cache (which already holds them): token t of a row sits at
// cache position pos0 + t and attends to keys [0 | pos0 + t + 1 - window, pos0 + t]
void launch_attention_heads(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache, bf16* out,
                            int batch, int seq, int n_head, int n_kv, int d, int tcap, int window, int pos0, cudaStream_t st);
void launch_attention_decode(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache, bf16* out,
                             float* partial, const GenState* state, int batch, int n_head, int n_kv, int d, int tcap,
                             int nsplit, int window, cudaStream_t st);
// RoPE in place on the q and k parts of packed qkv rows [rows][qkv_cols] (StarCoder2, rotate_half convention);
// cos/sin tables are bf16 [max_pos][D/2]; position of row r = pos0 + (r % seq) or state->cur_len when state != nullptr.
void launch_rope(bf16* qkv, int rows, int seq, int qkv_cols, int n_rot_heads, int d, const bf16* cos_t, const bf16* sin_t,
                 const GenState* state, int max_pos, int pos0, cudaStream_t st);
void launch_rope_append(bf16* qkv, int batch, int qkv_cols, int n_head, int n_kv, int d, const bf16* cos_t,
                        const bf16* sin_t, bf16* kcache, bf16* vtcache, const GenState* state, int tcap, int max_pos,
                        bool pdl, cudaStream_t st);
void launch_rope_table(bf16* cos_t, bf16* sin_t, int max_pos, int d, float theta, cudaStream_t st);

// decode attention (PDL-ready): the ncta <= 8 CTAs of one image form a thread-block cluster
int attention_decode_cluster_ncta(int total_len);
cudaError_t attention_decode_cluster_init();
cudaError_t launch_attention_decode_cluster(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache,
                                            bf16* out, const GenState* state, int batch, int n_head, int n_kv, int d,
                                            int tcap, int ncta, int window, bool pdl, cudaStream_t st);

// ---- sv_decode_fused.cu : token selection fused with the next step's embedding, PDL-ready
void launch_select_fused(const bf16* logits, int vocab, int batch, const float* amax_val, const int* amax_idx,
                         int ntiles, GenState* state, const GenParamsDev* params, uint8_t* seen, int32_t* next_ids,
                         int32_t* out_ids, int advance_len, const bf16* wte, const bf16* wpe, bf16* x, int h,
                         int n_positions, bool pdl, cudaStream_t st);

// ---- sv_decode_mega.cu : per-phase weight-ring decode GEMV; layer descriptor shared with sv_decode_flow.cu
struct MegaLayer {
  const bf16 *ln1_w, *ln1_b, *attn_w, *attn_b, *proj_w, *proj_b, *ln2_w, *ln2_b, *fc_w, *fc_b, *fc2_w, *fc2_b;
  bf16 *kc, *vc;
  const bf16 *attn_t, *proj_t, *fc_t, *fc2_t;   // slab-tiled copies for the dataflow decode kernel (sv_decode_flow.cu flow_repack_kernel)
};
// one-phase weight-ring GEMV (same device code as the persistent kernel's GEMV phases)
struct RingGemvLaunch {
  const bf16 *X, *W, *bias, *res, *ln_w, *ln_b;
  const uint8_t* Wt;              // slab-tiled copy of W (flow_repack_kernel) or nullptr: then W's rows are copied one by one
  bf16* Y;
  int B, N, K, act, epi;          // epi: 0 plain, 1 QKV (+KV append), 2 lm_head (+argmax partials)
  float ln_eps;
  int n_head, n_kv, tcap;
  const GenState* state;
  bf16 *kcache, *vtcache;
  float* amax_val;
  int* amax_idx;
  bool pdl;
};
cudaError_t gemv_ring_init();
bool gemv_ring_supported(int K, bool has_ln);
int gemv_ring_ntiles(int N);
int gemv_ring_ncta();
void launch_gemv_ring(const RingGemvLaunch& g, cudaStream_t st);
// ---- sv_decode_flow.cu : dataflow persistent decode kernel (flagged activation words through L2, no grid barriers)
struct FlowLaunch {
  const MegaLayer* layers_dev;
  int n_layer, B, H, I, n_head, n_kv, qkv_cols, vocab, tcap, n_positions;
  float ln_eps;
  const bf16 *wte, *wpe, *lnf_w, *lnf_b, *lm_head, *lm_head_t;
  bf16 *x_plain, *logits;
  uint32_t *xa, *xb, *qkv, *att, *hb;          // flagged bf16 words
  unsigned long long *part, *amax;             // flagged fp32 words / argmax partials
  GenState* state;
  const GenParamsDev* params;
  uint8_t* seen;
  int32_t *next_ids, *out_ids;
  int nsteps;          // tokens in this launch
  int step0;           // phase-tag epoch of the first step (monotonic since the exchange buffers were cleared)
  int cur_len0;        // tokens in the KV cache when the launch starts
  int first_plain;     // 1: the first step's input is x_plain (plain bf16) and gets converted to flagged words
  int do_select;       // 1: greedy select + embed after every step; 0: stop after the logits (teacher forcing)
  int l2_ahead;        // weight slabs per CTA prefetched into L2 ahead of the shared-memory ring (0 = off)
  long long* dbg;
  bool realloc;
};
cudaError_t decode_flow_init();
int decode_flow_ncta();
int decode_flow_max_splits();
int decode_flow_partial_floats();
const char* decode_flow_status();
bool decode_flow_supported(int H, int I, int head_dim, int max_batch, int window, bool rope);
bool decode_flow_realloc_supported();
cudaError_t launch_decode_flow(const FlowLaunch& m, cudaStream_t st);
size_t flow_tiled_bytes(int N, int K, int ncta);      // bytes of the slab-tiled copy of a [N][K] decode weight matrix
void launch_flow_repack(const bf16* W, const bf16* bias, void* T, int N, int K, int ncta, cudaStream_t st);

// ---- sv_beam.cu : beam search / beam-sample bookkeeping inside the decode graph (state structs: sv_beam_core.h)
size_t beam_candidates_smem(int vocab);
cudaError_t beam_init(int vocab);          // cudaErrorInvalidValue: a logits row does not fit the SM's shared memory
void launch_beam_candidates(const bf16* logits, int vocab, int rows, const svbeam::Params* p, const svbeam::State* st,
                            const int32_t* run_seq, float* cand_key, float* cand_val, int32_t* cand_tok, cudaStream_t st_);
void launch_beam_step(const svbeam::Params* p, svbeam::State* st, svbeam::Plan* plan, const float* cand_key,
                      const float* cand_val, const int32_t* cand_tok, int32_t* run_seq, int32_t* fin_seq, GenState* gs,
                      int advance, const bf16* wte, const bf16* wpe, bf16* x, int h, int n_positions,
                      int32_t* next_ids, cudaStream_t st_);
void launch_beam_kv_copy(bf16* kc, bf16* vc, bf16* kc2, bf16* vc2, int64_t layer_stride, int n_layer, int rows, int n_kv,
                         int tcap, int D, const svbeam::Plan* plan, cudaStream_t st_);

}  // namespace sv
