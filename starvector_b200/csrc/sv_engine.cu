// C-ABI of the im2svg engine (include/starvector_b200.h): engine state, weight registry, the
// encode -> prefill -> decode orchestration and the CUDA-graph generation loop.
//
// Reference path being replaced: StarVectorBase.generate_im2svg
// (starvector/model/models/starvector_base.py:203-259) = ImageEncoder (image_encoder.py:91-94,
// clip_model.py:181-191) -> Adapter (adapters/adapter.py:33-39) -> prompt concat -> HF
// GenerationMixin.generate over GPTBigCodeForCausalLM (SURVEY.md §3.1, App. A/B).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/starvector_b200.h"
#include "sv_kernels.h"

using namespace sv;

namespace {

constexpr int kMaxPrompt = 64;
constexpr int kStreamChunk = 1024;   // tokens per row handed to a streaming callback at once
constexpr int kMaxSplit = 128;
constexpr int kScoreRows = 4096;     // GEMM rows per sv_extend chunk (B rows x 4096 / B tokens): ~32 x 385 lm_head tiles fill 148 SMs

std::string g_create_error;

struct Weight {
  bf16* p = nullptr;
  std::vector<int64_t> shape;      // shape expected from the caller (reference layout)
  int64_t numel = 0;
  bool loaded = false;
  bool optional = false;
};

struct VitLayer { bf16 *ln1_w, *ln1_b, *qkv_w, *qkv_b, *out_w, *out_b, *ln2_w, *ln2_b, *fc_w, *fc_b, *proj_w, *proj_b; };
struct DecLayer { bf16 *ln1_w, *ln1_b, *attn_w, *attn_b, *proj_w, *proj_b, *ln2_w, *ln2_b, *fc_w, *fc_b, *fc2_w, *fc2_b; };

struct GraphEntry { cudaGraphExec_t exec = nullptr; int kernels = 0; };

}  // namespace

struct sv_engine {
  sv_model_desc d{};
  int device = 0;
  std::string err, describe;
  int64_t launches = 0;
  int linear_impl = SV_LINEAR_AUTO;

  int Q = 0, NP = 0, Kp = 0, Lpad = 0, qkv_cols = 0, tcap = 0;
  bool v2 = false;                 // SigLIP + StarCoder2 (StarVector-8B family)
  float vit_eps = 1e-5f;
  int vit_act = SV_ACT_QUICKGELU, window = 0;
  bf16 *conv_b = nullptr, *rope_cos = nullptr, *rope_sin = nullptr;
  std::map<std::string, Weight> w;
  std::vector<void*> allocs;

  // resolved weights
  bf16 *conv_w = nullptr, *conv_raw = nullptr, *cls = nullptr, *pos = nullptr, *lnpre_w = nullptr, *lnpre_b = nullptr;
  bf16 *lnv_w = nullptr, *lnv_b = nullptr;
  std::vector<VitLayer> vit;
  bf16 *afc_w = nullptr, *afc_b = nullptr, *aproj_w = nullptr, *aproj_b = nullptr, *anorm_w = nullptr, *anorm_b = nullptr,
       *anorm_rm = nullptr, *anorm_rv = nullptr;
  bf16 *wte = nullptr, *wpe = nullptr, *lnf_w = nullptr, *lnf_b = nullptr, *lm_head = nullptr;
  std::vector<DecLayer> dec;

  // activations / workspaces
  bf16 *v_patches, *v_pe, *v_x, *v_ln, *v_qkv, *v_vt, *v_attn, *v_h, *v_out, *a_h, *a_z, *visual;
  float* slab_partial;
  bf16 *p_x, *p_ln, *p_qkv, *p_attn, *p_h;
  bf16 *d_x, *d_ln, *d_qkv, *d_attn, *d_h, *d_last, *logits;
  float *logits_f32, *attn_partial, *amax_val;
  int* amax_idx;
  bool fused_decode = true, use_pdl = true;
  MegaLayer* mega_layers = nullptr;
  long long* mega_dbg = nullptr;
  bool mega_debug = false;
  // dataflow persistent decode kernel (sv_decode_flow.cu): flagged exchange buffers in one allocation
  bool use_flow = false, flow_realloc = false;
  bool use_tiles = false;           // slab-tiled weight copies exist (the dataflow kernel streams them)
  bool ring_tiles = false;          // SV_TILED=1: the ring GEMVs of the graph path stream them too
  uint8_t* flow_mem = nullptr;
  size_t flow_bytes = 0;
  uint32_t *f_xa = nullptr, *f_xb = nullptr, *f_qkv = nullptr, *f_att = nullptr, *f_hb = nullptr;
  unsigned long long *f_part = nullptr, *f_amax = nullptr;
  int flow_l2_ahead = 0;            // SV_FLOW_L2AHEAD: weight slabs per CTA prefetched into L2 ahead of the ring (measured: no gain, off)
  // slab-tiled copies of the decoder matrices for the dataflow kernel (made from the reference-layout weights when they change)
  std::vector<uint8_t*> t_attn, t_proj, t_fc, t_fc2;
  uint8_t* t_lm_head = nullptr;
  const bf16* t_lm_src = nullptr;   // which lm_head tensor t_lm_head was made from
  bool tiles_dirty = true;
  int flow_epoch = 0;               // phase-tag epoch: steps run through the flow kernel since the buffers were cleared
  bf16 *kscratch = nullptr, *vscratch = nullptr;   // one layer of cache, for beam-search reorders
  // device-resident beam search (sv_beam.cu), allocated by the first sv_beam_search call
  svbeam::Params* beam_params = nullptr;
  svbeam::State* beam_state = nullptr;
  svbeam::Plan* beam_plan = nullptr;
  float *beam_key = nullptr, *beam_val = nullptr;
  int32_t *beam_tok = nullptr, *beam_run_seq = nullptr, *beam_fin_seq = nullptr;
  bf16 *kstage = nullptr, *vstage = nullptr;        // staging copy of the cache for the KV suffix moves (all layers)
  std::map<long long, GraphEntry> beam_graphs;
  // scoring (sv_extend) workspaces for kScoreRows rows, allocated by the first sv_extend
  bf16 *s_x = nullptr, *s_ln = nullptr, *s_qkv = nullptr, *s_attn = nullptr, *s_h = nullptr;
  float2* s_part = nullptr;
  float* s_tlogit = nullptr;
  int32_t *s_tgt = nullptr, *s_lg_row = nullptr, *s_lp_idx = nullptr;
  bf16 *kcache, *vtcache;           // [layer][max_batch][n_kv][tcap][D] / [layer][max_batch][n_kv][D][tcap]
  int64_t cache_layer_stride = 0;
  GenState* state = nullptr;
  GenParamsDev* params = nullptr;
  uint8_t* seen = nullptr;
  int32_t *next_ids = nullptr, *out_ids = nullptr, *ids_tmp = nullptr;
  bf16* im2svg_px = nullptr;        // staging of sv_generate_im2svg_host (pixels in, ids + lengths out): allocated by its first
  int32_t* im2svg_out = nullptr;    //   call, sized for max_batch rows, kept for the engine's lifetime
  int32_t* host_flag = nullptr;     // pinned
  int32_t* host_stream = nullptr;   // pinned staging of streamed tokens [max_batch][kStreamChunk], allocated on first use

  // run state (host mirror)
  int cur_batch = 0, prefix_len = 0, host_cur_len = 0;
  bool encoded = false, prefilled = false;

  cudaStream_t gen_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
  std::map<long long, GraphEntry> graphs;   // key = batch * 1000 + nsplit * 2 + do_sample
  float last_decode_ms = 0.f;
  int last_decode_steps = 0;
};

namespace {

int fail(sv_engine* e, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (e) e->err = buf; else g_create_error = buf;
  return code;
}

#define SV_CK(e, call)                                                                              \
  do {                                                                                              \
    cudaError_t _err = (call);                                                                      \
    if (_err != cudaSuccess)                                                                        \
      return fail((e), SV_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_err), __FILE__, __LINE__); \
  } while (0)

struct LaunchScope {   // routes count_launch() of this thread to the engine's counter
  explicit LaunchScope(sv_engine* e) { g_launch_counter = &e->launches; }
  ~LaunchScope() { g_launch_counter = nullptr; }
};

template <typename T>
cudaError_t dev_alloc(sv_engine* e, T** p, int64_t n) {
  void* q = nullptr;
  cudaError_t r = cudaMalloc(&q, (size_t)std::max<int64_t>(n, 1) * sizeof(T));
  if (r == cudaSuccess) { e->allocs.push_back(q); *p = reinterpret_cast<T*>(q); }
  return r;
}

// `external` != nullptr registers the name as a view into storage that another entry owns (v2 packs the reference's
// separate q_proj / k_proj / v_proj tensors into one [q|k|v] matrix so both families share the same kernels).
bf16* add_weight(sv_engine* e, const std::string& name, std::vector<int64_t> shape, int64_t alloc_numel = -1,
                 bool optional = false, bf16* external = nullptr) {
  Weight wt;
  wt.shape = shape;
  wt.numel = 1;
  for (auto s : shape) wt.numel *= s;
  wt.optional = optional;
  if (external) {
    wt.p = external;
  } else {
    int64_t n = alloc_numel > 0 ? alloc_numel : wt.numel;
    if (dev_alloc(e, &wt.p, n) != cudaSuccess) return nullptr;
    cudaMemset(wt.p, 0, (size_t)n * sizeof(bf16));
  }
  bf16* p = wt.p;
  e->w[name] = std::move(wt);
  return p;
}

const char* VIS = "model.image_encoder.visual_encoder.";
const char* LNV = "model.image_encoder.ln_vision.";
const char* ADP = "model.image_projection.";
const char* DEC = "model.svg_transformer.transformer.transformer.";
const char* LMH = "model.svg_transformer.transformer.lm_head.weight";

bool build_weights_v2(sv_engine* e);

bool build_weights(sv_engine* e) {
  if (e->v2) return build_weights_v2(e);
  const sv_model_desc& d = e->d;
  const int64_t W = d.vit_width, Q = e->Q, H = d.hidden, kv = (int64_t)d.n_kv_head * d.head_dim, I = d.n_inner;
  bool ok = true;
  auto A = [&](const std::string& n, std::vector<int64_t> s, int64_t alloc = -1, bool opt = false) {
    bf16* p = add_weight(e, n, std::move(s), alloc, opt);
    ok = ok && p != nullptr;
    return p;
  };
  std::string v = VIS;
  e->conv_raw = A(v + "conv1.weight", {W, 3, d.patch_size, d.patch_size});
  ok = ok && dev_alloc(e, &e->conv_w, W * e->Kp) == cudaSuccess;
  e->cls = A(v + "class_embedding", {W});
  e->pos = A(v + "positional_embedding", {Q, W});
  e->lnpre_w = A(v + "ln_pre.weight", {W});
  e->lnpre_b = A(v + "ln_pre.bias", {W});
  e->vit.resize(d.vit_layers);
  for (int i = 0; i < d.vit_layers; ++i) {
    std::string p = v + "transformer.resblocks." + std::to_string(i) + ".";
    VitLayer& L = e->vit[i];
    L.ln1_w = A(p + "ln_1.weight", {W}); L.ln1_b = A(p + "ln_1.bias", {W});
    L.qkv_w = A(p + "attn.in_proj_weight", {3 * W, W}); L.qkv_b = A(p + "attn.in_proj_bias", {3 * W});
    L.out_w = A(p + "attn.out_proj.weight", {W, W}); L.out_b = A(p + "attn.out_proj.bias", {W});
    L.ln2_w = A(p + "ln_2.weight", {W}); L.ln2_b = A(p + "ln_2.bias", {W});
    L.fc_w = A(p + "mlp.c_fc.weight", {(int64_t)d.vit_mlp, W}); L.fc_b = A(p + "mlp.c_fc.bias", {(int64_t)d.vit_mlp});
    L.proj_w = A(p + "mlp.c_proj.weight", {W, (int64_t)d.vit_mlp}); L.proj_b = A(p + "mlp.c_proj.bias", {W});
  }
  e->lnv_w = A(std::string(LNV) + "weight", {W});
  e->lnv_b = A(std::string(LNV) + "bias", {W});
  std::string a = ADP;
  e->afc_w = A(a + "c_fc.weight", {2 * W, W}); e->afc_b = A(a + "c_fc.bias", {2 * W});
  e->aproj_w = A(a + "c_proj.weight", {H, 2 * W}); e->aproj_b = A(a + "c_proj.bias", {H});
  if (d.adapter_norm == 0) {
    e->anorm_w = A(a + "norm.weight", {Q, H}); e->anorm_b = A(a + "norm.bias", {Q, H});
  } else {
    e->anorm_w = A(a + "norm.weight", {Q}); e->anorm_b = A(a + "norm.bias", {Q});
    e->anorm_rm = A(a + "norm.running_mean", {Q}); e->anorm_rv = A(a + "norm.running_var", {Q});
  }
  std::string t = DEC;
  e->wte = A(t + "wte.weight", {(int64_t)d.vocab, H});
  e->wpe = A(t + "wpe.weight", {(int64_t)d.n_positions, H});
  e->dec.resize(d.n_layer);
  for (int i = 0; i < d.n_layer; ++i) {
    std::string p = t + "h." + std::to_string(i) + ".";
    DecLayer& L = e->dec[i];
    L.ln1_w = A(p + "ln_1.weight", {H}); L.ln1_b = A(p + "ln_1.bias", {H});
    L.attn_w = A(p + "attn.c_attn.weight", {H + 2 * kv, H}); L.attn_b = A(p + "attn.c_attn.bias", {H + 2 * kv});
    L.proj_w = A(p + "attn.c_proj.weight", {H, H}); L.proj_b = A(p + "attn.c_proj.bias", {H});
    L.ln2_w = A(p + "ln_2.weight", {H}); L.ln2_b = A(p + "ln_2.bias", {H});
    L.fc_w = A(p + "mlp.c_fc.weight", {I, H}); L.fc_b = A(p + "mlp.c_fc.bias", {I});
    L.fc2_w = A(p + "mlp.c_proj.weight", {H, I}); L.fc2_b = A(p + "mlp.c_proj.bias", {H});
  }
  e->lnf_w = A(t + "ln_f.weight", {H});
  e->lnf_b = A(t + "ln_f.bias", {H});
  e->lm_head = e->wte;   // tied (train/util.py:68-77); an explicit lm_head.weight un-ties it
  return ok;
}

// StarVector v2 (8B family) state dict: SiglipVisionTransformer keys under model.image_encoder.visual_encoder.
// (image_encoder.py:32-48,108-109), the same Adapter, Starcoder2ForCausalLM keys under
// model.svg_transformer.transformer. (llm/starcoder2.py:19-32).  q/k/v projections are packed [q|k|v] at load.
bool build_weights_v2(sv_engine* e) {
  const sv_model_desc& d = e->d;
  const int64_t W = d.vit_width, Q = e->Q, H = d.hidden, D = d.head_dim, kv = (int64_t)d.n_kv_head * D, I = d.n_inner;
  const int64_t HQ = (int64_t)d.n_head * D;
  bool ok = true;
  auto A = [&](const std::string& n, std::vector<int64_t> s, bf16* ext = nullptr, bool opt = false) {
    bf16* p = add_weight(e, n, std::move(s), -1, opt, ext);
    ok = ok && p != nullptr;
    return p;
  };
  auto raw = [&](int64_t n) { bf16* p = nullptr; ok = ok && dev_alloc(e, &p, n) == cudaSuccess; if (p) cudaMemset(p, 0, (size_t)n * 2); return p; };
  std::string v = VIS;
  e->conv_raw = A(v + "embeddings.patch_embedding.weight", {W, 3, d.patch_size, d.patch_size});
  ok = ok && dev_alloc(e, &e->conv_w, W * e->Kp) == cudaSuccess;
  e->conv_b = A(v + "embeddings.patch_embedding.bias", {W});
  e->pos = A(v + "embeddings.position_embedding.weight", {Q, W});
  e->vit.resize(d.vit_layers);
  for (int i = 0; i < d.vit_layers; ++i) {
    std::string p = v + "encoder.layers." + std::to_string(i) + ".";
    VitLayer& L = e->vit[i];
    L.ln1_w = A(p + "layer_norm1.weight", {W}); L.ln1_b = A(p + "layer_norm1.bias", {W});
    L.qkv_w = raw(3 * W * W); L.qkv_b = raw(3 * W);
    if (!ok) return false;
    const char* nm[3] = {"q_proj", "k_proj", "v_proj"};
    for (int j = 0; j < 3; ++j) {
      A(p + "self_attn." + nm[j] + ".weight", {W, W}, L.qkv_w + j * W * W);
      A(p + "self_attn." + nm[j] + ".bias", {W}, L.qkv_b + j * W);
    }
    L.out_w = A(p + "self_attn.out_proj.weight", {W, W}); L.out_b = A(p + "self_attn.out_proj.bias", {W});
    L.ln2_w = A(p + "layer_norm2.weight", {W}); L.ln2_b = A(p + "layer_norm2.bias", {W});
    L.fc_w = A(p + "mlp.fc1.weight", {(int64_t)d.vit_mlp, W}); L.fc_b = A(p + "mlp.fc1.bias", {(int64_t)d.vit_mlp});
    L.proj_w = A(p + "mlp.fc2.weight", {W, (int64_t)d.vit_mlp}); L.proj_b = A(p + "mlp.fc2.bias", {W});
  }
  e->lnv_w = A(v + "post_layernorm.weight", {W});
  e->lnv_b = A(v + "post_layernorm.bias", {W});
  std::string a = ADP;
  e->afc_w = A(a + "c_fc.weight", {2 * W, W}); e->afc_b = A(a + "c_fc.bias", {2 * W});
  e->aproj_w = A(a + "c_proj.weight", {H, 2 * W}); e->aproj_b = A(a + "c_proj.bias", {H});
  if (d.adapter_norm == 0) {
    e->anorm_w = A(a + "norm.weight", {Q, H}); e->anorm_b = A(a + "norm.bias", {Q, H});
  } else {
    e->anorm_w = A(a + "norm.weight", {Q}); e->anorm_b = A(a + "norm.bias", {Q});
    e->anorm_rm = A(a + "norm.running_mean", {Q}); e->anorm_rv = A(a + "norm.running_var", {Q});
  }
  std::string t = "model.svg_transformer.transformer.model.";
  e->wte = A(t + "embed_tokens.weight", {(int64_t)d.vocab, H});
  e->wpe = nullptr;
  e->dec.resize(d.n_layer);
  for (int i = 0; i < d.n_layer; ++i) {
    std::string p = t + "layers." + std::to_string(i) + ".";
    DecLayer& L = e->dec[i];
    L.ln1_w = A(p + "input_layernorm.weight", {H}); L.ln1_b = A(p + "input_layernorm.bias", {H});
    L.attn_w = raw((HQ + 2 * kv) * H); L.attn_b = raw(HQ + 2 * kv);
    if (!ok) return false;
    A(p + "self_attn.q_proj.weight", {HQ, H}, L.attn_w); A(p + "self_attn.q_proj.bias", {HQ}, L.attn_b);
    A(p + "self_attn.k_proj.weight", {kv, H}, L.attn_w + HQ * H); A(p + "self_attn.k_proj.bias", {kv}, L.attn_b + HQ);
    A(p + "self_attn.v_proj.weight", {kv, H}, L.attn_w + (HQ + kv) * H); A(p + "self_attn.v_proj.bias", {kv}, L.attn_b + HQ + kv);
    L.proj_w = A(p + "self_attn.o_proj.weight", {H, HQ}); L.proj_b = A(p + "self_attn.o_proj.bias", {H});
    L.ln2_w = A(p + "post_attention_layernorm.weight", {H}); L.ln2_b = A(p + "post_attention_layernorm.bias", {H});
    L.fc_w = A(p + "mlp.c_fc.weight", {I, H}); L.fc_b = A(p + "mlp.c_fc.bias", {I});
    L.fc2_w = A(p + "mlp.c_proj.weight", {H, I}); L.fc2_b = A(p + "mlp.c_proj.bias", {H});
  }
  e->lnf_w = A(t + "norm.weight", {H});
  e->lnf_b = A(t + "norm.bias", {H});
  e->lm_head = e->wte;
  // RoPE tables [n_positions][D/2]: computed on device at create; a host may overwrite them with its own values
  e->rope_cos = A("engine.rope_cos", {(int64_t)d.n_positions, D / 2}, nullptr, true);
  e->rope_sin = A("engine.rope_sin", {(int64_t)d.n_positions, D / 2}, nullptr, true);
  return ok;
}

bool build_buffers(sv_engine* e) {
  const sv_model_desc& d = e->d;
  const int64_t B = d.max_batch, W = d.vit_width, H = d.hidden, I = d.n_inner, D = d.head_dim;
  const int64_t Mv = B * e->Q, Mp = B * (e->Q + kMaxPrompt), heads = d.vit_heads;
  bool ok = true;
#define AL(ptr, n) ok = ok && (dev_alloc(e, &e->ptr, (n)) == cudaSuccess)
  AL(v_patches, B * e->NP * e->Kp); AL(v_pe, B * e->NP * W); AL(v_x, Mv * W); AL(v_ln, Mv * W);
  AL(v_qkv, Mv * 3 * W); AL(v_vt, B * heads * 64 * e->Lpad); AL(v_attn, Mv * W); AL(v_h, Mv * d.vit_mlp);
  AL(v_out, Mv * W); AL(a_h, Mv * 2 * W); AL(a_z, Mv * H); AL(visual, Mv * H);
  AL(slab_partial, B * 64 * 2);
  AL(p_x, Mp * H); AL(p_ln, Mp * H); AL(p_qkv, Mp * e->qkv_cols); AL(p_attn, Mp * H); AL(p_h, Mp * I);
  AL(d_x, B * H); AL(d_ln, B * H); AL(d_qkv, B * e->qkv_cols); AL(d_attn, B * H); AL(d_h, B * I); AL(d_last, B * H);
  AL(logits, B * d.vocab); AL(logits_f32, B * d.vocab);
  AL(attn_partial, B * d.n_kv_head * kMaxSplit * (32 + 16 * D));
  const int64_t amax_rows = gemv_ring_ntiles(d.vocab);
  AL(amax_val, amax_rows * 8); AL(amax_idx, amax_rows * 8);
  AL(mega_layers, d.n_layer); AL(mega_dbg, 8192);
  {
    // flagged exchange buffers of the dataflow decode kernel, cleared together when a sequence starts
    // a flagged word per value, one 8-value fragment per 256-byte chunk (sv_decode_flow.cu FRAG_STRIDE): 32 bytes per value
    const size_t n_x = (size_t)B * H * 32, n_qkv = (size_t)B * e->qkv_cols * 32, n_hb = (size_t)B * I * 32;
    const size_t n_part = (size_t)B * d.n_kv_head * decode_flow_max_splits() * decode_flow_partial_floats() * 8;
    const size_t n_amax = (size_t)gemv_ring_ntiles(d.vocab) * 8 * 8;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    e->flow_bytes = 3 * up(n_x) + up(n_qkv) + up(n_hb) + up(n_part) + up(n_amax);
    AL(flow_mem, (int64_t)e->flow_bytes);
    if (ok) {
      uint8_t* q = e->flow_mem;
      e->f_xa = reinterpret_cast<uint32_t*>(q); q += up(n_x);
      e->f_xb = reinterpret_cast<uint32_t*>(q); q += up(n_x);
      e->f_att = reinterpret_cast<uint32_t*>(q); q += up(n_x);
      e->f_qkv = reinterpret_cast<uint32_t*>(q); q += up(n_qkv);
      e->f_hb = reinterpret_cast<uint32_t*>(q); q += up(n_hb);
      e->f_part = reinterpret_cast<unsigned long long*>(q); q += up(n_part);
      e->f_amax = reinterpret_cast<unsigned long long*>(q);
    }
  }
  e->cache_layer_stride = B * d.n_kv_head * (int64_t)e->tcap * D;
  AL(kcache, e->cache_layer_stride * d.n_layer); AL(vtcache, e->cache_layer_stride * d.n_layer);
  AL(kscratch, e->cache_layer_stride); AL(vscratch, e->cache_layer_stride);
  AL(state, 1); AL(params, 1); AL(seen, B * d.vocab); AL(next_ids, B); AL(out_ids, B * (int64_t)d.max_len);
  AL(ids_tmp, B * kMaxPrompt);
#undef AL
  if (!ok) return false;
  // zero the caches once: masked keys are never read as NaN (sv_attention.cu, P == 0 there)
  cudaMemset(e->kcache, 0, (size_t)e->cache_layer_stride * d.n_layer * sizeof(bf16));
  cudaMemset(e->vtcache, 0, (size_t)e->cache_layer_stride * d.n_layer * sizeof(bf16));
  cudaMemset(e->state, 0, sizeof(GenState));
  cudaMemset(e->flow_mem, 0, e->flow_bytes);
  return cudaMallocHost(reinterpret_cast<void**>(&e->host_flag), 64) == cudaSuccess;
}

int do_linear(sv_engine* e, int impl, const bf16* x, const bf16* w, const bf16* bias, const bf16* res, bf16* y, int M,
              int N, int K, int act, cudaStream_t st) {
  if (impl == SV_LINEAR_AUTO) impl = (M > 32 && tc05_supported(M, N, K)) ? SV_LINEAR_TCGEN05 : SV_LINEAR_ROWGROUP;
  if (impl == SV_LINEAR_TCGEN05) {
    if (!tc05_supported(M, N, K)) return fail(e, SV_ERR_INVALID, "tcgen05 linear needs N%%8==0, K%%64==0 (M=%d N=%d K=%d)", M, N, K);
    cudaError_t r = launch_linear_tc05(x, w, bias, res, y, M, N, K, act, st);
    if (r != cudaSuccess) return fail(e, SV_ERR_CUDA, "tcgen05 linear launch failed: %s", cudaGetErrorString(r));
    return SV_OK;
  }
  if (K % 32 != 0) return fail(e, SV_ERR_INVALID, "rowgroup linear needs K%%32==0 (K=%d)", K);
  launch_linear_rowgroup(x, w, bias, res, y, M, N, K, act, st);
  return SV_OK;
}
#define LIN(...)                                   \
  do {                                             \
    int _r = do_linear(e, e->linear_impl, __VA_ARGS__); \
    if (_r != SV_OK) return _r;                    \
  } while (0)

// ---- stage: ViT + adapter -------------------------------------------------------------------
int run_encode(sv_engine* e, const bf16* pixels, int B, cudaStream_t st) {
  const sv_model_desc& d = e->d;
  const int W = d.vit_width, Q = e->Q, NP = e->NP, M = B * Q, H = d.hidden;
  const float veps = e->vit_eps;
  launch_im2col(pixels, e->v_patches, B, d.image_size, d.patch_size, e->Kp, st);
  LIN(e->v_patches, e->conv_w, e->conv_b, nullptr, e->v_pe, B * NP, W, e->Kp, SV_ACT_NONE, st);   // patch conv (bias: SigLIP only)
  if (e->v2) {
    launch_vit_assemble(e->v_pe, nullptr, e->pos, e->v_x, B, NP, W, st);                           // + position_embedding
  } else {
    launch_vit_assemble(e->v_pe, e->cls, e->pos, e->v_ln, B, NP, W, st);                           // cat cls + pos
    launch_layernorm(e->v_ln, e->lnpre_w, e->lnpre_b, e->v_x, M, W, veps, W, st);                  // ln_pre
  }
  for (int i = 0; i < d.vit_layers; ++i) {
    const VitLayer& L = e->vit[i];
    launch_layernorm(e->v_x, L.ln1_w, L.ln1_b, e->v_ln, M, W, veps, W, st);
    LIN(e->v_ln, L.qkv_w, L.qkv_b, nullptr, e->v_qkv, M, 3 * W, W, SV_ACT_NONE, st);
    launch_vit_transpose_v(e->v_qkv, e->v_vt, B, Q, d.vit_heads, e->Lpad, st);
    launch_attention_vit(e->v_qkv, e->v_vt, e->v_attn, B, Q, d.vit_heads, e->Lpad, st);
    LIN(e->v_attn, L.out_w, L.out_b, e->v_x, e->v_x, M, W, W, SV_ACT_NONE, st);                    // x += attn
    launch_layernorm(e->v_x, L.ln2_w, L.ln2_b, e->v_ln, M, W, veps, W, st);
    LIN(e->v_ln, L.fc_w, L.fc_b, nullptr, e->v_h, M, d.vit_mlp, W, e->vit_act, st);
    LIN(e->v_h, L.proj_w, L.proj_b, e->v_x, e->v_x, M, W, d.vit_mlp, SV_ACT_NONE, st);             // x += mlp
  }
  launch_layernorm(e->v_x, e->lnv_w, e->lnv_b, e->v_out, M, W, veps, W, st);                       // ln_vision | post_layernorm
  LIN(e->v_out, e->afc_w, e->afc_b, nullptr, e->a_h, M, 2 * W, W, SV_ACT_SILU, st);
  LIN(e->a_h, e->aproj_w, e->aproj_b, nullptr, e->a_z, M, H, 2 * W, SV_ACT_NONE, st);
  if (d.adapter_norm == 0)
    launch_slab_layernorm(e->a_z, e->anorm_w, e->anorm_b, e->visual, e->slab_partial, B, (int64_t)Q * H, 1e-5f, st);
  else
    launch_batchnorm_tokens(e->a_z, e->anorm_w, e->anorm_b, e->anorm_rm, e->anorm_rv, e->visual, B, Q, H, 1e-5f, st);
  return SV_OK;
}

// ---- stage: decoder prefill -----------------------------------------------------------------
// `prefix` is [B, q, H] embeddings (the resident visual prefix, or caller-provided inputs_embeds);
// `prompt_ids` [B, P] are embedded through wte and appended (P may be 0).
int run_prefill(sv_engine* e, const bf16* prefix, int q, const int32_t* prompt_ids, int B, int P, cudaStream_t st) {
  const sv_model_desc& d = e->d;
  const int H = d.hidden, T0 = q + P, M = B * T0, D = d.head_dim;
  launch_embed_prefix(prefix, prompt_ids, e->wte, e->wpe, e->p_x, B, q, P, H, d.vocab, st);
  for (int i = 0; i < d.n_layer; ++i) {
    const DecLayer& L = e->dec[i];
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    launch_layernorm(e->p_x, L.ln1_w, L.ln1_b, e->p_ln, M, H, d.ln_eps, H, st);
    LIN(e->p_ln, L.attn_w, L.attn_b, nullptr, e->p_qkv, M, e->qkv_cols, H, SV_ACT_NONE, st);
    if (e->v2)   // RoPE on q and k (positions 0..T0-1), modeling_starcoder2.py:167-168
      launch_rope(e->p_qkv, M, T0, e->qkv_cols, d.n_head + d.n_kv_head, D, e->rope_cos, e->rope_sin, nullptr, d.n_positions, 0, st);
    launch_kv_scatter(e->p_qkv, kc, vc, B, T0, d.n_head * D, d.n_kv_head, D, e->tcap, 0, st);
    launch_attention_heads(e->p_qkv, e->qkv_cols, kc, vc, e->p_attn, B, T0, d.n_head, d.n_kv_head, D, e->tcap, e->window, 0, st);
    LIN(e->p_attn, L.proj_w, L.proj_b, e->p_x, e->p_x, M, H, H, SV_ACT_NONE, st);
    launch_layernorm(e->p_x, L.ln2_w, L.ln2_b, e->p_ln, M, H, d.ln_eps, H, st);
    LIN(e->p_ln, L.fc_w, L.fc_b, nullptr, e->p_h, M, d.n_inner, H, SV_ACT_GELU_TANH, st);
    LIN(e->p_h, L.fc2_w, L.fc2_b, e->p_x, e->p_x, M, H, d.n_inner, SV_ACT_NONE, st);
  }
  // last-position logits only (HF computes all T0 positions; only [:, -1] is consumed)
  launch_gather_rows(e->p_x, e->d_last, B, T0, T0 - 1, H, st);
  launch_layernorm(e->d_last, e->lnf_w, e->lnf_b, e->d_ln, B, H, d.ln_eps, H, st);
  launch_linear_rowgroup(e->d_ln, e->lm_head, nullptr, nullptr, e->logits, B, d.vocab, H, SV_ACT_NONE, st);
  return SV_OK;
}

// ---- stage: teacher forcing over a chunk (sv_extend) ------------------------------------------
// run_prefill at a position offset: tokens ids[b][t0 .. t0 + n) of the call's [B][T] ids go to cache positions
// pos0 .. pos0 + n (pos0 = the cache length before the call + t0).  The final LayerNorm and the lm_head with the fused log-prob
// epilogue run on every row; the fp32 logits are stored for the rows lg_row maps (kept positions / the call's last position).
int run_extend_chunk(sv_engine* e, const int32_t* ids, int T, int t0, int n, int pos0, int keep, float* logits_out, float* logps,
                     float inv_temp, cudaStream_t st) {
  const sv_model_desc& d = e->d;
  const int B = e->cur_batch, H = d.hidden, M = B * n, D = d.head_dim;
  launch_embed_chunk(ids + t0, T, e->wte, e->wpe, e->s_x, B, n, pos0, H, d.vocab, d.n_positions, st);
  for (int i = 0; i < d.n_layer; ++i) {
    const DecLayer& L = e->dec[i];
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    launch_layernorm(e->s_x, L.ln1_w, L.ln1_b, e->s_ln, M, H, d.ln_eps, H, st);
    LIN(e->s_ln, L.attn_w, L.attn_b, nullptr, e->s_qkv, M, e->qkv_cols, H, SV_ACT_NONE, st);
    if (e->v2)
      launch_rope(e->s_qkv, M, n, e->qkv_cols, d.n_head + d.n_kv_head, D, e->rope_cos, e->rope_sin, nullptr, d.n_positions, pos0, st);
    launch_kv_scatter(e->s_qkv, kc, vc, B, n, d.n_head * D, d.n_kv_head, D, e->tcap, pos0, st);
    launch_attention_heads(e->s_qkv, e->qkv_cols, kc, vc, e->s_attn, B, n, d.n_head, d.n_kv_head, D, e->tcap, e->window, pos0, st);
    LIN(e->s_attn, L.proj_w, L.proj_b, e->s_x, e->s_x, M, H, H, SV_ACT_NONE, st);
    launch_layernorm(e->s_x, L.ln2_w, L.ln2_b, e->s_ln, M, H, d.ln_eps, H, st);
    LIN(e->s_ln, L.fc_w, L.fc_b, nullptr, e->s_h, M, d.n_inner, H, SV_ACT_GELU_TANH, st);
    LIN(e->s_h, L.fc2_w, L.fc2_b, e->s_x, e->s_x, M, H, d.n_inner, SV_ACT_NONE, st);
  }
  // the lm_head runs where a log-prob, a kept logit or the call's last position needs it
  const bool kept = (keep > 0 && t0 + n > T - keep) || t0 + n == T;
  if (!logps && !kept) return SV_OK;
  launch_layernorm(e->s_x, e->lnf_w, e->lnf_b, e->s_ln, M, H, d.ln_eps, H, st);
  launch_score_maps(ids, T, B, n, t0, keep, d.vocab, logps != nullptr, e->s_tgt, e->s_lg_row, e->s_lp_idx, st);
  LogpsEpilogue lp{e->s_tgt, e->s_lg_row, keep > 0 ? logits_out : e->logits_f32, e->s_part, e->s_tlogit, inv_temp};
  cudaError_t r = launch_lm_head_logps(e->s_ln, e->lm_head, M, d.vocab, H, lp, e->s_lp_idx, logps, st);
  if (r != cudaSuccess) return fail(e, SV_ERR_CUDA, "lm_head log-prob launch failed: %s", cudaGetErrorString(r));
  return SV_OK;
}

// ---- one decode step: token ids (device) at position state->cur_len -> logits ----------------
int run_decode_layers(sv_engine* e, const int32_t* ids, int B, int nsplit, cudaStream_t st) {
  const sv_model_desc& d = e->d;
  const int H = d.hidden, D = d.head_dim;
  launch_embed_tokens(ids, e->wte, e->wpe, e->state, e->d_x, B, H, d.vocab, d.n_positions, st);
  for (int i = 0; i < d.n_layer; ++i) {
    const DecLayer& L = e->dec[i];
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    launch_layernorm(e->d_x, L.ln1_w, L.ln1_b, e->d_ln, B, H, d.ln_eps, H, st);
    launch_linear_rowgroup(e->d_ln, L.attn_w, L.attn_b, nullptr, e->d_qkv, B, e->qkv_cols, H, SV_ACT_NONE, st);
    if (e->v2)
      launch_rope(e->d_qkv, B, 1, e->qkv_cols, d.n_head + d.n_kv_head, D, e->rope_cos, e->rope_sin, e->state, d.n_positions, 0, st);
    launch_kv_append(e->d_qkv, kc, vc, e->state, B, d.n_head * D, d.n_kv_head, D, e->tcap, st);
    launch_attention_decode(e->d_qkv, e->qkv_cols, kc, vc, e->d_attn, e->attn_partial, e->state, B, d.n_head,
                            d.n_kv_head, D, e->tcap, nsplit, e->window, st);
    launch_linear_rowgroup(e->d_attn, L.proj_w, L.proj_b, e->d_x, e->d_x, B, H, H, SV_ACT_NONE, st);
    launch_layernorm(e->d_x, L.ln2_w, L.ln2_b, e->d_ln, B, H, d.ln_eps, H, st);
    launch_linear_rowgroup(e->d_ln, L.fc_w, L.fc_b, nullptr, e->d_h, B, d.n_inner, H, SV_ACT_GELU_TANH, st);
    launch_linear_rowgroup(e->d_h, L.fc2_w, L.fc2_b, e->d_x, e->d_x, B, H, d.n_inner, SV_ACT_NONE, st);
  }
  launch_layernorm(e->d_x, e->lnf_w, e->lnf_b, e->d_ln, B, H, d.ln_eps, H, st);
  launch_linear_rowgroup(e->d_ln, e->lm_head, nullptr, nullptr, e->logits, B, d.vocab, H, SV_ACT_NONE, st);
  return SV_OK;
}

// Fused decode step: 5 kernels per layer (4 weight-ring GEMVs with fused LayerNorm / bias / GELU / residual / KV append,
// 1 cluster attention) + lm_head, chained with programmatic dependent launch.  `ids` != nullptr embeds those tokens first
// (teacher forcing / sampling); with nullptr, d_x was already written by select_fused.
// Leaves bf16 logits in e->logits and per-tile argmax partials in e->amax_*.
int run_decode_layers_fused(sv_engine* e, const int32_t* ids, int B, int ncta, bool pdl, cudaStream_t st) {
  const sv_model_desc& d = e->d;
  const int H = d.hidden, D = d.head_dim;
  if (ids) launch_embed_tokens(ids, e->wte, e->wpe, e->state, e->d_x, B, H, d.vocab, d.n_positions, st);
  bool first = true;
  RingGemvLaunch g{};
  g.B = B; g.ln_eps = d.ln_eps; g.n_head = d.n_head; g.n_kv = d.n_kv_head; g.tcap = e->tcap; g.state = e->state;
  g.amax_val = e->amax_val; g.amax_idx = e->amax_idx;
  auto gemv = [&](const bf16* X, const bf16* W, const uint8_t* Wt, const bf16* bias, const bf16* res, bf16* Y, int N, int K, int act,
                  const bf16* lw, const bf16* lb, int epi, bf16* kc, bf16* vc, bool p) {
    g.X = X; g.W = W; g.Wt = e->ring_tiles ? Wt : nullptr; g.bias = bias; g.res = res; g.Y = Y; g.N = N; g.K = K; g.act = act; g.ln_w = lw; g.ln_b = lb;
    g.epi = epi; g.kcache = kc; g.vtcache = vc; g.pdl = p;
    launch_gemv_ring(g, st);
  };
  for (int i = 0; i < d.n_layer; ++i) {
    const DecLayer& L = e->dec[i];
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    const bool tl = e->ring_tiles;
    gemv(e->d_x, L.attn_w, tl ? e->t_attn[i] : nullptr, L.attn_b, nullptr, e->d_qkv, e->qkv_cols, H, SV_ACT_NONE, L.ln1_w, L.ln1_b, e->v2 ? 0 : 1, kc, vc,
         pdl && !first);
    first = false;
    if (e->v2)   // RoPE on q,k then append (the GEMV epilogue cannot rotate: the pair element lives in another tile)
      launch_rope_append(e->d_qkv, B, e->qkv_cols, d.n_head, d.n_kv_head, D, e->rope_cos, e->rope_sin, kc, vc, e->state,
                         e->tcap, d.n_positions, pdl, st);
    launch_attention_decode_cluster(e->d_qkv, e->qkv_cols, kc, vc, e->d_attn, e->state, B, d.n_head, d.n_kv_head, D, e->tcap,
                                    std::min(ncta, 8), e->window, pdl, st);
    gemv(e->d_attn, L.proj_w, tl ? e->t_proj[i] : nullptr, L.proj_b, e->d_x, e->d_x, H, H, SV_ACT_NONE, nullptr, nullptr, 0, nullptr, nullptr, pdl);
    gemv(e->d_x, L.fc_w, tl ? e->t_fc[i] : nullptr, L.fc_b, nullptr, e->d_h, d.n_inner, H, SV_ACT_GELU_TANH, L.ln2_w, L.ln2_b, 0, nullptr, nullptr, pdl);
    gemv(e->d_h, L.fc2_w, tl ? e->t_fc2[i] : nullptr, L.fc2_b, e->d_x, e->d_x, H, d.n_inner, SV_ACT_NONE, nullptr, nullptr, 0, nullptr, nullptr, pdl);
  }
  gemv(e->d_x, e->lm_head, (e->ring_tiles && e->t_lm_src == e->lm_head) ? e->t_lm_head : nullptr, nullptr, nullptr, e->logits, d.vocab, H, SV_ACT_NONE, e->lnf_w, e->lnf_b, 2, nullptr, nullptr, pdl);
  return SV_OK;
}

// (re)build the slab-tiled copies the dataflow kernel streams, after any weight changed
void ensure_flow_tiles(sv_engine* e, cudaStream_t st) {
  if (!e->use_tiles || (!e->tiles_dirty && e->t_lm_src == e->lm_head)) return;
  const sv_model_desc& d = e->d;
  const int nc = decode_flow_ncta();
  for (int i = 0; i < d.n_layer; ++i) {
    const DecLayer& L = e->dec[i];
    launch_flow_repack(L.attn_w, L.attn_b, e->t_attn[i], e->qkv_cols, d.hidden, nc, st);
    launch_flow_repack(L.proj_w, L.proj_b, e->t_proj[i], d.hidden, d.hidden, nc, st);
    launch_flow_repack(L.fc_w, L.fc_b, e->t_fc[i], d.n_inner, d.hidden, nc, st);
    launch_flow_repack(L.fc2_w, L.fc2_b, e->t_fc2[i], d.hidden, d.n_inner, nc, st);
  }
  launch_flow_repack(e->lm_head, nullptr, e->t_lm_head, d.vocab, d.hidden, nc, st);
  e->t_lm_src = e->lm_head;
  e->tiles_dirty = false;
}

FlowLaunch flow_launch_desc(sv_engine* e, int B) {
  FlowLaunch m{};
  m.layers_dev = e->mega_layers; m.n_layer = e->d.n_layer; m.B = B; m.H = e->d.hidden; m.I = e->d.n_inner;
  m.n_head = e->d.n_head; m.n_kv = e->d.n_kv_head; m.qkv_cols = e->qkv_cols; m.vocab = e->d.vocab; m.tcap = e->tcap;
  m.n_positions = e->d.n_positions; m.ln_eps = e->d.ln_eps; m.wte = e->wte; m.wpe = e->wpe; m.lnf_w = e->lnf_w;
  m.lnf_b = e->lnf_b; m.lm_head = e->lm_head; m.lm_head_t = reinterpret_cast<const bf16*>(e->t_lm_head); m.x_plain = e->d_x; m.logits = e->logits;
  m.xa = e->f_xa; m.xb = e->f_xb; m.qkv = e->f_qkv; m.att = e->f_att; m.hb = e->f_hb; m.part = e->f_part; m.amax = e->f_amax;
  m.state = e->state; m.params = e->params; m.seen = e->seen; m.next_ids = e->next_ids; m.out_ids = e->out_ids;
  m.dbg = e->mega_debug ? e->mega_dbg : nullptr;
  m.realloc = e->flow_realloc;
  m.l2_ahead = e->flow_l2_ahead;
  return m;
}

int nsplit_for(const sv_engine* e, int total_len) {
  int blocks = (total_len + 31) / 32;
  return std::max(1, std::min(kMaxSplit, blocks));
}

void launch_select(sv_engine* e, int B, int do_sample, cudaStream_t st) {
  if (do_sample)
    launch_select_sample(e->logits, e->d.vocab, B, e->state, e->params, e->seen, e->next_ids, e->out_ids,
                         e->logits_f32, st);
  else
    launch_select_greedy(e->logits, e->d.vocab, B, e->state, e->params, e->seen, e->next_ids, e->out_ids, st);
}

int check_ready(sv_engine* e) {
  for (auto& kv : e->w)
    if (!kv.second.loaded && !kv.second.optional) return fail(e, SV_ERR_STATE, "weight not loaded: %s", kv.first.c_str());
  return SV_OK;
}

}  // namespace

static int finish_prefill_impl(sv_engine* e, int batch, int prefix_len, float* last_logits, cudaStream_t st) {
  e->prefix_len = prefix_len;
  e->host_cur_len = e->prefix_len;
  GenState hs;
  memset(&hs, 0, sizeof(hs));
  hs.cur_len = e->prefix_len;
  for (int b = 0; b < batch; ++b) hs.unfinished[b] = 1;
  SV_CK(e, cudaMemcpyAsync(e->state, &hs, sizeof(hs), cudaMemcpyHostToDevice, st));   // pageable: staged synchronously
  ensure_flow_tiles(e, st);          // (no-op unless a weight changed since the last sequence)
  if (e->use_flow) {                 // new sequence: no word of the exchange buffers may carry a tag of the coming epochs
    SV_CK(e, cudaMemsetAsync(e->flow_mem, 0, e->flow_bytes, st));
    e->flow_epoch = 0;
  }
  if (last_logits) launch_logits_to_float(e->logits, last_logits, (int64_t)batch * e->d.vocab, st);
  SV_CK(e, cudaGetLastError());
  e->prefilled = true;
  return SV_OK;
}

static int finish_prefill(sv_engine* e, int batch, int prefix_len, float* last_logits, cudaStream_t st) {
  LaunchScope scope(e);
  return finish_prefill_impl(e, batch, prefix_len, last_logits, st);
}

// =============================================================================================
extern "C" {

int sv_abi_version(void) { return SV_ABI_VERSION; }

const char* sv_last_error(const sv_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int sv_engine_create(const sv_model_desc* desc, int device, sv_engine** out) {
  if (!desc || !out) return fail(nullptr, SV_ERR_INVALID, "null argument");
  *out = nullptr;
  const sv_model_desc& d = *desc;
  if (d.variant != 0 && d.variant != 1) return fail(nullptr, SV_ERR_UNSUPPORTED, "unknown model variant %d", d.variant);
  if (d.variant == 1 && !(d.rope_theta > 1.0f)) return fail(nullptr, SV_ERR_INVALID, "variant 1 (StarCoder2) needs rope_theta > 1");
  if (d.variant == 1 && d.sliding_window < 0) return fail(nullptr, SV_ERR_INVALID, "sliding_window must be >= 0");
  if (d.vit_width != d.vit_heads * 64) return fail(nullptr, SV_ERR_INVALID, "ViT head dim must be 64");
  if (d.head_dim != 128 || d.hidden != d.n_head * d.head_dim) return fail(nullptr, SV_ERR_INVALID, "decoder head dim must be 128 and hidden == n_head*128");
  if (d.hidden % 64 || d.n_inner % 64) return fail(nullptr, SV_ERR_INVALID, "decoder widths must be multiples of 64");
  if (d.n_kv_head < 1 || d.n_head % d.n_kv_head || d.n_head / d.n_kv_head > 16) return fail(nullptr, SV_ERR_INVALID, "need 1 <= n_head/n_kv_head <= 16");
  if (d.image_size % d.patch_size) return fail(nullptr, SV_ERR_INVALID, "image_size %% patch_size != 0");
  if (d.vit_width % 64 || d.vit_mlp % 64 || d.hidden % 64 || d.n_inner % 64) return fail(nullptr, SV_ERR_INVALID, "widths must be multiples of 64");
  if (d.max_batch < 1 || d.max_batch > 8) return fail(nullptr, SV_ERR_INVALID, "max_batch must be in [1,8] (decode kernels hold 8 rows per MMA)");
  if (d.adapter_norm != 0 && d.adapter_norm != 1) return fail(nullptr, SV_ERR_INVALID, "adapter_norm must be 0 or 1");
  if (d.vocab < 8 || d.vocab > (1 << 20)) return fail(nullptr, SV_ERR_INVALID, "vocab out of range");

  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev <= device)
    return fail(nullptr, SV_ERR_CUDA, "no CUDA device %d (%s): this engine has no CPU fallback", device,
                r == cudaSuccess ? "device count too small" : cudaGetErrorString(r));
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10)
    return fail(nullptr, SV_ERR_CUDA, "device %d is sm_%d%d; kernels are built for sm_100a (B200) only", device, prop.major, prop.minor);
  if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, SV_ERR_CUDA, "cudaSetDevice(%d) failed", device);

  sv_engine* e = new sv_engine();
  e->d = d;
  e->device = device;
  const int g = d.image_size / d.patch_size;
  e->NP = g * g;
  e->v2 = d.variant == 1;
  e->Q = e->NP + (e->v2 ? 0 : 1);                       // SigLIP has no class token
  if (e->v2) {
    e->vit_eps = d.vit_ln_eps > 0.f ? d.vit_ln_eps : 1e-6f;
    e->vit_act = SV_ACT_GELU_TANH;
    e->window = d.sliding_window;
  }
  e->Kp = (3 * d.patch_size * d.patch_size + 63) / 64 * 64;
  e->Lpad = (e->Q + 31) / 32 * 32;
  e->qkv_cols = d.hidden + 2 * d.n_kv_head * d.head_dim;
  int max_len = std::min(d.max_len, d.n_positions);
  if (max_len < e->Q + 2) { delete e; return fail(nullptr, SV_ERR_INVALID, "max_len %d smaller than the visual prefix", d.max_len); }
  e->d.max_len = max_len;
  e->tcap = (max_len + 1 + 31) / 32 * 32;
  const char* impl = getenv("SV_LINEAR_IMPL");
  if (impl && !strcmp(impl, "rowgroup")) e->linear_impl = SV_LINEAR_ROWGROUP;
  if (impl && !strcmp(impl, "tcgen05")) e->linear_impl = SV_LINEAR_TCGEN05;
  const char* dec = getenv("SV_DECODE");          // "legacy" = the unfused per-op kernels (A/B checks)
  if (dec && !strcmp(dec, "legacy")) e->fused_decode = false;
  const char* pdl = getenv("SV_PDL");             // "0" = plain stream order between decode kernels
  if (pdl && !strcmp(pdl, "0")) e->use_pdl = false;
  e->mega_debug = getenv("SV_MEGA_DEBUG") != nullptr;
  { const char* fl = getenv("SV_FLOW");          // "1": dataflow persistent kernel for greedy decode / teacher forcing (opt-in: the
    // per-phase CUDA graph is still faster, DESIGN.md §4); "3": the same without setmaxnreg register reallocation
    e->use_flow = fl && (!strcmp(fl, "1") || !strcmp(fl, "2") || !strcmp(fl, "3")); 
    e->flow_realloc = !(fl && !strcmp(fl, "3"));
    const char* la = getenv("SV_FLOW_L2AHEAD");
    if (la) e->flow_l2_ahead = std::max(0, std::min(64, atoi(la))); }
  if (!gemv_ring_supported(d.hidden, true) || !gemv_ring_supported(d.n_inner, false)) e->fused_decode = false;
  // v2 at full size: the per-op kernels measure faster (4.4 vs 5.8 ms/token at 8B; 768-wide slabs + per-slab LayerNorm
  // on the consumer path), so the fused ring step is opt-in for v2 (SV_DECODE=fused) until that is fixed.
  if (e->v2 && !(dec && !strcmp(dec, "fused"))) e->fused_decode = false;
  if (!build_weights(e) || !build_buffers(e)) {
    std::string msg = std::string("device allocation failed: ") + cudaGetErrorString(cudaGetLastError());
    sv_engine_destroy(e);
    return fail(nullptr, SV_ERR_CUDA, "%s", msg.c_str());
  }
  if (e->v2) {
    launch_rope_table(e->rope_cos, e->rope_sin, d.n_positions, d.head_dim, d.rope_theta, nullptr);
    if (cudaDeviceSynchronize() != cudaSuccess) {
      sv_engine_destroy(e);
      return fail(nullptr, SV_ERR_CUDA, "RoPE table setup failed");
    }
  }
  {
    std::vector<MegaLayer> ml(d.n_layer);
    for (int i = 0; i < d.n_layer; ++i) {
      const DecLayer& L = e->dec[i];
      ml[i] = MegaLayer{L.ln1_w, L.ln1_b, L.attn_w, L.attn_b, L.proj_w, L.proj_b, L.ln2_w, L.ln2_b, L.fc_w, L.fc_b,
                        L.fc2_w, L.fc2_b, e->kcache + e->cache_layer_stride * i, e->vtcache + e->cache_layer_stride * i,
                        nullptr, nullptr, nullptr, nullptr};
    }
    // slab-tiled copies of the decode weights (one bulk copy per ring slot instead of one per weight row): what the dataflow
    // kernel streams (SV_FLOW=1), and optionally the ring GEMVs of the graph path (SV_TILED=1).  In the streaming
    // microbenchmark one 30 KB copy per slot beats 16 row copies (7.1 vs 6.1 TB/s, profiles/r02_ring_stream.txt), but inside
    // the decode step the row-major weights measured 2 % faster (0.932 vs 0.954 ms/token, profiles/r02_summary.md), so the
    // default keeps ONE copy of the decoder in HBM.
    const char* tl = getenv("SV_TILED");
    const bool want_tiles = e->use_flow || (tl && !strcmp(tl, "1"));
    if (want_tiles && decode_flow_init() == cudaSuccess && e->fused_decode && decode_flow_ncta() == gemv_ring_ncta()) {
      const int nc = decode_flow_ncta();
      e->use_tiles = true;
      e->ring_tiles = tl && !strcmp(tl, "1");
      bool ok = true;
      auto tiled = [&](int N, int K) -> uint8_t* {
        uint8_t* p = nullptr;
        ok = ok && dev_alloc(e, &p, (int64_t)flow_tiled_bytes(N, K, nc)) == cudaSuccess;
        return p;
      };
      e->t_attn.resize(d.n_layer); e->t_proj.resize(d.n_layer); e->t_fc.resize(d.n_layer); e->t_fc2.resize(d.n_layer);
      for (int i = 0; i < d.n_layer; ++i) {
        e->t_attn[i] = tiled(e->qkv_cols, d.hidden); e->t_proj[i] = tiled(d.hidden, d.hidden);
        e->t_fc[i] = tiled(d.n_inner, d.hidden); e->t_fc2[i] = tiled(d.hidden, d.n_inner);
        ml[i].attn_t = reinterpret_cast<const bf16*>(e->t_attn[i]); ml[i].proj_t = reinterpret_cast<const bf16*>(e->t_proj[i]);
        ml[i].fc_t = reinterpret_cast<const bf16*>(e->t_fc[i]); ml[i].fc2_t = reinterpret_cast<const bf16*>(e->t_fc2[i]);
      }
      e->t_lm_head = tiled(d.vocab, d.hidden);
      if (!ok) { sv_engine_destroy(e); return fail(nullptr, SV_ERR_CUDA, "allocation of the tiled decode weights failed"); }
    }
    if (cudaMemcpy(e->mega_layers, ml.data(), ml.size() * sizeof(MegaLayer), cudaMemcpyHostToDevice) != cudaSuccess ||
        decode_flow_init() != cudaSuccess || gemv_ring_init() != cudaSuccess) {
      sv_engine_destroy(e);
      return fail(nullptr, SV_ERR_CUDA, "persistent decode kernel setup failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!decode_flow_supported(d.hidden, d.n_inner, d.head_dim, d.max_batch, e->window, e->v2) || !e->fused_decode || d.n_layer > 24 || !e->use_tiles) e->use_flow = false;
    if (e->flow_realloc && !decode_flow_realloc_supported()) e->flow_realloc = false;
  }
  if (attention_decode_cluster_init() != cudaSuccess) {
    sv_engine_destroy(e);
    return fail(nullptr, SV_ERR_CUDA, "cannot raise the shared-memory limit of the decode attention kernel");
  }
  if (cudaStreamCreateWithFlags(&e->gen_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&e->ev_t0) != cudaSuccess || cudaEventCreate(&e->ev_t1) != cudaSuccess) {
    sv_engine_destroy(e);
    return fail(nullptr, SV_ERR_CUDA, "stream/event creation failed");
  }
  *out = e;
  return SV_OK;
}

void sv_engine_destroy(sv_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (auto& g : e->graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
  for (auto& g : e->beam_graphs) if (g.second.exec) cudaGraphExecDestroy(g.second.exec);
  for (void* p : e->allocs) cudaFree(p);
  if (e->host_flag) cudaFreeHost(e->host_flag);
  if (e->host_stream) cudaFreeHost(e->host_stream);
  if (e->gen_stream) cudaStreamDestroy(e->gen_stream);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->ev_t0) cudaEventDestroy(e->ev_t0);
  if (e->ev_t1) cudaEventDestroy(e->ev_t1);
  delete e;
}

int sv_engine_load_weight(sv_engine* e, const char* hf_name, const void* data, const int64_t* shape, int32_t ndim,
                          int32_t dtype) {
  if (!e || !hf_name || !data || !shape) return fail(e, SV_ERR_INVALID, "null argument");
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  std::string name = hf_name;
  auto ends_with = [&](const char* s) { size_t n = strlen(s); return name.size() >= n && !name.compare(name.size() - n, n, s); };
  if (ends_with("num_batches_tracked") || ends_with(".attn.bias") || ends_with("transformer.bias") ||
      ends_with(".attn.masked_bias") || ends_with("rotary_emb.inv_freq") || ends_with("embeddings.position_ids"))
    return SV_OK;   // buffers that carry no parameters
  if (name.find("visual_encoder.head.") != std::string::npos)
    return SV_OK;   // SigLIP pooling head: computed and discarded by the reference (image_encoder.py:109)
  int64_t numel = 1;
  for (int i = 0; i < ndim; ++i) numel *= shape[i];
  if (name == LMH && e->w.find(name) == e->w.end()) {   // explicit (un-tied) lm_head
    const sv_model_desc& d = e->d;
    bf16* p = add_weight(e, name, {(int64_t)d.vocab, (int64_t)d.hidden}, -1, true);
    if (!p) return fail(e, SV_ERR_CUDA, "allocation failed for lm_head");
    e->lm_head = p;
  }
  auto it = e->w.find(name);
  if (it == e->w.end()) return fail(e, SV_ERR_INVALID, "unknown weight name: %s", hf_name);
  Weight& wt = it->second;
  if (numel != wt.numel || ndim != (int)wt.shape.size())
    return fail(e, SV_ERR_INVALID, "shape mismatch for %s: got %lld elements / %d dims, expected %lld / %zu", hf_name,
                (long long)numel, ndim, (long long)wt.numel, wt.shape.size());
  for (int i = 0; i < ndim; ++i)
    if (shape[i] != wt.shape[i]) return fail(e, SV_ERR_INVALID, "shape mismatch for %s at dim %d", hf_name, i);
  if (dtype == SV_DTYPE_BF16) {
    SV_CK(e, cudaMemcpy(wt.p, data, (size_t)numel * 2, cudaMemcpyDefault));
  } else if (dtype == SV_DTYPE_F32 || dtype == SV_DTYPE_F16) {
    const size_t es = dtype == SV_DTYPE_F32 ? 4 : 2;
    void* tmp = nullptr;
    SV_CK(e, cudaMalloc(&tmp, (size_t)numel * es));
    cudaError_t r = cudaMemcpy(tmp, data, (size_t)numel * es, cudaMemcpyDefault);
    if (r == cudaSuccess) {
      launch_convert_to_bf16(tmp, dtype, wt.p, numel, nullptr);
      r = cudaDeviceSynchronize();
    }
    cudaFree(tmp);
    SV_CK(e, r);
  } else {
    return fail(e, SV_ERR_INVALID, "unsupported dtype %d", dtype);
  }
  if (wt.p == e->conv_raw) {   // [W,3,p,p] -> [W, Kp] zero padded GEMM operand
    launch_pad_rows(e->conv_raw, e->conv_w, e->d.vit_width, 3 * e->d.patch_size * e->d.patch_size, e->Kp, nullptr);
    SV_CK(e, cudaDeviceSynchronize());
  }
  wt.loaded = true;
  e->tiles_dirty = true;
  return SV_OK;
}

int sv_engine_missing_weights(sv_engine* e) {
  if (!e) return SV_ERR_INVALID;
  int n = 0;
  std::string names;
  for (auto& kv : e->w)
    if (!kv.second.loaded && !kv.second.optional) { ++n; names += kv.first + "\n"; }
  e->err = names;
  return n;
}

int sv_encode_images(sv_engine* e, const void* pixels, int32_t batch, void* out_embeds, void* vit_out, void* stream) {
  if (!e || !pixels) return fail(e, SV_ERR_INVALID, "null argument");
  if (batch < 1 || batch > e->d.max_batch) return fail(e, SV_ERR_INVALID, "batch %d outside [1,%d]", batch, e->d.max_batch);
  int r = check_ready(e);
  if (r != SV_OK) return r;
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  r = run_encode(e, (const bf16*)pixels, batch, st);
  if (r != SV_OK) return r;
  const size_t M = (size_t)batch * e->Q;
  if (out_embeds) SV_CK(e, cudaMemcpyAsync(out_embeds, e->visual, M * e->d.hidden * 2, cudaMemcpyDeviceToDevice, st));
  if (vit_out) SV_CK(e, cudaMemcpyAsync(vit_out, e->v_out, M * e->d.vit_width * 2, cudaMemcpyDeviceToDevice, st));
  SV_CK(e, cudaGetLastError());
  e->cur_batch = batch;
  e->encoded = true;
  e->prefilled = false;
  return SV_OK;
}

int sv_prefill(sv_engine* e, const int32_t* prompt_ids, int32_t batch, int32_t prompt_len, float* last_logits,
               void* stream) {
  if (!e || !prompt_ids) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->encoded || batch != e->cur_batch) return fail(e, SV_ERR_STATE, "sv_prefill needs sv_encode_images with the same batch first");
  if (prompt_len < 1 || prompt_len > kMaxPrompt) return fail(e, SV_ERR_INVALID, "prompt_len %d outside [1,%d]", prompt_len, kMaxPrompt);
  if (e->Q + prompt_len + 1 > e->d.max_len) return fail(e, SV_ERR_INVALID, "prefix longer than max_len");
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  int r = run_prefill(e, e->visual, e->Q, prompt_ids, batch, prompt_len, st);
  if (r != SV_OK) return r;
  return finish_prefill(e, batch, e->Q + prompt_len, last_logits, st);
}

int sv_prefill_embeds(sv_engine* e, const void* inputs_embeds, int32_t batch, int32_t seq_len, float* last_logits,
                      void* stream) {
  if (!e || !inputs_embeds) return fail(e, SV_ERR_INVALID, "null argument");
  if (batch < 1 || batch > e->d.max_batch) return fail(e, SV_ERR_INVALID, "batch %d outside [1,%d]", batch, e->d.max_batch);
  if (seq_len < 1 || seq_len > e->Q + kMaxPrompt) return fail(e, SV_ERR_INVALID, "seq_len %d outside [1,%d]", seq_len, e->Q + kMaxPrompt);
  if (seq_len + 1 > e->d.max_len) return fail(e, SV_ERR_INVALID, "prefix longer than max_len");
  int r = check_ready(e);
  if (r != SV_OK) return r;
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  r = run_prefill(e, (const bf16*)inputs_embeds, seq_len, nullptr, batch, 0, st);
  if (r != SV_OK) return r;
  e->cur_batch = batch;
  return finish_prefill(e, batch, seq_len, last_logits, st);
}

int sv_decode_step(sv_engine* e, const int32_t* ids, float* logits, void* stream) {
  if (!e || !ids) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(e, SV_ERR_STATE, "sv_decode_step needs sv_prefill first");
  if (e->host_cur_len + 1 > e->d.max_len) return fail(e, SV_ERR_INVALID, "KV cache full (max_len %d)", e->d.max_len);
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  int r = SV_OK;
  if (e->use_flow) {
    // one token through the dataflow kernel: embed (plain) -> all layers -> logits, no selection
    const sv_model_desc& d = e->d;
    launch_embed_tokens(ids, e->wte, e->wpe, e->state, e->d_x, e->cur_batch, d.hidden, d.vocab, d.n_positions, st);
    ensure_flow_tiles(e, st);
    FlowLaunch m = flow_launch_desc(e, e->cur_batch);
    m.nsteps = 1; m.step0 = e->flow_epoch; m.cur_len0 = e->host_cur_len; m.first_plain = 1; m.do_select = 0;
    cudaError_t ce = launch_decode_flow(m, st);
    if (ce != cudaSuccess) return fail(e, SV_ERR_CUDA, "dataflow decode launch failed: %s", cudaGetErrorString(ce));
    e->flow_epoch += 1;
    launch_advance_len(e->state, st);
  } else {
    r = e->fused_decode
            ? run_decode_layers_fused(e, ids, e->cur_batch, attention_decode_cluster_ncta(e->host_cur_len + 1), e->use_pdl, st)
            : run_decode_layers(e, ids, e->cur_batch, nsplit_for(e, e->host_cur_len + 1), st);
    if (r != SV_OK) return r;
    launch_advance_len(e->state, st);
  }
  if (logits) launch_logits_to_float(e->logits, logits, (int64_t)e->cur_batch * e->d.vocab, st);
  SV_CK(e, cudaGetLastError());
  e->host_cur_len += 1;
  return SV_OK;
}

int sv_extend(sv_engine* e, const int32_t* ids, int32_t T, float* logits, int32_t keep, float* logps, float temperature,
              void* stream) {
  if (!e || !ids) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->prefilled)
    return fail(e, SV_ERR_STATE, "sv_extend needs sv_prefill / sv_prefill_embeds first (a finished generation cannot be extended)");
  const sv_model_desc& d = e->d;
  if (T < 1 || e->host_cur_len + T + 1 > d.max_len)
    return fail(e, SV_ERR_INVALID, "T = %d outside [1, %d] (%d tokens cached, max_len %d)", T, d.max_len - e->host_cur_len - 1,
                e->host_cur_len, d.max_len);
  if (keep < 0 || keep > T) return fail(e, SV_ERR_INVALID, "keep = %d outside [0, T = %d]", keep, T);
  if (keep > 0 && !logits) return fail(e, SV_ERR_INVALID, "keep = %d needs a logits buffer", keep);
  if (!(temperature > 0.f) || !std::isfinite(temperature)) return fail(e, SV_ERR_INVALID, "temperature must be a finite value > 0");
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  if (!e->s_x) {
    const int64_t R = kScoreRows;
    bool ok = true;
#define SAL(ptr, n) ok = ok && (dev_alloc(e, &e->ptr, (n)) == cudaSuccess)
    SAL(s_x, R * d.hidden); SAL(s_ln, R * d.hidden); SAL(s_qkv, R * e->qkv_cols); SAL(s_attn, R * d.hidden);
    SAL(s_h, R * d.n_inner); SAL(s_part, R * lm_head_logps_ntiles(d.vocab)); SAL(s_tlogit, R);
    SAL(s_tgt, R); SAL(s_lg_row, R); SAL(s_lp_idx, R);
#undef SAL
    if (!ok) { e->s_x = nullptr; return fail(e, SV_ERR_CUDA, "allocation of the scoring workspaces failed: %s", cudaGetErrorString(cudaGetLastError())); }
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int B = e->cur_batch, V = d.vocab, C = kScoreRows / B;
  const float inv_temp = 1.0f / temperature;
  if (logps) launch_row_logp(e->logits, V, B, ids, T, inv_temp, logps, T, st);    // token 0: the logits held before the call
  for (int t0 = 0; t0 < T; t0 += C) {
    const int r = run_extend_chunk(e, ids, T, t0, std::min(C, T - t0), e->host_cur_len + t0, keep, logits, logps, inv_temp, st);
    if (r != SV_OK) return r;
  }
  // the call's last position becomes the held last-position logits (bf16-exact fp32 values -> bf16)
  if (keep > 0) launch_float_rows_to_bf16(logits + (int64_t)(keep - 1) * V, (int64_t)keep * V, e->logits, B, V, st);
  else launch_float_rows_to_bf16(e->logits_f32, V, e->logits, B, V, st);
  const int32_t len = e->host_cur_len + T;
  SV_CK(e, cudaMemcpyAsync(&e->state->cur_len, &len, sizeof(len), cudaMemcpyHostToDevice, st));   // pageable: staged synchronously
  SV_CK(e, cudaStreamSynchronize(st));
  SV_CK(e, cudaGetLastError());
  e->host_cur_len = len;
  return SV_OK;
}

// The generate loop.  `cb` (optional) receives the new tokens of every row each time the host polls the device
// (sv_generate_stream); with cb == NULL the code path is exactly sv_generate's.
static int generate_impl(sv_engine* e, const sv_gen_params* p, int32_t* out_ids, int32_t* out_len, void* stream,
                         sv_token_callback cb, void* cb_user) {
  if (!e || !p || !out_ids) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(e, SV_ERR_STATE, "sv_generate needs sv_prefill first");
  if (e->host_cur_len != e->prefix_len) return fail(e, SV_ERR_STATE, "sv_generate must directly follow sv_prefill");
  const int B = e->cur_batch, max_new = p->max_new_tokens;
  if (max_new < 1) return fail(e, SV_ERR_INVALID, "max_new_tokens must be >= 1");
  if (e->prefix_len + max_new > e->d.max_len)
    return fail(e, SV_ERR_INVALID, "prefix %d + max_new_tokens %d exceeds max_len %d", e->prefix_len, max_new, e->d.max_len);
  if (p->n_stop_ids < 0 || p->n_stop_ids > 8) return fail(e, SV_ERR_INVALID, "n_stop_ids outside [0,8]");
  if (p->do_sample && !(p->temperature > 0.f)) return fail(e, SV_ERR_INVALID, "temperature must be > 0");
  if (!(p->repetition_penalty > 0.f)) return fail(e, SV_ERR_INVALID, "repetition_penalty must be > 0");
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t caller = (cudaStream_t)stream, st = e->gen_stream;
  SV_CK(e, cudaEventRecord(e->ev_in, caller));
  SV_CK(e, cudaStreamWaitEvent(st, e->ev_in, 0));

  GenParamsDev hp;
  memset(&hp, 0, sizeof(hp));
  hp.max_new = max_new; hp.do_sample = p->do_sample; hp.eos_id = p->eos_token_id; hp.pad_id = p->pad_token_id;
  hp.n_stop = p->n_stop_ids;
  for (int i = 0; i < p->n_stop_ids; ++i) hp.stop_ids[i] = p->stop_ids[i];
  hp.stop_row0_only = p->stop_row0_only; hp.out_stride = e->d.max_len;
  hp.temperature = p->temperature; hp.top_p = p->top_p; hp.rep_penalty = p->repetition_penalty; hp.seed = p->seed;
  SV_CK(e, cudaMemcpyAsync(e->params, &hp, sizeof(hp), cudaMemcpyHostToDevice, st));
  SV_CK(e, cudaMemsetAsync(e->seen, 0, (size_t)B * e->d.vocab, st));
  launch_fill_i32(e->out_ids, p->pad_token_id, B * e->d.max_len, st);

  // token 0 comes from the prefill logits.  Greedy on the fused path: one kernel selects, applies the
  // HF stop rules and embeds the token for the first decode step.
  const bool fused = e->fused_decode;
  const bool fused_select = fused && !p->do_sample;
  const int ntiles = gemv_ring_ntiles(e->d.vocab);
  auto select_step = [&](int advance_len, bool have_partials, bool pdl) {
    if (fused_select) {
      launch_select_fused(e->logits, e->d.vocab, B, have_partials ? e->amax_val : nullptr, e->amax_idx, ntiles, e->state,
                          e->params, e->seen, e->next_ids, e->out_ids, advance_len, e->wte, e->wpe, e->d_x, e->d.hidden,
                          e->d.n_positions, pdl, st);
    } else {
      launch_select(e, B, p->do_sample, st);
      launch_gen_finalize(e->state, e->params, B, advance_len, st);
    }
  };
  select_step(/*advance_len=*/0, /*have_partials=*/false, /*pdl=*/false);

  const int nsplit = fused ? attention_decode_cluster_ncta(e->prefix_len + max_new) : nsplit_for(e, e->prefix_len + max_new);
  const long long key = (long long)B * 100000 + nsplit * 8 + (p->do_sample ? 1 : 0) + (fused ? 2 : 0) + (e->use_pdl ? 4 : 0);
  GraphEntry& ge = e->graphs[key];
  const bool flow = e->use_flow && fused_select;
  if (!ge.exec && max_new > 1 && !flow) {
    for (int attempt = 0; attempt < 2 && !ge.exec; ++attempt) {
      const bool pdl = e->use_pdl && fused && attempt == 0;
      int64_t counted = 0;
      g_launch_counter = &counted;
      cudaGraph_t graph = nullptr;
      SV_CK(e, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      int r;
      if (fused) r = run_decode_layers_fused(e, fused_select ? nullptr : e->next_ids, B, nsplit, pdl, st);
      else r = run_decode_layers(e, e->next_ids, B, nsplit, st);
      select_step(/*advance_len=*/1, /*have_partials=*/fused, pdl);
      cudaError_t ce = cudaStreamEndCapture(st, &graph);
      g_launch_counter = &e->launches;
      if (r != SV_OK) { if (graph) cudaGraphDestroy(graph); return r; }
      if (ce == cudaSuccess) ce = cudaGraphInstantiate(&ge.exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        ge.exec = nullptr;
        cudaGetLastError();
        if (!pdl) SV_CK(e, ce);          // plain capture failed: a real error
        e->use_pdl = false;              // programmatic edges refused by this driver: plain stream order
        continue;
      }
      ge.kernels = (int)counted;
    }
  }

  const int poll = p->poll_interval > 0 ? p->poll_interval : 16;
  const bool can_stop = p->eos_token_id >= 0 || p->n_stop_ids > 0;
  // streaming: at every poll, tokens [emitted, step) of every row go to the callback through a pinned staging buffer
  int emitted = 0;
  bool cancelled = false;
  auto emit_upto = [&](int upto) -> int {          // `st` must be idle (synchronised) when this is called
    while (cb && emitted < upto) {
      const int n = std::min(upto - emitted, kStreamChunk);
      if (!e->host_stream) SV_CK(e, cudaMallocHost(reinterpret_cast<void**>(&e->host_stream), (size_t)e->d.max_batch * kStreamChunk * 4));
      SV_CK(e, cudaMemcpy2DAsync(e->host_stream, (size_t)n * 4, e->out_ids + emitted, (size_t)e->d.max_len * 4, (size_t)n * 4, B,
                                 cudaMemcpyDeviceToHost, st));
      SV_CK(e, cudaStreamSynchronize(st));
      if (cb(cb_user, e->host_stream, B, emitted, n) != 0) cancelled = true;
      emitted += n;
    }
    return SV_OK;
  };
  auto poll_device = [&](bool& done_flag) -> int {  // done flag (+ step count when streaming), then the new tokens
    SV_CK(e, cudaMemcpyAsync(e->host_flag, &e->state->step, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));   // {step, done}
    SV_CK(e, cudaStreamSynchronize(st));
    done_flag = e->host_flag[1] != 0;
    const int r = emit_upto(std::min(e->host_flag[0], max_new));
    if (cancelled) done_flag = true;
    return r;
  };
  SV_CK(e, cudaEventRecord(e->ev_t0, st));
  int steps = 0;
  bool done = false;
  if (flow) {
    // dataflow persistent kernel: up to `chunk` whole tokens per cooperative launch, no host work in between
    const int chunk = (can_stop || cb) ? poll : 512;
    ensure_flow_tiles(e, st);
    FlowLaunch m = flow_launch_desc(e, B);
    m.do_select = 1;
    if (e->mega_debug) cudaMemsetAsync(e->mega_dbg, 0, 8192 * sizeof(long long), st);
    int left = max_new - 1;
    bool first = true;
    while (left > 0 && !done) {
      m.nsteps = std::min(left, chunk);
      m.step0 = e->flow_epoch; m.cur_len0 = e->prefix_len + steps; m.first_plain = first ? 1 : 0;
      cudaError_t ce = launch_decode_flow(m, st);
      if (ce != cudaSuccess) return fail(e, SV_ERR_CUDA, "dataflow decode launch failed: %s", cudaGetErrorString(ce));
      first = false;
      m.dbg = nullptr;
      e->flow_epoch += m.nsteps;
      left -= m.nsteps;
      steps += m.nsteps;
      if (cb && left > 0) {
        const int r = poll_device(done);
        if (r != SV_OK) return r;
      } else if (can_stop && left > 0) {
        SV_CK(e, cudaMemcpyAsync(e->host_flag, &e->state->done, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        SV_CK(e, cudaStreamSynchronize(st));
        done = e->host_flag[0] != 0;
      }
    }
  }
  for (int s = 1; s < max_new && !done && !flow; ++s) {
    SV_CK(e, cudaGraphLaunch(ge.exec, st));
    e->launches += ge.kernels;
    ++steps;
    if (cb && (s % poll == 0)) {
      const int r = poll_device(done);
      if (r != SV_OK) return r;
    } else if (can_stop && (s % poll == 0)) {
      SV_CK(e, cudaMemcpyAsync(e->host_flag, &e->state->done, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      SV_CK(e, cudaStreamSynchronize(st));
      done = e->host_flag[0] != 0;
    }
  }
  SV_CK(e, cudaEventRecord(e->ev_t1, st));
  // rectangular result: [B, n_generated] new tokens, padded (HF returns the same rectangle)
  SV_CK(e, cudaMemcpyAsync(e->host_flag, &e->state->step, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  SV_CK(e, cudaStreamSynchronize(st));
  const int n_gen = std::min(e->host_flag[0], max_new);
  if (cb) {
    const int r = emit_upto(n_gen);
    if (r != SV_OK) return r;
  }
  SV_CK(e, cudaMemcpy2DAsync(out_ids, (size_t)max_new * 4, e->out_ids, (size_t)e->d.max_len * 4, (size_t)max_new * 4, B,
                             cudaMemcpyDeviceToDevice, st));
  if (out_len) launch_fill_i32(out_len, n_gen, B, st);
  SV_CK(e, cudaStreamSynchronize(st));
  SV_CK(e, cudaGetLastError());
  SV_CK(e, cudaEventElapsedTime(&e->last_decode_ms, e->ev_t0, e->ev_t1));
  e->last_decode_steps = steps;
  e->host_cur_len = e->prefix_len + std::max(0, n_gen - 1);
  e->prefilled = false;   // the cache now holds a finished generation; a new prefill is required
  return SV_OK;
}

int sv_generate(sv_engine* e, const sv_gen_params* p, int32_t* out_ids, int32_t* out_len, void* stream) {
  return generate_impl(e, p, out_ids, out_len, stream, nullptr, nullptr);
}

int sv_generate_stream(sv_engine* e, const sv_gen_params* p, int32_t* out_ids, int32_t* out_len, sv_token_callback on_tokens,
                       void* user, void* stream) {
  if (!on_tokens) return fail(e, SV_ERR_INVALID, "sv_generate_stream needs a callback (use sv_generate otherwise)");
  return generate_impl(e, p, out_ids, out_len, stream, on_tokens, user);
}

int sv_generate_im2svg_host(sv_engine* e, const void* pixels_host, int32_t batch, const int32_t* prompt_ids_host,
                            int32_t prompt_len, const sv_gen_params* p, int32_t* out_ids_host, int32_t* out_len_host,
                            void* stream) {
  if (!e || !pixels_host || !prompt_ids_host || !p || !out_ids_host) return fail(e, SV_ERR_INVALID, "null argument");
  if (batch < 1 || batch > e->d.max_batch) return fail(e, SV_ERR_INVALID, "batch %d outside [1,%d]", batch, e->d.max_batch);
  if (prompt_len < 1 || prompt_len > kMaxPrompt) return fail(e, SV_ERR_INVALID, "prompt_len outside [1,%d]", kMaxPrompt);
  SV_CK(e, cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (p->max_new_tokens < 1 || p->max_new_tokens > e->d.max_len)
    return fail(e, SV_ERR_INVALID, "max_new_tokens %d outside [1,%d]", p->max_new_tokens, e->d.max_len);
  const size_t px_bytes = (size_t)batch * 3 * e->d.image_size * e->d.image_size * 2;
  // device staging of the host entry point: one allocation for the engine's lifetime (no cudaMalloc / cudaFree per call)
  if (!e->im2svg_px && dev_alloc(e, &e->im2svg_px, (int64_t)e->d.max_batch * 3 * e->d.image_size * e->d.image_size) != cudaSuccess)
    return fail(e, SV_ERR_CUDA, "allocation of the pixel staging buffer failed: %s", cudaGetErrorString(cudaGetLastError()));
  if (!e->im2svg_out && dev_alloc(e, &e->im2svg_out, (int64_t)e->d.max_batch * (e->d.max_len + 1)) != cudaSuccess)
    return fail(e, SV_ERR_CUDA, "allocation of the output staging buffer failed: %s", cudaGetErrorString(cudaGetLastError()));
  bf16* px = e->im2svg_px;
  int32_t* dout = e->im2svg_out;
  int32_t* dlen = dout + (size_t)batch * p->max_new_tokens;
  int r = SV_OK;
  cudaError_t ce = cudaMemcpyAsync(px, pixels_host, px_bytes, cudaMemcpyHostToDevice, st);
  if (ce == cudaSuccess) ce = cudaMemcpyAsync(e->ids_tmp, prompt_ids_host, (size_t)batch * prompt_len * 4, cudaMemcpyHostToDevice, st);
  if (ce != cudaSuccess) r = fail(e, SV_ERR_CUDA, "H2D copy failed: %s", cudaGetErrorString(ce));
  if (r == SV_OK) r = sv_encode_images(e, px, batch, nullptr, nullptr, stream);
  if (r == SV_OK) r = sv_prefill(e, e->ids_tmp, batch, prompt_len, nullptr, stream);
  if (r == SV_OK) r = sv_generate(e, p, dout, dlen, stream);
  if (r == SV_OK) {
    ce = cudaMemcpyAsync(out_ids_host, dout, (size_t)batch * p->max_new_tokens * 4, cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess && out_len_host) ce = cudaMemcpyAsync(out_len_host, dlen, (size_t)batch * 4, cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
    if (ce != cudaSuccess) r = fail(e, SV_ERR_CUDA, "D2H copy failed: %s", cudaGetErrorString(ce));
  }
  cudaStreamSynchronize(st);
  return r;
}

// Beam search with the whole loop on the device.  Graph body = one decode step over the batch * num_beams cache rows, then
// candidates -> bookkeeping (+ next-token embeddings) -> KV suffix copies; the host replays it and polls `done`.
int sv_beam_search(sv_engine* e, const sv_beam_params* bp, int32_t batch, int32_t* out_ids, int32_t* out_len, void* stream) {
  if (!e || !bp || !out_ids) return fail(e, SV_ERR_INVALID, "null argument");
  if (sv_beam_params_check(bp, batch) != SV_OK)
    return fail(e, SV_ERR_INVALID, "bad beam parameters (need num_beams >= 2, batch * num_beams <= 8, max_new_tokens >= 1, "
                                   "n_stop_ids in [0,8], early_stopping in {0,1,2}, temperature > 0, repetition_penalty > 0)");
  if (!e->prefilled) return fail(e, SV_ERR_STATE, "sv_beam_search needs sv_prefill first");
  if (e->host_cur_len != e->prefix_len) return fail(e, SV_ERR_STATE, "sv_beam_search must directly follow sv_prefill");
  const sv_model_desc& d = e->d;
  const int nb = bp->num_beams, R = batch * nb, max_new = bp->max_new_tokens, K = 2 * nb;
  if (R != e->cur_batch) return fail(e, SV_ERR_STATE, "prefilled rows %d != batch %d x num_beams %d", e->cur_batch, batch, nb);
  if (e->prefix_len + max_new > d.max_len)
    return fail(e, SV_ERR_INVALID, "prefix %d + max_new_tokens %d exceeds max_len %d", e->prefix_len, max_new, d.max_len);
  SV_CK(e, cudaSetDevice(e->device));
  if (beam_init(d.vocab) != cudaSuccess) {
    cudaGetLastError();
    return fail(e, SV_ERR_UNSUPPORTED, "a logits row of %d entries does not fit the SM's shared memory: use the host-stepped beam loop", d.vocab);
  }
  LaunchScope scope(e);
  const int stride = d.max_len;
  if (!e->beam_state) {
    bool ok = true;
    const int MR = svbeam::kMaxRows, MK = svbeam::kMaxK;
#define BAL(ptr, n) ok = ok && (dev_alloc(e, &e->ptr, (n)) == cudaSuccess)
    BAL(beam_params, 1); BAL(beam_state, 1); BAL(beam_plan, 1);
    BAL(beam_key, MR * MK); BAL(beam_val, MR * MK); BAL(beam_tok, MR * MK);
    BAL(beam_run_seq, (int64_t)2 * MR * stride); BAL(beam_fin_seq, (int64_t)2 * MR * stride);
    BAL(kstage, e->cache_layer_stride * d.n_layer); BAL(vstage, e->cache_layer_stride * d.n_layer);
#undef BAL
    if (!ok) { e->beam_state = nullptr; return fail(e, SV_ERR_CUDA, "allocation of the beam-search state failed: %s", cudaGetErrorString(cudaGetLastError())); }
  }
  cudaStream_t caller = (cudaStream_t)stream, st = e->gen_stream;
  SV_CK(e, cudaEventRecord(e->ev_in, caller));
  SV_CK(e, cudaStreamWaitEvent(st, e->ev_in, 0));

  svbeam::Params hp;
  memset(&hp, 0, sizeof(hp));
  hp.B = batch; hp.nb = nb; hp.K = K; hp.vocab = d.vocab; hp.max_length = max_new; hp.eos_id = bp->eos_token_id;
  hp.pad_id = bp->pad_token_id;
  hp.n_stop = bp->n_stop_ids;
  for (int i = 0; i < bp->n_stop_ids; ++i) hp.stop_ids[i] = bp->stop_ids[i];
  hp.do_sample = bp->do_sample; hp.early_stopping = bp->early_stopping;
  hp.min_keep = std::max(2, 1 + (bp->eos_token_id >= 0 ? 1 : 0));
  hp.seq_stride = stride;
  hp.temperature = bp->temperature; hp.top_p = bp->top_p; hp.rep_penalty = bp->repetition_penalty;
  hp.length_penalty = bp->length_penalty; hp.seed = bp->seed;
  svbeam::State hs;
  memset(&hs, 0, sizeof(hs));
  svbeam::init_state(hp, hs, e->prefix_len);
  SV_CK(e, cudaMemcpyAsync(e->beam_params, &hp, sizeof(hp), cudaMemcpyHostToDevice, st));   // pageable: staged synchronously
  SV_CK(e, cudaMemcpyAsync(e->beam_state, &hs, sizeof(hs), cudaMemcpyHostToDevice, st));
  SV_CK(e, cudaMemsetAsync(e->beam_plan, 0, sizeof(svbeam::Plan), st));
  launch_fill_i32(e->beam_run_seq, bp->pad_token_id, 2 * R * stride, st);
  launch_fill_i32(e->beam_fin_seq, bp->pad_token_id, 2 * R * stride, st);

  const bool fused = e->fused_decode;
  auto bookkeeping = [&](int advance) {
    launch_beam_candidates(e->logits, d.vocab, R, e->beam_params, e->beam_state, e->beam_run_seq, e->beam_key, e->beam_val,
                           e->beam_tok, st);
    launch_beam_step(e->beam_params, e->beam_state, e->beam_plan, e->beam_key, e->beam_val, e->beam_tok, e->beam_run_seq,
                     e->beam_fin_seq, e->state, advance, e->wte, e->wpe, e->d_x, d.hidden, d.n_positions, e->next_ids, st);
    launch_beam_kv_copy(e->kcache, e->vtcache, e->kstage, e->vstage, e->cache_layer_stride, d.n_layer, R, d.n_kv_head,
                        e->tcap, d.head_dim, e->beam_plan, st);
  };
  bookkeeping(/*advance=*/0);                       // step 0: candidates from the prefill logits

  const int nsplit = fused ? attention_decode_cluster_ncta(e->prefix_len + max_new) : nsplit_for(e, e->prefix_len + max_new);
  const long long key = (long long)R * 100000 + nsplit * 8 + (fused ? 2 : 0) + (e->use_pdl ? 4 : 0);
  GraphEntry& ge = e->beam_graphs[key];
  if (!ge.exec && max_new > 1) {
    for (int attempt = 0; attempt < 2 && !ge.exec; ++attempt) {
      const bool pdl = e->use_pdl && fused && attempt == 0;
      int64_t counted = 0;
      g_launch_counter = &counted;
      cudaGraph_t graph = nullptr;
      SV_CK(e, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      int r;
      if (fused) r = run_decode_layers_fused(e, nullptr, R, nsplit, pdl, st);
      else r = run_decode_layers(e, e->next_ids, R, nsplit, st);
      bookkeeping(/*advance=*/1);
      cudaError_t ce = cudaStreamEndCapture(st, &graph);
      g_launch_counter = &e->launches;
      if (r != SV_OK) { if (graph) cudaGraphDestroy(graph); return r; }
      if (ce == cudaSuccess) ce = cudaGraphInstantiate(&ge.exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {
        ge.exec = nullptr;
        cudaGetLastError();
        if (!pdl) SV_CK(e, ce);
        e->use_pdl = false;
        continue;
      }
      ge.kernels = (int)counted;
    }
  }
  const int poll = bp->poll_interval > 0 ? bp->poll_interval : 16;
  SV_CK(e, cudaEventRecord(e->ev_t0, st));
  int steps = 0;
  bool done = false;
  for (int s = 1; s < max_new && !done; ++s) {
    SV_CK(e, cudaGraphLaunch(ge.exec, st));
    e->launches += ge.kernels;
    ++steps;
    if (s % poll == 0) {
      SV_CK(e, cudaMemcpyAsync(e->host_flag, &e->beam_state->done, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      SV_CK(e, cudaStreamSynchronize(st));
      done = e->host_flag[0] != 0;
    }
  }
  SV_CK(e, cudaEventRecord(e->ev_t1, st));
  SV_CK(e, cudaMemcpyAsync(&hs, e->beam_state, sizeof(hs), cudaMemcpyDeviceToHost, st));
  SV_CK(e, cudaStreamSynchronize(st));
  SV_CK(e, cudaGetLastError());
  if (!hs.done) return fail(e, SV_ERR_STATE, "beam search did not terminate within max_new_tokens steps (internal error)");
  int n_gen = 0;
  for (int b = 0; b < batch; ++b) n_gen = std::max(n_gen, hs.fin_len[b * nb]);     // HF: max_generated over the best beams
  n_gen = std::min(n_gen, max_new);
  launch_fill_i32(out_ids, bp->pad_token_id, batch * max_new, st);
  // best hypothesis of image b = finished slot 0 = row b * nb of the live half of fin_seq
  SV_CK(e, cudaMemcpy2DAsync(out_ids, (size_t)max_new * 4, e->beam_fin_seq + ((int64_t)hs.parity * R) * stride, (size_t)nb * stride * 4,
                             (size_t)std::max(n_gen, 1) * 4, batch, cudaMemcpyDeviceToDevice, st));
  if (out_len) launch_fill_i32(out_len, n_gen, batch, st);
  SV_CK(e, cudaStreamSynchronize(st));
  SV_CK(e, cudaGetLastError());
  SV_CK(e, cudaEventElapsedTime(&e->last_decode_ms, e->ev_t0, e->ev_t1));
  e->last_decode_steps = steps;
  e->host_cur_len = e->prefix_len + hs.cur_len;
  e->prefilled = false;
  return SV_OK;
}

int sv_reorder_cache(sv_engine* e, const int32_t* src_rows, void* stream) {
  if (!e || !src_rows) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->prefilled) return fail(e, SV_ERR_STATE, "sv_reorder_cache needs a prefilled cache");
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  const sv_model_desc& d = e->d;
  const int B = e->cur_batch, len = e->host_cur_len;
  for (int i = 0; i < d.n_layer; ++i) {
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    launch_kv_gather(kc, vc, e->kscratch, e->vscratch, src_rows, B, d.n_kv_head, e->tcap, d.head_dim, len, st);
    launch_kv_gather(e->kscratch, e->vscratch, kc, vc, nullptr, B, d.n_kv_head, e->tcap, d.head_dim, len, st);
  }
  SV_CK(e, cudaGetLastError());
  return SV_OK;
}

int sv_expand_batch(sv_engine* e, const int32_t* src_rows_host, int32_t new_batch, void* stream) {
  if (!e || !src_rows_host) return fail(e, SV_ERR_INVALID, "null argument");
  if (!e->prefilled || e->host_cur_len != e->prefix_len) return fail(e, SV_ERR_STATE, "sv_expand_batch must directly follow sv_prefill");
  if (new_batch < 1 || new_batch > e->d.max_batch) return fail(e, SV_ERR_INVALID, "new_batch %d outside [1,%d]", new_batch, e->d.max_batch);
  for (int r = 0; r < new_batch; ++r)
    if (src_rows_host[r] < 0 || src_rows_host[r] >= e->cur_batch) return fail(e, SV_ERR_INVALID, "src_rows[%d] = %d is not a prefilled row", r, src_rows_host[r]);
  SV_CK(e, cudaSetDevice(e->device));
  LaunchScope scope(e);
  cudaStream_t st = (cudaStream_t)stream;
  const sv_model_desc& d = e->d;
  const int len = e->host_cur_len;
  SV_CK(e, cudaMemcpyAsync(e->ids_tmp, src_rows_host, (size_t)new_batch * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  for (int i = 0; i < d.n_layer; ++i) {          // cache rows: gather through the one-layer scratch (as sv_reorder_cache)
    bf16* kc = e->kcache + e->cache_layer_stride * i;
    bf16* vc = e->vtcache + e->cache_layer_stride * i;
    launch_kv_gather(kc, vc, e->kscratch, e->vscratch, e->ids_tmp, new_batch, d.n_kv_head, e->tcap, d.head_dim, len, st);
    launch_kv_gather(e->kscratch, e->vscratch, kc, vc, nullptr, new_batch, d.n_kv_head, e->tcap, d.head_dim, len, st);
  }
  // the prefill's last-position logits (token 0 is selected from them) and the last hidden row, staged through logits_f32
  const size_t row = (size_t)d.vocab * sizeof(bf16);
  uint8_t* stage = reinterpret_cast<uint8_t*>(e->logits_f32);
  for (int r = 0; r < new_batch; ++r)
    SV_CK(e, cudaMemcpyAsync(stage + r * row, reinterpret_cast<uint8_t*>(e->logits) + src_rows_host[r] * row, row, cudaMemcpyDeviceToDevice, st));
  SV_CK(e, cudaMemcpyAsync(e->logits, stage, new_batch * row, cudaMemcpyDeviceToDevice, st));
  e->cur_batch = new_batch;
  return finish_prefill_impl(e, new_batch, e->prefix_len, nullptr, st);     // fresh GenState for the new rows, exchange buffers cleared
}

int64_t sv_launch_count(const sv_engine* e) { return e ? e->launches : 0; }

int sv_debug_read_timeline(sv_engine* e, long long* out_host, int32_t n) {
  if (!e || !out_host || n < 1 || n > 8192) return SV_ERR_INVALID;
  cudaError_t r = cudaMemcpy(out_host, e->mega_dbg, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost);
  return r == cudaSuccess ? SV_OK : SV_ERR_CUDA;
}

const char* sv_engine_describe(sv_engine* e) {
  if (!e) return "";
  char buf[512];
  snprintf(buf, sizeof(buf), "decode=%s weights=%s attn=cluster-dsmem pdl=%d linear_impl=%d flow[%s]",
           !e->fused_decode ? "legacy-kernels" : e->use_flow ? (e->flow_realloc ? "dataflow-kernel-setmaxnreg" : "dataflow-kernel") : "ring-gemv-graph",
           e->ring_tiles ? "slab-tiled" : "row-major", (int)e->use_pdl, e->linear_impl, decode_flow_status());
  e->describe = buf;
  return e->describe.c_str();
}

int sv_last_decode_timing(const sv_engine* e, float* ms, int32_t* steps) {
  if (!e) return SV_ERR_INVALID;
  if (ms) *ms = e->last_decode_ms;
  if (steps) *steps = e->last_decode_steps;
  return SV_OK;
}

// ---- single-kernel entry points ---------------------------------------------------------------
static std::string g_op_error;
static int op_fail(const char* what, cudaError_t r) {
  g_create_error = std::string(what) + ": " + cudaGetErrorString(r);
  return SV_ERR_CUDA;
}

int sv_op_layernorm(const void* x, const void* w, const void* b, void* y, int32_t rows, int32_t cols, float eps,
                    void* stream) {
  if (!x || !w || !b || !y || cols % 8) return fail(nullptr, SV_ERR_INVALID, "bad layernorm arguments");
  launch_layernorm((const bf16*)x, (const bf16*)w, (const bf16*)b, (bf16*)y, rows, cols, eps, cols, (cudaStream_t)stream);
  cudaError_t r = cudaGetLastError();
  return r == cudaSuccess ? SV_OK : op_fail("layernorm", r);
}

int sv_op_linear(int32_t impl, const void* x, const void* w, const void* bias, const void* residual, void* y, int32_t M,
                 int32_t N, int32_t K, int32_t act, void* stream) {
  if (!x || !w || !y || M < 1 || N < 1 || K < 32) return fail(nullptr, SV_ERR_INVALID, "bad linear arguments");
  int r = do_linear(nullptr, impl, (const bf16*)x, (const bf16*)w, (const bf16*)bias, (const bf16*)residual, (bf16*)y, M,
                    N, K, act, (cudaStream_t)stream);
  if (r != SV_OK) return r;
  cudaError_t ce = cudaGetLastError();
  return ce == cudaSuccess ? SV_OK : op_fail("linear", ce);
}

int sv_op_attention_vit(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t heads, void* stream) {
  if (!qkv || !out || batch < 1 || seq < 1 || heads < 1) return fail(nullptr, SV_ERR_INVALID, "bad attention arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int seq_pad = (seq + 31) / 32 * 32;
  bf16* vt = nullptr;
  cudaError_t r = cudaMalloc(reinterpret_cast<void**>(&vt), (size_t)batch * heads * 64 * seq_pad * 2);
  if (r != cudaSuccess) return op_fail("attention_vit alloc", r);
  launch_vit_transpose_v((const bf16*)qkv, vt, batch, seq, heads, seq_pad, st);
  launch_attention_vit((const bf16*)qkv, vt, (bf16*)out, batch, seq, heads, seq_pad, st);
  r = cudaStreamSynchronize(st);
  cudaFree(vt);
  return r == cudaSuccess ? SV_OK : op_fail("attention_vit", r);
}

int sv_op_attention_mqa(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t heads, void* stream) {
  if (!qkv || !out || batch < 1 || seq < 1 || heads < 1 || heads > 16) return fail(nullptr, SV_ERR_INVALID, "bad attention arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int D = 128, tcap = (seq + 31) / 32 * 32;
  const size_t n = (size_t)batch * tcap * D;
  bf16* kc = nullptr;
  cudaError_t r = cudaMalloc(reinterpret_cast<void**>(&kc), 2 * n * 2);
  if (r != cudaSuccess) return op_fail("attention_mqa alloc", r);
  bf16* vc = kc + n;
  cudaMemsetAsync(kc, 0, 2 * n * 2, st);
  launch_kv_scatter((const bf16*)qkv, kc, vc, batch, seq, heads * D, 1, D, tcap, 0, st);
  launch_attention_heads((const bf16*)qkv, heads * D + 2 * D, kc, vc, (bf16*)out, batch, seq, heads, 1, D, tcap, 0, 0, st);
  r = cudaStreamSynchronize(st);
  cudaFree(kc);
  return r == cudaSuccess ? SV_OK : op_fail("attention_mqa", r);
}

int sv_op_attention_prefill(const void* qkv, void* out, int32_t batch, int32_t seq, int32_t n_head, int32_t n_kv,
                            int32_t window, void* stream) {
  if (!qkv || !out || batch < 1 || seq < 1 || n_kv < 1 || n_head < n_kv || n_head % n_kv || n_head / n_kv > 16 || window < 0)
    return fail(nullptr, SV_ERR_INVALID, "bad attention_prefill arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int D = 128, tcap = (seq + 31) / 32 * 32, cols = (n_head + 2 * n_kv) * D;
  const size_t n = (size_t)batch * n_kv * tcap * D;
  bf16* kc = nullptr;
  cudaError_t r = cudaMalloc(reinterpret_cast<void**>(&kc), 2 * n * 2);
  if (r != cudaSuccess) return op_fail("attention_prefill alloc", r);
  bf16* vc = kc + n;
  cudaMemsetAsync(kc, 0, 2 * n * 2, st);
  launch_kv_scatter((const bf16*)qkv, kc, vc, batch, seq, n_head * D, n_kv, D, tcap, 0, st);
  launch_attention_heads((const bf16*)qkv, cols, kc, vc, (bf16*)out, batch, seq, n_head, n_kv, D, tcap, window, 0, st);
  r = cudaStreamSynchronize(st);
  cudaFree(kc);
  return r == cudaSuccess ? SV_OK : op_fail("attention_prefill", r);
}

// Scratch of the decode-step entry points: one allocation, freed on every path out.
namespace {
struct OpScratch {
  void* p = nullptr;
  ~OpScratch() { if (p) cudaFree(p); }
};
GenState op_state(int cur_len, int step) {
  GenState hs;
  memset(&hs, 0, sizeof(hs));
  hs.cur_len = cur_len;
  hs.step = step;
  for (int b = 0; b < 8; ++b) hs.unfinished[b] = 1;
  return hs;
}
}  // namespace

int sv_op_attention_decode(int32_t impl, const void* q, const void* kcache, const void* vtcache, void* out, int32_t batch,
                           int32_t n_head, int32_t n_kv, int32_t tcap, int32_t nkeys, int32_t window, int32_t nparts,
                           void* stream) {
  if (!q || !kcache || !vtcache || !out) return fail(nullptr, SV_ERR_INVALID, "attention_decode: null pointer");
  if (impl != SV_ATTN_DECODE_CLUSTER && impl != SV_ATTN_DECODE_SPLIT) return fail(nullptr, SV_ERR_INVALID, "attention_decode: unknown impl %d", impl);
  if (batch < 1 || batch > 8) return fail(nullptr, SV_ERR_INVALID, "attention_decode: batch %d not in [1,8]", batch);
  if (n_kv < 1 || n_head < n_kv || n_head % n_kv || n_head / n_kv > 16)
    return fail(nullptr, SV_ERR_INVALID, "attention_decode: need n_head %% n_kv == 0 and a group of 1..16");
  if (tcap < 32 || tcap % 32) return fail(nullptr, SV_ERR_INVALID, "attention_decode: tcap %d must be a positive multiple of 32", tcap);
  if (nkeys < 1 || nkeys > tcap) return fail(nullptr, SV_ERR_INVALID, "attention_decode: nkeys %d not in [1, tcap=%d]", nkeys, tcap);
  if (window < 0) return fail(nullptr, SV_ERR_INVALID, "attention_decode: window < 0");
  const int max_parts = impl == SV_ATTN_DECODE_CLUSTER ? 8 : kMaxSplit;
  if (nparts < 0 || nparts > max_parts) return fail(nullptr, SV_ERR_INVALID, "attention_decode: %d parts not in [0,%d]", nparts, max_parts);
  if (nparts == 0)   // the engine's choice for this length
    nparts = impl == SV_ATTN_DECODE_CLUSTER ? attention_decode_cluster_ncta(nkeys) : std::max(1, std::min(kMaxSplit, (nkeys + 31) / 32));
  cudaStream_t st = (cudaStream_t)stream;
  const int D = 128;
  const size_t part_bytes = impl == SV_ATTN_DECODE_SPLIT ? (size_t)batch * n_kv * nparts * (32 + 16 * D) * sizeof(float) : 0;
  OpScratch s;
  cudaError_t r = cudaMalloc(&s.p, sizeof(GenState) + part_bytes);
  if (r != cudaSuccess) return op_fail("attention_decode alloc", r);
  GenState* state = reinterpret_cast<GenState*>(s.p);
  const GenState hs = op_state(nkeys - 1, 0);      // the kernels attend over keys [.., cur_len] = the new token's own K/V
  r = cudaMemcpyAsync(state, &hs, sizeof(hs), cudaMemcpyHostToDevice, st);
  if (r != cudaSuccess) return op_fail("attention_decode state", r);
  if (impl == SV_ATTN_DECODE_CLUSTER) {
    r = attention_decode_cluster_init();
    if (r == cudaSuccess)
      r = launch_attention_decode_cluster((const bf16*)q, n_head * D, (const bf16*)kcache, (const bf16*)vtcache, (bf16*)out,
                                          state, batch, n_head, n_kv, D, tcap, nparts, window, false, st);
  } else {
    float* part = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s.p) + sizeof(GenState));
    launch_attention_decode((const bf16*)q, n_head * D, (const bf16*)kcache, (const bf16*)vtcache, (bf16*)out, part, state,
                            batch, n_head, n_kv, D, tcap, nparts, window, st);
  }
  if (r == cudaSuccess) r = cudaGetLastError();
  if (r == cudaSuccess) r = cudaStreamSynchronize(st);
  return r == cudaSuccess ? SV_OK : op_fail("attention_decode", r);
}

int sv_op_gemv_ring(const void* x, const void* w, const void* bias, const void* residual, const void* ln_w, const void* ln_b,
                    void* y, int32_t batch, int32_t N, int32_t K, int32_t act, float ln_eps, int32_t epi, int32_t tiled,
                    void* kcache, void* vtcache, int32_t n_head, int32_t n_kv, int32_t tcap, int32_t pos, float* amax_val,
                    int32_t* amax_idx, int32_t amax_capacity, int32_t* ntiles_out, void* stream) {
  if (!x || !w || !y) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: null pointer");
  if (batch < 1 || batch > 8) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: batch %d not in [1,8]", batch);
  if (N < 1 || K < 32 || K % 32) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: need N >= 1 and K a positive multiple of 32");
  if (act < SV_ACT_NONE || act > SV_ACT_SILU) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: unknown act %d", act);
  if ((ln_w == nullptr) != (ln_b == nullptr)) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: LayerNorm needs both weight and bias");
  if (tiled != 0 && tiled != 1) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: tiled must be 0 or 1");
  const int D = 128;
  const int ntiles = gemv_ring_ntiles(N);
  if (ntiles_out) *ntiles_out = ntiles;
  if (epi == SV_GEMV_EPI_QKV) {
    if (!kcache || !vtcache) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: QKV epilogue needs both caches");
    if (n_kv < 1 || n_head < n_kv || n_head % n_kv || N != (n_head + 2 * n_kv) * D)
      return fail(nullptr, SV_ERR_INVALID, "gemv_ring: QKV epilogue needs N == (n_head + 2*n_kv)*128");
    if (tcap < 1 || pos < 0 || pos >= tcap) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: pos %d not in [0, tcap=%d)", pos, tcap);
  } else if (epi == SV_GEMV_EPI_LMHEAD) {
    if (!amax_val || !amax_idx) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: lm_head epilogue needs the partial buffers");
    if (amax_capacity < ntiles) return fail(nullptr, SV_ERR_INVALID, "gemv_ring: %d partial tiles needed, capacity %d", ntiles, amax_capacity);
  } else if (epi != SV_GEMV_EPI_PLAIN) {
    return fail(nullptr, SV_ERR_INVALID, "gemv_ring: unknown epilogue %d", epi);
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int ncta = gemv_ring_ncta();
  const size_t tile_bytes = tiled ? flow_tiled_bytes(N, K, ncta) : 0;
  OpScratch s;
  cudaError_t r = cudaMalloc(&s.p, 512 + tile_bytes);
  if (r != cudaSuccess) return op_fail("gemv_ring alloc", r);
  GenState* state = reinterpret_cast<GenState*>(s.p);
  uint8_t* wt = tiled ? reinterpret_cast<uint8_t*>(s.p) + 512 : nullptr;
  const GenState hs = op_state(epi == SV_GEMV_EPI_QKV ? pos : 0, 0);
  r = cudaMemcpyAsync(state, &hs, sizeof(hs), cudaMemcpyHostToDevice, st);
  if (r == cudaSuccess) r = gemv_ring_init();
  if (r != cudaSuccess) return op_fail("gemv_ring setup", r);
  if (tiled) launch_flow_repack((const bf16*)w, (const bf16*)bias, wt, N, K, ncta, st);
  RingGemvLaunch g{};
  g.X = (const bf16*)x; g.W = (const bf16*)w; g.Wt = wt; g.bias = (const bf16*)bias; g.res = (const bf16*)residual;
  g.ln_w = (const bf16*)ln_w; g.ln_b = (const bf16*)ln_b; g.Y = (bf16*)y;
  g.B = batch; g.N = N; g.K = K; g.act = act; g.epi = epi; g.ln_eps = ln_eps;
  g.n_head = n_head; g.n_kv = n_kv; g.tcap = tcap; g.state = state;
  g.kcache = (bf16*)kcache; g.vtcache = (bf16*)vtcache; g.amax_val = amax_val; g.amax_idx = amax_idx; g.pdl = false;
  launch_gemv_ring(g, st);
  r = cudaGetLastError();
  if (r == cudaSuccess) r = cudaStreamSynchronize(st);
  return r == cudaSuccess ? SV_OK : op_fail("gemv_ring", r);
}

int sv_op_select(int32_t mode, const void* logits, const uint8_t* seen, const sv_gen_params* p, int32_t batch, int32_t vocab,
                 int32_t step, int32_t cur_len, const float* amax_val, const int32_t* amax_idx, int32_t ntiles,
                 const void* wte, const void* wpe, int32_t h, int32_t n_positions, void* x_out, int32_t* tokens,
                 void* stream) {
  if (!logits || !seen || !p || !tokens) return fail(nullptr, SV_ERR_INVALID, "select: null pointer");
  if (mode < SV_SELECT_GREEDY || mode > SV_SELECT_SAMPLE) return fail(nullptr, SV_ERR_INVALID, "select: unknown mode %d", mode);
  if (batch < 1 || batch > 8) return fail(nullptr, SV_ERR_INVALID, "select: batch %d not in [1,8]", batch);
  if (vocab < 1 || step < 0 || cur_len < 0) return fail(nullptr, SV_ERR_INVALID, "select: bad vocab / step / cur_len");
  if (p->n_stop_ids < 0 || p->n_stop_ids > 8) return fail(nullptr, SV_ERR_INVALID, "select: n_stop_ids not in [0,8]");
  if (mode == SV_SELECT_SAMPLE && !(p->temperature > 0.f && p->top_p > 0.f && p->top_p <= 1.f))
    return fail(nullptr, SV_ERR_INVALID, "select: sampling needs temperature > 0 and top_p in (0,1]");
  const bool fused = mode == SV_SELECT_FUSED || mode == SV_SELECT_FUSED_PARTIALS;
  if (fused && (!wte || !x_out || h < 8 || h % 8 || (wpe && n_positions < 1)))
    return fail(nullptr, SV_ERR_INVALID, "select: the fused kernel needs wte, x_out and h a multiple of 8");
  if (mode == SV_SELECT_FUSED_PARTIALS && (!amax_val || !amax_idx || ntiles < 1))
    return fail(nullptr, SV_ERR_INVALID, "select: partials mode needs amax_val, amax_idx and ntiles >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  // scratch: GenState | params | out_ids [batch][step + 1] | next_ids [8] | seen copy [batch][vocab] | probs [batch][vocab]
  const size_t off_par = 512, off_out = off_par + 512, out_bytes = (size_t)batch * (step + 1) * 4;
  const size_t off_next = (off_out + out_bytes + 255) / 256 * 256, off_seen = off_next + 256;
  const size_t off_probs = (off_seen + (size_t)batch * vocab + 255) / 256 * 256;
  const size_t bytes = off_probs + (mode == SV_SELECT_SAMPLE ? (size_t)batch * vocab * 4 : 0);
  OpScratch s;
  cudaError_t r = cudaMalloc(&s.p, bytes);
  if (r != cudaSuccess) return op_fail("select alloc", r);
  uint8_t* base = reinterpret_cast<uint8_t*>(s.p);
  GenState* state = reinterpret_cast<GenState*>(base);
  GenParamsDev* par = reinterpret_cast<GenParamsDev*>(base + off_par);
  int32_t* out_ids = reinterpret_cast<int32_t*>(base + off_out);
  int32_t* next_ids = reinterpret_cast<int32_t*>(base + off_next);
  uint8_t* seen_w = base + off_seen;                  // the kernels mark the chosen id: work on a copy
  float* probs = reinterpret_cast<float*>(base + off_probs);
  const GenState hs = op_state(cur_len, step);
  GenParamsDev hp;
  memset(&hp, 0, sizeof(hp));
  hp.max_new = step + 1; hp.do_sample = p->do_sample; hp.eos_id = p->eos_token_id; hp.pad_id = p->pad_token_id;
  hp.n_stop = p->n_stop_ids;
  for (int i = 0; i < p->n_stop_ids; ++i) hp.stop_ids[i] = p->stop_ids[i];
  hp.stop_row0_only = p->stop_row0_only; hp.out_stride = step + 1;
  hp.temperature = p->temperature; hp.top_p = p->top_p; hp.rep_penalty = p->repetition_penalty; hp.seed = p->seed;
  if ((r = cudaMemcpyAsync(state, &hs, sizeof(hs), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (r = cudaMemcpyAsync(par, &hp, sizeof(hp), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (r = cudaMemsetAsync(out_ids, 0xff, out_bytes, st)) != cudaSuccess ||
      (r = cudaMemcpyAsync(seen_w, seen, (size_t)batch * vocab, cudaMemcpyDefault, st)) != cudaSuccess)
    return op_fail("select setup", r);
  if (mode == SV_SELECT_GREEDY)
    launch_select_greedy((const bf16*)logits, vocab, batch, state, par, seen_w, next_ids, out_ids, st);
  else if (mode == SV_SELECT_SAMPLE)
    launch_select_sample((const bf16*)logits, vocab, batch, state, par, seen_w, next_ids, out_ids, probs, st);
  else
    launch_select_fused((const bf16*)logits, vocab, batch, mode == SV_SELECT_FUSED_PARTIALS ? amax_val : nullptr, amax_idx,
                        ntiles, state, par, seen_w, next_ids, out_ids, 1, (const bf16*)wte, (const bf16*)wpe, (bf16*)x_out, h,
                        n_positions, false, st);
  r = cudaGetLastError();
  if (r == cudaSuccess) r = cudaMemcpyAsync(tokens, next_ids, (size_t)batch * 4, cudaMemcpyDefault, st);
  if (r == cudaSuccess) r = cudaStreamSynchronize(st);
  return r == cudaSuccess ? SV_OK : op_fail("select", r);
}

int sv_op_lm_head_logps(const void* x, const void* w, const int32_t* ids, float* logps, float* logits, int32_t M, int32_t N,
                        int32_t K, float temperature, void* stream) {
  if (!x || !w || !ids || !logps) return fail(nullptr, SV_ERR_INVALID, "lm_head_logps: null pointer");
  if (M < 1 || N < 1 || K < 64 || K % 64) return fail(nullptr, SV_ERR_INVALID, "lm_head_logps: need M, N >= 1 and K a positive multiple of 64");
  if (!(temperature > 0.f) || !std::isfinite(temperature)) return fail(nullptr, SV_ERR_INVALID, "lm_head_logps: temperature must be a finite value > 0");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t part_bytes = (size_t)M * lm_head_logps_ntiles(N) * sizeof(float2);
  OpScratch s;
  cudaError_t r = cudaMalloc(&s.p, part_bytes + (size_t)M * sizeof(float));
  if (r != cudaSuccess) return op_fail("lm_head_logps alloc", r);
  float2* part = reinterpret_cast<float2*>(s.p);
  float* tlogit = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s.p) + part_bytes);
  LogpsEpilogue lp{ids, nullptr, logits, part, tlogit, 1.0f / temperature};
  r = launch_lm_head_logps((const bf16*)x, (const bf16*)w, M, N, K, lp, nullptr, logps, st);
  if (r == cudaSuccess) r = cudaStreamSynchronize(st);
  return r == cudaSuccess ? SV_OK : op_fail("lm_head_logps", r);
}

}  // extern "C"
