// Elementwise / normalisation / layout kernels of the im2svg path (all HBM-bound, bf16 storage,
// fp32 math).  Reference semantics are cited per kernel; rounding points follow DESIGN.md.
#include "sv_kernels.h"

namespace sv {

thread_local int64_t* g_launch_counter = nullptr;

// ------------------------------------------------------------------------------------------
// block reductions
template <int NT>
SV_DEVINL float block_sum(float v, float* sm) {
  v = warp_sum(v);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sm[w] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < NT / 32; ++i) r += sm[i];
  return r;
}

// ------------------------------------------------------------------------------------------
// LayerNorm over the last dim (clip_model.py:117-124; nn.LayerNorm in GPTBigCode blocks):
// fp32 statistics (two-pass), y = bf16((x-mean)*rstd*w + b).
__global__ void __launch_bounds__(128) layernorm_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w,
                                                        const bf16* __restrict__ b, bf16* __restrict__ y, int cols,
                                                        float eps, int64_t x_row_stride) {
  __shared__ float sm[4];
  const bf16* xr = x + (int64_t)blockIdx.x * x_row_stride;
  bf16* yr = y + (int64_t)blockIdx.x * cols;
  const int nvec = cols >> 3;
  float s = 0.f;
  for (int i = threadIdx.x; i < nvec; i += 128) {
    float f[8];
    unpack8(ldg_cached(xr + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s += f[j];
  }
  const float mean = block_sum<128>(s, sm) / (float)cols;
  float q = 0.f;
  for (int i = threadIdx.x; i < nvec; i += 128) {
    float f[8];
    unpack8(ldg_cached(xr + i * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { float d = f[j] - mean; q += d * d; }
  }
  const float var = block_sum<128>(q, sm) / (float)cols;
  const float rstd = 1.0f / sqrtf(var + eps);
  for (int i = threadIdx.x; i < nvec; i += 128) {
    float f[8], wf[8], bf[8];
    unpack8(ldg_cached(xr + i * 8), f);
    unpack8(ldg_cached(w + i * 8), wf);
    unpack8(ldg_cached(b + i * 8), bf);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean) * rstd * wf[j] + bf[j];
    *reinterpret_cast<uint4*>(yr + i * 8) = pack8(f);
  }
}

void launch_layernorm(const bf16* x, const bf16* w, const bf16* b, bf16* y, int rows, int cols, float eps,
                      int64_t x_row_stride, cudaStream_t st) {
  if (rows <= 0) return;
  layernorm_kernel<<<rows, 128, 0, st>>>(x, w, b, y, cols, eps, x_row_stride);
  count_launch();
}

// ------------------------------------------------------------------------------------------
__global__ void convert_kernel(const void* __restrict__ src, int dtype, bf16* __restrict__ dst, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float v = dtype == 1 ? reinterpret_cast<const float*>(src)[i]
                         : __half2float(reinterpret_cast<const __half*>(src)[i]);
    dst[i] = __float2bfloat16_rn(v);
  }
}
void launch_convert_to_bf16(const void* src, int dtype, bf16* dst, int64_t n, cudaStream_t st) {
  if (n <= 0) return;
  int blocks = (int)((n + 255) / 256 > 4096 ? 4096 : (n + 255) / 256);
  convert_kernel<<<blocks, 256, 0, st>>>(src, dtype, dst, n);
  count_launch();
}

__global__ void pad_rows_kernel(const bf16* __restrict__ src, bf16* __restrict__ dst, int src_cols, int dst_cols) {
  const int r = blockIdx.x;
  for (int c = threadIdx.x; c < dst_cols; c += blockDim.x)
    dst[(int64_t)r * dst_cols + c] = c < src_cols ? src[(int64_t)r * src_cols + c] : __float2bfloat16_rn(0.f);
}
void launch_pad_rows(const bf16* src, bf16* dst, int rows, int src_cols, int dst_cols, cudaStream_t st) {
  pad_rows_kernel<<<rows, 128, 0, st>>>(src, dst, src_cols, dst_cols);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Patch extraction for conv1 (clip_model.py:174,182): stride == kernel, so the conv is a GEMM over
// [B*G*G, 3*p*p] patches; K is zero-padded to a multiple of 64 for the TMA/UMMA tile.
__global__ void im2col_kernel(const bf16* __restrict__ px, bf16* __restrict__ out, int image, int patch, int kpad) {
  const int g = image / patch;
  const int np = g * g;
  const int b = blockIdx.x / np, pi = blockIdx.x % np;
  const int py = pi / g, pxi = pi % g;
  const int pp = patch * patch;
  for (int k = threadIdx.x; k < kpad; k += blockDim.x) {
    bf16 v = __float2bfloat16_rn(0.f);
    if (k < 3 * pp) {
      int c = k / pp, r = k % pp, iy = r / patch, ix = r % patch;
      v = px[(((int64_t)b * 3 + c) * image + (py * patch + iy)) * image + (pxi * patch + ix)];
    }
    out[(int64_t)blockIdx.x * kpad + k] = v;
  }
}
void launch_im2col(const bf16* pixels, bf16* patches, int batch, int image, int patch, int kpad, cudaStream_t st) {
  int g = image / patch;
  im2col_kernel<<<batch * g * g, 128, 0, st>>>(pixels, patches, image, patch, kpad);
  count_launch();
}

// cat([class_embedding, patches]) + positional_embedding (clip_model.py:185-186); bf16 add.
__global__ void vit_assemble_kernel(const bf16* __restrict__ pe, const bf16* __restrict__ cls,
                                    const bf16* __restrict__ pos, bf16* __restrict__ x, int np, int width) {
  const int off = cls ? 1 : 0;                     // SigLIP has no class token (modeling_siglip.py:178-187)
  const int q = np + off;
  const int b = blockIdx.x / q, t = blockIdx.x % q;
  const bf16* src = (cls && t == 0) ? cls : pe + ((int64_t)b * np + (t - off)) * width;
  for (int c = threadIdx.x; c < width; c += blockDim.x)
    x[(int64_t)blockIdx.x * width + c] =
        __float2bfloat16_rn(__bfloat162float(src[c]) + __bfloat162float(pos[(int64_t)t * width + c]));
}
void launch_vit_assemble(const bf16* pe, const bf16* cls, const bf16* pos, bf16* x, int batch, int np, int width,
                         cudaStream_t st) {
  vit_assemble_kernel<<<batch * (np + (cls ? 1 : 0)), 128, 0, st>>>(pe, cls, pos, x, np, width);
  count_launch();
}

// V^T per (image, head): vt[b][h][d][l] = qkv[b*L+l][2W + h*64 + d], zero for l >= L (keeps P.V clean).
__global__ void vit_transpose_v_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ vt, int seq, int heads,
                                       int seq_pad) {
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int W = heads * 64;
  const int total = 64 * seq_pad;
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    int d = i / seq_pad, l = i % seq_pad;
    bf16 v = __float2bfloat16_rn(0.f);
    if (l < seq) v = qkv[((int64_t)b * seq + l) * (3 * W) + 2 * W + h * 64 + d];
    vt[((int64_t)blockIdx.x * 64 + d) * seq_pad + l] = v;
  }
}
void launch_vit_transpose_v(const bf16* qkv, bf16* vt, int batch, int seq, int heads, int seq_pad, cudaStream_t st) {
  vit_transpose_v_kernel<<<batch * heads, 256, 0, st>>>(qkv, vt, seq, heads, seq_pad);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Adapter norm, LayerNorm([Q,H]) flavour (adapters/adapter.py:25-26,37): statistics over the whole
// [Q,H] slab of one image, elementwise affine of the same shape.  Two kernels: per-chunk partial
// (sum, sumsq) then normalise (each block recombines the 64 partials in double).
constexpr int kSlabChunks = 64;
__global__ void __launch_bounds__(256) slab_stats_kernel(const bf16* __restrict__ z, float* __restrict__ partial,
                                                         int64_t slab) {
  __shared__ float sm[8];
  const int b = blockIdx.y, c = blockIdx.x;
  const int64_t per = (slab + kSlabChunks - 1) / kSlabChunks;
  const int64_t lo = c * per, hi = (lo + per < slab) ? lo + per : slab;
  const bf16* zr = z + (int64_t)b * slab;
  float s = 0.f, q = 0.f;
  for (int64_t i = lo + threadIdx.x; i < hi; i += 256) {
    float v = __bfloat162float(zr[i]);
    s += v; q += v * v;
  }
  s = block_sum<256>(s, sm);
  q = block_sum<256>(q, sm);
  if (threadIdx.x == 0) {
    partial[((int64_t)b * kSlabChunks + c) * 2 + 0] = s;
    partial[((int64_t)b * kSlabChunks + c) * 2 + 1] = q;
  }
}
__global__ void __launch_bounds__(256) slab_norm_kernel(const bf16* __restrict__ z, const bf16* __restrict__ w,
                                                        const bf16* __restrict__ bb, bf16* __restrict__ y,
                                                        const float* __restrict__ partial, int64_t slab, float eps) {
  __shared__ float stat[2];
  const int b = blockIdx.y;
  if (threadIdx.x == 0) {
    double s = 0.0, q = 0.0;
    for (int c = 0; c < kSlabChunks; ++c) {
      s += (double)partial[((int64_t)b * kSlabChunks + c) * 2 + 0];
      q += (double)partial[((int64_t)b * kSlabChunks + c) * 2 + 1];
    }
    double mean = s / (double)slab;
    double var = q / (double)slab - mean * mean;
    if (var < 0.0) var = 0.0;
    stat[0] = (float)mean;
    stat[1] = (float)(1.0 / sqrt(var + (double)eps));
  }
  __syncthreads();
  const float mean = stat[0], rstd = stat[1];
  const int64_t i = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 8;
  if (i >= slab) return;
  float f[8], wf[8], bf[8];
  unpack8(ldg_cached(z + (int64_t)b * slab + i), f);
  unpack8(ldg_cached(w + i), wf);
  unpack8(ldg_cached(bb + i), bf);
#pragma unroll
  for (int j = 0; j < 8; ++j) f[j] = (f[j] - mean) * rstd * wf[j] + bf[j];
  *reinterpret_cast<uint4*>(y + (int64_t)b * slab + i) = pack8(f);
}
void launch_slab_layernorm(const bf16* z, const bf16* w, const bf16* b, bf16* y, float* partial, int batch,
                           int64_t slab, float eps, cudaStream_t st) {
  slab_stats_kernel<<<dim3(kSlabChunks, batch), 256, 0, st>>>(z, partial, slab);
  int64_t nvec = slab / 8;
  slab_norm_kernel<<<dim3((unsigned)((nvec + 255) / 256), batch), 256, 0, st>>>(z, w, b, y, partial, slab, eps);
  count_launch(2);
}

// Adapter norm, BatchNorm1d(Q) eval flavour (adapter.py:27-28): channel = token index q.
__global__ void batchnorm_tokens_kernel(const bf16* __restrict__ z, const bf16* __restrict__ w,
                                        const bf16* __restrict__ b, const bf16* __restrict__ rmean,
                                        const bf16* __restrict__ rvar, bf16* __restrict__ y, int q, int h, float eps) {
  const int t = blockIdx.x % q;
  const float mean = __bfloat162float(rmean[t]);
  const float invstd = 1.0f / sqrtf(__bfloat162float(rvar[t]) + eps);
  const float ww = __bfloat162float(w[t]), bb = __bfloat162float(b[t]);
  for (int c = threadIdx.x; c < h; c += blockDim.x) {
    float v = __bfloat162float(z[(int64_t)blockIdx.x * h + c]);
    y[(int64_t)blockIdx.x * h + c] = __float2bfloat16_rn((v - mean) * invstd * ww + bb);
  }
}
void launch_batchnorm_tokens(const bf16* z, const bf16* w, const bf16* b, const bf16* rmean, const bf16* rvar, bf16* y,
                             int batch, int q, int h, float eps, cudaStream_t st) {
  batchnorm_tokens_kernel<<<batch * q, 128, 0, st>>>(z, w, b, rmean, rvar, y, q, h, eps);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// inputs_embeds = cat([visual, wte(prompt)]) (starvector_base.py:218-219) + wpe[position]
// (GPTBigCodeModel.forward: hidden = inputs_embeds + position_embeds), bf16 add.
__global__ void embed_prefix_kernel(const bf16* __restrict__ visual, const int32_t* __restrict__ prompt,
                                    const bf16* __restrict__ wte, const bf16* __restrict__ wpe, bf16* __restrict__ x,
                                    int q, int p, int h, int vocab) {
  const int t0 = q + p;
  const int b = blockIdx.x / t0, t = blockIdx.x % t0;
  const bf16* src;
  if (t < q) {
    src = visual + ((int64_t)b * q + t) * h;
  } else {
    int id = prompt[b * p + (t - q)];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    src = wte + (int64_t)id * h;
  }
  const bf16* pos = wpe ? wpe + (int64_t)t * h : nullptr;   // RoPE models (StarCoder2) have no learned positions
  for (int c = threadIdx.x * 8; c < h; c += blockDim.x * 8) {
    float a[8], d[8];
    unpack8(ldg_cached(src + c), a);
    if (pos) {
      unpack8(ldg_cached(pos + c), d);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += d[j];
    }
    *reinterpret_cast<uint4*>(x + (int64_t)blockIdx.x * h + c) = pack8(a);
  }
}
void launch_embed_prefix(const bf16* visual, const int32_t* prompt_ids, const bf16* wte, const bf16* wpe, bf16* x,
                         int batch, int q, int p, int h, int vocab, cudaStream_t st) {
  embed_prefix_kernel<<<batch * (q + p), 128, 0, st>>>(visual, prompt_ids, wte, wpe, x, q, p, h, vocab);
  count_launch();
}

__global__ void embed_chunk_kernel(const int32_t* __restrict__ ids, int ids_ld, const bf16* __restrict__ wte,
                                   const bf16* __restrict__ wpe, bf16* __restrict__ x, int seq, int pos0, int h, int vocab,
                                   int n_positions) {
  const int b = blockIdx.x / seq, t = blockIdx.x % seq;
  int id = ids[(int64_t)b * ids_ld + t];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  const int pos = min(pos0 + t, n_positions - 1);
  const bf16* src = wte + (int64_t)id * h;
  const bf16* pe = wpe ? wpe + (int64_t)pos * h : nullptr;
  for (int c = threadIdx.x * 8; c < h; c += blockDim.x * 8) {
    float a[8], d[8];
    unpack8(ldg_cached(src + c), a);
    if (pe) {
      unpack8(ldg_cached(pe + c), d);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += d[j];
    }
    *reinterpret_cast<uint4*>(x + (int64_t)blockIdx.x * h + c) = pack8(a);
  }
}
void launch_embed_chunk(const int32_t* ids, int ids_ld, const bf16* wte, const bf16* wpe, bf16* x, int batch, int seq, int pos0,
                        int h, int vocab, int n_positions, cudaStream_t st) {
  embed_chunk_kernel<<<batch * seq, 128, 0, st>>>(ids, ids_ld, wte, wpe, x, seq, pos0, h, vocab, n_positions);
  count_launch();
}

// Row r = b*seq + t of a scoring chunk holds call position t0 + t; its logits predict token t0 + t + 1 of the row.
//   tgt    : that token's id (clamped as the embedding clamps), -1 past the end
//   lp_idx : where its log-prob goes in logps [B][T], -1 past the end or when no log-probs are wanted
//   lg_row : output row of its fp32 logits: the last `keep` positions go to [B][keep]; with keep == 0 only the call's last
//            position is stored, to row b of a [B][V] staging buffer (it becomes the engine's held last-position logits)
__global__ void score_maps_kernel(const int32_t* __restrict__ ids, int T, int rows, int seq, int t0, int keep, int vocab,
                                  int want_logps, int32_t* __restrict__ tgt, int32_t* __restrict__ lg_row,
                                  int32_t* __restrict__ lp_idx) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int b = r / seq, t = t0 + r % seq;
  int id = -1;
  if (t + 1 < T) {
    id = ids[(int64_t)b * T + t + 1];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  }
  tgt[r] = id;
  lp_idx[r] = (want_logps && t + 1 < T) ? b * T + t + 1 : -1;
  lg_row[r] = keep > 0 ? (t >= T - keep ? b * keep + t - (T - keep) : -1) : (t == T - 1 ? b : -1);
}
void launch_score_maps(const int32_t* ids, int T, int batch, int seq, int t0, int keep, int vocab, bool want_logps,
                       int32_t* tgt, int32_t* lg_row, int32_t* lp_idx, cudaStream_t st) {
  const int rows = batch * seq;
  score_maps_kernel<<<(rows + 255) / 256, 256, 0, st>>>(ids, T, rows, seq, t0, keep, vocab, want_logps ? 1 : 0, tgt, lg_row,
                                                        lp_idx);
  count_launch();
}

// log_softmax(bf16 row / T)[id] with the lm_head epilogue's arithmetic: x = bf16 value * (1/T) in fp32, fp32 max and sum.
__global__ void row_logp_kernel(const bf16* __restrict__ logits, int vocab, const int32_t* __restrict__ ids, int ids_ld,
                                float inv_temp, float* __restrict__ logps, int lp_ld) {
  __shared__ float red[32];
  const int b = blockIdx.x, nw = blockDim.x >> 5, w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bf16* row = logits + (int64_t)b * vocab;
  float m = -INFINITY;
  for (int i = threadIdx.x; i < vocab; i += blockDim.x) m = fmaxf(m, __bfloat162float(row[i]) * inv_temp);
  m = warp_max(m);
  if (lane == 0) red[w] = m;
  __syncthreads();
  m = -INFINITY;
  for (int i = 0; i < nw; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float s = 0.f;
  for (int i = threadIdx.x; i < vocab; i += blockDim.x) s += expf(__bfloat162float(row[i]) * inv_temp - m);
  s = warp_sum(s);
  if (lane == 0) red[w] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    s = 0.f;
    for (int i = 0; i < nw; ++i) s += red[i];
    int id = ids[(int64_t)b * ids_ld];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    logps[(int64_t)b * lp_ld] = __bfloat162float(row[id]) * inv_temp - (m + logf(s));
  }
}
void launch_row_logp(const bf16* logits, int vocab, int batch, const int32_t* ids, int ids_ld, float inv_temp, float* logps,
                     int lp_ld, cudaStream_t st) {
  row_logp_kernel<<<batch, 256, 0, st>>>(logits, vocab, ids, ids_ld, inv_temp, logps, lp_ld);
  count_launch();
}

__global__ void float_rows_to_bf16_kernel(const float* __restrict__ src, int64_t src_ld, bf16* __restrict__ dst, int n) {
  const int b = blockIdx.y;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    dst[(int64_t)b * n + i] = __float2bfloat16_rn(src[b * src_ld + i]);
}
void launch_float_rows_to_bf16(const float* src, int64_t src_ld, bf16* dst, int batch, int n, cudaStream_t st) {
  float_rows_to_bf16_kernel<<<dim3((n + 255) / 256 < 64 ? (n + 255) / 256 : 64, batch), 256, 0, st>>>(src, src_ld, dst, n);
  count_launch();
}

__global__ void embed_tokens_kernel(const int32_t* __restrict__ ids, const bf16* __restrict__ wte,
                                    const bf16* __restrict__ wpe, const GenState* __restrict__ state,
                                    bf16* __restrict__ x, int h, int vocab, int n_positions) {
  const int b = blockIdx.x;
  int id = ids[b];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  int pos = state->cur_len;
  pos = pos >= n_positions ? n_positions - 1 : pos;
  const bf16* src = wte + (int64_t)id * h;
  const bf16* pe = wpe ? wpe + (int64_t)pos * h : nullptr;
  for (int c = threadIdx.x * 8; c < h; c += blockDim.x * 8) {
    float a[8], d[8];
    unpack8(ldg_cached(src + c), a);
    if (pe) {
      unpack8(ldg_cached(pe + c), d);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += d[j];
    }
    *reinterpret_cast<uint4*>(x + (int64_t)b * h + c) = pack8(a);
  }
}
void launch_embed_tokens(const int32_t* ids, const bf16* wte, const bf16* wpe, const GenState* state, bf16* x,
                         int batch, int h, int vocab, int n_positions, cudaStream_t st) {
  embed_tokens_kernel<<<batch, 128, 0, st>>>(ids, wte, wpe, state, x, h, vocab, n_positions);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// KV cache write.  Layout per layer: K [max_batch][n_kv][tcap][d] (rows), V^T [max_batch][n_kv][d][tcap]
// (so the P.V tensor-core operand is a contiguous 16-byte load per lane; see sv_attention.cu).
// The reference re-allocates and copies the whole cache every step (torch.cat, SURVEY.md K15).
__global__ void kv_write_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ kcache, bf16* __restrict__ vtcache,
                                const GenState* __restrict__ state, int seq, int q_cols, int n_kv, int d, int tcap, int pos0) {
  const int b = blockIdx.y, ts = blockIdx.x;
  const int t = (state ? state->cur_len : pos0) + ts;
  if (t >= tcap) return;
  const int cols = q_cols + 2 * n_kv * d;
  const bf16* row = qkv + ((int64_t)b * seq + ts) * cols;
  for (int i = threadIdx.x; i < n_kv * d; i += blockDim.x) {
    int kvh = i / d, dim = i % d;
    kcache[(((int64_t)b * n_kv + kvh) * tcap + t) * d + dim] = row[q_cols + i];
    vtcache[(((int64_t)b * n_kv + kvh) * d + dim) * tcap + t] = row[q_cols + n_kv * d + i];
  }
}
void launch_kv_scatter(const bf16* qkv, bf16* kcache, bf16* vtcache, int batch, int seq, int q_cols, int n_kv, int d,
                       int tcap, int pos0, cudaStream_t st) {
  kv_write_kernel<<<dim3(seq, batch), 128, 0, st>>>(qkv, kcache, vtcache, nullptr, seq, q_cols, n_kv, d, tcap, pos0);
  count_launch();
}
void launch_kv_append(const bf16* qkv, bf16* kcache, bf16* vtcache, const GenState* state, int batch, int q_cols,
                      int n_kv, int d, int tcap, cudaStream_t st) {
  kv_write_kernel<<<dim3(1, batch), 128, 0, st>>>(qkv, kcache, vtcache, state, 1, q_cols, n_kv, d, tcap, 0);
  count_launch();
}

// Beam search cache reorder (HF `_reorder_cache` / `Cache.reorder_cache`, generation/utils.py beam loop): image row r of
// the destination takes the first `len` tokens of source row idx[r].  One layer at a time through a scratch layer
// (gather), then copied back with idx == nullptr (identity).  grid = (n_kv * 2, rows); 16-byte vectors.
__global__ void kv_gather_kernel(const bf16* __restrict__ ksrc, const bf16* __restrict__ vsrc, bf16* __restrict__ kdst,
                                 bf16* __restrict__ vdst, const int32_t* __restrict__ idx, int n_kv, int tcap, int d,
                                 int len) {
  const int r = blockIdx.y, kvh = blockIdx.x >> 1, which = blockIdx.x & 1;
  const int sr = idx ? idx[r] : r;
  if (which == 0) {            // K rows: contiguous [len][d]
    const uint4* s = reinterpret_cast<const uint4*>(ksrc + ((int64_t)sr * n_kv + kvh) * tcap * d);
    uint4* t = reinterpret_cast<uint4*>(kdst + ((int64_t)r * n_kv + kvh) * tcap * d);
    const int n = len * d / 8;
    for (int i = threadIdx.x; i < n; i += blockDim.x) t[i] = s[i];
  } else {                     // V^T: d rows of `len` (rounded up to 8) keys
    const int per = (len + 7) / 8;
    for (int i = threadIdx.x; i < d * per; i += blockDim.x) {
      const int dim = i / per, c = i % per;
      const int64_t off = (((int64_t)0 * n_kv + kvh) * d + dim) * tcap + c * 8;
      *reinterpret_cast<uint4*>(vdst + ((int64_t)r * n_kv * d) * tcap + off) =
          *reinterpret_cast<const uint4*>(vsrc + ((int64_t)sr * n_kv * d) * tcap + off);
    }
  }
}
void launch_kv_gather(const bf16* ksrc, const bf16* vsrc, bf16* kdst, bf16* vdst, const int32_t* idx, int rows, int n_kv,
                      int tcap, int d, int len, cudaStream_t st) {
  kv_gather_kernel<<<dim3(n_kv * 2, rows), 256, 0, st>>>(ksrc, vsrc, kdst, vdst, idx, n_kv, tcap, d, len);
  count_launch();
}

__global__ void gather_rows_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int seq, int row, int h) {
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < h; c += blockDim.x) y[(int64_t)b * h + c] = x[((int64_t)b * seq + row) * h + c];
}
void launch_gather_rows(const bf16* x, bf16* y, int batch, int seq, int row, int h, cudaStream_t st) {
  gather_rows_kernel<<<batch, 256, 0, st>>>(x, y, seq, row, h);
  count_launch();
}

__global__ void logits_to_float_kernel(const bf16* __restrict__ l, float* __restrict__ o, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = __bfloat162float(l[i]);
}
void launch_logits_to_float(const bf16* logits, float* out, int64_t n, cudaStream_t st) {
  logits_to_float_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(logits, out, n);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Token selection = the body of HF `_sample` (SURVEY.md App. B.3-6): fp32 cast of the bf16 logits,
// repetition penalty over generated ids, argmax with lowest-index tie-break, EOS->pad for finished
// rows, append, EOS / '</svg>' stop bookkeeping.  One block per batch row.
struct ArgMax { float v; int i; };
SV_DEVINL ArgMax better(ArgMax a, ArgMax b) { return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a; }

SV_DEVINL void append_token(int b, int tok, GenState* state, const GenParamsDev* p, uint8_t* seen, int vocab,
                            int32_t* next_ids, int32_t* out_ids) {
  const int step = state->step;
  const bool unfinished = state->unfinished[b] != 0;
  if (p->eos_id >= 0 && !unfinished) tok = p->pad_id;                 // next*unfinished + pad*(1-unfinished)
  int32_t* row = out_ids + (int64_t)b * p->out_stride;
  row[step] = tok;
  next_ids[b] = tok;
  if (tok >= 0 && tok < vocab) seen[(int64_t)b * vocab + tok] = 1;
  if (p->eos_id >= 0 && tok == p->eos_id) state->unfinished[b] = 0;   // EosTokenCriteria
  const int n = p->n_stop;
  if (n > 0 && step + 1 >= n && (b == 0 || !p->stop_row0_only)) {     // StoppingCriteriaSub (row 0 only)
    bool match = true;
    for (int j = 0; j < n; ++j) match = match && (row[step + 1 - n + j] == p->stop_ids[j]);
    if (match) {
      if (p->stop_row0_only) state->row0_stop = 1;
      else state->unfinished[b] = 0;
    }
  }
}

__global__ void __launch_bounds__(1024) select_greedy_kernel(const bf16* __restrict__ logits, int vocab,
                                                             GenState* state, const GenParamsDev* __restrict__ p,
                                                             uint8_t* seen, int32_t* next_ids, int32_t* out_ids) {
  if (state->done) return;
  __shared__ ArgMax sm[32];
  const int b = blockIdx.x;
  const bf16* lr = logits + (int64_t)b * vocab;
  const uint8_t* sr = seen + (int64_t)b * vocab;
  const float rp = p->rep_penalty;
  const bool use_rp = rp != 1.0f;
  ArgMax best{-INFINITY, 0x7fffffff};
  for (int i = threadIdx.x; i < vocab; i += 1024) {
    float v = __bfloat162float(lr[i]);
    if (use_rp && sr[i]) v = v < 0.f ? v * rp : v / rp;               // RepetitionPenaltyLogitsProcessor
    best = better(best, ArgMax{v, i});
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ArgMax other{__shfl_xor_sync(0xffffffffu, best.v, o), __shfl_xor_sync(0xffffffffu, best.i, o)};
    best = better(best, other);
  }
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 32; ++w) best = better(best, sm[w]);
    int tok = best.i == 0x7fffffff ? 0 : best.i;
    append_token(b, tok, state, p, seen, vocab, next_ids, out_ids);
  }
}
void launch_select_greedy(const bf16* logits, int vocab, int batch, GenState* state, const GenParamsDev* params,
                          uint8_t* seen, int32_t* next_ids, int32_t* out_ids, cudaStream_t st) {
  select_greedy_kernel<<<batch, 1024, 0, st>>>(logits, vocab, state, params, seen, next_ids, out_ids);
  count_launch();
}

// ---- sampling: repetition penalty -> temperature -> top-p -> multinomial (App. B.3), Philox stream.
SV_DEVINL uint32_t mulhilo(uint32_t a, uint32_t b, uint32_t* hi) {
  unsigned long long p = (unsigned long long)a * b;
  *hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
}
SV_DEVINL float philox_uniform(unsigned long long seed, uint32_t c0, uint32_t c1) {   // Philox4x32-10
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t x0 = c0, x1 = c1, x2 = 0x5356u, x3 = 0x42323030u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    uint32_t lo0 = mulhilo(0xD2511F53u, x0, &hi0);
    uint32_t lo1 = mulhilo(0xCD9E8D57u, x2, &hi1);
    uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
    x0 = y0; x1 = y1; x2 = y2; x3 = y3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return ((float)(x0 >> 8) + 0.5f) * (1.0f / 16777216.0f);
}

constexpr int kSampleThreads = 1024;
// `probs` is an fp32 scratch row [B][vocab] (L2 resident): the kernel makes ~34 passes over it.
__global__ void __launch_bounds__(kSampleThreads) select_sample_kernel(const bf16* __restrict__ logits, int vocab,
                                                                       GenState* state,
                                                                       const GenParamsDev* __restrict__ p,
                                                                       uint8_t* seen, int32_t* next_ids,
                                                                       int32_t* out_ids, float* __restrict__ probs) {
  if (state->done) return;
  __shared__ float smf[32];
  __shared__ float s_bcast;
  __shared__ int s_tok;
  const int b = blockIdx.x, tid = threadIdx.x;
  const bf16* lr = logits + (int64_t)b * vocab;
  const uint8_t* sr = seen + (int64_t)b * vocab;
  float* pr = probs + (int64_t)b * vocab;
  const float rp = p->rep_penalty, invT = 1.0f / p->temperature;
  float mx = -INFINITY;
  for (int i = tid; i < vocab; i += kSampleThreads) {
    float v = __bfloat162float(lr[i]);
    if (rp != 1.0f && sr[i]) v = v < 0.f ? v * rp : v / rp;            // RepetitionPenaltyLogitsProcessor
    v *= invT;                                                         // TemperatureLogitsWarper
    pr[i] = v;
    mx = fmaxf(mx, v);
  }
  mx = warp_max(mx);
  if ((tid & 31) == 0) smf[tid >> 5] = mx;
  __syncthreads();
  mx = smf[0];
  for (int w = 1; w < 32; ++w) mx = fmaxf(mx, smf[w]);
  float z = 0.f;
  for (int i = tid; i < vocab; i += kSampleThreads) { float e = __expf(pr[i] - mx); pr[i] = e; z += e; }
  z = block_sum<kSampleThreads>(z, smf);
  const float invz = 1.0f / z;
  // TopPLogitsWarper: keep a token iff the mass of strictly more probable tokens is < top_p.
  // Bisection on the probability threshold: find (the infimum of) q with mass(p > q) < top_p.
  float lo = 0.f, hi = 1.f;
  const float top_p = p->top_p;
  if (top_p < 1.0f) {
    for (int it = 0; it < 30; ++it) {
      const float mid = 0.5f * (lo + hi);
      float m = 0.f;
      for (int i = tid; i < vocab; i += kSampleThreads) { float q = pr[i] * invz; m += q > mid ? q : 0.f; }
      m = block_sum<kSampleThreads>(m, smf);
      if (m < top_p) hi = mid; else lo = mid;
    }
  } else {
    lo = -1.f;
  }
  // kept set = { p > lo }.  Thread `tid` owns ids [tid*per, tid*per+per) so the scan runs in id order.
  const int per = (vocab + kSampleThreads - 1) / kSampleThreads;
  const int i0 = tid * per, i1 = min(i0 + per, vocab);
  float own = 0.f;
  for (int i = i0; i < i1; ++i) { float q = pr[i] * invz; own += q > lo ? q : 0.f; }
  float incl = own;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { float n = __shfl_up_sync(0xffffffffu, incl, o); if ((tid & 31) >= o) incl += n; }
  __syncthreads();
  if ((tid & 31) == 31) smf[tid >> 5] = incl;
  __syncthreads();
  float base = 0.f, total = 0.f;
  for (int w = 0; w < 32; ++w) { if (w < (tid >> 5)) base += smf[w]; total += smf[w]; }
  if (tid == 0) { s_bcast = philox_uniform(p->seed, (uint32_t)b, (uint32_t)state->step) * total; s_tok = -1; }
  __syncthreads();
  const float target = s_bcast;
  const float excl = base + incl - own;
  if (own > 0.f && target >= excl && target < excl + own) {            // torch.multinomial(probs, 1)
    float acc = excl; int tok = -1;
    for (int i = i0; i < i1; ++i) {
      float q = pr[i] * invz;
      if (q > lo) { tok = i; acc += q; if (target < acc) break; }
    }
    atomicMax(&s_tok, tok);
  }
  __syncthreads();
  if (tid == 0) {
    int tok = s_tok;
    if (tok < 0) {                                                     // fp rounding fell off the end: last kept id
      for (int i = vocab - 1; i >= 0; --i) if (pr[i] * invz > lo) { tok = i; break; }
      if (tok < 0) tok = 0;
    }
    append_token(b, tok, state, p, seen, vocab, next_ids, out_ids);
  }
}
void launch_select_sample(const bf16* logits, int vocab, int batch, GenState* state, const GenParamsDev* params,
                          uint8_t* seen, int32_t* next_ids, int32_t* out_ids, float* probs, cudaStream_t st) {
  select_sample_kernel<<<batch, kSampleThreads, 0, st>>>(logits, vocab, state, params, seen, next_ids, out_ids, probs);
  count_launch();
}

// unfinished &= ~stop; this_peer_finished = unfinished.max()==0; then advance the step counter.
__global__ void gen_finalize_kernel(GenState* state, const GenParamsDev* __restrict__ p, int batch, int advance_len) {
  if (threadIdx.x != 0 || state->done) return;
  if (state->row0_stop) {
    for (int b = 0; b < batch; ++b) state->unfinished[b] = 0;
    state->row0_stop = 0;
  }
  state->step += 1;
  if (advance_len) state->cur_len += 1;
  int any = 0;
  for (int b = 0; b < batch; ++b) any |= state->unfinished[b];
  if (!any || state->step >= p->max_new) state->done = 1;
}
void launch_gen_finalize(GenState* state, const GenParamsDev* params, int batch, int advance_len, cudaStream_t st) {
  gen_finalize_kernel<<<1, 32, 0, st>>>(state, params, batch, advance_len);
  count_launch();
}
__global__ void advance_len_kernel(GenState* state) {
  if (threadIdx.x == 0) state->cur_len += 1;
}
void launch_advance_len(GenState* state, cudaStream_t st) {
  advance_len_kernel<<<1, 32, 0, st>>>(state);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Rotary position embedding of StarCoder2 (transformers modeling_starcoder2.py:72-107,265-329): cos/sin are computed
// in fp32, CAST TO bf16, and  q*cos + rotate_half(q)*sin  runs as three bf16 tensor ops (two products, one sum).
__global__ void rope_table_kernel(bf16* __restrict__ cos_t, bf16* __restrict__ sin_t, int max_pos, int half, float theta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= max_pos * half) return;
  const int pos = i / half, j = i % half;
  const float inv_freq = 1.0f / powf(theta, (float)(2 * j) / (float)(2 * half));
  const float ang = (float)pos * inv_freq;
  cos_t[i] = __float2bfloat16_rn(cosf(ang));
  sin_t[i] = __float2bfloat16_rn(sinf(ang));
}
void launch_rope_table(bf16* cos_t, bf16* sin_t, int max_pos, int d, float theta, cudaStream_t st) {
  const int n = max_pos * (d / 2);
  rope_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(cos_t, sin_t, max_pos, d / 2, theta);
  count_launch();
}
__global__ void rope_kernel(bf16* __restrict__ qkv, int seq, int qkv_cols, int n_rot_heads, int d,
                            const bf16* __restrict__ cos_t, const bf16* __restrict__ sin_t,
                            const GenState* __restrict__ state, int max_pos, int pos0) {
  const int row = blockIdx.x, half = d >> 1;
  int pos = state ? state->cur_len : pos0 + (row % seq);
  pos = pos >= max_pos ? max_pos - 1 : pos;
  bf16* base = qkv + (int64_t)row * qkv_cols;
  for (int i = threadIdx.x; i < n_rot_heads * half; i += blockDim.x) {
    const int h = i / half, j = i % half;
    bf16* v = base + h * d;
    const float c = __bfloat162float(cos_t[(int64_t)pos * half + j]), s = __bfloat162float(sin_t[(int64_t)pos * half + j]);
    const float x1 = __bfloat162float(v[j]), x2 = __bfloat162float(v[j + half]);
    v[j] = __float2bfloat16_rn(bf16_round(x1 * c) + bf16_round(-x2 * s));
    v[j + half] = __float2bfloat16_rn(bf16_round(x2 * c) + bf16_round(x1 * s));
  }
}
// Decode-step companion of the fused QKV GEMV for RoPE models: rotate q in place, rotate k and append it (and v) to the
// KV cache at position cur_len.  One block per image.
__global__ void rope_append_kernel(bf16* __restrict__ qkv, int qkv_cols, int n_head, int n_kv, int d,
                                   const bf16* __restrict__ cos_t, const bf16* __restrict__ sin_t,
                                   bf16* __restrict__ kcache, bf16* __restrict__ vtcache,
                                   const GenState* __restrict__ state, int tcap, int max_pos) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const int b = blockIdx.x, half = d >> 1;
  const int pos = state->cur_len;
  const int tp = pos >= max_pos ? max_pos - 1 : pos;
  bf16* base = qkv + (int64_t)b * qkv_cols;
  for (int i = threadIdx.x; i < (n_head + n_kv) * half; i += blockDim.x) {
    const int h = i / half, j = i % half;
    bf16* v = base + h * d;
    const float c = __bfloat162float(cos_t[(int64_t)tp * half + j]), s = __bfloat162float(sin_t[(int64_t)tp * half + j]);
    const float x1 = __bfloat162float(__ldcg(v + j)), x2 = __bfloat162float(__ldcg(v + j + half));
    const bf16 o1 = __float2bfloat16_rn(bf16_round(x1 * c) + bf16_round(-x2 * s));
    const bf16 o2 = __float2bfloat16_rn(bf16_round(x2 * c) + bf16_round(x1 * s));
    if (h < n_head) {
      v[j] = o1; v[j + half] = o2;
    } else if (pos < tcap) {
      const int kvh = h - n_head;
      bf16* kr = kcache + (((int64_t)b * n_kv + kvh) * tcap + pos) * d;
      kr[j] = o1; kr[j + half] = o2;
    }
  }
  if (pos < tcap) {
    const bf16* vsrc = base + (n_head + n_kv) * d;
    for (int i = threadIdx.x; i < n_kv * d; i += blockDim.x) {
      const int kvh = i / d, dim = i % d;
      vtcache[(((int64_t)b * n_kv + kvh) * d + dim) * tcap + pos] = __ldcg(vsrc + i);
    }
  }
}
void launch_rope_append(bf16* qkv, int batch, int qkv_cols, int n_head, int n_kv, int d, const bf16* cos_t,
                        const bf16* sin_t, bf16* kcache, bf16* vtcache, const GenState* state, int tcap, int max_pos,
                        bool pdl, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(batch); cfg.blockDim = dim3(256); cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, rope_append_kernel, qkv, qkv_cols, n_head, n_kv, d, cos_t, sin_t, kcache, vtcache, state, tcap,
                     max_pos);
  count_launch();
}

void launch_rope(bf16* qkv, int rows, int seq, int qkv_cols, int n_rot_heads, int d, const bf16* cos_t, const bf16* sin_t,
                 const GenState* state, int max_pos, int pos0, cudaStream_t st) {
  rope_kernel<<<rows, 256, 0, st>>>(qkv, seq, qkv_cols, n_rot_heads, d, cos_t, sin_t, state, max_pos, pos0);
  count_launch();
}

__global__ void fill_i32_kernel(int32_t* p, int32_t v, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
void launch_fill_i32(int32_t* p, int32_t v, int n, cudaStream_t st) {
  fill_i32_kernel<<<(n + 255) / 256, 256, 0, st>>>(p, v, n);
  count_launch();
}

}  // namespace sv
