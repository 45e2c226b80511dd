// Attention for the three places the im2svg path needs it, on one register-resident core:
//   * ViT self-attention (clip_model.py:134,148-150; 16 heads x 64, seq 257, no mask),
//   * decoder prefill: causal multi-query attention over the Q+P prefix (GPTBigCodeAttention),
//   * decode: one new token per image against the KV cache, split over the key axis.
//
// One warp owns a 16-row tile of the score matrix and walks the keys 32 at a time with
// mma.sync m16n8k16 (bf16 in, fp32 accumulate) and an online softmax in the exp2 domain.
// The reduction over the single shared KV head is done with warp shuffles (quad_max/quad_sum).
// For the decoder the 16 rows are the (up to 16) QUERY HEADS that share one KV head, so a K/V
// block loaded once serves every head (multi-query), and all rows share one causal bound.
//
// No shared memory and no ldmatrix: both MMA operands are 128-bit global loads.
//   Q.K^T : the dot product over head_dim is invariant under a permutation of the dim index applied
//           to both operands, so lane (g,t) feeds dims 32j+8t..+7 of its row to k-steps 2j,2j+1.
//   P.V   : V is kept TRANSPOSED ([dim][key]) so the "B" fragment (two consecutive keys for one
//           dim) is contiguous; keys inside a 32-block are permuted consistently between the S
//           accumulator columns and the V^T load: S tile j, column i  <->  key 8*(i/2) + 2j + (i%2).
#include <algorithm>

#include "sv_kernels.h"

namespace sv {

// CG = true: L2-only loads (ld.global.cg) for data produced by the immediately preceding kernel when
// kernels overlap under Programmatic Dependent Launch (a co-resident CTA may hold stale L1 lines).
template <bool CG>
SV_DEVINL uint4 ld16(const void* p) {
  if constexpr (CG) return __ldcg(reinterpret_cast<const uint4*>(p));
  else return ldg_cached(p);
}

template <int D, bool CG = false>
SV_DEVINL void load_q_frag(uint32_t (&qa)[D / 16][4], const bf16* row_lo, bool ok_lo, const bf16* row_hi, bool ok_hi,
                           int t) {
#pragma unroll
  for (int jj = 0; jj < D / 32; ++jj) {
    uint4 a = make_uint4(0u, 0u, 0u, 0u), b = make_uint4(0u, 0u, 0u, 0u);
    if (ok_lo) a = ld16<CG>(row_lo + 32 * jj + 8 * t);
    if (ok_hi) b = ld16<CG>(row_hi + 32 * jj + 8 * t);
    qa[2 * jj][0] = a.x; qa[2 * jj][1] = b.x; qa[2 * jj][2] = a.y; qa[2 * jj][3] = b.y;
    qa[2 * jj + 1][0] = a.z; qa[2 * jj + 1][1] = b.z; qa[2 * jj + 1][2] = a.w; qa[2 * jj + 1][3] = b.w;
  }
}

// Processes keys [key_begin, key_end) (key_begin % 32 == 0).  acc/m/l are running (unnormalised)
// output, row max (log2 domain) and per-lane partial row sums for rows g (index 0) and g+8 (1).
// HOIST_V: issue the block's V^T loads together with its K loads (one dependent memory round instead of two;
// costs 64 more live registers, used by the latency-critical single-token decode kernel).
template <int D, bool CG = false, bool HOIST_V = false>
SV_DEVINL void attn_core(const uint32_t (&qa)[D / 16][4], const bf16* __restrict__ kbase, int64_t k_row_stride,
                         const bf16* __restrict__ vtbase, int64_t vt_dim_stride, int key_begin, int key_end,
                         float scale_log2, float (&acc)[D / 8][4], float (&mrow)[2], float (&lrow)[2], int lane,
                         int key_lo = 0) {   // keys < key_lo are masked (sliding-window attention, StarCoder2)
  const int g = lane >> 2, t = lane & 3;
  for (int kb = key_begin; kb < key_end; kb += 32) {
    float s[4][4];
    uint4 vpre[HOIST_V ? D / 8 : 1];
    if constexpr (HOIST_V) {
#pragma unroll
      for (int nd = 0; nd < D / 8; ++nd) vpre[nd] = ld16<CG>(vtbase + (int64_t)(8 * nd + g) * vt_dim_stride + kb + 8 * t);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
      int key = kb + 8 * (g >> 1) + 2 * j + (g & 1);
      key = key < key_end ? key : key_end - 1;          // clamp: stays inside valid rows, masked below
      const bf16* kp = kbase + (int64_t)key * k_row_stride + 8 * t;
#pragma unroll
      for (int jj = 0; jj < D / 32; ++jj) {
        const uint4 w = ld16<CG>(kp + 32 * jj);
        mma_bf16_16816(s[j], qa[2 * jj][0], qa[2 * jj][1], qa[2 * jj][2], qa[2 * jj][3], w.x, w.y);
        mma_bf16_16816(s[j], qa[2 * jj + 1][0], qa[2 * jj + 1][1], qa[2 * jj + 1][2], qa[2 * jj + 1][3], w.z, w.w);
      }
    }
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int kidx = kb + 8 * t + 2 * j + e;
        const bool valid = kidx < key_end && kidx >= key_lo;
        s[j][e] = valid ? s[j][e] * scale_log2 : -INFINITY;
        s[j][2 + e] = valid ? s[j][2 + e] * scale_log2 : -INFINITY;
        mx0 = fmaxf(mx0, s[j][e]);
        mx1 = fmaxf(mx1, s[j][2 + e]);
      }
    }
    mx0 = quad_max(mx0);
    mx1 = quad_max(mx1);
    const float mn0 = fmaxf(mrow[0], mx0), mn1 = fmaxf(mrow[1], mx1);
    const float corr0 = exp2f(mrow[0] - mn0), corr1 = exp2f(mrow[1] - mn1);
    mrow[0] = mn0; mrow[1] = mn1;
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      s[j][0] = exp2f(s[j][0] - mn0); s[j][1] = exp2f(s[j][1] - mn0);
      s[j][2] = exp2f(s[j][2] - mn1); s[j][3] = exp2f(s[j][3] - mn1);
      rs0 += s[j][0] + s[j][1];
      rs1 += s[j][2] + s[j][3];
    }
    lrow[0] = lrow[0] * corr0 + rs0;
    lrow[1] = lrow[1] * corr1 + rs1;
    uint32_t pa[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      pa[h][0] = pack_bf16x2(s[2 * h][0], s[2 * h][1]);
      pa[h][1] = pack_bf16x2(s[2 * h][2], s[2 * h][3]);
      pa[h][2] = pack_bf16x2(s[2 * h + 1][0], s[2 * h + 1][1]);
      pa[h][3] = pack_bf16x2(s[2 * h + 1][2], s[2 * h + 1][3]);
    }
#pragma unroll
    for (int nd = 0; nd < D / 8; ++nd) {
      acc[nd][0] *= corr0; acc[nd][1] *= corr0; acc[nd][2] *= corr1; acc[nd][3] *= corr1;
      uint4 w;
      if constexpr (HOIST_V) w = vpre[nd];
      else w = ld16<CG>(vtbase + (int64_t)(8 * nd + g) * vt_dim_stride + kb + 8 * t);
      mma_bf16_16816(acc[nd], pa[0][0], pa[0][1], pa[0][2], pa[0][3], w.x, w.y);
      mma_bf16_16816(acc[nd], pa[1][0], pa[1][1], pa[1][2], pa[1][3], w.z, w.w);
    }
  }
}

template <int D>
SV_DEVINL void attn_init(float (&acc)[D / 8][4], float (&mrow)[2], float (&lrow)[2]) {
#pragma unroll
  for (int nd = 0; nd < D / 8; ++nd) acc[nd][0] = acc[nd][1] = acc[nd][2] = acc[nd][3] = 0.f;
  mrow[0] = mrow[1] = -INFINITY;
  lrow[0] = lrow[1] = 0.f;
}

// ------------------------------------------------------------------------------------------
// ViT: rows of a tile are 16 consecutive queries of one (image, head).  qkv is [B*L, 3W] packed
// (in_proj output, q|k|v), vt is V^T [B][heads][64][seq_pad].
constexpr int kAttnWarps = 4;
__global__ void __launch_bounds__(kAttnWarps * 32) attention_vit_kernel(const bf16* __restrict__ qkv,
                                                                        const bf16* __restrict__ vt,
                                                                        bf16* __restrict__ out, int batch, int seq,
                                                                        int heads, int seq_pad, float scale_log2) {
  constexpr int D = 64;
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int qtiles = (seq + 15) / 16;
  const int tile = blockIdx.x * kAttnWarps + (threadIdx.x >> 5);
  if (tile >= batch * heads * qtiles) return;
  const int qt = tile % qtiles, bh = tile / qtiles, h = bh % heads, b = bh / heads;
  const int W = heads * D;
  const int64_t ld = 3 * W;
  const bf16* base = qkv + (int64_t)b * seq * ld;
  const int q_lo = qt * 16 + g, q_hi = q_lo + 8;
  uint32_t qa[D / 16][4];
  load_q_frag<D>(qa, base + (int64_t)q_lo * ld + h * D, q_lo < seq, base + (int64_t)q_hi * ld + h * D, q_hi < seq, t);
  float acc[D / 8][4], mrow[2], lrow[2];
  attn_init<D>(acc, mrow, lrow);
  attn_core<D>(qa, base + W + h * D, ld, vt + (int64_t)bh * D * seq_pad, seq_pad, 0, seq, scale_log2, acc, mrow, lrow,
               lane);
  const float inv0 = 1.0f / quad_sum(lrow[0]), inv1 = 1.0f / quad_sum(lrow[1]);
  bf16* o = out + (int64_t)b * seq * W + h * D;
#pragma unroll
  for (int nd = 0; nd < D / 8; ++nd) {
    if (q_lo < seq)
      *reinterpret_cast<uint32_t*>(o + (int64_t)q_lo * W + 8 * nd + 2 * t) = pack_bf16x2(acc[nd][0] * inv0, acc[nd][1] * inv0);
    if (q_hi < seq)
      *reinterpret_cast<uint32_t*>(o + (int64_t)q_hi * W + 8 * nd + 2 * t) = pack_bf16x2(acc[nd][2] * inv1, acc[nd][3] * inv1);
  }
}

void launch_attention_vit(const bf16* qkv, const bf16* vt, bf16* out, int batch, int seq, int heads, int seq_pad,
                          cudaStream_t st) {
  const int tiles = batch * heads * ((seq + 15) / 16);
  const float scale_log2 = 1.4426950408889634f / sqrtf(64.f);
  attention_vit_kernel<<<(tiles + kAttnWarps - 1) / kAttnWarps, kAttnWarps * 32, 0, st>>>(qkv, vt, out, batch, seq,
                                                                                       heads, seq_pad, scale_log2);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Decoder (prefill / scoring chunk): a tile = the `group` query heads of one (image, token, kv head); the token sits at
// cache position pos0 + token and takes keys [0, pos0 + token] from the cache (causal).  qkv rows are [n_head*D | n_kv*D | n_kv*D].
template <int D>
__global__ void __launch_bounds__(kAttnWarps * 32) attention_heads_kernel(
    const bf16* __restrict__ qkv, int ld, const bf16* __restrict__ kcache, const bf16* __restrict__ vtcache,
    bf16* __restrict__ out, int batch, int seq, int n_head, int n_kv, int tcap, float scale_log2, int window, int pos0) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int tile = blockIdx.x * kAttnWarps + (threadIdx.x >> 5);
  if (tile >= batch * seq * n_kv) return;
  const int kvh = tile % n_kv, bt = tile / n_kv, tok = bt % seq, b = bt / seq;
  const int group = n_head / n_kv;
  const bf16* qrow = qkv + (int64_t)bt * ld + (int64_t)kvh * group * D;
  uint32_t qa[D / 16][4];
  load_q_frag<D>(qa, qrow + (int64_t)g * D, g < group, qrow + (int64_t)(g + 8) * D, g + 8 < group, t);
  float acc[D / 8][4], mrow[2], lrow[2];
  attn_init<D>(acc, mrow, lrow);
  const int64_t bk = (int64_t)b * n_kv + kvh;
  const int qpos = pos0 + tok;
  const int key_lo = window > 0 ? max(0, qpos + 1 - window) : 0;    // HF sliding window: keys in (q - window, q]
  attn_core<D>(qa, kcache + bk * tcap * D, D, vtcache + bk * D * tcap, tcap, (key_lo / 32) * 32, qpos + 1, scale_log2, acc,
               mrow, lrow, lane, key_lo);
  const float inv0 = 1.0f / quad_sum(lrow[0]), inv1 = 1.0f / quad_sum(lrow[1]);
  bf16* o = out + (int64_t)bt * n_head * D + (int64_t)kvh * group * D;
#pragma unroll
  for (int nd = 0; nd < D / 8; ++nd) {
    if (g < group)
      *reinterpret_cast<uint32_t*>(o + (int64_t)g * D + 8 * nd + 2 * t) = pack_bf16x2(acc[nd][0] * inv0, acc[nd][1] * inv0);
    if (g + 8 < group)
      *reinterpret_cast<uint32_t*>(o + (int64_t)(g + 8) * D + 8 * nd + 2 * t) =
          pack_bf16x2(acc[nd][2] * inv1, acc[nd][3] * inv1);
  }
}

void launch_attention_heads(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache, bf16* out,
                            int batch, int seq, int n_head, int n_kv, int d, int tcap, int window, int pos0, cudaStream_t st) {
  const int tiles = batch * seq * n_kv;
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)d);
  const int ld = q_cols_total;
  attention_heads_kernel<128><<<(tiles + kAttnWarps - 1) / kAttnWarps, kAttnWarps * 32, 0, st>>>(
      qkv, ld, kcache, vtcache, out, batch, seq, n_head, n_kv, tcap, scale_log2, window, pos0);
  count_launch();
}

// ------------------------------------------------------------------------------------------
// Decode: one token per image; the key axis [0, cur_len] is split over `nsplit` warps (one CTA
// each) so every SM pulls a slice of the cache; partial (m, l, acc) go to an fp32 scratch and a
// second small kernel merges them in a fixed order (deterministic).
//   partial layout: [b][kvh][split][ 16 (m) | 16 (l) | 16*D (acc) ]
template <int D>
__global__ void __launch_bounds__(32) attention_decode_split_kernel(
    const bf16* __restrict__ qkv, int ld, const bf16* __restrict__ kcache, const bf16* __restrict__ vtcache,
    float* __restrict__ partial, const GenState* __restrict__ state, int n_head, int n_kv, int tcap, int nsplit,
    float scale_log2, int window) {
  const int lane = threadIdx.x, g = lane >> 2, t = lane & 3;
  const int split = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z;
  const int group = n_head / n_kv;
  const int nkeys = state->cur_len + 1;                       // the new token's K/V is already appended
  const int key_lo = window > 0 ? max(0, nkeys - window) : 0;
  const int blk_lo = key_lo / 32;
  const int blocks = (nkeys + 31) / 32 - blk_lo;
  const int per = (blocks + nsplit - 1) / nsplit;
  const int kb0 = (blk_lo + split * per) * 32;
  const int kb1 = min(nkeys, (blk_lo + (split + 1) * per) * 32);
  if (kb0 >= kb1) return;                                     // inactive split: the merge skips it too
  float* pout = partial + (((int64_t)b * n_kv + kvh) * nsplit + split) * (32 + 16 * D);
  float acc[D / 8][4], mrow[2], lrow[2];
  attn_init<D>(acc, mrow, lrow);
  {
    const bf16* qrow = qkv + (int64_t)b * ld + (int64_t)kvh * group * D;
    uint32_t qa[D / 16][4];
    load_q_frag<D>(qa, qrow + (int64_t)g * D, g < group, qrow + (int64_t)(g + 8) * D, g + 8 < group, t);
    const int64_t bk = (int64_t)b * n_kv + kvh;
    attn_core<D>(qa, kcache + bk * tcap * D, D, vtcache + bk * D * tcap, tcap, kb0, kb1, scale_log2, acc, mrow, lrow,
                 lane, key_lo);
  }
  const float l0 = quad_sum(lrow[0]), l1 = quad_sum(lrow[1]);
  if (t == 0) {
    pout[g] = mrow[0]; pout[g + 8] = mrow[1];
    pout[16 + g] = l0; pout[16 + g + 8] = l1;
  }
#pragma unroll
  for (int nd = 0; nd < D / 8; ++nd) {
    *reinterpret_cast<float2*>(pout + 32 + g * D + 8 * nd + 2 * t) = make_float2(acc[nd][0], acc[nd][1]);
    *reinterpret_cast<float2*>(pout + 32 + (g + 8) * D + 8 * nd + 2 * t) = make_float2(acc[nd][2], acc[nd][3]);
  }
}

template <int D>
__global__ void __launch_bounds__(D) attention_decode_merge_kernel(const float* __restrict__ partial,
                                                                   bf16* __restrict__ out,
                                                                   const GenState* __restrict__ state, int n_head,
                                                                   int n_kv, int nsplit, int window) {
  const int r = blockIdx.x, kvh = blockIdx.y, b = blockIdx.z, dim = threadIdx.x;
  const int group = n_head / n_kv;
  if (r >= group) return;
  const int nkeys = state->cur_len + 1;
  const int blocks = (nkeys + 31) / 32 - (window > 0 ? max(0, nkeys - window) : 0) / 32;
  const int per = (blocks + nsplit - 1) / nsplit;
  const int nact = (blocks + per - 1) / per;                  // splits that had keys (same rule as above)
  const float* p = partial + ((int64_t)b * n_kv + kvh) * nsplit * (32 + 16 * D);
  float M = -INFINITY;
  for (int s = 0; s < nact; ++s) M = fmaxf(M, p[(int64_t)s * (32 + 16 * D) + r]);
  float L = 0.f, A = 0.f;
  for (int s = 0; s < nact; ++s) {
    const float* ps = p + (int64_t)s * (32 + 16 * D);
    const float m = ps[r];
    const float w = (m == -INFINITY) ? 0.f : exp2f(m - M);
    L += ps[16 + r] * w;
    A += ps[32 + r * D + dim] * w;
  }
  out[(int64_t)b * n_head * D + ((int64_t)kvh * group + r) * D + dim] = __float2bfloat16_rn(A / L);
}

void launch_attention_decode(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache, bf16* out,
                             float* partial, const GenState* state, int batch, int n_head, int n_kv, int d, int tcap,
                             int nsplit, int window, cudaStream_t st) {
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)d);
  attention_decode_split_kernel<128><<<dim3(nsplit, n_kv, batch), 32, 0, st>>>(qkv, q_cols_total, kcache, vtcache,
                                                                              partial, state, n_head, n_kv, tcap,
                                                                              nsplit, scale_log2, window);
  attention_decode_merge_kernel<128><<<dim3(n_head / n_kv, n_kv, batch), 128, 0, st>>>(partial, out, state, n_head,
                                                                                      n_kv, nsplit, window);
  count_launch(2);
}

constexpr int kDecWarps = 8;

// ------------------------------------------------------------------------------------------
// Decode attention on a THREAD-BLOCK CLUSTER: the CTAs that split one image's key axis form a cluster
// (<= 8 CTAs x 8 warps = 64 key blocks per pass) and merge their partials through DISTRIBUTED SHARED
// MEMORY: no global scratch, no __threadfence, no atomic ticket, no second dependent trip to L2.
//   warp partial -> own smem -> CTA partial (own smem) -> barrier.cluster -> every CTA reads all CTA
//   partials with ld.shared::cluster for its slice of the 16x128 outputs -> bf16 store.
SV_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
SV_DEVINL float ld_dsmem(uint32_t local_addr, uint32_t cta_rank) {
  uint32_t remote;
  float v;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(cta_rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(remote) : "memory");
  return v;
}

template <int D>
__global__ void __launch_bounds__(kDecWarps * 32, 1) attention_decode_cluster_kernel(
    const bf16* __restrict__ qkv, int ld, const bf16* __restrict__ kcache, const bf16* __restrict__ vtcache,
    bf16* __restrict__ out, const GenState* __restrict__ state, int n_head, int n_kv, int tcap, float scale_log2,
    int window) {
  extern __shared__ float dsm[];                               // [kDecWarps][PSZ] warp partials | [PSZ] CTA partial
  constexpr int PSZ = 32 + 16 * D;
  float* cta_part = dsm + kDecWarps * PSZ;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // cur_len was written by the previous token's select kernel (long complete): read it before the PDL wait
  const int nkeys = state->cur_len + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int cta = blockIdx.x, ncta = gridDim.x, kvh = blockIdx.y, b = blockIdx.z;
  const int group = n_head / n_kv;
  const int key_lo = window > 0 ? max(0, nkeys - window) : 0;    // sliding window (StarCoder2): keys in (q - window, q]
  const int blk_lo = key_lo / 32, blk_hi = (nkeys + 31) / 32;
  const int per = (blk_hi - blk_lo + ncta - 1) / ncta;
  const int blk0 = blk_lo + cta * per, blk1 = min(blk_hi, blk0 + per);
  const int64_t bk = (int64_t)b * n_kv + kvh;
  asm volatile("griddepcontrol.wait;" ::: "memory");

  float acc[D / 8][4], mrow[2], lrow[2];
  attn_init<D>(acc, mrow, lrow);
  if (blk0 + warp < blk1) {
    const bf16* qrow = qkv + (int64_t)b * ld + (int64_t)kvh * group * D;
    uint32_t qa[D / 16][4];
    load_q_frag<D, true>(qa, qrow + (int64_t)g * D, g < group, qrow + (int64_t)(g + 8) * D, g + 8 < group, t);
    for (int blk = blk0 + warp; blk < blk1; blk += kDecWarps)
      attn_core<D, true, true>(qa, kcache + bk * tcap * D, D, vtcache + bk * D * tcap, tcap, blk * 32,
                               min(nkeys, blk * 32 + 32), scale_log2, acc, mrow, lrow, lane, key_lo);
  }
  float* ws = dsm + warp * PSZ;
  const float l0 = quad_sum(lrow[0]), l1 = quad_sum(lrow[1]);
  if (t == 0) { ws[g] = mrow[0]; ws[g + 8] = mrow[1]; ws[16 + g] = l0; ws[16 + g + 8] = l1; }
#pragma unroll
  for (int nd = 0; nd < D / 8; ++nd) {
    *reinterpret_cast<float2*>(ws + 32 + g * D + 8 * nd + 2 * t) = make_float2(acc[nd][0], acc[nd][1]);
    *reinterpret_cast<float2*>(ws + 32 + (g + 8) * D + 8 * nd + 2 * t) = make_float2(acc[nd][2], acc[nd][3]);
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 16 * D; idx += kDecWarps * 32) {      // CTA-level merge of the 8 warp partials
    const int r = idx / D;
    float M = -INFINITY;
#pragma unroll
    for (int w = 0; w < kDecWarps; ++w) M = fmaxf(M, dsm[w * PSZ + r]);
    float L = 0.f, A = 0.f;
#pragma unroll
    for (int w = 0; w < kDecWarps; ++w) {
      const float m = dsm[w * PSZ + r];
      const float sc = (m == -INFINITY) ? 0.f : exp2f(m - M);
      L += dsm[w * PSZ + 16 + r] * sc;
      A += dsm[w * PSZ + 32 + idx] * sc;
    }
    cta_part[32 + idx] = A;
    if (idx % D == 0) { cta_part[r] = M; cta_part[16 + r] = L; }
  }
  cluster_sync_all();                                           // every CTA's partial is complete and visible
  bf16* orow = out + (int64_t)b * n_head * D + (int64_t)kvh * group * D;
  const uint32_t base = (uint32_t)__cvta_generic_to_shared(cta_part);
  for (int idx = cta * (kDecWarps * 32) + threadIdx.x; idx < group * D; idx += ncta * kDecWarps * 32) {
    const int r = idx / D;
    float m_c[8], l_c[8], a_c[8];
    float M = -INFINITY;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (c < ncta) {
        m_c[c] = ld_dsmem(base + 4u * r, c);
        l_c[c] = ld_dsmem(base + 4u * (16 + r), c);
        a_c[c] = ld_dsmem(base + 4u * (32 + idx), c);
        M = fmaxf(M, m_c[c]);
      }
    }
    float L = 0.f, A = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (c < ncta) {
        const float sc = (m_c[c] == -INFINITY) ? 0.f : exp2f(m_c[c] - M);
        L += l_c[c] * sc;
        A += a_c[c] * sc;
      }
    }
    orow[idx] = __float2bfloat16_rn(A / L);
  }
  cluster_sync_all();                                           // nobody exits while its smem may still be read
}

int attention_decode_cluster_ncta(int total_len) {
  const int blocks = (total_len + 31) / 32;
  return std::max(1, std::min(8, (blocks + kDecWarps - 1) / kDecWarps));
}

cudaError_t attention_decode_cluster_init() {
  return cudaFuncSetAttribute(attention_decode_cluster_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (kDecWarps + 1) * (32 + 16 * 128) * (int)sizeof(float));
}

cudaError_t launch_attention_decode_cluster(const bf16* qkv, int q_cols_total, const bf16* kcache, const bf16* vtcache,
                                            bf16* out, const GenState* state, int batch, int n_head, int n_kv, int d,
                                            int tcap, int ncta, int window, bool pdl, cudaStream_t st) {
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)d);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(ncta, n_kv, batch); cfg.blockDim = dim3(kDecWarps * 32);
  cfg.dynamicSmemBytes = (kDecWarps + 1) * (32 + 16 * 128) * sizeof(float); cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = ncta; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, attention_decode_cluster_kernel<128>, qkv, q_cols_total, kcache, vtcache, out,
                                     state, n_head, n_kv, tcap, scale_log2, window);
  count_launch();
  return e;
}

}  // namespace sv
