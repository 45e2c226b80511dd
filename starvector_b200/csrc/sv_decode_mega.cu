// Per-phase decode GEMV on a shared-memory weight ring (the kernels of the CUDA-graph decode step):
//   Y[B,N] = epilogue( LayerNorm?(X)[B,K] . W[N,K]^T ),  B <= 8 image rows, one CTA per SM.
//
//   warp 8 (producer, one elected lane per row): copies [R rows x 1024 k] weight slabs into a 5-slot shared-memory ring with
//       cp.async.bulk (completion on the slot's "full" mbarrier).  It starts BEFORE the programmatic-dependency wait --
//       weights are immutable -- so ~165 KB per SM of HBM reads are in flight while the previous kernel drains.
//   warps 0-7 (consumers): LayerNorm prologue on register-resident activation fragments, 128-bit MMA fragments from the slot
//       (row pitch = 2 KB + 64 B, bank-conflict free), mma.sync m16n8k16 (weights = A, the <= 8 image rows = B), slot
//       release ("empty" mbarrier, one arrive per warp), deterministic cross-warp split-K reduction and the reference's
//       bf16 epilogue (bias, gelu, residual, KV-cache append, argmax partials).
//
// Work split: N output rows are tiled R <= 16 rows at a time so that every CTA owns the same number of rows
// (2048 -> 147 x 14, 2304 -> 144 x 16, 8192 -> 147 x 4 x 14, 49156 -> 147 x 21 x 16).  Every wait is bounded and traps.
// (Round 1's barrier-synchronised persistent kernel lived here too; the dataflow kernel in sv_decode_flow.cu replaces it.)
#include <cstdio>
#include <cstdlib>

#include "sv_kernels.h"
#include "sv_ring.cuh"
#include "sv_select.cuh"

namespace sv {
namespace mega {


enum { EPI_PLAIN = 0, EPI_QKV = 1, EPI_LMHEAD = 2 };

struct Ctx {
  const Args* a;
  uint8_t* smem;
  int cta, ncta, warp, lane, g, t;
  float* red;     // [2][NWC][16][8]
  float* stat;    // [NWC][8]
  // optional (per-phase ring kernels): parameters staged into shared memory BEFORE the programmatic-dependency wait, so that
  // their HBM misses overlap the previous kernel's tail instead of sitting on this kernel's critical path
  uint32_t ln_s = 0;            // shared address of [ln_w row | ln_b row] (K bf16 each), 0 = read them from global
  const float* bias_s = nullptr;   // [tile][16] biases of this CTA's output rows
};

// ---- consumer: one GEMV phase  Y[B,N] = epi( LN?(X)[B,K] . W[N,K]^T )
// LN_BIGK compiles in the LayerNorm path for phases of more than two slabs (K > 2048, or a K only a narrow slab divides);
// the other kernels are instantiated without it so their register allocation is untouched.
template <bool HAS_LN, int EPI, bool LN_BIGK = false>
SV_DEVINL void gemv_phase(const Ctx& cx, Ring& r, const bf16* __restrict__ X, const bf16* __restrict__ bias,
                          const bf16* res, bf16* Y, int N, int K, int act, const bf16* __restrict__ ln_w,
                          const bf16* __restrict__ ln_b, const Layer* L) {
  const Args& a = *cx.a;
  const Plan p = make_plan(N, K, cx.cta, cx.ncta);
  const int warp = cx.warp, g = cx.g, t = cx.t;
  const int cps = p.KS >> 5;                         // 32-wide chunks per slot row
  const int cpws = (cps + NWC - 1) / NWC;            // chunks per warp per slot (<= CPW)
  const bool row_ok = g < a.B;
  const bf16* xp = X + (int64_t)(row_ok ? g : 0) * K + 8 * t;
  const bool big_k = p.nstg > 2;

  // activations for the whole phase live in registers when K <= 2048 (8 fragments per lane)
  uint4 xr[2 * CPW];
#pragma unroll
  for (int i = 0; i < 2 * CPW; ++i) xr[i] = make_uint4(0u, 0u, 0u, 0u);
  if (!big_k && p.ntile > 0) {
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
      for (int j = 0; j < CPW; ++j) {
        const int cl = warp + NWC * j;
        const bool okc = ks < p.nstg && j < cpws && cl < cps;
        if (okc && row_ok) xr[ks * CPW + j] = ldcg16(xp + (ks * cps + cl) * 32);
      }
    }
    if constexpr (HAS_LN) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 2 * CPW; ++i) {
        float f[8];
        unpack8(xr[i], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += f[j];
      }
      s = quad_sum(s);
      if (t == 0) cx.stat[warp * 8 + g] = s;
      consumer_sync();
      float mean = 0.f;
#pragma unroll
      for (int w = 0; w < NWC; ++w) mean += cx.stat[w * 8 + g];
      mean /= (float)K;
      float q = 0.f;
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const bool okc = ks < p.nstg && j < cpws && (warp + NWC * j) < cps;
          if (okc) {
            float f[8];
            unpack8(xr[ks * CPW + j], f);
#pragma unroll
            for (int e = 0; e < 8; ++e) { const float dlt = f[e] - mean; q += dlt * dlt; }
          }
        }
      }
      q = quad_sum(q);
      consumer_sync();
      if (t == 0) cx.stat[warp * 8 + g] = q;
      consumer_sync();
      float var = 0.f;
#pragma unroll
      for (int w = 0; w < NWC; ++w) var += cx.stat[w * 8 + g];
      const float rstd = 1.0f / sqrtf(var / (float)K + a.ln_eps);
      // (the weight ring keeps HBM busy on its own, so the LN affine is fetched late to save registers)
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int cl = warp + NWC * j;
          const bool okc = ks < p.nstg && j < cpws && cl < cps;
          float f[8], wf[8], bfv[8];
          unpack8(xr[ks * CPW + j], f);
          const int ch = okc ? ks * cps + cl : 0;
          if (cx.ln_s) {
            unpack8(lds16(cx.ln_s + (ch * 32 + 8 * t) * 2), wf);
            unpack8(lds16(cx.ln_s + (K + ch * 32 + 8 * t) * 2), bfv);
          } else {
            unpack8(ldg_cached(ln_w + ch * 32 + 8 * t), wf);
            unpack8(ldg_cached(ln_b + ch * 32 + 8 * t), bfv);
          }
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = (row_ok && okc) ? (f[e] - mean) * rstd * wf[e] + bfv[e] : 0.f;
          xr[ks * CPW + j] = pack8(f);       // ln output is a bf16 tensor in the reference; 0 on padded chunks
        }
      }
    }
  }

  // LayerNorm with K > 2048 (StarCoder2: H = 4608): row statistics in two streaming passes over x (L2 resident),
  // the normalisation itself happens per slab inside the MMA loop.
  float ln_mean = 0.f, ln_rstd = 1.f;
  if constexpr (HAS_LN && LN_BIGK) {
    if (big_k && p.ntile > 0) {
      float sv = 0.f;
      for (int ks = 0; ks < p.nstg; ++ks) {
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int cl = warp + NWC * j;
          if (row_ok && j < cpws && cl < cps) {
            float f[8];
            unpack8(ldcg16(xp + (ks * cps + cl) * 32), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) sv += f[e];
          }
        }
      }
      sv = quad_sum(sv);
      if (t == 0) cx.stat[warp * 8 + g] = sv;
      consumer_sync();
#pragma unroll
      for (int w = 0; w < NWC; ++w) ln_mean += cx.stat[w * 8 + g];
      ln_mean /= (float)K;
      float q = 0.f;
      for (int ks = 0; ks < p.nstg; ++ks) {
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int cl = warp + NWC * j;
          if (row_ok && j < cpws && cl < cps) {
            float f[8];
            unpack8(ldcg16(xp + (ks * cps + cl) * 32), f);
#pragma unroll
            for (int e = 0; e < 8; ++e) { const float dlt = f[e] - ln_mean; q += dlt * dlt; }
          }
        }
      }
      q = quad_sum(q);
      consumer_sync();
      if (t == 0) cx.stat[warp * 8 + g] = q;
      consumer_sync();
      float var = 0.f;
#pragma unroll
      for (int w = 0; w < NWC; ++w) var += cx.stat[w * 8 + g];
      ln_rstd = 1.0f / sqrtf(var / (float)K + a.ln_eps);
    }
  }

  float c[4] = {0.f, 0.f, 0.f, 0.f};
  int pos_now = 0;
  if constexpr (EPI == EPI_QKV) pos_now = __ldcg(&a.state->cur_len);         // read here, not behind the last MMA
  for (int tl = 0; tl < p.ntile; ++tl) {
    const int tile = p.tile0 + tl;
    // the epilogue thread's residual value: requested now, used after the MMAs (an L2 round trip off the tail)
    float res_pre = 0.f;
    {
      const int n_ = threadIdx.x & 15, mm_ = threadIdx.x >> 4, col_ = tile * p.R + n_;
      if (res != nullptr && threadIdx.x < 128 && n_ < p.R && col_ < N && mm_ < a.B) res_pre = __bfloat162float(__ldcg(res + (int64_t)mm_ * N + col_));
    }
    if (!big_k) {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        if (ks < p.nstg) {
          mbar_wait(r.full0 + 8u * r.slot, r.phase);
          const uint32_t sb = r.base + r.slot * SLOT_BYTES + g * p.pitch + t * 16;
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            const int cl = warp + NWC * j;
            if (j < cpws && cl < cps) {
              const uint4 lo = lds16(sb + cl * 64), hi = lds16(sb + 8 * p.pitch + cl * 64);
              const uint4 xv = xr[ks * CPW + j];
              mma_bf16_16816(c, lo.x, hi.x, lo.y, hi.y, xv.x, xv.y);
              mma_bf16_16816(c, lo.z, hi.z, lo.w, hi.w, xv.z, xv.w);
            }
          }
          __syncwarp();
          if (cx.lane == 0) mbar_arrive(r.empty0 + 8u * r.slot);
          r.advance();
        }
      }
    } else {
      // K > 2048: activation fragments are fetched per slab from L2, one slab ahead of their use (with HAS_LN the
      // LayerNorm affine of the same columns rides along and the fragment is normalised after the slab's MMAs).
      constexpr bool LNB = HAS_LN && LN_BIGK;
      uint4 xc[CPW], xn[CPW], wn[LNB ? CPW : 1], bn[LNB ? CPW : 1];
      auto fetch = [&](int ks) {
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int cl = warp + NWC * j;
          const bool okc = ks < p.nstg && j < cpws && cl < cps;
          const int ch = okc ? ks * cps + cl : 0;
          xn[j] = (row_ok && okc) ? ldcg16(xp + ch * 32) : make_uint4(0u, 0u, 0u, 0u);
          if constexpr (LNB) {
            wn[j] = okc ? ldg_cached(ln_w + ch * 32 + 8 * t) : make_uint4(0u, 0u, 0u, 0u);
            bn[j] = okc ? ldg_cached(ln_b + ch * 32 + 8 * t) : make_uint4(0u, 0u, 0u, 0u);
          }
        }
      };
      auto promote = [&](int ks) {             // xn (raw) -> xc (what the MMAs consume)
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          if constexpr (LNB) {
            const bool okc = ks < p.nstg && j < cpws && (warp + NWC * j) < cps;
            float f[8], wf[8], bfv[8];
            unpack8(xn[j], f); unpack8(wn[j], wf); unpack8(bn[j], bfv);
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = (row_ok && okc) ? (f[e] - ln_mean) * ln_rstd * wf[e] + bfv[e] : 0.f;
            xc[j] = pack8(f);
          } else {
            xc[j] = xn[j];
          }
        }
      };
      fetch(0);
      promote(0);
      for (int ks = 0; ks < p.nstg; ++ks) {
        fetch(ks + 1);
        mbar_wait(r.full0 + 8u * r.slot, r.phase);
        const uint32_t sb = r.base + r.slot * SLOT_BYTES + g * p.pitch + t * 16;
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          const int cl = warp + NWC * j;
          if (j < cpws && cl < cps) {
            const uint4 lo = lds16(sb + cl * 64), hi = lds16(sb + 8 * p.pitch + cl * 64);
            mma_bf16_16816(c, lo.x, hi.x, lo.y, hi.y, xc[j].x, xc[j].y);
            mma_bf16_16816(c, lo.z, hi.z, lo.w, hi.w, xc[j].z, xc[j].w);
          }
        }
        __syncwarp();
        if (cx.lane == 0) mbar_arrive(r.empty0 + 8u * r.slot);
        r.advance();
        promote(ks + 1);
      }
    }
    // ---- tile finished: deterministic cross-warp split-K reduction + epilogue
    float* rd = cx.red + (tl & 1) * (NWC * 16 * 8);
    rd[(warp * 16 + g) * 8 + 2 * t] = c[0]; rd[(warp * 16 + g) * 8 + 2 * t + 1] = c[1];
    rd[(warp * 16 + g + 8) * 8 + 2 * t] = c[2]; rd[(warp * 16 + g + 8) * 8 + 2 * t + 1] = c[3];
    c[0] = c[1] = c[2] = c[3] = 0.f;
    consumer_sync();
    if (threadIdx.x < 128) {
      const int n = threadIdx.x & 15, mm = threadIdx.x >> 4;
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < NWC; ++w) acc += rd[(w * 16 + n) * 8 + mm];
      const int col = tile * p.R + n;
      const bool ok = n < p.R && col < N && mm < a.B;
      float v = 0.f, v_bf = 0.f;          // v_bf: the value as the bf16 logits tensor holds it
      if (ok) {
        const float bv = bias ? (cx.bias_s ? cx.bias_s[tl * 16 + n] : __bfloat162float(bias[col])) : 0.f;
        const float rv = res_pre;
        v = epilogue_elem(acc, bv, act, res != nullptr, rv);
        const bf16 vb = __float2bfloat16_rn(v);
        v_bf = __bfloat162float(vb);
        Y[(int64_t)mm * N + col] = vb;
        if constexpr (EPI == EPI_QKV) {
          const int q_cols = a.n_head * D, j = col - q_cols;
          const int pos = pos_now;
          if (j >= 0 && pos < a.tcap) {
            if (j < a.n_kv * D) {
              const int kvh = j / D, dim = j % D;
              L->kc[(((int64_t)mm * a.n_kv + kvh) * a.tcap + pos) * D + dim] = vb;
            } else {
              const int jj = j - a.n_kv * D, kvh = jj / D, dim = jj % D;
              L->vc[(((int64_t)mm * a.n_kv + kvh) * D + dim) * a.tcap + pos] = vb;
            }
          }
        }
      }
      if constexpr (EPI == EPI_LMHEAD) {
        // greedy = argmax over the bf16 logits cast to float, lowest index wins ties (HF _sample): reduce the ROUNDED value
        float bv = ok ? v_bf : -INFINITY;
        int bi = ok ? col : 0x7fffffff;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if (n == 0 && mm < a.B) {
          a.amax_val[(int64_t)tile * 8 + mm] = bv;
          a.amax_idx[(int64_t)tile * 8 + mm] = bi;
        }
      }
    }
    // red[] is double-buffered by tile parity: one barrier per tile
  }
}


// ------------------------------------------------------------------------------------------
// One-phase kernels of the per-phase CUDA-graph decode path: a producer warp
// streams this GEMV's slabs through shared memory (starting before the PDL dependency wait, weights
// are immutable), 8 consumer warps do LayerNorm prologue / MMA / epilogue.  ~165 KB of HBM reads
// in flight per SM instead of the 64 KB a register-landing GEMV can hold.
struct RingGemvArgs {
  Args a;            // B, ln_eps, n_head, n_kv, tcap, state, amax_* (fields the epilogues read)
  Layer L;           // kc / vc for the QKV epilogue
  const bf16 *X, *W, *bias, *res, *ln_w, *ln_b;
  const uint8_t* Wt; // slab-tiled copy of W (one bulk copy per ring slot) or nullptr
  bf16* Y;
  int N, K, act;
  int nslots;        // ring depth of THIS launch
};

// The c_attn GEMV's producer warp is idle once its two slabs are on their way: it pulls the K / V^T rows the NEXT kernel (the
// decode attention) will read into L2 -- one 4-byte ld.global.cg with the L2::128B prefetch size per 128-byte line, the lines
// dealt round-robin over all CTAs and lanes (scripts/l2_prefetch_test.cu: this, unlike cp.async.bulk.prefetch.L2, leaves the
// region L2-resident).  The attention's dependent K -> softmax -> V loads then cost L2, not HBM, latency.
SV_DEVINL void l2_prefetch_kv(const bf16* kc, const bf16* vc, int nkeys, int nbk, int tcap, int cta, int ncta, int lane) {
  if (nkeys <= 0) return;
  const int klines = (nkeys * D * 2 + 127) >> 7;                 // per (image, kv head): K rows are contiguous
  const int vlines_row = (nkeys * 2 + 127) >> 7, vlines = D * vlines_row;
  const int per_bk = klines + vlines, total = nbk * per_bk;
  uint32_t acc = 0;
  for (int i = cta + ncta * lane; i < total; i += ncta * 32) {
    const int bk = i / per_bk, r = i % per_bk;
    const char* p = r < klines ? reinterpret_cast<const char*>(kc + (int64_t)bk * tcap * D) + (int64_t)r * 128
                               : reinterpret_cast<const char*>(vc + ((int64_t)bk * D + (r - klines) / vlines_row) * tcap) + (int64_t)((r - klines) % vlines_row) * 128;
    uint32_t v;
    asm volatile("ld.global.cg.L2::128B.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    acc ^= v;
  }
  if (acc == 0x9e3779b9u && nkeys < 0) asm volatile("trap;");     // (never: keeps the loads' results alive)
}
constexpr int RING_BIAS_TILES = 8;     // biases staged for up to this many tiles per CTA (mlp.c_fc has 4)
SV_DEVINL constexpr int ring_smem_bytes(int nslots) {
  return nslots * SLOT_BYTES + RED_BYTES + NWC * 8 * 4 + 2 * 8 * 8 + 16 + 2 * 2 * KS_MAX * 2 + RING_BIAS_TILES * 16 * 4 + 256;
}

// (A 2-CTA/SM register budget (96 regs) so that consecutive kernels co-reside under PDL was measured 25% slower.)
template <bool HAS_LN, int EPI, bool LN_BIGK = false>
__global__ void __launch_bounds__(NTHREADS, RING_MINBLOCKS) gemv_ring_kernel(const RingGemvArgs ra) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cta = blockIdx.x, ncta = gridDim.x;
  const int off_red = ra.nslots * SLOT_BYTES, off_stat = off_red + RED_BYTES, off_bar = off_stat + NWC * 8 * 4;
  Ring ring;
  ring.base = smem_u32(smem);
  ring.full0 = smem_u32(smem + off_bar);
  ring.empty0 = ring.full0 + 8u * 8;
  ring.slot = 0; ring.phase = 0; ring.nslots = (uint32_t)ra.nslots;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ra.nslots; ++s) { mbar_init(ring.full0 + 8u * s, 1); mbar_init(ring.empty0 + 8u * s, NWC); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == NWC) {
    if (ra.Wt != nullptr) produce_phase_tiled(ring, ra.Wt, ra.N, ra.K, cta, ncta, lane);
    else produce_phase(ring, ra.W, ra.N, ra.K, cta, ncta, lane);     // no dependency on the previous kernel
    if constexpr (EPI == EPI_QKV)
      l2_prefetch_kv(ra.L.kc, ra.L.vc, ra.a.state->cur_len, ra.a.B * ra.a.n_kv, ra.a.tcap, cta, ncta, lane);
    return;
  }
  Ctx cx;
  cx.a = &ra.a; cx.smem = smem; cx.cta = cta; cx.ncta = ncta; cx.warp = warp; cx.lane = lane; cx.g = lane >> 2; cx.t = lane & 3;
  cx.red = reinterpret_cast<float*>(smem + off_red);
  cx.stat = reinterpret_cast<float*>(smem + off_stat);
  // immutable parameters (LayerNorm affine, biases of this CTA's rows) are staged into shared memory before the wait on the
  // previous kernel: their HBM misses (~1 us each, two per LayerNorm kernel, one per epilogue) overlap that kernel's tail
  {
    const int off_par = (off_bar + 2 * 8 * 8 + 15) & ~15;
    if (HAS_LN && !LN_BIGK && ra.K <= 2 * KS_MAX) {
      cx.ln_s = smem_u32(smem + off_par);
      const int nv = ra.K / 8;                                   // 16-byte vectors per row
      for (int i = threadIdx.x; i < 2 * nv; i += NCT)
        *reinterpret_cast<uint4*>(smem + off_par + i * 16) = ldg_cached((i < nv ? ra.ln_w : ra.ln_b) + (i % nv) * 8);
    }
    if (ra.bias != nullptr) {
      float* bs = reinterpret_cast<float*>(smem + off_par + 2 * 2 * KS_MAX * 2);
      const Plan p = make_plan(ra.N, ra.K, cta, ncta);
      if (p.tpc <= RING_BIAS_TILES) {
        for (int i = threadIdx.x; i < p.ntile * 16; i += NCT) {
          const int col = (p.tile0 + i / 16) * p.R + (i % 16);
          bs[i] = (i % 16) < p.R && col < ra.N ? __bfloat162float(ra.bias[col]) : 0.f;
        }
        cx.bias_s = bs;
      }
    }
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  gemv_phase<HAS_LN, EPI, LN_BIGK>(cx, ring, ra.X, ra.bias, ra.res, ra.Y, ra.N, ra.K, ra.act, ra.ln_w, ra.ln_b, &ra.L);
}

}  // namespace mega

// ---- host side
// ---- per-phase ring GEMV launchers (used by the CUDA-graph decode path)
template <bool HAS_LN, int EPI, bool LN_BIGK = false>
static void launch_ring_t(const mega::RingGemvArgs& ra, int ncta, bool pdl, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(ncta); cfg.blockDim = dim3(mega::NTHREADS); cfg.stream = st;
  cfg.dynamicSmemBytes = mega::ring_smem_bytes(ra.nslots);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, mega::gemv_ring_kernel<HAS_LN, EPI, LN_BIGK>, ra);
  count_launch();
}

cudaError_t gemv_ring_init() {   // set the shared-memory opt-in outside of any stream capture
  cudaError_t e;
#define SV_RING_ATTR(LN, EPI)                                                                                          \
  e = cudaFuncSetAttribute(mega::gemv_ring_kernel<LN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, mega::SMEM_BYTES); \
  if (e != cudaSuccess) return e;
  SV_RING_ATTR(true, mega::EPI_QKV) SV_RING_ATTR(true, mega::EPI_PLAIN) SV_RING_ATTR(true, mega::EPI_LMHEAD)
  SV_RING_ATTR(false, mega::EPI_PLAIN)
#undef SV_RING_ATTR
  e = cudaFuncSetAttribute(mega::gemv_ring_kernel<true, mega::EPI_QKV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mega::SMEM_BYTES);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(mega::gemv_ring_kernel<true, mega::EPI_PLAIN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mega::SMEM_BYTES);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(mega::gemv_ring_kernel<true, mega::EPI_LMHEAD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mega::SMEM_BYTES);
  if (e != cudaSuccess) return e;
  return cudaSuccess;
}

bool gemv_ring_supported(int K, bool has_ln) { (void)has_ln; return K >= 32 && K % 32 == 0; }

// CTAs of one ring GEMV: one per SM in every build.  With RING_MINBLOCKS = 2 the CTA is small enough for two per SM, and
// the second slot is deliberately left free: it is where the NEXT kernel's CTA (launched early through PDL) becomes
// resident and starts filling its ring while this kernel is still computing.
int gemv_ring_ncta() {
  int dev = 0, nsm = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  return nsm;
}

int gemv_ring_ntiles(int N) {
  const int nsm = gemv_ring_ncta();
  const int rows_per_cta = (N + nsm - 1) / nsm, tpc = (rows_per_cta + 15) / 16, R = (rows_per_cta + tpc - 1) / tpc;
  return (N + R - 1) / R;
}

void launch_gemv_ring(const RingGemvLaunch& g, cudaStream_t st) {
  mega::RingGemvArgs ra{};
  ra.a.B = g.B; ra.a.ln_eps = g.ln_eps; ra.a.n_head = g.n_head; ra.a.n_kv = g.n_kv; ra.a.tcap = g.tcap; ra.a.state = const_cast<GenState*>(g.state);
  ra.a.amax_val = g.amax_val; ra.a.amax_idx = g.amax_idx;
  ra.L.kc = g.kcache; ra.L.vc = g.vtcache;
  ra.X = g.X; ra.W = g.W; ra.Wt = g.Wt; ra.bias = g.bias; ra.res = g.res; ra.ln_w = g.ln_w; ra.ln_b = g.ln_b; ra.Y = g.Y;
  ra.N = g.N; ra.K = g.K; ra.act = g.act;
  const int nsm = gemv_ring_ncta();
  int nstg = 1;
  {   // ring depth: what this CTA will stream, capped so the next kernel's CTA can co-reside (227 KB per SM)
    static int cap = 0;
    if (cap == 0) { const char* c = getenv("SV_RING_SLOTS"); cap = c ? atoi(c) : mega::STAGES; if (cap < 1 || cap > 6) cap = mega::STAGES; }
    const int rows_per_cta = (g.N + nsm - 1) / nsm, tpc = (rows_per_cta + 15) / 16;
    int ks = 32;
    for (int c : {1024, 768, 512, 256, 128, 64}) if (c <= g.K && g.K % c == 0) { ks = c; break; }
    nstg = g.K / ks;
    const int need = tpc * nstg;
    ra.nslots = need < cap ? need : cap;
    if (ra.nslots < 1) ra.nslots = 1;
  }
  const bool ln = g.ln_w != nullptr;
  // More than two slabs (every K > 2048, and narrower K that only a small slab divides, e.g. 640 = 5 x 128): the activations
  // are streamed per slab, and only the LN_BIGK instantiations normalise them there.
  if (ln && nstg > 2) {
    if (g.epi == mega::EPI_LMHEAD) launch_ring_t<true, mega::EPI_LMHEAD, true>(ra, nsm, g.pdl, st);
    else if (g.epi == mega::EPI_QKV) launch_ring_t<true, mega::EPI_QKV, true>(ra, nsm, g.pdl, st);
    else launch_ring_t<true, mega::EPI_PLAIN, true>(ra, nsm, g.pdl, st);
    return;
  }
  if (ln && g.epi == mega::EPI_QKV) launch_ring_t<true, mega::EPI_QKV>(ra, nsm, g.pdl, st);
  else if (ln && g.epi == mega::EPI_LMHEAD) launch_ring_t<true, mega::EPI_LMHEAD>(ra, nsm, g.pdl, st);
  else if (ln) launch_ring_t<true, mega::EPI_PLAIN>(ra, nsm, g.pdl, st);
  else launch_ring_t<false, mega::EPI_PLAIN>(ra, nsm, g.pdl, st);
}

}  // namespace sv
