// Large-M linear layer on the 5th-gen tensor cores: y[M,N] = epilogue(x[M,K] . w[N,K]^T + bias).
// Used by the ViT blocks, the adapter and the decoder prefill (every GEMM with M >= ~64 rows).
//
// Structure (one 128 x BN output tile per CTA, warp-specialised, 192 threads):
//   warp 0   : TMA producer - cp.async.bulk.tensor.2d loads of the 128x64 activation tile and the
//              BNx64 weight tile (both K-major, 128-byte swizzle) into a STAGES-deep smem ring,
//              completion signalled on per-stage "full" mbarriers (expect_tx).
//   warp 1   : TMEM owner + MMA issuer - one elected lane issues 4 x tcgen05.mma (128 x BN x 16,
//              kind::f16, bf16 in / fp32 accumulate in TMEM) per stage and releases the stage with
//              tcgen05.commit on its "empty" mbarrier; a final commit signals the epilogue.
//   warps 2-5: epilogue - tcgen05.ld (32 lanes x 32 columns per warp-instruction) TMEM -> registers,
//              bias / activation / residual with the reference's bf16 rounding points, 16-byte
//              global stores.  Warp w may only touch TMEM lanes 32*(w%4)..+31, so warps 2,3,4,5 own
//              row quadrants 2,3,0,1 of the tile.
// Rows beyond M and weight rows beyond N are zero-filled by TMA (OOB fill) and masked at the store.
// Every mbarrier wait is bounded: a protocol bug traps (CUDA error) instead of hanging the GPU.
//
// A second epilogue kind (EPI_LOGPS, the scoring lm_head) keeps the same producer / MMA warps and replaces the bf16 store:
// each accumulator is rounded to bf16 (the reference lm_head's output), scaled by 1/temperature in fp32 and reduced per
// row to a partial (max, sum exp(x - max)) over the tile's columns < N; the row's target logit is written by the one
// tile that holds it, and the unscaled fp32 logits optionally go to a row-mapped output.  logps_merge_kernel combines the
// partials in a fixed tile order (deterministic).
#include <cuda.h>

#include <cstdlib>
#include <map>
#include <mutex>
#include <tuple>

#include "sv_kernels.h"

namespace sv {

namespace tc05 {

constexpr int BM = 128;
constexpr int BK = 64;                 // 64 bf16 = 128 bytes = one swizzle row
constexpr int kThreads = 192;

template <int BN> struct Cfg {
  static constexpr int kStageBytes = BM * BK * 2 + BN * BK * 2;
#ifndef SV_TC05_STAGES64
#define SV_TC05_STAGES64 4
#define SV_TC05_STAGES128 3
#define SV_TC05_MINCTAS 2
#endif
  static constexpr int kStages = (BN == 128) ? SV_TC05_STAGES128 : SV_TC05_STAGES64;   // ~96 KB per CTA: CTAs share an SM
  static constexpr int kBarBytes = 256;
  static constexpr int kSmemBytes = kStages * kStageBytes + kBarBytes + 1024;   // +1024: manual 1 KiB alignment
  static constexpr uint32_t kTmemCols = BN < 32 ? 32 : BN;                      // power of two >= 32
};

SV_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

SV_DEVINL void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
SV_DEVINL void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
SV_DEVINL void mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t it = 0;; ++it) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) return;
    if (it > (1u << 20)) __trap();   // ~seconds: pipeline protocol broken -> fail loudly, never hang
  }
}
SV_DEVINL void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(x), "r"(y) : "memory");
}
SV_DEVINL void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
SV_DEVINL void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
SV_DEVINL void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 128 x BN x 16, bf16 -> fp32.
SV_DEVINL void tcgen05_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor (PTX "matrix descriptor", sm_100 format):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major) | SBO>>4 [32,46) = 1024 B between
// 8-row groups | version=1 [46,48) | layout_type=2 (SWIZZLE_128B) [61,64).
SV_DEVINL uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor, kind::f16: D=f32 (bits 4-5 = 1), A=B=bf16 (bits 7-9, 10-12 = 1), both
// K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29).
SV_DEVINL constexpr uint32_t make_idesc(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

SV_DEVINL void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

enum { EPI_LINEAR = 0, EPI_LOGPS = 1 };

template <int BN, int EPI>
__global__ void __launch_bounds__(kThreads, SV_TC05_MINCTAS) linear_tc05_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                  const __grid_constant__ CUtensorMap tmap_w,
                                                                  const bf16* __restrict__ bias,
                                                                  const bf16* __restrict__ res, bf16* __restrict__ Y,
                                                                  int M, int N, int K, int act, const LogpsEpilogue lp) {
  using C = Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars = base + C::kStages * C::kStageBytes;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (C::kStages + s); };
  const uint32_t accum_bar = bars + 8u * (2 * C::kStages);
  const uint32_t tmem_slot = bars + 8u * (2 * C::kStages + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_blk = blockIdx.x, m_blk = blockIdx.y;
  const int nk = K / BK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
  }
  if (warp == 1) {   // whole warp: allocate the accumulator columns, publish the TMEM base address
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(C::kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < nk; ++kb) {
        const int s = kb % C::kStages;
        const uint32_t ph = (uint32_t)(kb / C::kStages) & 1u;
        mbar_wait(empty_bar(s), ph ^ 1u);
        const uint32_t a_smem = base + s * C::kStageBytes;
        const uint32_t b_smem = a_smem + BM * BK * 2;
        mbar_expect_tx(full_bar(s), C::kStageBytes);
        tma_load_2d(a_smem, &tmap_x, full_bar(s), kb * BK, m_blk * BM);
        tma_load_2d(b_smem, &tmap_w, full_bar(s), kb * BK, n_blk * BN);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BM, BN);
      for (int kb = 0; kb < nk; ++kb) {
        const int s = kb % C::kStages;
        const uint32_t ph = (uint32_t)(kb / C::kStages) & 1u;
        mbar_wait(full_bar(s), ph);
        tcgen05_fence_after();
        const uint32_t a_smem = base + s * C::kStageBytes;
        const uint32_t b_smem = a_smem + BM * BK * 2;
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // advance 16 elements (32 bytes) along K inside the 128-byte swizzle row
          const uint64_t a_desc = make_sw128_desc(a_smem + k * 32);
          const uint64_t b_desc = make_sw128_desc(b_smem + k * 32);
          tcgen05_mma_f16(tmem_base, a_desc, b_desc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
        }
        tcgen05_commit(empty_bar(s));      // smem stage reusable once these MMAs have read it
      }
      tcgen05_commit(accum_bar);           // accumulator complete
    }
  } else {
    mbar_wait(accum_bar, 0);
    tcgen05_fence_after();
    const int quad = warp & 3;             // TMEM lane quadrant this warp may access
    const int row = m_blk * BM + quad * 32 + lane;
    const bool has_res = res != nullptr;
    if constexpr (EPI == EPI_LOGPS) {      // one thread = one row of the tile: no cross-thread reduction
      const bool live = row < M;
      const int tgt = live ? lp.tgt[row] : -1;
      const int lrow = (live && lp.logits) ? (lp.lg_row ? lp.lg_row[row] : row) : -1;
      float* lout = lrow >= 0 ? lp.logits + (int64_t)lrow * N : nullptr;
      float mx = -INFINITY, sum = 0.f, tval = 0.f;
      bool found = false;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);   // whole warp (sync.aligned)
        const int col0 = n_blk * BN + c0;
        if (!live || col0 >= N) continue;
        float lg[32];
        float cm = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          lg[j] = bf16_round(__uint_as_float(r[j]));
          if (col0 + j < N) cm = fmaxf(cm, lg[j] * lp.inv_temp);
        }
        if (cm > mx) { sum *= expf(mx - cm); mx = cm; }
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float xs = lg[j] * lp.inv_temp;
          if (col0 + j < N) sum += expf(xs - mx);
          if (col0 + j == tgt) { tval = xs; found = true; }
        }
        if (lout) {
          if (col0 + 32 <= N && (N & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(lout + col0 + j) = make_float4(lg[j], lg[j + 1], lg[j + 2], lg[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < N) lout[col0 + j] = lg[j];
          }
        }
      }
      if (live) {
        lp.part[(int64_t)row * gridDim.x + n_blk] = make_float2(mx, sum);
        if (found) lp.tlogit[row] = tval;
      }
      tcgen05_fence_before();
    } else {
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, r);
      const int col0 = n_blk * BN + c0;
      if (row < M) {
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int col = col0 + 8 * v;
          if (col + 8 <= N) {
            float bv[8], rv[8], o[8];
            if (bias) unpack8(ldg_cached(bias + col), bv);
            else { for (int j = 0; j < 8; ++j) bv[j] = 0.f; }
            if (has_res) unpack8(ldg_cached(res + (int64_t)row * N + col), rv);
            else { for (int j = 0; j < 8; ++j) rv[j] = 0.f; }
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = epilogue_elem(__uint_as_float(r[8 * v + j]), bv[j], act, has_res, rv[j]);
            *reinterpret_cast<uint4*>(Y + (int64_t)row * N + col) = pack8(o);
          }
        }
      }
    }
    tcgen05_fence_before();
    }
  }
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::kTmemCols) : "memory");
  }
}

// ---- host side: tensor maps through the driver entry point (no link-time libcuda dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2-D bf16 row-major [rows, cols] tensor, box = [box_rows, 64 cols], 128-byte swizzle, zero OOB fill.
static bool make_map(CUtensorMap* m, const void* ptr, int64_t rows, int64_t cols, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

struct MapKey {
  const void* p; int64_t rows, cols; int box;
  bool operator<(const MapKey& o) const { return std::tie(p, rows, cols, box) < std::tie(o.p, o.rows, o.cols, o.box); }
};
static std::mutex g_map_mu;
static std::map<MapKey, CUtensorMap> g_maps;

static bool cached_map(CUtensorMap* out, const void* ptr, int64_t rows, int64_t cols, int box_rows) {
  std::lock_guard<std::mutex> lk(g_map_mu);
  MapKey k{ptr, rows, cols, box_rows};
  auto it = g_maps.find(k);
  if (it == g_maps.end()) {
    CUtensorMap m;
    if (!make_map(&m, ptr, rows, cols, box_rows)) return false;
    if (g_maps.size() > 4096) g_maps.clear();
    it = g_maps.emplace(k, m).first;
  }
  *out = it->second;
  return true;
}

template <int BN, int EPI = EPI_LINEAR>
static cudaError_t launch(const bf16* x, const bf16* w, const bf16* bias, const bf16* res, bf16* y, int M, int N,
                          int K, int act, cudaStream_t st, const LogpsEpilogue& lp = LogpsEpilogue{}) {
  CUtensorMap mx, mw;
  if (!cached_map(&mx, x, M, K, BM) || !cached_map(&mw, w, N, K, BN)) return cudaErrorInvalidValue;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(linear_tc05_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg<BN>::kSmemBytes);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM);
  linear_tc05_kernel<BN, EPI><<<grid, kThreads, Cfg<BN>::kSmemBytes, st>>>(mx, mw, bias, res, y, M, N, K, act, lp);
  count_launch();
  return cudaGetLastError();
}

// One warp per row: lse = m + log(sum_i s_i * exp(m_i - m)) over the row's tile partials, lanes taking tiles lane,
// lane + 32, ... and a fixed shuffle tree after that (the same bits on every run); logp = target logit - lse.
SV_DEVINL void lse_combine(float& m, float& s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  if (mn == -INFINITY) return;
  s = s * expf(m - mn) + s2 * expf(m2 - mn);
  m = mn;
}
__global__ void logps_merge_kernel(const float2* __restrict__ part, const float* __restrict__ tlogit,
                                   const int32_t* __restrict__ tgt, const int32_t* __restrict__ lp_idx,
                                   float* __restrict__ logps, int M, int N, int ntiles) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= M) return;
  float m = -INFINITY, s = 0.f;
  for (int i = lane; i < ntiles; i += 32) {
    const float2 p = part[(int64_t)row * ntiles + i];
    lse_combine(m, s, p.x, p.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_down_sync(0xffffffffu, m, o), s2 = __shfl_down_sync(0xffffffffu, s, o);
    lse_combine(m, s, m2, s2);
  }
  if (lane != 0) return;
  const int out = lp_idx ? lp_idx[row] : row;
  if (out < 0) return;
  const int t = tgt[row];
  logps[out] = (t >= 0 && t < N) ? tlogit[row] - (m + logf(s)) : __int_as_float(0x7fc00000);   // no target: NaN
}

}  // namespace tc05

bool tc05_supported(int M, int N, int K) { return M >= 1 && N >= 8 && (N % 8) == 0 && K >= 64 && (K % 64) == 0; }

cudaError_t launch_linear_tc05(const bf16* x, const bf16* w, const bf16* bias, const bf16* res, bf16* y, int M, int N,
                               int K, int act, cudaStream_t st) {
  if (!tc05_supported(M, N, K)) return cudaErrorInvalidValue;
  // Tile-count heuristic for the small-M GEMMs of this path (M = 257..2072): every CTA pays ~10 us of fixed cost
  // (launch, TMEM alloc, pipeline fill, epilogue), so never spill into a second wave if a wider tile avoids it:
  // BN=64 while its tile count fits one wave of SMs, else BN=128.
  const int mt = (M + tc05::BM - 1) / tc05::BM;
  static int nsm = 0;
  if (nsm == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev); if (nsm <= 0) nsm = 148; }
  static int per_sm = 0;                       // CTAs of this kernel that fit one SM (2 with the 96 KB ring)
  if (per_sm == 0) { const char* c = getenv("SV_TC05_PER_SM"); per_sm = c ? atoi(c) : 2; if (per_sm < 1) per_sm = 1; }
  const bool wide = (N % 128 == 0) && ((int64_t)mt * ((N + 63) / 64) > (int64_t)nsm * per_sm);
  return wide ? tc05::launch<128>(x, w, bias, res, y, M, N, K, act, st)
              : tc05::launch<64>(x, w, bias, res, y, M, N, K, act, st);
}

int lm_head_logps_ntiles(int N) { return (N + 127) / 128; }

cudaError_t launch_lm_head_logps(const bf16* x, const bf16* w, int M, int N, int K, const LogpsEpilogue& lp,
                                 const int32_t* lp_idx, float* logps, cudaStream_t st) {
  if (M < 1 || N < 1 || K < 64 || K % 64) return cudaErrorInvalidValue;
  cudaError_t r = tc05::launch<128, tc05::EPI_LOGPS>(x, w, nullptr, nullptr, nullptr, M, N, K, /*act=*/0, st, lp);
  if (r != cudaSuccess || !logps) return r;
  constexpr int kRowsPerBlock = 8;
  tc05::logps_merge_kernel<<<(M + kRowsPerBlock - 1) / kRowsPerBlock, 32 * kRowsPerBlock, 0, st>>>(
      lp.part, lp.tlogit, lp.tgt, lp_idx, logps, M, N, lm_head_logps_ntiles(N));
  count_launch();
  return cudaGetLastError();
}

}  // namespace sv
