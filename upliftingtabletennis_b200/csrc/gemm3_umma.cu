// fp32-class GEMM on the 5th-generation tensor cores ("3xTF32") for the uplifting transformer's Linear layers (K = 128):
//     C[m][n] = act( sum_k A'[m][k] W[n][k] + bias[n] ) (+ R[m][n]),      A' = A or LayerNorm(A)
// Reference: the nn.Linear / LayerNorm calls of uplifting/model.py:10-36 (Mlp), :161-229 (attention qkv / proj), :278-300 (layer).
// The reference multiplies in fp32 on a GPU (torch keeps TF32 off for matmul), so one TF32 product is not enough.  Every operand is
// split into two TF32 numbers, x = x_hi + x_lo with x_hi = tf32(x) and x_lo = x - x_hi (exact in fp32), and three tensor-core
// products are accumulated in the fp32 TMEM accumulator:  A_hi W_hi + A_lo W_hi + A_hi W_lo.  The dropped A_lo W_lo term is 2^-22
// relative, kind::tf32 truncating A_lo / W_lo to 11 significant bits costs another 2^-22: fp32-level results (tests: 1e-4 bar of the
// strict path, measured ~1e-6) at 1/3 of the TF32 tensor rate instead of the SIMT FMA rate.
//
// Tile 128 x 128, K = 128 as four 32-column chunks (128-byte swizzled rows).  A CTA owns one N tile and walks M tiles:
//   * the N tile's weights, W_hi and W_lo (split once on the host), stay resident in shared memory (128 KB);
//   * warp 0 streams raw fp32 A chunks by TMA through a 3-stage ring;
//   * warps 2-5 (transform) turn a raw chunk into A_hi (in place) and A_lo (second buffer) -- element-wise, so the swizzled layout
//     TMA produced is kept -- and apply the LayerNorm of the layer on the way when asked to: (a - mean[m]) * rstd[m] * gamma[k] + beta[k]
//     with per-row statistics that the epilogue of the GEMM which produced A wrote (no LayerNorm kernels, no normalised copy in HBM);
//   * warp 1 issues the 48 MMAs of a tile (4 chunks x 4 K8 steps x 3 products), accumulators double buffered in TMEM;
//   * warps 6-13 (epilogue, thread = row x column half): the residual is requested before the accumulators are waited for, the
//     accumulators are released as soon as they sit in registers; bias, ReLU, residual add, fp32 row-contiguous 256-bit stores, and
//     for N = 128 the row's mean / rstd for the next LayerNorm (chunk-wise two-pass + Chan merge, halves exchanged in shared memory).
#include "umma_prims.h"
#include "uplift.h"

namespace {

using namespace umma;

constexpr int BM = 128, BN = 128, KD = 128, KC = 32, NKC = KD / KC;
#ifndef TTK_GEMM3_STAGES
#define TTK_GEMM3_STAGES 3      // tools/run_sanitizer.sh builds a 2-stage variant for synccheck, whose own bookkeeping needs shared memory
#endif
constexpr int STAGES = TTK_GEMM3_STAGES;
constexpr int CHUNK_BYTES = BM * KC * 4;                 // 16 KB: 128 rows x 128 bytes
constexpr int W_BYTES = 2 * NKC * CHUNK_BYTES;           // hi | lo, four chunks each
constexpr int STAGE_BYTES = 2 * CHUNK_BYTES;             // raw -> hi (in place) | lo
constexpr int THREADS = 448;                             // TMA warp, MMA warp, 4 transform warps, 8 epilogue warps
constexpr int SMEM_BYTES = W_BYTES + STAGES * STAGE_BYTES + 3 * KD * 4 + 2 * BM * 4 + 128;      // 232 064 of the 232 448 bytes a CTA can have
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct G3Maps {
  CUtensorMap a, whi, wlo;
};

__device__ __forceinline__ float tf32_hi(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

__global__ void __launch_bounds__(THREADS, 1) gemm3_umma_kernel(const __grid_constant__ G3Maps maps, const Gemm3Args g, int tiles_m, int tiles_n) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();          // the swizzled tiles need 1024-byte alignment (no static shared memory precedes them)
  uint8_t* sW = smem;                                   // [hi | lo][chunk][128 rows][128 B]
  uint8_t* ring = smem + W_BYTES;
  float* sGamma = reinterpret_cast<float*>(ring + STAGES * STAGE_BYTES);
  float* sBeta = sGamma + KD;
  float* sBias = sBeta + KD;
  float2* sHalf = reinterpret_cast<float2*>(sBias + KD);  // statistics of the upper column half of every row (epilogue exchange)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sHalf + BM);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 5);
  const uint32_t bar_raw = smem_u32(bars), bar_ready = bar_raw + 8 * STAGES, bar_empty = bar_ready + 8 * STAGES, bar_tfull = bar_empty + 8 * STAGES,
                 bar_tempty = bar_tfull + 16, bar_w = bar_tempty + 16;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tn = blockIdx.x % tiles_n, tm0 = blockIdx.x / tiles_n;
  const int tm_step = (gridDim.x - tn + tiles_n - 1) / tiles_n;
  const bool ln = g.ln_stats != nullptr;

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(bar_raw + 8 * s, 1);
      mbar_init(bar_ready + 8 * s, 4);                  // one arrival per transform warp
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, 8);
    }
    mbar_init(bar_w, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < KD; i += THREADS) {
    sGamma[i] = ln ? __ldg(g.ln_gamma + i) : 1.f;
    sBeta[i] = ln ? __ldg(g.ln_beta + i) : 0.f;
    sBias[i] = g.bias ? __ldg(g.bias + tn * BN + i) : 0.f;
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), 256);
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0 && tm0 < tiles_m) {
      mbar_expect_tx(bar_w, W_BYTES);
      for (int kc = 0; kc < NKC; ++kc) {
        tma_load_2d(smem_u32(sW + kc * CHUNK_BYTES), &maps.whi, bar_w, kc * KC, tn * BN);
        tma_load_2d(smem_u32(sW + (NKC + kc) * CHUNK_BYTES), &maps.wlo, bar_w, kc * KC, tn * BN);
      }
      // The ring holds three 16 KB chunks, too little to cover the DRAM latency: the rows of the tile after the next are prefetched into
      // L2 (TMA prefetch, no shared memory needed), so the ring's loads are L2 hits.
      constexpr int AHEAD = 2;
      for (int a = 0; a < AHEAD; ++a)
        if (tm0 + a * tm_step < tiles_m)
          for (int kc = 0; kc < NKC; ++kc) tma_prefetch_2d(&maps.a, kc * KC, (tm0 + a * tm_step) * BM);
      uint32_t it = 0;
      for (int tm = tm0; tm < tiles_m; tm += tm_step) {
        if (tm + AHEAD * tm_step < tiles_m)
          for (int kc = 0; kc < NKC; ++kc) tma_prefetch_2d(&maps.a, kc * KC, (tm + AHEAD * tm_step) * BM);
        for (int kc = 0; kc < NKC; ++kc, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_raw + 8 * s, CHUNK_BYTES);
          tma_load_2d(smem_u32(ring + s * STAGE_BYTES), &maps.a, bar_raw + 8 * s, kc * KC, tm * BM);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: whole warp, warp-uniform operands, one elected lane issues (see conv_umma.cu) =====
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc_tf32(BM, BN);
    const uint32_t w16 = smem_u32(sW) >> 4, ring16 = smem_u32(ring) >> 4;
    uint32_t it = 0, tcount = 0;
    if (tm0 < tiles_m) mbar_wait(bar_w, 0);
    for (int tm = tm0; tm < tiles_m; tm += tm_step, ++tcount) {
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      mbar_wait(bar_tempty + 8 * acc, aph ^ 1);          // accumulator drained by the epilogue (passes at once the first two times)
      fence_after();
      const uint32_t d = tmem_u + acc * BN;
      for (int kc = 0; kc < NKC; ++kc, ++it) {
        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
        mbar_wait(bar_ready + 8 * s, ph);
        fence_after();
        const uint32_t ahi = ring16 + s * (STAGE_BYTES / 16), alo = ahi + CHUNK_BYTES / 16;
        const uint32_t whi = w16 + kc * (CHUNK_BYTES / 16), wlo = whi + NKC * (CHUNK_BYTES / 16);
#pragma unroll
        for (int ks = 0; ks < KC / 8; ++ks) {
          if (leader) {
            mma_tf32(d, make_desc16<1024, 2>(ahi + ks * 2), make_desc16<1024, 2>(whi + ks * 2), idesc, (kc | ks) ? 1u : 0u);
            mma_tf32(d, make_desc16<1024, 2>(alo + ks * 2), make_desc16<1024, 2>(whi + ks * 2), idesc, 1u);
            mma_tf32(d, make_desc16<1024, 2>(ahi + ks * 2), make_desc16<1024, 2>(wlo + ks * 2), idesc, 1u);
          }
        }
        if (leader) commit(bar_empty + 8 * s);
      }
      if (leader) commit(bar_tfull + 8 * acc);
      __syncwarp();
    }
  } else if (warp < 6) {
    // ===== transform warps 2..5: raw chunk -> (LayerNorm ->) hi in place, lo beside it =====
    const int t = tid - 64;                              // 0..127
    uint32_t it = 0, tcount = 0;
    for (int tm = tm0; tm < tiles_m; tm += tm_step, ++tcount) {
      // per-row statistics of the eight rows this thread touches in every chunk (rows t / 8 + 16 i)
      float mu[8], rs[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int m = tm * BM + (t >> 3) + 16 * i;
        float2 st = make_float2(0.f, 1.f);
        if (ln && m < g.M) st = __ldg(reinterpret_cast<const float2*>(g.ln_stats) + m);
        mu[i] = st.x;
        rs[i] = st.y;
      }
      for (int kc = 0; kc < NKC; ++kc, ++it) {
        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1;
        mbar_wait(bar_raw + 8 * s, ph);
        uint8_t* hi = ring + s * STAGE_BYTES;
        uint8_t* lo = hi + CHUNK_BYTES;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int idx = t + 128 * i;                   // 16-byte chunk index in the tile: row = idx / 8, stored position = idx % 8
          float4 v = *reinterpret_cast<const float4*>(hi + idx * 16);
          if (ln) {
            const int r = idx >> 3, c = ((idx & 7) ^ (r & 7)) * 4 + kc * KC;      // 128-byte swizzle: logical chunk = position ^ (row & 7)
            const float4 ga = *reinterpret_cast<const float4*>(sGamma + c), be = *reinterpret_cast<const float4*>(sBeta + c);
            v.x = (v.x - mu[i]) * rs[i] * ga.x + be.x;
            v.y = (v.y - mu[i]) * rs[i] * ga.y + be.y;
            v.z = (v.z - mu[i]) * rs[i] * ga.z + be.z;
            v.w = (v.w - mu[i]) * rs[i] * ga.w + be.w;
          }
          float4 h, l;
          h.x = tf32_hi(v.x), h.y = tf32_hi(v.y), h.z = tf32_hi(v.z), h.w = tf32_hi(v.w);
          l.x = v.x - h.x, l.y = v.y - h.y, l.z = v.z - h.z, l.w = v.w - h.w;
          *reinterpret_cast<float4*>(hi + idx * 16) = h;
          *reinterpret_cast<float4*>(lo + idx * 16) = l;
        }
        fence_async_smem();                              // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_ready + 8 * s);
      }
    }
  } else {
    // ===== epilogue warps 6..13: TMEM lane quarter q = warp % 4 (thread = row), column half = (warp - 6) / 4 =====
    const int q = warp & 3, half = (warp - 6) >> 2;
    const uint32_t lane_base = tmem + ((uint32_t)(q * 32) << 16);
    const int relu = g.relu;
    const float* __restrict__ gR = g.R;
    float* const gC = g.C;
    float* const gStats = g.out_stats;
    const int N = g.N;
    const int rt = q * 32 + lane;                        // row within the tile
    uint32_t tcount = 0;
    for (int tm = tm0; tm < tiles_m; tm += tm_step, ++tcount) {
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      const int m = tm * BM + rt;
      const bool live = m < g.M;
      const size_t off = (size_t)m * N + tn * BN + half * 64;
      // the residual of both 32-column chunks is in flight before the accumulators are waited for
      uint32_t r[2][32];
      if (gR && live) {
#pragma unroll
        for (int j = 0; j < 8; ++j) ld256(gR + off + 8 * j, &r[j >> 2][8 * (j & 3)]);      // coherent loads: R may be C (x += ...), each element is read before this thread writes it
      }
      mbar_wait(bar_tfull + 8 * acc, aph);
      fence_after();
      uint32_t v[2][32];
      tmem_ld32(lane_base + acc * BN + half * 64, v[0]);
      tmem_ld32(lane_base + acc * BN + half * 64 + 32, v[1]);
      tmem_wait_ld();
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);  // the accumulator is in registers: the MMA warp may overwrite it
      // mean / sum of squared deviations of this thread's 64 columns (Chan merge of two 32-wide chunks), taken about `shift` (the first
      // value): chunk means of rows with a large mean and a small spread would otherwise carry the rounding of a sum of large values
      // (1e-5 of a mean of 50 against a spread of 0.05), and the merge term delta^2 inherits it
      float shift = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[c][j]) + sBias[half * 64 + c * 32 + j];
        if (relu) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
        }
        if (gR && live) {
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] += __uint_as_float(r[c][j]);
        }
        if (gStats) {
          if (c == 0) shift = f[0];
          float s = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) s += f[j] - shift;
          const float cm = s * (1.f / 32.f);
          const float center = shift + cm;               // any centre near the mean gives the squared deviations to second order
          float cq = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) cq = fmaf(f[j] - center, f[j] - center, cq);
          if (c == 0) {
            mean = cm;
            m2 = cq;
          } else {
            const float delta = cm - mean;
            mean += 0.5f * delta;
            m2 += cq + delta * delta * 16.f;
          }
        }
        if (live) {
          uint32_t o[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) o[j] = __float_as_uint(f[j]);
#pragma unroll
          for (int j = 0; j < 4; ++j) stg256(gC + off + c * 32 + 8 * j, o + 8 * j);
        }
      }
      if (gStats) {
        // the two column halves of a row meet in shared memory (N = 128: the tile holds whole rows)
        if (half == 1) sHalf[rt] = make_float2(shift + mean, m2);
        asm volatile("bar.sync 3, 256;" ::: "memory");
        if (half == 0 && live) {
          const float2 h1 = sHalf[rt];
          const float delta = (h1.x - shift) - mean;
          const float mu = shift + (mean + 0.5f * delta);
          const float q2 = m2 + h1.y + delta * delta * 32.f;
          *reinterpret_cast<float2*>(gStats + 2 * (size_t)m) = make_float2(mu, rsqrtf(q2 * (1.f / KD) + 1e-5f));
        }
        asm volatile("bar.sync 3, 256;" ::: "memory");   // sHalf is free for the next tile
      }
    }
  }
  fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, 256);
}

bool encode_f32_2d(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols) {
  EncodeFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 4};
  cuuint32_t box[2] = {KC, BM};
  cuuint32_t es[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

int ttk_gemm3(const Gemm3Args& g, cudaStream_t st) {
  if (g.M <= 0 || g.N % BN != 0 || (g.out_stats && g.N != BN)) {
    ttk_set_error("ttk_gemm3: unsupported shape M %d N %d (K is 128, N a multiple of 128; row statistics need N = 128)", g.M, g.N);
    return TTK_ERR_UNSUPPORTED;
  }
  // TMA reads A and W from 16-byte aligned rows; the epilogue reads R and writes C with 256-bit accesses
  const auto misaligned = [](const void* p, uintptr_t a) { return ((uintptr_t)p & (a - 1)) != 0; };
  if (misaligned(g.A, 16) || misaligned(g.W_hi, 16) || misaligned(g.W_lo, 16) || misaligned(g.C, 32) || misaligned(g.R, 32)) {
    ttk_set_error("ttk_gemm3: A and W must be 16-byte aligned, C and R 32-byte aligned");
    return TTK_ERR_ARG;
  }
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(gemm3_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  }
  G3Maps maps;
  if (!encode_f32_2d(&maps.a, g.A, (uint64_t)g.M, KD) || !encode_f32_2d(&maps.whi, g.W_hi, (uint64_t)g.N, KD) ||
      !encode_f32_2d(&maps.wlo, g.W_lo, (uint64_t)g.N, KD)) {
    ttk_set_error("ttk_gemm3: cuTensorMapEncodeTiled failed (M %d N %d)", g.M, g.N);
    return TTK_ERR_CUDA;
  }
  const int tiles_m = ttk_cdiv(g.M, BM), tiles_n = g.N / BN;
  const int grid = std::max(1, std::min(tiles_m * tiles_n, ttk_num_sms() / tiles_n * tiles_n));
  gemm3_umma_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(maps, g, tiles_m, tiles_n);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_uplift_debug_gemm3(const float* a_dev, const float* w_hi_dev, const float* w_lo_dev, const float* bias_dev, const float* res_dev,
                                      float* c_dev, int m, int n, int relu, const float* ln_stats_dev, const float* ln_gamma_dev,
                                      const float* ln_beta_dev, float* out_stats_dev, void* stream) {
  TTK_CHECK_ARG(a_dev && w_hi_dev && w_lo_dev && c_dev, "ttk_uplift_debug_gemm3: null pointer");
  TTK_CHECK_ARG(!ln_stats_dev || (ln_gamma_dev && ln_beta_dev), "ttk_uplift_debug_gemm3: LayerNorm statistics need gamma and beta");
  const Gemm3Args g{a_dev, w_hi_dev, w_lo_dev, bias_dev, res_dev, c_dev, m, n, relu, ln_stats_dev, ln_gamma_dev, ln_beta_dev, out_stats_dev};
  return ttk_gemm3(g, (cudaStream_t)stream);
}
