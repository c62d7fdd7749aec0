// Uplifting transformer, bf16 tensor-core path: one fused kernel per stage (table-token layers, temporal
// layers, second stage) with every Linear layer on tcgen05.mma.
// Reference: uplifting/model.py:278-300 (SimpleStaticLayer), :186-229 (rotary attention), :335-390, :529-571.
//
// A CTA owns 128 token rows (8 table-token sequences of 14 in 16-row slots, or 2 temporal sequences of <= 64) for
// ALL layers of a stage:
//   * the fp32 residual stream lives in TMEM (128 lanes x 128 columns) for the whole stage; four threads (one per
//     warp group) own 32 columns of row r each, so LayerNorm is a per-thread reduction over tcgen05.ld'ed registers
//     plus a four-way exchange, and the residual adds are TMEM read-modify-writes by the same thread;
//   * GEMM A operands (LayerNorm output, attention output, ReLU(fc1)) are written as bf16 into 128-byte-swizzled
//     K-major shared tiles, B operands are the weight matrices' own (out, in) rows streamed by TMA from one
//     [layers*768][128] bf16 matrix through a 3-slot ring, accumulators go to TMEM columns 0..383;
//   * attention runs on the tensor cores as well: per head, scores = Q_h K_h^T (128 x 128 block, the rows' own
//     sequence block is the valid part) land in TMEM, the row-owning thread applies masks + safe softmax and writes
//     un-normalised probabilities as a bf16 A operand, O_h = P V_h accumulates into TMEM and is scaled by 1/sum in
//     the epilogue (V is stored transposed, keys contiguous, so it is a K-major B operand);
//   * bias + RoPE + bf16 packing of q/k/v run on CUDA cores straight out of TMEM;
//   * 16 warps: every CUDA-core phase is split between four warp groups (warps q, q+4, q+8, q+12 share TMEM lane
//     quarter q): the softmax by key columns (partial maxima / sums exchanged through shared memory and a 128-thread
//     named barrier), the q/k/v and attention-output epilogues by heads, everything else by 32-column quarters.  The
//     kernel is latency bound (one CTA per SM, dependent TMEM-load -> math -> store chains), so four warps per
//     scheduler instead of two is what hides it; the scores of head h+1 are issued together with P V of head h, so a
//     head costs one MMA round trip.
#include <cuda.h>

#include "uplift.h"
#include "umma_prims.h"

namespace {

using namespace umma;      // mbarriers, TMA loads, descriptors, tcgen05 wrappers shared by all tensor-core kernels

constexpr int D = 128, HEADS = 4, HD = 32, NF = 16, NTAB = 13;
constexpr int NG = 4;                                // warp groups: warps 4g .. 4g+3 cover the four TMEM lane quarters
constexpr int TC_THREADS = 128 * NG;
constexpr int CW = 128 / NG;                        // columns of every 128-column phase per thread
constexpr int ROWS = 128;
constexpr int CHUNK_BYTES = 32768;                 // 128 weight rows x 128 K bf16 = two 16 KB K-halves
constexpr int SA_BYTES = 32768, SQ_BYTES = 128 * 384 * 2, SW_BYTES = 3 * CHUNK_BYTES;
constexpr int TC_SMEM = SA_BYTES + SQ_BYTES + SW_BYTES;
constexpr int LAYER_ROWS = 768;                    // qkv 384 | proj 128 | fc1 128 | fc2 128

enum { MODE_POS = 0, MODE_TEMPORAL = 1, MODE_SECOND = 2 };

__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t addr) { return make_desc(addr, 1024, 2); }     // 8 rows x 128 B between core-matrix groups
__device__ __forceinline__ uint64_t make_desc_sw64(uint32_t addr) { return make_desc(addr, 512, 4); }       // 8 rows x 64 B
constexpr uint32_t IDESC_128x32 = make_idesc(128, 32), IDESC_128x128 = make_idesc(128, 128);
__device__ __forceinline__ void tc_fence_before() { fence_before(); }
__device__ __forceinline__ void tc_fence_after() { fence_after(); }
__device__ __forceinline__ void proxy_fence() { fence_async_smem(); }

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]), "=r"(u[9]),
        "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]), "=r"(u[17]), "=r"(u[18]),
        "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]), "=r"(u[25]), "=r"(u[26]), "=r"(u[27]),
        "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4_nowait(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float* v) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]), "=r"(u[9]),
                 "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 128-thread named barrier of the four warps that share a TMEM lane quarter (ids 1..4; 0 is __syncthreads)
__device__ __forceinline__ void quad_barrier(int quarter) { asm volatile("bar.sync %0, 128;" ::"r"(quarter + 1) : "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
  const uint32_t* u = reinterpret_cast<const uint32_t*>(v);
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
      "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]), "r"(u[10]),
      "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15]), "r"(u[16]), "r"(u[17]), "r"(u[18]), "r"(u[19]), "r"(u[20]),
      "r"(u[21]), "r"(u[22]), "r"(u[23]), "r"(u[24]), "r"(u[25]), "r"(u[26]), "r"(u[27]), "r"(u[28]), "r"(u[29]), "r"(u[30]),
      "r"(u[31])
      : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}

// byte offset of element (row, col) of a [128 x 128] bf16 A/B operand stored as two 128-byte-swizzled K-halves
__device__ __forceinline__ uint32_t a_off(int row, int col) {
  const int kh = col >> 6, b = (col & 63) * 2;
  return kh * 16384 + row * 128 + ((((b >> 4) ^ (row & 7)) << 4) | (b & 15));
}

struct TcParams {
  const LayerW* layers;
  int n_layers, layer_first;      // index of the stage's first layer in the weight matrix
  int batch, T;
  float* X;
  const float* table_emb;
  const float* table;
  const float* mask;
  const float* times;
  const float* cls;
  const float* second_in;
  float* out_rows;                // POS/TEMPORAL: X; SECOND: [batch][128] cls rows
  // Hand-over between the table-token stage and the temporal stage.  Only the ball token of a table-token sequence is used
  // afterwards (model.py:375-378), so the last table-token layer stops after its attention: the ball rows' residual stream
  // (-> X) and normalised attention output (-> attn_rows, bf16) leave the kernel, and the temporal kernel, whose 128 rows are
  // exactly such ball rows, starts with that layer's projection + MLP ("tail") before its own layers.  1/14 of the rows
  // pay for the tail instead of all of them.
  __nv_bfloat16* attn_rows;
};

// ADD_MASK: p.mask holds the additive values themselves ({-1e9, 0}) instead of {0, 1} (TEMPORAL / SECOND only).  A template argument
// rather than a run-time flag so that the {0, 1} instantiation keeps its registers (the additive softmax holds more of them).
template <int MODE, bool ADD_MASK = false>
__global__ void __launch_bounds__(TC_THREADS, 1) uplift_tc_kernel(const __grid_constant__ CUtensorMap wmap, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();  // the swizzled operand tiles need 1024-byte alignment
  uint8_t* sA = smem;                           // LN output / probabilities P / attention output (A operands, 2 x SW128 halves)
  uint8_t* sQh = sA + SA_BYTES;                 // 4 heads x [128 rows][64 B] SW64 (q); later the fc2 A operand
  uint8_t* sKh = sQh + 32768;                   // 4 heads x [128 rows][64 B] SW64 (k)
  uint8_t* sVt = sKh + 32768;                   // 4 heads x [32 dims][128 keys] as 2 SW128 halves (v transposed)
  uint8_t* sW = sVt + 32768;                    // weight ring, 3 slots
  // 227 KB - 224 KB of operand tiles leave 3 KB of static shared memory, so the exchange buffers overlay dead storage:
  // ring slot 2 is empty between the QKV GEMM and the end of the attention (the fc2 weights are fetched after it),
  // k is dead whenever LayerNorm runs.
  float(*sMax)[ROWS] = reinterpret_cast<float(*)[ROWS]>(sW + 2 * CHUNK_BYTES);                        // [NG][ROWS] partial row maxima
  float(*sSum)[NG][ROWS] = reinterpret_cast<float(*)[NG][ROWS]>(sW + 2 * CHUNK_BYTES + NG * ROWS * 4);  // [HEADS][NG][ROWS] partial row sums
  float2(*sRed)[ROWS] = reinterpret_cast<float2(*)[ROWS]>(sKh);                                        // [NG][ROWS] LayerNorm partial sums
  __shared__ float sMask[ROWS];                 // additive key masks and times of the rows (-inf: never attended)
  __shared__ float sTime[ROWS];
  __shared__ uint64_t bars[4];                  // full[3], mma
  __shared__ uint32_t tmem_slot;
  const uint32_t bar_full = smem_u32(bars), bar_mma = bar_full + 24;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int grp = warp >> 2, quarter = warp & 3;           // warps q, q+4, q+8, q+12 share TMEM lane quarter q
  const int row = quarter * 32 + lane;                      // TMEM lane of this thread
  const int cq = grp * CW;                                  // this thread's 32 columns of every 128-column phase
  const int T = p.T;
  const int S = MODE == MODE_POS ? NTAB + 1 : (MODE == MODE_TEMPORAL ? T : T + 1);
  constexpr int SSTRIDE = MODE == MODE_POS ? 16 : 64;      // rows per sequence slot: a warp's 32 rows hold whole slots
  constexpr int G = ROWS / SSTRIDE;
  const long long n_seq = MODE == MODE_POS ? (long long)p.batch * T : p.batch;
  const long long seq0 = (long long)blockIdx.x * G;
  const float NEG_INF = -INFINITY;

  if (tid == 0) {
    for (int i = 0; i < 3; ++i) mbar_init(bar_full + 8 * i, 1);
    mbar_init(bar_mma, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  // per-row sequence bookkeeping
  const int g_row = row / SSTRIDE, s_row = row - g_row * SSTRIDE;
  const long long seq_row = seq0 + g_row;
  const bool valid = s_row < S && seq_row < n_seq;
  if (tid < ROWS) {
    float m = NEG_INF, t_row = __int_as_float(0x7fc00000);     // NaN time: no rotation (cls token / padding row)
    if (valid) {
      m = 0.f;
      if (MODE == MODE_POS) {
        if (s_row > 0) {
          const long long b = seq_row / T;
          m = p.table[(b * NTAB + (s_row - 1)) * 3 + 2] == 1.f ? 0.f : NEG_INF;
          t_row = (float)(s_row - 1) / 100.f;
        }
      } else if (MODE == MODE_TEMPORAL || s_row > 0) {
        const float mv = p.mask[seq_row * T + s_row - (MODE == MODE_SECOND)];
        m = ADD_MASK ? mv : (mv == 0.f ? NEG_INF : 0.f);
        t_row = p.times[seq_row * T + s_row - (MODE == MODE_SECOND)];
      }
    }
    sMask[row] = m;
    sTime[row] = t_row;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  // MMA issue: warp 0 walks the issue code with warp-uniform operands (TMEM base broadcast, addresses from shared-memory symbols) and
  // its elected lane executes tcgen05.mma / commit / the TMA loads.  Under `if (tid == 0)` the compiler wrapped every MMA in an
  // ELECT / R2UR loop (16 instructions each) -- issue latency that sat on each of the nine MMA round trips of a layer.
  const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
  const bool issuer = elect_one() && warp == 0;
  auto issue_mma = [&](uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate, uint32_t idesc) {
    if (issuer) mma(tmem_d, da, db, idesc, accumulate);
  };
  const uint32_t lane_base = tmem + ((uint32_t)(quarter * 32) << 16);
  constexpr uint32_t COL_X = 384, COL_S = 0, COL_O = 128, COL_PROJ = 256, COL_FC1 = 0, COL_FC2 = 128;
  const int k_lo = g_row * SSTRIDE, k_hi = k_lo + S;        // this row's key block
  const bool q_live = sMask[row] != NEG_INF;

  // rotary table of this thread's row (every warp group keeps a copy): angle = rint(t / 0.002) * inv_freq
  float rc[NF], rs[NF];
  {
    const float t = sTime[row];
    const float* invf = p.layers[0].invf;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      rc[f] = 1.f;
      rs[f] = 0.f;
      if (t == t) {
        const float pos = rintf(__fdiv_rn(t, 0.002f));
        sincosf(__fmul_rn(pos, __ldg(invf + f)), &rs[f], &rc[f]);
      }
    }
  }

  // weight chunks of 128 rows: 6 per layer (qkv 3, proj, fc1, fc2).  The temporal stage starts with chunks -3, -2, -1: proj, fc1 and
  // fc2 of the last table-token layer (the layer before layer_first); ring slot and mbarrier parity follow gchunk + 3.
  constexpr bool TAIL = MODE == MODE_TEMPORAL, HEADLESS_LAST = MODE == MODE_POS;
  const int total_chunks = p.n_layers * 6;
  auto issue_load = [&](int gchunk) {           // warp 0; the elected lane issues
    if (gchunk >= total_chunks || !issuer) return;
    const int slot = (gchunk + 3) % 3;
    const int wrow = gchunk >= 0 ? (p.layer_first + gchunk / 6) * LAYER_ROWS + (gchunk % 6) * 128 : (p.layer_first - 1) * LAYER_ROWS + (6 + gchunk) * 128;
    mbar_expect_tx(bar_full + 8 * slot, CHUNK_BYTES);
    const uint32_t dst = smem_u32(sW + slot * CHUNK_BYTES);
    tma_load_2d(dst, &wmap, bar_full + 8 * slot, 0, wrow);
    tma_load_2d(dst + 16384, &wmap, bar_full + 8 * slot, 64, wrow);
  };
  auto gemm = [&](int gchunk, uint32_t a_base, uint32_t col) {   // warp 0: D[128 x 128] at TMEM column `col`
    const int slot = (gchunk + 3) % 3;
    mbar_wait(bar_full + 8 * slot, ((gchunk + (TAIL ? 3 : 0)) / 3) & 1);
    tc_fence_after();
    const uint32_t b_base = smem_u32(sW + slot * CHUNK_BYTES);
#pragma unroll
    for (int kh = 0; kh < 2; ++kh)
#pragma unroll
      for (int k16 = 0; k16 < 4; ++k16)
        issue_mma(tmem_u + col, make_desc_sw128(a_base + kh * 16384 + k16 * 32), make_desc_sw128(b_base + kh * 16384 + k16 * 32),
                  (kh | k16) != 0 ? 1u : 0u, IDESC_128x128);
  };
  uint32_t mma_phase = 0;
  auto mma_sync = [&]() {                       // all threads: wait for the committed MMAs
    mbar_wait(bar_mma, mma_phase);
    mma_phase ^= 1;
    tc_fence_after();
  };
  // x (+= delta [+ bias]) -> TMEM, then LayerNorm -> sA.  ALL threads: the four warps of a lane quarter own 32 columns
  // of row `row` each and exchange their partial (sum, sum of squares) through shared memory.
  auto residual_ln = [&](bool add, uint32_t col_delta, const float* bias, const float* lnw, const float* lnb, bool do_ln, float* out_global) {
    float v[CW];
    tmem_ld32_nowait(lane_base + COL_X + cq, v);
    if (add) {
      float a[CW];
      tmem_ld32_nowait(lane_base + col_delta + cq, a);
      tmem_ld_wait();
      if (bias) {
#pragma unroll
        for (int j = 0; j < CW; j += 4) {
          const float4 bz = __ldg(reinterpret_cast<const float4*>(bias + cq + j));
          v[j] += a[j] + bz.x, v[j + 1] += a[j + 1] + bz.y, v[j + 2] += a[j + 2] + bz.z, v[j + 3] += a[j + 3] + bz.w;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] += a[j];
      }
      tmem_st32(lane_base + COL_X + cq, v);
    } else {
      tmem_ld_wait();
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < CW; ++j) {
      s1 += v[j];
      s2 = fmaf(v[j], v[j], s2);
    }
    if (add) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    if (out_global) {
#pragma unroll
      for (int c = 0; c < CW; c += 4) *reinterpret_cast<float4*>(out_global + cq + c) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
    }
    if (!do_ln) return;
    sRed[grp][row] = make_float2(s1, s2);
    quad_barrier(quarter);
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int g = 0; g < NG; ++g) {                // every group adds in the same order
      const float2 t = sRed[g][row];
      t1 += t.x;
      t2 += t.y;
    }
    const float mean = t1 * (1.f / D);
    const float var = fmaxf(t2 * (1.f / D) - mean * mean, 0.f);
    const float rstd = rsqrtf(var + 1e-5f);
#pragma unroll
    for (int c = 0; c < CW; c += 8) {
      uint32_t w[4];
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(lnw + cq + c)), g1 = __ldg(reinterpret_cast<const float4*>(lnw + cq + c + 4));
      const float4 h0 = __ldg(reinterpret_cast<const float4*>(lnb + cq + c)), h1 = __ldg(reinterpret_cast<const float4*>(lnb + cq + c + 4));
      const float gw[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w}, gb[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = c + 2 * j;
        const float y0 = (v[i] - mean) * rstd * gw[2 * j] + gb[2 * j];
        const float y1 = (v[i + 1] - mean) * rstd * gw[2 * j + 1] + gb[2 * j + 1];
        w[j] = pack_bf16(y0, y1);
      }
      *reinterpret_cast<uint4*>(sA + a_off(row, cq + c)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  };
  // ReLU(fc1 + b) -> bf16 A operand of fc2 (in the q buffer); 32 columns per warp group
  auto relu_fc1 = [&](const float* fc1b) {
    float a[CW];
    tmem_ld32_nowait(lane_base + COL_FC1 + cq, a);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < CW; j += 4) {
      const float4 bz = __ldg(reinterpret_cast<const float4*>(fc1b + cq + j));
      a[j] = fmaxf(a[j] + bz.x, 0.f), a[j + 1] = fmaxf(a[j + 1] + bz.y, 0.f), a[j + 2] = fmaxf(a[j + 2] + bz.z, 0.f), a[j + 3] = fmaxf(a[j + 3] + bz.w, 0.f);
    }
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4)
      *reinterpret_cast<uint4*>(sQh + a_off(row, cq + 8 * q4)) =
          make_uint4(pack_bf16(a[8 * q4], a[8 * q4 + 1]), pack_bf16(a[8 * q4 + 2], a[8 * q4 + 3]),
                     pack_bf16(a[8 * q4 + 4], a[8 * q4 + 5]), pack_bf16(a[8 * q4 + 6], a[8 * q4 + 7]));
  };
  // Softmax work split.  The keys of a row are its own slot's (k_lo .. k_hi); the warp groups take a quarter of the
  // slot's columns each: NC = 4 of 16 (table-token stage) or 16 of 64 (temporal stages) score columns per thread,
  // starting at key `col0`.  The valid ones are a per-thread bit mask that is fixed for the whole stage.
  constexpr int NC = SSTRIDE / NG;
  const int col0 = k_lo + grp * NC;
  uint32_t key_bits = 0u;
  for (int j = 0; j < NC; ++j) {
    const int key = col0 + j;
    if (q_live && key < k_hi && sMask[key] != NEG_INF) key_bits |= 1u << j;
  }

  if (warp == 0) {
    issue_load(TAIL ? -3 : 0);
    issue_load(TAIL ? -2 : 1);
    issue_load(TAIL ? -1 : 2);
  }

  // ---- prologue: residual rows -> TMEM, first LayerNorm -> sA --------------------------------
  {
    const float* src = nullptr;
    if (valid) {
      if (MODE == MODE_POS) {
        const long long b = seq_row / T;
        src = s_row == 0 ? p.X + seq_row * D : p.table_emb + (b * NTAB + (s_row - 1)) * D;
      } else if (MODE == MODE_TEMPORAL) {
        src = p.X + (seq_row * T + s_row) * D;
      } else {
        src = s_row == 0 ? p.cls : p.second_in + (seq_row * T + (s_row - 1)) * D;
      }
    }
    float a[CW];
#pragma unroll
    for (int j = 0; j < CW; j += 4) {
      float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
      if (src) q = __ldg(reinterpret_cast<const float4*>(src + cq + j));
      a[j] = q.x; a[j + 1] = q.y; a[j + 2] = q.z; a[j + 3] = q.w;
    }
    tmem_st32(lane_base + COL_X + cq, a);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    if constexpr (!TAIL) {
      residual_ln(false, 0, nullptr, p.layers[0].ln1w, p.layers[0].ln1b, true, nullptr);
    } else {
      // ---- tail of the last table-token layer on its ball rows: x += attn Wproj^T; x += fc2(ReLU(fc1(LN2(x)))) -------------
      const LayerW tw = p.layers[-1];
      {
        uint4 o[4] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
        if (valid) {
          const uint4* ap = reinterpret_cast<const uint4*>(p.attn_rows + (seq_row * T + s_row) * D + cq);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) o[q4] = __ldg(ap + q4);
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) *reinterpret_cast<uint4*>(sA + a_off(row, cq + 8 * q4)) = o[q4];
      }
      proxy_fence();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        gemm(-3, smem_u32(sA), COL_PROJ);
        if (issuer) commit(bar_mma);
      }
      mma_sync();
      if (warp == 0) issue_load(0);
      residual_ln(true, COL_PROJ, nullptr, tw.ln2w, tw.ln2b, true, nullptr);
      proxy_fence();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        gemm(-2, smem_u32(sA), COL_FC1);
        if (issuer) commit(bar_mma);
      }
      mma_sync();
      if (warp == 0) issue_load(1);
      relu_fc1(tw.fc1b);
      proxy_fence();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        gemm(-1, smem_u32(sQh), COL_FC2);
        if (issuer) commit(bar_mma);
      }
      mma_sync();
      if (warp == 0) issue_load(2);
      residual_ln(true, COL_FC2, tw.fc2b, p.layers[0].ln1w, p.layers[0].ln1b, true, nullptr);
    }
  }

  const float scale = 0.17677669529663687f;     // 1/sqrt(32)
  for (int l = 0; l < p.n_layers; ++l) {
    const LayerW lw = p.layers[l];
    const int g0 = l * 6;
    // ---- QKV GEMM ---------------------------------------------------------------------------
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      gemm(g0 + 0, smem_u32(sA), 0);
      gemm(g0 + 1, smem_u32(sA), 128);
      gemm(g0 + 2, smem_u32(sA), 256);
      if (issuer) commit(bar_mma);
    }
    mma_sync();
    const bool headless = HEADLESS_LAST && l + 1 == p.n_layers;     // last table-token layer: stops after the attention (see TcParams)
    if (warp == 0 && !headless) {                  // proj, fc1; ring slot 2 stays empty (scratch) until the attention is done
      issue_load(g0 + 3);
      issue_load(g0 + 4);
    }
    // ---- q/k/v epilogue: bias, RoPE (q, k), bf16 operands; warp group g takes head g of q, of k and of v -----------
#pragma unroll 1
    for (int i = 0; i < 3; ++i) {
      const int c0 = i * D + cq;
      float a[CW];
      tmem_ld32_nowait(lane_base + c0, a);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < CW; j += 4) {
        const float4 bz = __ldg(reinterpret_cast<const float4*>(lw.qkvb + c0 + j));
        a[j] += bz.x, a[j + 1] += bz.y, a[j + 2] += bz.z, a[j + 3] += bz.w;
      }
      if (i < 2) {
#pragma unroll
        for (int f = 0; f < NF; ++f) {                           // rotate pairs (2f, 2f+1)
          const float x0 = a[2 * f], x1 = a[2 * f + 1];
          a[2 * f] = x0 * rc[f] - x1 * rs[f];
          a[2 * f + 1] = x0 * rs[f] + x1 * rc[f];
        }
        uint8_t* base = (i == 0 ? sQh : sKh) + grp * 8192 + row * 64;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4)                           // 64-byte swizzle: 16-byte chunk ^= (row >> 1) & 3
          *reinterpret_cast<uint4*>(base + ((q4 ^ ((row >> 1) & 3)) << 4)) =
              make_uint4(pack_bf16(a[8 * q4], a[8 * q4 + 1]), pack_bf16(a[8 * q4 + 2], a[8 * q4 + 3]),
                         pack_bf16(a[8 * q4 + 4], a[8 * q4 + 5]), pack_bf16(a[8 * q4 + 6], a[8 * q4 + 7]));
      } else {
        // v transposed: element (dim n, key = row) of head grp; keys contiguous, two 128-byte-swizzled halves
        uint8_t* base = sVt + grp * 8192 + (row >> 6) * 4096;
        const int b = (row & 63) * 2;
#pragma unroll
        for (int n = 0; n < 32; ++n)
          *reinterpret_cast<__nv_bfloat16*>(base + n * 128 + ((((b >> 4) ^ (n & 7)) << 4) | (b & 15))) = __float2bfloat16_rn(a[n]);
      }
    }
    // ---- attention per head on the tensor cores ---------------------------------------------------
    auto issue_scores = [&](int hh) {             // warp 0: S = Q_h K_h^T (K = 32 = two K16 steps)
      const uint32_t qa = smem_u32(sQh + hh * 8192), ka = smem_u32(sKh + hh * 8192);
      issue_mma(tmem_u + COL_S, make_desc_sw64(qa), make_desc_sw64(ka), 0u, IDESC_128x128);
      issue_mma(tmem_u + COL_S, make_desc_sw64(qa + 32), make_desc_sw64(ka + 32), 1u, IDESC_128x128);
    };
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      issue_scores(0);
      if (issuer) commit(bar_mma);
    }
#pragma unroll 1
    for (int hh = 0; hh < HEADS; ++hh) {
      mma_sync();       // S_hh is complete; for hh > 0 so is O_{hh-1}, and P (sA) is free again
      {
        // masks + safe softmax of this row; each warp group takes NC of the row's key columns, the partial maxima meet
        // in shared memory; un-normalised bf16 probabilities -> sA, partial sums -> sSum (used by the O epilogue)
        float e[NC];
        if constexpr (MODE == MODE_POS) {
          float a0[4], a1[4];                      // the warp's rows sit in two 16-row slots: load both, keep the own one
          const uint32_t c = lane_base + COL_S + quarter * 32 + grp * 4;
          tmem_ld4_nowait(c, a0);
          tmem_ld4_nowait(c + 16, a1);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 4; ++j) e[j] = (lane & 16) ? a1[j] : a0[j];
        } else {
          tmem_ld16_nowait(lane_base + COL_S + (quarter >> 1) * 64 + grp * 16, e);
          tmem_ld_wait();
        }
        float mx = NEG_INF;
        if constexpr (ADD_MASK) {
          // finite additive masks: score * scale + (m_k + m_q) like model.py:218-224; a padded query row then attends uniformly
          // over the valid keys (-1e9 absorbs the score)
          const float mq = sMask[row];
#pragma unroll
          for (int j = 0; j < NC; ++j) {
            e[j] = ((key_bits >> j) & 1u) ? e[j] * scale + (sMask[col0 + j] + mq) : NEG_INF;
            mx = fmaxf(mx, e[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < NC; ++j) {
            e[j] = ((key_bits >> j) & 1u) ? e[j] * scale : NEG_INF;
            mx = fmaxf(mx, e[j]);
          }
        }
        sMax[grp][row] = mx;
        quad_barrier(quarter);
#pragma unroll
        for (int g = 0; g < NG; ++g) mx = fmaxf(mx, sMax[g][row]);
        if (mx == NEG_INF) mx = 0.f;              // fully masked row: every exponential below is exp(-inf) = 0 (safe softmax)
        float sum = 0.f;
#pragma unroll
        for (int j = 0; j < NC; ++j) {
          e[j] = __expf(e[j] - mx);
          sum += e[j];
        }
        sSum[hh][grp][row] = sum;
        if constexpr (MODE == MODE_POS) {
          *reinterpret_cast<uint2*>(sA + a_off(row, col0)) = make_uint2(pack_bf16(e[0], e[1]), pack_bf16(e[2], e[3]));
        } else {
#pragma unroll
          for (int jj = 0; jj < NC; jj += 8)
            *reinterpret_cast<uint4*>(sA + a_off(row, col0 + jj)) =
                make_uint4(pack_bf16(e[jj], e[jj + 1]), pack_bf16(e[jj + 2], e[jj + 3]), pack_bf16(e[jj + 4], e[jj + 5]), pack_bf16(e[jj + 6], e[jj + 7]));
        }
        if (hh == 0) {
          // columns outside the row's slot are zero for every head: written once per layer (sA held the LayerNorm output)
          if constexpr (MODE == MODE_POS) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int ch = 4 * i + grp;          // 8-column chunks grp, grp + 4, ...; the slot's own two hold the probabilities
              if ((ch >> 1) != g_row) *reinterpret_cast<uint4*>(sA + a_off(row, ch * 8)) = make_uint4(0, 0, 0, 0);
            }
          } else {
            const int zb = ((quarter >> 1) ? 0 : 64) + grp * 16;
            *reinterpret_cast<uint4*>(sA + a_off(row, zb)) = make_uint4(0, 0, 0, 0);
            *reinterpret_cast<uint4*>(sA + a_off(row, zb + 8)) = make_uint4(0, 0, 0, 0);
          }
        }
      }
      proxy_fence();
      tc_fence_before();
      __syncthreads();
      if (warp == 0) {
        tc_fence_after();
        const uint32_t pa = smem_u32(sA), va = smem_u32(sVt + hh * 8192);
#pragma unroll
        for (int k16 = 0; k16 < 8; ++k16)
          issue_mma(tmem_u + COL_O + hh * HD, make_desc_sw128(pa + (k16 >> 2) * 16384 + (k16 & 3) * 32),
                    make_desc_sw128(va + (k16 >> 2) * 4096 + (k16 & 3) * 32), k16 != 0 ? 1u : 0u, IDESC_128x32);
        if (hh + 1 < HEADS) issue_scores(hh + 1);  // every thread has drained S_hh; one round trip per head
        if (issuer) commit(bar_mma);
      }
    }
    mma_sync();         // O of the last head is complete
    // ---- attention output: O_h / sum -> bf16 A operand of the projection; warp group g normalises head g -------------
    {
      float a[32];
      tmem_ld32_nowait(lane_base + COL_O + grp * HD, a);
      float sum = 0.f;
#pragma unroll
      for (int g = 0; g < NG; ++g) sum += sSum[grp][g][row];
      const float is = sum > 0.f ? 1.f / sum : 0.f;      // a fully masked row sums to zero -> zero output (safe softmax)
      tmem_ld_wait();
      if (headless) {
        // hand the ball rows over to the temporal kernel: attention output (bf16, as the projection would read it) and residual stream
        float x[CW];
        tmem_ld32_nowait(lane_base + COL_X + cq, x);      // warp-collective: every lane loads, the ball rows store
        tmem_ld_wait();
        if (valid && s_row == 0) {
          uint4* ap = reinterpret_cast<uint4*>(p.attn_rows + seq_row * D + grp * HD);
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4)
            ap[q4] = make_uint4(pack_bf16(a[8 * q4] * is, a[8 * q4 + 1] * is), pack_bf16(a[8 * q4 + 2] * is, a[8 * q4 + 3] * is),
                                pack_bf16(a[8 * q4 + 4] * is, a[8 * q4 + 5] * is), pack_bf16(a[8 * q4 + 6] * is, a[8 * q4 + 7] * is));
          float* xp = p.out_rows + seq_row * D + cq;
#pragma unroll
          for (int c = 0; c < CW; c += 4) *reinterpret_cast<float4*>(xp + c) = make_float4(x[c], x[c + 1], x[c + 2], x[c + 3]);
        }
        break;
      }
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4)
        *reinterpret_cast<uint4*>(sA + a_off(row, grp * HD + 8 * q4)) =
            make_uint4(pack_bf16(a[8 * q4] * is, a[8 * q4 + 1] * is), pack_bf16(a[8 * q4 + 2] * is, a[8 * q4 + 3] * is),
                       pack_bf16(a[8 * q4 + 4] * is, a[8 * q4 + 5] * is), pack_bf16(a[8 * q4 + 6] * is, a[8 * q4 + 7] * is));
    }
    // ---- projection GEMM (no bias, model.py:268) -------------------------------------------
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      issue_load(g0 + 5);                         // fc2 weights into ring slot 2: the softmax scratch in it is dead now
      gemm(g0 + 3, smem_u32(sA), COL_PROJ);
      if (issuer) commit(bar_mma);
    }
    mma_sync();
    if (warp == 0) issue_load(g0 + 6);
    // ---- x += proj ; LayerNorm 2 -> sA ---------------------------------------------------
    residual_ln(true, COL_PROJ, nullptr, lw.ln2w, lw.ln2b, true, nullptr);
    // ---- fc1 GEMM ---------------------------------------------------------------------------
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      gemm(g0 + 4, smem_u32(sA), COL_FC1);
      if (issuer) commit(bar_mma);
    }
    mma_sync();
    if (warp == 0) issue_load(g0 + 7);
    // ---- ReLU(fc1 + b) -> bf16 A operand (in the q buffer); 32 columns per warp group ----------
    relu_fc1(lw.fc1b);
    // ---- fc2 GEMM ---------------------------------------------------------------------------
    proxy_fence();
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      gemm(g0 + 5, smem_u32(sQh), COL_FC2);
      if (issuer) commit(bar_mma);
    }
    mma_sync();
    if (warp == 0) issue_load(g0 + 8);
    // ---- x += fc2 + b ; next layer's LayerNorm 1 -> sA, or the stage's output rows ---------------------
    {
      const bool last = l + 1 == p.n_layers;
      float* dst = nullptr;
      if (last && valid) {
        if (MODE == MODE_POS) {
          if (s_row == 0) dst = p.out_rows + seq_row * D;
        } else if (MODE == MODE_TEMPORAL) {
          dst = p.out_rows + (seq_row * T + s_row) * D;
        } else if (s_row == 0) {
          dst = p.out_rows + seq_row * D;
        }
      }
      const LayerW& nx = p.layers[last ? l : l + 1];
      residual_ln(true, COL_FC2, lw.fc2b, nx.ln1w, nx.ln1b, !last, dst);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

__global__ void pack_weights_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}

}  // namespace

// Build the [layers*768][128] bf16 weight matrix (qkv | proj | fc1 | fc2 per layer, torch (out, in) rows = K-major).
int ttk_uplift_tc_prepare(ttk_uplift* h) {
  const int n_layers = h->depth + 4;
  const size_t elems = (size_t)n_layers * LAYER_ROWS * D;
  if (!h->wmat_dev) TTK_CUDA(cudaMalloc((void**)&h->wmat_dev, elems * sizeof(__nv_bfloat16)));
  std::vector<std::string> prefixes;
  char buf[96];
  for (int i = 0; i < 4; ++i) { snprintf(buf, sizeof(buf), "firststage.pos_layers.%d.", i); prefixes.push_back(buf); }
  for (int i = 0; i < h->depth - 4; ++i) { snprintf(buf, sizeof(buf), "firststage.layers.%d.", i); prefixes.push_back(buf); }
  for (int i = 0; i < 4; ++i) { snprintf(buf, sizeof(buf), "secondstage.%d.", i); prefixes.push_back(buf); }
  const float* inv0 = nullptr;
  for (int l = 0; l < n_layers; ++l) {
    const std::string& p = prefixes[l];
    const char* names[4] = {"attn.qkv.weight", "attn.proj.weight", "mlp1.fc1.weight", "mlp1.fc2.weight"};
    const int rows[4] = {384, 128, 128, 128};
    size_t off = (size_t)l * LAYER_ROWS * D;
    for (int m = 0; m < 4; ++m) {
      const int n = rows[m] * D;
      pack_weights_kernel<<<ttk_cdiv(n, 256), 256>>>(h->dev(p + names[m]), h->wmat_dev + off, n);
      TTK_LAUNCH_CHECK();
      off += n;
    }
    if (!inv0) inv0 = h->dev(p + "attn.rotary_emb.inv_freq");
  }
  TTK_CUDA(cudaDeviceSynchronize());
  // the kernels build each row's rotary table once per stage from the first layer's inv_freq (a non-trainable buffer)
  std::vector<float> a(NF), b(NF);
  TTK_CUDA(cudaMemcpy(a.data(), inv0, NF * sizeof(float), cudaMemcpyDeviceToHost));
  for (int l = 1; l < n_layers; ++l) {
    TTK_CUDA(cudaMemcpy(b.data(), h->dev(prefixes[l] + "attn.rotary_emb.inv_freq"), NF * sizeof(float), cudaMemcpyDeviceToHost));
    for (int f = 0; f < NF; ++f)
      if (a[f] != b[f]) {
        ttk_set_error("bf16 uplift path: layers carry different rotary inv_freq tables, which this path does not support");
        return TTK_ERR_UNSUPPORTED;
      }
  }
  h->wmat_ready = true;
  return TTK_OK;
}

int ttk_uplift_tc_stage(ttk_uplift* h, int mode, const UpliftIO& io, cudaStream_t st) {
  EncodeFn encode = get_encode();
  if (!encode) {
    ttk_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return TTK_ERR_CUDA;
  }
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(uplift_tc_kernel<MODE_POS>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    TTK_CUDA(cudaFuncSetAttribute(uplift_tc_kernel<MODE_TEMPORAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    TTK_CUDA(cudaFuncSetAttribute(uplift_tc_kernel<MODE_SECOND>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    TTK_CUDA(cudaFuncSetAttribute(uplift_tc_kernel<MODE_TEMPORAL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    TTK_CUDA(cudaFuncSetAttribute(uplift_tc_kernel<MODE_SECOND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  }
  const int n_layers_total = h->depth + 4;
  CUtensorMap wmap;
  cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)n_layers_total * LAYER_ROWS};
  cuuint64_t strides[1] = {(cuuint64_t)D * 2};
  cuuint32_t box[2] = {64, 128};
  cuuint32_t es[2] = {1, 1};
  const CUresult r = encode(&wmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h->wmat_dev, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    ttk_set_error("cuTensorMapEncodeTiled failed (%d) for the uplift weight matrix", (int)r);
    return TTK_ERR_CUDA;
  }
  TcParams p;
  p.batch = io.batch;
  p.T = io.T;
  p.X = io.X;
  p.table_emb = io.table_emb;
  p.table = io.table;
  p.mask = io.mask;
  p.times = io.times;
  p.cls = h->dev("cls_token");
  p.second_in = h->skip ? io.X : io.second_emb;
  p.attn_rows = (__nv_bfloat16*)io.attn_rows;
  const long long ntok = (long long)io.batch * io.T;
  if (mode == MODE_POS) {
    p.layers = h->layers_dev;
    p.n_layers = 4;
    p.layer_first = 0;
    p.out_rows = io.X;
    uplift_tc_kernel<MODE_POS><<<ttk_cdiv(ntok, 8), TC_THREADS, TC_SMEM, st>>>(wmap, p);
  } else if (mode == MODE_TEMPORAL) {
    p.layers = h->layers_dev + 4;
    p.n_layers = h->depth - 4;
    p.layer_first = 4;
    p.out_rows = io.X;
    if (io.mask_additive)
      uplift_tc_kernel<MODE_TEMPORAL, true><<<ttk_cdiv(io.batch, 2), TC_THREADS, TC_SMEM, st>>>(wmap, p);
    else
      uplift_tc_kernel<MODE_TEMPORAL><<<ttk_cdiv(io.batch, 2), TC_THREADS, TC_SMEM, st>>>(wmap, p);
  } else {
    p.layers = h->layers_dev + h->depth;
    p.n_layers = 4;
    p.layer_first = h->depth;
    p.out_rows = io.table_emb;        // dead by now: receives the [batch][128] cls rows
    if (io.mask_additive)
      uplift_tc_kernel<MODE_SECOND, true><<<ttk_cdiv(io.batch, 2), TC_THREADS, TC_SMEM, st>>>(wmap, p);
    else
      uplift_tc_kernel<MODE_SECOND><<<ttk_cdiv(io.batch, 2), TC_THREADS, TC_SMEM, st>>>(wmap, p);
  }
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}
