// 2D->3D uplifting transformer (MultiStageModel 'multistage' / 'connectstage', dim 128, 4 heads,
// tabletoken_mode 'dynamic', time_rotation 'new').
// Reference: uplifting/model.py:529-571 (MultiStageModel.forward), :335-390 (FirstStage),
// :278-300 (SimpleStaticLayer), :186-229 (rotary attention), :56-102 (RoPE), :105-158 (embeddings),
// :232-261 (heads).
//
// fp32 path.  Whole layer stacks are fused: a CTA keeps its sequences' residual stream in shared
// memory across all layers of a stage (4 table-token layers on 14-token sequences, 12 temporal
// layers, 4 second-stage layers), so activations touch HBM only between stages:
//   embed (ball, table)  ->  stack<POS>  ->  stack<TEMPORAL> (+ position head)  ->  stack<SECOND> (+ rotation head)
// Layer weights (393 KB fp32 each) stream from L2 through a shared-memory tile.
#include <string>
#include <vector>

#include "uplift.h"

namespace {

constexpr int D = 128;          // model width
constexpr int HEADS = 4;
constexpr int HD = 32;          // head dim
constexpr int NF = 16;          // rotary frequencies per head
constexpr int NTAB = 13;        // table keypoints
constexpr int MT = 64;          // token rows per CTA
constexpr int LDX = 132;        // padded row strides (floats)
constexpr int LDQ = 388;
constexpr int LDW = 132;
constexpr int THREADS = 256;
constexpr size_t SMEM_FLOATS = (size_t)MT * (LDX + LDX + LDQ + LDW) + MT * 2 * NF + MT * 2;
constexpr size_t SMEM_BYTES = SMEM_FLOATS * sizeof(float);

enum { MODE_POS = 0, MODE_TEMPORAL = 1, MODE_SECOND = 2 };

struct StackParams {
  const LayerW* layers;   // device array
  int n_layers;
  int batch, T;
  float* X;               // [batch*T][128] residual stream between stages (in/out)
  const float* table_emb; // [batch][13][128]           (POS)
  const float* table;     // [batch][13][3] raw input    (POS: visibility)
  const float* mask;      // [batch][T] {0,1}, or additive {-1e9, 0} values when mask_additive (TEMPORAL, SECOND)
  int mask_additive;
  const float* times;     // [batch][T] seconds          (TEMPORAL, SECOND)
  const float* cls;       // [128]                       (SECOND)
  const float* second_in; // [batch*T][128]              (SECOND: X (skip connection) or embed(pos))
  HeadW head;             // position head (TEMPORAL) / rotation head (SECOND)
  float* head_out;        // pos [batch][T][3] / rot [batch][3]
};

// C[64 x N] = A[64 x 128] * W[N x 128]^T, W row-major in global memory (torch Linear layout).
// 256 threads, each 4 rows x 4 columns per 64-column chunk; epi(m, n, acc) consumes the result.
template <typename Epi>
__device__ __forceinline__ void gemm64(const float* __restrict__ sA, int lda, const float* __restrict__ Wg, int N,
                                       float* __restrict__ sW, Epi epi) {
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  for (int n0 = 0; n0 < N; n0 += 64) {
    for (int i = tid; i < 64 * 32; i += THREADS) {
      const int nn = i >> 5, k4 = i & 31;
      const float4 v = __ldg(reinterpret_cast<const float4*>(Wg + (size_t)(n0 + nn) * D) + k4);
      *reinterpret_cast<float4*>(sW + nn * LDW + k4 * 4) = v;
    }
    __syncthreads();
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < D; k += 4) {
      float4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(sA + (ty * 4 + i) * lda + k);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4*>(sW + (tx + 16 * j) * LDW + k);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]);
          acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
          acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]);
          acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) epi(ty * 4 + i, n0 + tx + 16 * j, acc[i][j]);
    __syncthreads();
  }
}

// LayerNorm(eps 1e-5) of rows [0, M) of sX into sH; one warp per row.
__device__ __forceinline__ void layer_norm(const float* sX, float* sH, int M, const float* __restrict__ w,
                                           const float* __restrict__ b) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < M; r += THREADS / 32) {
    const float4 v = *reinterpret_cast<const float4*>(sX + r * LDX + lane * 4);
    float s = v.x + v.y + v.z + v.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s * (1.f / D);
    const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
    float q = dx * dx + dy * dy + dz * dz + dw * dw;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q * (1.f / D) + 1e-5f);
    const float4 g = __ldg(reinterpret_cast<const float4*>(w) + lane);
    const float4 be = __ldg(reinterpret_cast<const float4*>(b) + lane);
    float4 o4;
    o4.x = dx * rstd * g.x + be.x;
    o4.y = dy * rstd * g.y + be.y;
    o4.z = dz * rstd * g.z + be.z;
    o4.w = dw * rstd * g.w + be.w;
    *reinterpret_cast<float4*>(sH + r * LDX + lane * 4) = o4;
  }
}

// MyHead (128 -> 64 -> 32 -> 3, ReLU between) on one row held in shared memory; one warp.
__device__ __forceinline__ void head_row(const float* row, const HeadW& hw, float* out3, float* scratch /*>=96 floats per warp*/) {
  const int lane = threadIdx.x & 31;
  for (int o = lane; o < 64; o += 32) {
    float acc = __ldg(hw.b1 + o);
    const float4* wr = reinterpret_cast<const float4*>(hw.w1 + (size_t)o * D);
    for (int k = 0; k < D / 4; ++k) {
      const float4 wv = __ldg(wr + k);
      const float4 xv = *reinterpret_cast<const float4*>(row + 4 * k);
      acc = fmaf(xv.x, wv.x, acc);
      acc = fmaf(xv.y, wv.y, acc);
      acc = fmaf(xv.z, wv.z, acc);
      acc = fmaf(xv.w, wv.w, acc);
    }
    scratch[o] = fmaxf(acc, 0.f);
  }
  __syncwarp();
  {
    float acc = __ldg(hw.b2 + lane);
    for (int k = 0; k < 64; ++k) acc = fmaf(scratch[k], __ldg(hw.w2 + lane * 64 + k), acc);
    scratch[64 + lane] = fmaxf(acc, 0.f);
  }
  __syncwarp();
  if (lane < 3) {
    float acc = __ldg(hw.b3 + lane);
    for (int k = 0; k < 32; ++k) acc = fmaf(scratch[64 + k], __ldg(hw.w3 + lane * 32 + k), acc);
    out3[lane] = acc;
  }
  __syncwarp();
}

template <int MODE>
__global__ void __launch_bounds__(THREADS, 1) uplift_stack_kernel(StackParams p) {
  extern __shared__ __align__(16) float smem[];
  float* sX = smem;
  float* sH = sX + MT * LDX;
  float* sQ = sH + MT * LDX;
  float* sW = sQ + MT * LDQ;
  float* sCos = sW + MT * LDW;      // [MT][NF]
  float* sSin = sCos + MT * NF;
  float* sMask = sSin + MT * NF;    // additive mask per row (0 / -inf, or the caller's additive values)
  float* sTime = sMask + MT;        // time per row; NaN = no rotation (cls token)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = p.T;
  const int S = MODE == MODE_POS ? NTAB + 1 : (MODE == MODE_TEMPORAL ? T : T + 1);
  const int G = MODE == MODE_POS ? 4 : 1;
  const long long n_seq = MODE == MODE_POS ? (long long)p.batch * T : p.batch;
  const long long seq0 = (long long)blockIdx.x * G;
  const int g_here = (int)min((long long)G, n_seq - seq0);
  const int M = g_here * S;
  const float NEG_INF = -INFINITY;
  const float NO_ROPE = __int_as_float(0x7fc00000);

  // ---- prologue: residual stream rows, masks, times --------------------------------------
  for (int i = tid; i < MT * (D / 4); i += THREADS) {
    const int r = i / (D / 4), c4 = i % (D / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < M) {
      const int g = r / S, s = r - g * S;
      const long long seq = seq0 + g;
      const float* src;
      if (MODE == MODE_POS) {
        const long long b = seq / T;
        src = s == 0 ? p.X + seq * D : p.table_emb + (b * NTAB + (s - 1)) * D;
      } else if (MODE == MODE_TEMPORAL) {
        src = p.X + (seq * T + s) * D;
      } else {
        src = s == 0 ? p.cls : p.second_in + (seq * T + (s - 1)) * D;
      }
      v = __ldg(reinterpret_cast<const float4*>(src) + c4);
    }
    *reinterpret_cast<float4*>(sX + r * LDX + c4 * 4) = v;
  }
  for (int r = tid; r < MT; r += THREADS) {
    float m = 0.f, t = NO_ROPE;
    if (r < M) {
      const int g = r / S, s = r - g * S;
      const long long seq = seq0 + g;
      if (MODE == MODE_POS) {
        if (s > 0) {
          const long long b = seq / T;
          m = p.table[(b * NTAB + (s - 1)) * 3 + 2] == 1.f ? 0.f : NEG_INF;    // model.py:363
          t = (float)(s - 1) / 100.f;                                           // model.py:367, arange / (MAX_FPS / 5)
        }
      } else if (MODE == MODE_TEMPORAL || s > 0) {
        const float mv = p.mask[seq * T + s - (MODE == MODE_SECOND)];
        m = p.mask_additive ? mv : (mv == 0.f ? NEG_INF : 0.f);                 // model.py:541-546
        t = p.times[seq * T + s - (MODE == MODE_SECOND)];
      }
    }
    sMask[r] = m;
    sTime[r] = t;
  }
  __syncthreads();

  const float scale = 0.17677669529663687f;   // 1/sqrt(32), SDPA default

  for (int l = 0; l < p.n_layers; ++l) {
    const LayerW lw = p.layers[l];
    // rotary tables for this layer: pos = round(t / (1/500)) (model.py:72), angle = pos * inv_freq
    for (int i = tid; i < MT * NF; i += THREADS) {
      const int r = i / NF, f = i % NF;
      const float t = sTime[r];
      float c = 1.f, s = 0.f;
      if (t == t) {
        const float pos = rintf(__fdiv_rn(t, 0.002f));
        const float ang = __fmul_rn(pos, __ldg(lw.invf + f));
        sincosf(ang, &s, &c);
      }
      sCos[i] = c;
      sSin[i] = s;
    }
    layer_norm(sX, sH, M, lw.ln1w, lw.ln1b);
    __syncthreads();
    // qkv = LN(x) Wqkv^T + b ; rotary on q (cols 0..127) and k (cols 128..255), pairs (2f, 2f+1) per head
    gemm64(sH, LDX, lw.qkvw, 3 * D, sW, [&](int m, int n, float acc) { sQ[m * LDQ + n] = acc + __ldg(lw.qkvb + n); });
    for (int i = tid; i < M * 2 * HEADS * NF; i += THREADS) {
      const int f = i % NF, hh = (i / NF) % (2 * HEADS), r = i / (NF * 2 * HEADS);
      float* q = sQ + r * LDQ + hh * HD + 2 * f;     // hh 0..3: q heads, 4..7: k heads (contiguous columns)
      const float c = sCos[r * NF + f], s = sSin[r * NF + f];
      const float a = q[0], b = q[1];
      q[0] = a * c - b * s;
      q[1] = a * s + b * c;
    }
    __syncthreads();
    // attention: one warp per (sequence, head, query row); lanes over keys, then over head dims
    for (int item = warp; item < M * HEADS; item += THREADS / 32) {
      const int r = item / HEADS, hh = item % HEADS;
      const int g = r / S;
      const int k0 = g * S;
      const float* q = sQ + r * LDQ + hh * HD;
      const float mq = sMask[r];
      float sc[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = lane + 32 * u;
        float v = NEG_INF;
        if (j < S) {
          const float* kk = sQ + (k0 + j) * LDQ + D + hh * HD;
          float acc = 0.f;
#pragma unroll
          for (int d = 0; d < HD; d += 4) {
            const float4 qa = *reinterpret_cast<const float4*>(q + d);
            const float4 ka = *reinterpret_cast<const float4*>(kk + d);
            acc = fmaf(qa.x, ka.x, acc);
            acc = fmaf(qa.y, ka.y, acc);
            acc = fmaf(qa.z, ka.z, acc);
            acc = fmaf(qa.w, ka.w, acc);
          }
          v = acc * scale + (sMask[k0 + j] + mq);
        }
        sc[u] = v;
      }
      float mx = fmaxf(sc[0], sc[1]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      float e0 = 0.f, e1 = 0.f, inv = 0.f;
      if (mx != NEG_INF) {                       // fully masked row -> all-zero probabilities (safe softmax)
        e0 = sc[0] == NEG_INF ? 0.f : expf(sc[0] - mx);
        e1 = sc[1] == NEG_INF ? 0.f : expf(sc[1] - mx);
        float sum = e0 + e1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        inv = 1.f / sum;
      }
      e0 *= inv;
      e1 *= inv;
      float acc = 0.f;
      for (int j = 0; j < S; ++j) {
        const float pj = __shfl_sync(0xffffffffu, j < 32 ? e0 : e1, j & 31);
        acc = fmaf(pj, sQ[(k0 + j) * LDQ + 2 * D + hh * HD + lane], acc);
      }
      sH[r * LDX + hh * HD + lane] = acc;
    }
    __syncthreads();
    // x += attn Wproj^T (no bias: model.py:268 passes attn_drop_rate into the proj_bias slot)
    gemm64(sH, LDX, lw.projw, D, sW, [&](int m, int n, float acc) { sX[m * LDX + n] += acc; });
    layer_norm(sX, sH, M, lw.ln2w, lw.ln2b);
    __syncthreads();
    gemm64(sH, LDX, lw.fc1w, D, sW, [&](int m, int n, float acc) { sQ[m * LDQ + n] = fmaxf(acc + __ldg(lw.fc1b + n), 0.f); });
    gemm64(sQ, LDQ, lw.fc2w, D, sW, [&](int m, int n, float acc) { sX[m * LDX + n] += acc + __ldg(lw.fc2b + n); });
  }

  // ---- epilogue ----------------------------------------------------------------------------
  if (MODE == MODE_POS) {
    for (int i = tid; i < g_here * (D / 4); i += THREADS) {
      const int g = i / (D / 4), c4 = i % (D / 4);
      *(reinterpret_cast<float4*>(p.X + (seq0 + g) * D) + c4) = *reinterpret_cast<const float4*>(sX + g * S * LDX + c4 * 4);
    }
  } else if (MODE == MODE_TEMPORAL) {
    for (int i = tid; i < M * (D / 4); i += THREADS) {
      const int r = i / (D / 4), c4 = i % (D / 4);
      *(reinterpret_cast<float4*>(p.X + (seq0 * T + r) * D) + c4) = *reinterpret_cast<const float4*>(sX + r * LDX + c4 * 4);
    }
    float* scratch = sW + warp * 96;
    for (int r = warp; r < M; r += THREADS / 32) head_row(sX + r * LDX, p.head, p.head_out + (seq0 * T + r) * 3, scratch);
  } else {
    if (warp == 0) head_row(sX, p.head, p.head_out + seq0 * 3, sW);
  }
}

// MyHead on rows of a [n_rows][128] fp32 matrix in global memory (used by the bf16 path): 64 rows per CTA, fc1 through the
// register-tiled GEMM, fc2 / fc3 from shared memory.  (One warp per row re-read the 41 KB of head weights per row: 3.2 ms for
// the 204 800 rows of a 4096-trajectory batch; this form takes a fraction of that.)
constexpr int LDH1 = 68, LDW2 = 65, LDH2 = 33;
constexpr size_t HEAD_SMEM_BYTES = ((size_t)MT * (LDX + LDW + LDH1 + LDH2) + 32 * LDW2) * sizeof(float);
__global__ void __launch_bounds__(THREADS, 2) head_kernel(const float* __restrict__ rows, long long n_rows, HeadW hw, float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  float* sX = smem;                  // [64][LDX] input rows
  float* sW = sX + MT * LDX;         // [64][LDW] fc1 weight tile (gemm64)
  float* sH1 = sW + MT * LDW;        // [64][LDH1] ReLU(fc1)
  float* sH2 = sH1 + MT * LDH1;      // [64][LDH2] ReLU(fc2)
  float* sW2 = sH2 + MT * LDH2;      // [32][LDW2] fc2 weights
  const int tid = threadIdx.x;
  const long long r0 = (long long)blockIdx.x * MT;
  for (int i = tid; i < MT * (D / 4); i += THREADS) {
    const int r = i / (D / 4), c4 = i % (D / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < n_rows) v = __ldg(reinterpret_cast<const float4*>(rows + (r0 + r) * D) + c4);
    *reinterpret_cast<float4*>(sX + r * LDX + c4 * 4) = v;
  }
  for (int i = tid; i < 32 * 64; i += THREADS) sW2[(i >> 6) * LDW2 + (i & 63)] = __ldg(hw.w2 + i);
  __syncthreads();
  gemm64(sX, LDX, hw.w1, 64, sW, [&](int m, int n, float acc) { sH1[m * LDH1 + n] = fmaxf(acc + __ldg(hw.b1 + n), 0.f); });
  {
    // fc2: thread = (row, 8 of the 32 outputs); the fmaf chain over k ascends like the one-warp form
    const int m = tid >> 2, j0 = (tid & 3) * 8;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = __ldg(hw.b2 + j0 + j);
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      const float a = sH1[m * LDH1 + k];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(a, sW2[(j0 + j) * LDW2 + k], acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) sH2[m * LDH2 + j0 + j] = fmaxf(acc[j], 0.f);
  }
  __syncthreads();
  if (tid < MT * 3) {
    const int m = tid / 3, o = tid - m * 3;
    if (r0 + m < n_rows) {
      float acc = __ldg(hw.b3 + o);
#pragma unroll 8
      for (int k = 0; k < 32; ++k) acc = fmaf(sH2[m * LDH2 + k], __ldg(hw.w3 + o * 32 + k), acc);
      out[(r0 + m) * 3 + o] = acc;
    }
  }
}

// Two-layer embedding (Linear(in_dim,128) -> ReLU -> Linear(128,128)) for 64 tokens per CTA
// (BallEmbedding / TableEmbedding, model.py:105-158).
__global__ void __launch_bounds__(THREADS, 1) embed_kernel(const float* __restrict__ in, int in_dim, int in_stride,
                                                           long long n_tokens, const float* __restrict__ w1,
                                                           const float* __restrict__ b1, const float* __restrict__ w2,
                                                           const float* __restrict__ b2, float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  float* sX = smem;                 // output rows
  float* sH = sX + MT * LDX;        // hidden rows
  float* sW = sH + MT * LDX;
  const int tid = threadIdx.x;
  const long long t0 = (long long)blockIdx.x * MT;
  for (int i = tid; i < MT * D; i += THREADS) {
    const int r = i / D, c = i % D;
    float v = 0.f;
    if (t0 + r < n_tokens) {
      float acc = __ldg(b1 + c);
      for (int k = 0; k < in_dim; ++k) acc = fmaf(__ldg(in + (t0 + r) * in_stride + k), __ldg(w1 + c * in_dim + k), acc);
      v = fmaxf(acc, 0.f);
    }
    sH[r * LDX + c] = v;
  }
  __syncthreads();
  gemm64(sH, LDX, w2, D, sW, [&](int m, int n, float acc) { sX[m * LDX + n] = acc + __ldg(b2 + n); });
  for (int i = tid; i < MT * (D / 4); i += THREADS) {
    const int r = i / (D / 4), c4 = i % (D / 4);
    if (t0 + r < n_tokens) *(reinterpret_cast<float4*>(out + (t0 + r) * D) + c4) = *reinterpret_cast<const float4*>(sX + r * LDX + c4 * 4);
  }
}

}  // namespace

namespace {

void add_linear(ttk_uplift* h, const std::string& p, int in, int out) {
  h->params.push_back({p + ".weight", in * out});
  h->params.push_back({p + ".bias", out});
}

void add_layer(ttk_uplift* h, const std::string& p) {
  h->params.push_back({p + "attn.qkv.weight", 3 * D * D});
  h->params.push_back({p + "attn.qkv.bias", 3 * D});
  h->params.push_back({p + "attn.proj.weight", D * D});
  h->params.push_back({p + "attn.rotary_emb.inv_freq", NF});
  add_linear(h, p + "mlp1.fc1", D, D);
  add_linear(h, p + "mlp1.fc2", D, D);
  h->params.push_back({p + "norm1.weight", D});
  h->params.push_back({p + "norm1.bias", D});
  h->params.push_back({p + "norm2.weight", D});
  h->params.push_back({p + "norm2.bias", D});
}

void add_head(ttk_uplift* h, const std::string& p) {
  add_linear(h, p + ".fc1", D, D / 2);
  add_linear(h, p + ".fc2", D / 2, D / 4);
  add_linear(h, p + ".fc3", D / 4, 3);
}

LayerW layer_ptrs(const ttk_uplift* h, const std::string& p) {
  LayerW w;
  w.ln1w = h->dev(p + "norm1.weight");
  w.ln1b = h->dev(p + "norm1.bias");
  w.qkvw = h->dev(p + "attn.qkv.weight");
  w.qkvb = h->dev(p + "attn.qkv.bias");
  w.projw = h->dev(p + "attn.proj.weight");
  w.invf = h->dev(p + "attn.rotary_emb.inv_freq");
  w.fc1w = h->dev(p + "mlp1.fc1.weight");
  w.fc1b = h->dev(p + "mlp1.fc1.bias");
  w.fc2w = h->dev(p + "mlp1.fc2.weight");
  w.fc2b = h->dev(p + "mlp1.fc2.bias");
  w.ln2w = h->dev(p + "norm2.weight");
  w.ln2b = h->dev(p + "norm2.bias");
  return w;
}

HeadW head_ptrs(const ttk_uplift* h, const std::string& p) {
  HeadW w;
  w.w1 = h->dev(p + ".fc1.weight");
  w.b1 = h->dev(p + ".fc1.bias");
  w.w2 = h->dev(p + ".fc2.weight");
  w.b2 = h->dev(p + ".fc2.bias");
  w.w3 = h->dev(p + ".fc3.weight");
  w.b3 = h->dev(p + ".fc3.bias");
  return w;
}

std::string idx(const char* f, int i) {
  char b[96];
  snprintf(b, sizeof(b), f, i);
  return b;
}

int finalize_layers(ttk_uplift* h) {
  std::vector<LayerW> L;
  for (int i = 0; i < 4; ++i) L.push_back(layer_ptrs(h, idx("firststage.pos_layers.%d.", i)));
  for (int i = 0; i < h->depth - 4; ++i) L.push_back(layer_ptrs(h, idx("firststage.layers.%d.", i)));
  for (int i = 0; i < 4; ++i) L.push_back(layer_ptrs(h, idx("secondstage.%d.", i)));
  if (!h->layers_dev) TTK_CUDA(cudaMalloc((void**)&h->layers_dev, L.size() * sizeof(LayerW)));
  TTK_CUDA(cudaMemcpy(h->layers_dev, L.data(), L.size() * sizeof(LayerW), cudaMemcpyHostToDevice));
  h->layers_ready = true;
  return TTK_OK;
}

}  // namespace

extern "C" int ttk_uplift_create(int dim, int heads, int depth, int use_skipconnection, ttk_uplift** out) {
  TTK_CHECK_ARG(out, "ttk_uplift_create: null out");
  if (dim != D || heads != HEADS) {
    ttk_set_error("ttk_uplift_create: only the 'large' model (dim 128, 4 heads) has kernels (got dim %d, heads %d)", dim, heads);
    return TTK_ERR_UNSUPPORTED;
  }
  TTK_CHECK_ARG(depth > 4 && depth <= 64, "ttk_uplift_create: bad depth %d", depth);
  ttk_uplift* h = new ttk_uplift();
  h->dim = dim;
  h->heads = heads;
  h->depth = depth;
  h->skip = use_skipconnection ? 1 : 0;
  // order of oracle/uplift.py:state_dict_layout
  h->params.push_back({"cls_token", D});
  add_linear(h, "embed.fc1", 3, D);
  add_linear(h, "embed.fc2", D, D);
  add_linear(h, "firststage.ball_embed.fc1", 2, D);
  add_linear(h, "firststage.ball_embed.fc2", D, D);
  add_linear(h, "firststage.table_embed.fc1", 2, D);
  add_linear(h, "firststage.table_embed.fc2", D, D);
  for (int i = 0; i < 4; ++i) add_layer(h, idx("firststage.pos_layers.%d.", i));
  for (int i = 0; i < depth - 4; ++i) add_layer(h, idx("firststage.layers.%d.", i));
  add_head(h, "firststage.position_head");
  for (int i = 0; i < 4; ++i) add_layer(h, idx("secondstage.%d.", i));
  add_head(h, "rotation_head");
  *out = h;
  return TTK_OK;
}

extern "C" void ttk_uplift_destroy(ttk_uplift* h) {
  if (!h) return;
  for (UpliftParam& p : h->params) cudaFree(p.dev);
  cudaFree(h->wmat_dev);
  cudaFree(h->w3_hi);
  cudaFree(h->w3_lo);
  cudaFree(h->layers_dev);
  delete h;
}

extern "C" int ttk_uplift_num_params(const ttk_uplift* h) { return h ? (int)h->params.size() : 0; }

extern "C" int ttk_uplift_param_info(const ttk_uplift* h, int i, char* name, int* numel) {
  TTK_CHECK_ARG(h && i >= 0 && i < (int)h->params.size(), "ttk_uplift_param_info: bad index %d", i);
  if (name) snprintf(name, 128, "%s", h->params[i].name.c_str());
  if (numel) *numel = h->params[i].numel;
  return TTK_OK;
}

extern "C" int ttk_uplift_set_param(ttk_uplift* h, int i, const float* data_host, int numel) {
  TTK_CHECK_ARG(h && i >= 0 && i < (int)h->params.size(), "ttk_uplift_set_param: bad index %d", i);
  UpliftParam& p = h->params[i];
  TTK_CHECK_ARG(data_host && numel == p.numel, "ttk_uplift_set_param: %s expects %d elements, got %d", p.name.c_str(), p.numel, numel);
  if (int rc = ttk_bind_device(&h->device, "ttk_uplift_set_param")) return rc;
  if (!p.dev) TTK_CUDA(cudaMalloc((void**)&p.dev, (size_t)numel * sizeof(float)));
  TTK_CUDA(cudaMemcpy(p.dev, data_host, (size_t)numel * sizeof(float), cudaMemcpyHostToDevice));
  p.set = true;
  h->layers_ready = false;
  h->wmat_ready = false;
  h->w3_ready = false;
  return TTK_OK;
}

namespace {
// X [B*T][128] + table_emb [B*13][128] (+ embed(pos) [B*T][128] without skip connection) + bf16 attention rows [B*T][128]
size_t base_workspace_bytes(const ttk_uplift* h, int batch, int seq_len) {
  size_t tokens = (size_t)batch * seq_len * (h->skip ? 1 : 2) + (size_t)batch * NTAB;
  return (tokens * D * sizeof(float) + (size_t)batch * seq_len * D * 2 + 1024 + 1023) & ~(size_t)1023;
}
}  // namespace

extern "C" size_t ttk_uplift_workspace_bytes(const ttk_uplift* h, int batch, int seq_len, int dtype) {
  if (!h || batch <= 0 || seq_len <= 0) return 0;
  // the tf32x3 path keeps a layer's activations in HBM between its kernels (uplift3.cu)
  return base_workspace_bytes(h, batch, seq_len) + (dtype == TTK_TF32X3 ? ttk_uplift3_workspace_bytes(h, batch, seq_len) : 0);
}

extern "C" int ttk_uplift_forward(ttk_uplift* h, const float* ball_dev, const float* table_dev, const float* mask_dev,
                                  const float* times_dev, int batch, int seq_len, int mask_additive, int dtype, float* rot_out_dev,
                                  float* pos_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
  TTK_CHECK_ARG(h, "ttk_uplift_forward: null handle");
  h->launches = 0;
  if (int rc = ttk_bind_device(&h->device, "ttk_uplift_forward")) return rc;
  TTK_CHECK_ARG(dtype == TTK_F32 || dtype == TTK_BF16 || dtype == TTK_TF32X3, "ttk_uplift_forward: bad dtype %d", dtype);
  TTK_CHECK_ARG(batch >= 0 && seq_len >= 2 && seq_len + 1 <= MT, "ttk_uplift_forward: seq_len must be in [2, %d] (got %d)", MT - 1, seq_len);
  for (const UpliftParam& p : h->params)
    if (!p.set) {
      ttk_set_error("ttk_uplift_forward: parameter %s was never set", p.name.c_str());
      return TTK_ERR_STATE;
    }
  if (batch == 0) return TTK_OK;
  TTK_CHECK_ARG(ball_dev && table_dev && mask_dev && times_dev && rot_out_dev && pos_out_dev && workspace_dev,
                "ttk_uplift_forward: null pointer");
  TTK_CHECK_ARG(workspace_bytes >= ttk_uplift_workspace_bytes(h, batch, seq_len, dtype), "ttk_uplift_forward: workspace too small");
  if (!h->layers_ready) {
    int rc = finalize_layers(h);
    if (rc) return rc;
  }
  static TtkPerDevice attr_done;
  if (attr_done.first()) {
    TTK_CUDA(cudaFuncSetAttribute(uplift_stack_kernel<MODE_POS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    TTK_CUDA(cudaFuncSetAttribute(uplift_stack_kernel<MODE_TEMPORAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    TTK_CUDA(cudaFuncSetAttribute(uplift_stack_kernel<MODE_SECOND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    TTK_CUDA(cudaFuncSetAttribute(embed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    TTK_CUDA(cudaFuncSetAttribute(head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)HEAD_SMEM_BYTES));
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int T = seq_len;
  const long long ntok = (long long)batch * T;
  float* X = (float*)workspace_dev;
  float* table_emb = X + ntok * D;
  float* second_emb = table_emb + (long long)batch * NTAB * D;
  TTK_CHECK_ARG(ntok / 4 + 1 < 2147483647LL, "ttk_uplift_forward: batch too large for one launch");

  embed_kernel<<<ttk_cdiv(ntok, MT), THREADS, SMEM_BYTES, st>>>(ball_dev, 2, 2, ntok, h->dev("firststage.ball_embed.fc1.weight"),
                                                               h->dev("firststage.ball_embed.fc1.bias"),
                                                               h->dev("firststage.ball_embed.fc2.weight"),
                                                               h->dev("firststage.ball_embed.fc2.bias"), X);
  TTK_LAUNCH_CHECK();
  embed_kernel<<<ttk_cdiv((long long)batch * NTAB, MT), THREADS, SMEM_BYTES, st>>>(
      table_dev, 2, 3, (long long)batch * NTAB, h->dev("firststage.table_embed.fc1.weight"), h->dev("firststage.table_embed.fc1.bias"),
      h->dev("firststage.table_embed.fc2.weight"), h->dev("firststage.table_embed.fc2.bias"), table_emb);
  TTK_LAUNCH_CHECK();
  h->launches += 2;

  if (dtype == TTK_TF32X3) {
    // fp32-class tensor-core path: every Linear layer as three TF32 products of split operands (gemm3_umma.cu, uplift3.cu); heads stay SIMT
    if (!h->w3_ready) {
      int rc = ttk_uplift3_prepare(h);
      if (rc) return rc;
    }
    UpliftIO io;
    io.ball = ball_dev;
    io.table = table_dev;
    io.mask = mask_dev;
    io.mask_additive = mask_additive;
    io.times = times_dev;
    io.batch = batch;
    io.T = T;
    io.rot_out = rot_out_dev;
    io.pos_out = pos_out_dev;
    io.X = X;
    io.table_emb = table_emb;
    io.second_emb = second_emb;
    io.attn_rows = nullptr;
    void* ws3 = (char*)workspace_dev + base_workspace_bytes(h, batch, seq_len);
    int rc = ttk_uplift3_stage(h, MODE_POS, io, ws3, st);
    if (rc) return rc;
    rc = ttk_uplift3_stage(h, MODE_TEMPORAL, io, ws3, st);
    if (rc) return rc;
    head_kernel<<<ttk_cdiv(ntok, MT), THREADS, HEAD_SMEM_BYTES, st>>>(X, ntok, head_ptrs(h, "firststage.position_head"), pos_out_dev);
    TTK_LAUNCH_CHECK();
    h->launches += 1;
    if (!h->skip) {
      embed_kernel<<<ttk_cdiv(ntok, MT), THREADS, SMEM_BYTES, st>>>(pos_out_dev, 3, 3, ntok, h->dev("embed.fc1.weight"),
                                                                   h->dev("embed.fc1.bias"), h->dev("embed.fc2.weight"),
                                                                   h->dev("embed.fc2.bias"), second_emb);
      TTK_LAUNCH_CHECK();
      h->launches += 1;
    }
    rc = ttk_uplift3_stage(h, MODE_SECOND, io, ws3, st);
    if (rc) return rc;
    head_kernel<<<ttk_cdiv(batch, MT), THREADS, HEAD_SMEM_BYTES, st>>>(table_emb, batch, head_ptrs(h, "rotation_head"), rot_out_dev);
    TTK_LAUNCH_CHECK();
    h->launches += 1;
    return TTK_OK;
  }

  if (dtype == TTK_BF16) {
    // tensor-core path: tcgen05 GEMMs, residual stream in TMEM (uplift_tc.cu); heads stay fp32
    if (!h->wmat_ready) {
      int rc = ttk_uplift_tc_prepare(h);
      if (rc) return rc;
    }
    UpliftIO io;
    io.ball = ball_dev;
    io.table = table_dev;
    io.mask = mask_dev;
    io.mask_additive = mask_additive;
    io.times = times_dev;
    io.batch = batch;
    io.T = T;
    io.rot_out = rot_out_dev;
    io.pos_out = pos_out_dev;
    io.X = X;
    io.table_emb = table_emb;
    io.second_emb = second_emb;
    io.attn_rows = second_emb + (h->skip ? 0 : ntok * D);
    int rc = ttk_uplift_tc_stage(h, MODE_POS, io, st);
    if (rc) return rc;
    rc = ttk_uplift_tc_stage(h, MODE_TEMPORAL, io, st);
    if (rc) return rc;
    head_kernel<<<ttk_cdiv(ntok, MT), THREADS, HEAD_SMEM_BYTES, st>>>(X, ntok, head_ptrs(h, "firststage.position_head"), pos_out_dev);
    TTK_LAUNCH_CHECK();
    h->launches += 3;
    if (!h->skip) {
      embed_kernel<<<ttk_cdiv(ntok, MT), THREADS, SMEM_BYTES, st>>>(pos_out_dev, 3, 3, ntok, h->dev("embed.fc1.weight"),
                                                                   h->dev("embed.fc1.bias"), h->dev("embed.fc2.weight"),
                                                                   h->dev("embed.fc2.bias"), second_emb);
      TTK_LAUNCH_CHECK();
      h->launches += 1;
    }
    rc = ttk_uplift_tc_stage(h, MODE_SECOND, io, st);
    if (rc) return rc;
    head_kernel<<<ttk_cdiv(batch, MT), THREADS, HEAD_SMEM_BYTES, st>>>(table_emb, batch, head_ptrs(h, "rotation_head"), rot_out_dev);
    TTK_LAUNCH_CHECK();
    h->launches += 2;
    return TTK_OK;
  }

  StackParams p;
  p.batch = batch;
  p.T = T;
  p.X = X;
  p.table_emb = table_emb;
  p.table = table_dev;
  p.mask = mask_dev;
  p.mask_additive = mask_additive;
  p.times = times_dev;
  p.cls = h->dev("cls_token");
  p.second_in = X;
  p.head_out = nullptr;
  p.head = head_ptrs(h, "firststage.position_head");

  p.layers = h->layers_dev;
  p.n_layers = 4;
  uplift_stack_kernel<MODE_POS><<<ttk_cdiv(ntok, 4), THREADS, SMEM_BYTES, st>>>(p);
  TTK_LAUNCH_CHECK();

  p.layers = h->layers_dev + 4;
  p.n_layers = h->depth - 4;
  p.head_out = pos_out_dev;
  uplift_stack_kernel<MODE_TEMPORAL><<<batch, THREADS, SMEM_BYTES, st>>>(p);
  TTK_LAUNCH_CHECK();
  h->launches += 2;

  if (!h->skip) {
    // multistage: second stage embeds the predicted 3-D positions (model.py:551-559)
    embed_kernel<<<ttk_cdiv(ntok, MT), THREADS, SMEM_BYTES, st>>>(pos_out_dev, 3, 3, ntok, h->dev("embed.fc1.weight"),
                                                                 h->dev("embed.fc1.bias"), h->dev("embed.fc2.weight"),
                                                                 h->dev("embed.fc2.bias"), second_emb);
    TTK_LAUNCH_CHECK();
    h->launches += 1;
    p.second_in = second_emb;
  }
  p.layers = h->layers_dev + h->depth;
  p.n_layers = 4;
  p.head = head_ptrs(h, "rotation_head");
  p.head_out = rot_out_dev;
  uplift_stack_kernel<MODE_SECOND><<<batch, THREADS, SMEM_BYTES, st>>>(p);
  TTK_LAUNCH_CHECK();
  h->launches += 1;
  return TTK_OK;
}

extern "C" int ttk_uplift_last_launches(const ttk_uplift* h) { return h ? h->launches : 0; }
