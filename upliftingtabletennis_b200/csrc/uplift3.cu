// Uplifting transformer, fp32-class tensor-core path ("tf32x3"): every Linear layer runs as ttk_gemm3 (three TF32 tensor-core products
// per term, fp32-level results, LayerNorm applied while the A operand is split), attention in fp32 on CUDA cores.
// Reference: uplifting/model.py:529-571 (MultiStageModel.forward), :335-390 (FirstStage), :278-300 (SimpleStaticLayer),
// :186-229 (rotary attention), :56-102 (RoPE).
//
// Unlike the fused fp32 SIMT stacks (uplift.cu) the residual stream lives in HBM between the kernels of a layer:
//     x, stats --[LN1 on load] gemm3 qkv (+bias)--> qkv --attention3--> o --gemm3 proj (+x, stats)--> x
//       --[LN2 on load] gemm3 fc1 (+bias, ReLU)--> a --gemm3 fc2 (+bias, +x, stats)--> x
// i.e. 15 passes over a [rows][128] fp32 tensor per layer, which is what bounds it (the three-product GEMM of a 128 x 128 tile takes
// 3 k clk on the tensor pipe against ~8 k clk of HBM time); the fused SIMT stacks are bound by the fp32 FMA rate instead and are ~6x
// slower.  Row layouts: table-token stage rows = (b T + t) 14 + s (ball token s = 0, table tokens 1..13), temporal stage rows = b T + s,
// second stage rows = b (T + 1) + s (cls token s = 0).
#include <algorithm>

#include "uplift.h"

namespace {

constexpr int D = 128, HEADS = 4, HD = 32, NF = 16, NTAB = 13;
constexpr int LAYER_ROWS = 768;                    // qkv 384 | proj 128 | fc1 128 | fc2 128
constexpr int LDQ = 388;                           // padded row stride of the staged q | k | v rows (floats)
constexpr int ATT_ROWS = 64;                       // longest sequence the attention kernel takes (T + 1 <= 64)
constexpr size_t att_smem(int slots) { return ((size_t)slots * LDQ + 2 * slots * NF + 2 * slots) * sizeof(float); }

enum { MODE_POS = 0, MODE_TEMPORAL = 1, MODE_SECOND = 2 };

__global__ void split_weights_kernel(const float* __restrict__ src, float* __restrict__ hi, float* __restrict__ lo, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = src[i];
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  const float h = __uint_as_float(r);
  hi[i] = h;
  lo[i] = v - h;
}

// mean / rstd (eps 1e-5, two-pass like LayerNorm) of one 128-float row held as one float4 per lane
__device__ __forceinline__ float2 row_stats(const float4 v) {
  float s = v.x + v.y + v.z + v.w;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.f / D);
  const float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
  float q = dx * dx + dy * dy + dz * dz + dw * dw;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  return make_float2(mean, rsqrtf(q * (1.f / D) + 1e-5f));
}

// Stage input rows -> x (and their LayerNorm statistics).  One warp per row.
//   POS: x[(seq 14 + s)] = s == 0 ? X[seq] : table_emb[b][s - 1]      TEMPORAL: x aliases X (statistics only)
//   SECOND: x[b (T + 1) + s] = s == 0 ? cls : second_in[b T + s - 1]
template <int MODE>
__global__ void __launch_bounds__(256) assemble_kernel(const float* __restrict__ X, const float* __restrict__ table_emb, const float* __restrict__ cls,
                                                       float* __restrict__ x, float* __restrict__ stats, long long rows, int T) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* src;
  if (MODE == MODE_POS) {
    const long long seq = r / (NTAB + 1);
    const int s = (int)(r - seq * (NTAB + 1));
    src = s == 0 ? X + seq * D : table_emb + ((seq / T) * NTAB + (s - 1)) * D;
  } else if (MODE == MODE_TEMPORAL) {
    src = X + r * D;
  } else {
    const long long b = r / (T + 1);
    const int s = (int)(r - b * (T + 1));
    src = s == 0 ? cls : X + (b * T + (s - 1)) * D;
  }
  const float4 v = __ldg(reinterpret_cast<const float4*>(src) + lane);
  if (MODE != MODE_TEMPORAL) *(reinterpret_cast<float4*>(x + r * D) + lane) = v;
  const float2 st = row_stats(v);
  if (lane == 0) *reinterpret_cast<float2*>(stats + 2 * r) = st;
}

// rows r * stride of x -> out[r]  (the ball tokens of the table-token stage, the cls tokens of the second stage)
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, int stride) {
  const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= n) return;
  const int lane = threadIdx.x & 31;
  *(reinterpret_cast<float4*>(out + r * D) + lane) = __ldg(reinterpret_cast<const float4*>(x + r * stride * D) + lane);
}

// fp32 attention of whole sequences.  A CTA stages the q | k | v rows of G sequences (bias already added by the GEMM) in shared memory
// and rotates q and k there (RoPE with time-derived angles, pairs (2f, 2f+1); the cls / ball token is not rotated).  Then ONE THREAD
// per (row, head): its q in registers, one independent accumulator per key for the scores and one per head dimension for P V, keys and
// values read as float4 broadcasts (the threads of a warp share the head and sit in at most three sequences), masked safe softmax in
// registers.  (The first version, one warp per (row, head) with lanes over keys like uplift.cu's fused stack, was a chain of dependent
// FMAs and shuffles with 14 of 32 lanes busy: 4.9 ms per table-token layer against 1 ms of HBM time.)
// SMAX: compile-time bound of the sequence length (score registers); G: sequences per CTA; SLOTS: thread slots per head (>= G S rows).
// FIRST_ONLY: only token 0 of every sequence is a query and o has one row per SEQUENCE (last table-token layer: only the ball token is
// used afterwards, model.py:375-378).  mask_additive: `mask` holds the additive values themselves ({-1e9, 0}, model.py:543-544) instead of
// {0, 1}.
template <int MODE, int SMAX, int G, int SLOTS, bool FIRST_ONLY = false>
__global__ void __launch_bounds__(4 * SLOTS, SLOTS == 32 ? 4 : 2) attention3_kernel(const float* __restrict__ qkv, float* __restrict__ o, const float* __restrict__ table,
                                                                     const float* __restrict__ mask, const float* __restrict__ times,
                                                                     const float* __restrict__ invf, int batch, int T, int mask_additive) {
  extern __shared__ __align__(16) float smem[];
  float* sQ = smem;                        // [rows][LDQ]: q (0..127) | k (128..255) | v (256..383)
  float* sCos = sQ + SLOTS * LDQ;          // [rows][NF]
  float* sSin = sCos + SLOTS * NF;
  float* sMask = sSin + SLOTS * NF;        // additive key / query mask per row (0 / -inf, or the caller's additive values)
  float* sTime = sMask + SLOTS;
  constexpr int ATT_THREADS = 4 * SLOTS;
  const int tid = threadIdx.x;
  const int S = MODE == MODE_POS ? NTAB + 1 : (MODE == MODE_TEMPORAL ? T : T + 1);
  const long long n_seq = MODE == MODE_POS ? (long long)batch * T : batch;
  const long long seq0 = (long long)blockIdx.x * G;
  const int g_here = (int)min((long long)G, n_seq - seq0);
  const int M = g_here * S;
  const long long row0 = seq0 * S;
  const float NEG_INF = -INFINITY;
  const float NO_ROPE = __int_as_float(0x7fc00000);
  for (int i = tid; i < M * (3 * D / 4); i += ATT_THREADS) {
    const int r = i / (3 * D / 4), c4 = i % (3 * D / 4);
    *reinterpret_cast<float4*>(sQ + r * LDQ + c4 * 4) = __ldg(reinterpret_cast<const float4*>(qkv + (row0 + r) * 3 * D) + c4);
  }
  for (int r = tid; r < M; r += ATT_THREADS) {
    float m = 0.f, t = NO_ROPE;
    const int g = r / S, s = r - g * S;
    const long long seq = seq0 + g;
    if (MODE == MODE_POS) {
      if (s > 0) {
        const long long b = seq / T;
        m = table[(b * NTAB + (s - 1)) * 3 + 2] == 1.f ? 0.f : NEG_INF;        // model.py:363
        t = (float)(s - 1) / 100.f;                                               // model.py:367
      }
    } else if (MODE == MODE_TEMPORAL || s > 0) {
      const float mv = mask[seq * T + s - (MODE == MODE_SECOND)];
      m = mask_additive ? mv : (mv == 0.f ? NEG_INF : 0.f);                      // model.py:541-546
      t = times[seq * T + s - (MODE == MODE_SECOND)];
    }
    sMask[r] = m;
    sTime[r] = t;
  }
  __syncthreads();
  for (int i = tid; i < M * NF; i += ATT_THREADS) {
    const int r = i / NF, f = i % NF;
    const float t = sTime[r];
    float c = 1.f, s = 0.f;
    if (t == t) {
      const float pos = rintf(__fdiv_rn(t, 0.002f));                              // model.py:72: round(t / (1 / 500))
      sincosf(__fmul_rn(pos, __ldg(invf + f)), &s, &c);
    }
    sCos[i] = c;
    sSin[i] = s;
  }
  __syncthreads();
  for (int i = tid; i < M * 2 * HEADS * NF; i += ATT_THREADS) {
    const int f = i % NF, hh = (i / NF) % (2 * HEADS), r = i / (NF * 2 * HEADS);
    float* q = sQ + r * LDQ + hh * HD + 2 * f;          // hh 0..3: q heads, 4..7: k heads (contiguous columns)
    const float c = sCos[r * NF + f], s = sSin[r * NF + f];
    const float a = q[0], b = q[1];
    q[0] = a * c - b * s;
    q[1] = a * s + b * c;
  }
  __syncthreads();
  const float scale = 0.17677669529663687f;             // 1 / sqrt(32), SDPA default
  const int hh = tid / SLOTS, r = tid % SLOTS;          // SLOTS thread slots per head; a warp works on one head
  if (r >= M) return;
  if (FIRST_ONLY && r % S != 0) return;
  const int k0 = (r / S) * S;
  float q[HD];
#pragma unroll
  for (int d = 0; d < HD; d += 4) {
    const float4 t4 = *reinterpret_cast<const float4*>(sQ + r * LDQ + hh * HD + d);
    q[d] = t4.x, q[d + 1] = t4.y, q[d + 2] = t4.z, q[d + 3] = t4.w;
  }
  const float mq = sMask[r];
  float sc[SMAX];
  float mx = NEG_INF;
#pragma unroll
  for (int j = 0; j < SMAX; ++j) {
    sc[j] = NEG_INF;
    if (j < S) {
      const float* kk = sQ + (k0 + j) * LDQ + D + hh * HD;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
      for (int d = 0; d < HD; d += 4) {
        const float4 ka = *reinterpret_cast<const float4*>(kk + d);
        a0 = fmaf(q[d], ka.x, a0);
        a1 = fmaf(q[d + 1], ka.y, a1);
        a2 = fmaf(q[d + 2], ka.z, a2);
        a3 = fmaf(q[d + 3], ka.w, a3);
      }
      sc[j] = ((a0 + a1) + (a2 + a3)) * scale + (sMask[k0 + j] + mq);
      mx = fmaxf(mx, sc[j]);
    }
  }
  float sum = 0.f;
  if (mx != NEG_INF) {                                  // fully masked row -> all-zero probabilities (safe softmax)
#pragma unroll
    for (int j = 0; j < SMAX; ++j) {
      sc[j] = sc[j] == NEG_INF ? 0.f : expf(sc[j] - mx);
      sum += sc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < SMAX; ++j) sc[j] = 0.f;
  }
  const float inv = sum > 0.f ? 1.f / sum : 0.f;
  float acc[HD];
#pragma unroll
  for (int d = 0; d < HD; ++d) acc[d] = 0.f;
#pragma unroll
  for (int j = 0; j < SMAX; ++j) {
    if (j < S) {
      const float pj = sc[j] * inv;
      const float* vv = sQ + (k0 + j) * LDQ + 2 * D + hh * HD;
#pragma unroll
      for (int d = 0; d < HD; d += 4) {
        const float4 va = *reinterpret_cast<const float4*>(vv + d);
        acc[d] = fmaf(pj, va.x, acc[d]);
        acc[d + 1] = fmaf(pj, va.y, acc[d + 1]);
        acc[d + 2] = fmaf(pj, va.z, acc[d + 2]);
        acc[d + 3] = fmaf(pj, va.w, acc[d + 3]);
      }
    }
  }
  float4* op = reinterpret_cast<float4*>(o + (FIRST_ONLY ? seq0 + r / S : row0 + r) * D + hh * HD);      // 128 contiguous bytes per thread
#pragma unroll
  for (int d = 0; d < HD; d += 4) op[d / 4] = make_float4(acc[d], acc[d + 1], acc[d + 2], acc[d + 3]);
}

// The attention instantiation of a stage: SMAX (score registers) is the smallest bound that holds S keys, the table-token stage packs two
// sequences per CTA.  The stage and ttk_uplift_debug_attention3 both launch through here, so a test exercises the dispatch the model uses.
int launch_attention3(int mode, bool first_only, const float* qkv, float* o, const float* table, const float* mask, const float* times,
                      const float* invf, int batch, int T, int mask_additive, cudaStream_t st) {
  static TtkPerDevice attr;
  if (attr.first()) {
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_POS, NTAB + 1, 2, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(32)));
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_POS, NTAB + 1, 2, 32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(32)));
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_TEMPORAL, 52, 1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(64)));
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_TEMPORAL, 64, 1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(64)));
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_SECOND, 52, 1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(64)));
    TTK_CUDA(cudaFuncSetAttribute(attention3_kernel<MODE_SECOND, 64, 1, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem(64)));
  }
  const int S = mode == MODE_POS ? NTAB + 1 : (mode == MODE_TEMPORAL ? T : T + 1);
  const long long n_seq = mode == MODE_POS ? (long long)batch * T : batch;
  if (mode == MODE_POS && first_only)
    attention3_kernel<MODE_POS, NTAB + 1, 2, 32, true><<<ttk_cdiv(n_seq, 2), 128, att_smem(32), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  else if (mode == MODE_POS)
    attention3_kernel<MODE_POS, NTAB + 1, 2, 32><<<ttk_cdiv(n_seq, 2), 128, att_smem(32), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  else if (mode == MODE_TEMPORAL && S <= 52)
    attention3_kernel<MODE_TEMPORAL, 52, 1, 64><<<(int)n_seq, 256, att_smem(64), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  else if (mode == MODE_TEMPORAL)
    attention3_kernel<MODE_TEMPORAL, 64, 1, 64><<<(int)n_seq, 256, att_smem(64), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  else if (S <= 52)
    attention3_kernel<MODE_SECOND, 52, 1, 64><<<(int)n_seq, 256, att_smem(64), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  else
    attention3_kernel<MODE_SECOND, 64, 1, 64><<<(int)n_seq, 256, att_smem(64), st>>>(qkv, o, table, mask, times, invf, batch, T, mask_additive);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

const char* kLayerPrefix[3] = {"firststage.pos_layers.%d.", "firststage.layers.%d.", "secondstage.%d."};

std::string lname(int stage, int i, const char* suffix) {
  char b[128];
  snprintf(b, sizeof(b), kLayerPrefix[stage], i);
  return std::string(b) + suffix;
}

// stats [rows][2] rounded up to whole 256-byte blocks: qkv and o / a behind it are C operands of ttk_gemm3, whose 256-bit stores need
// 32-byte aligned rows (with an odd batch T the unpadded qkv started 16 bytes off)
size_t stats_floats(size_t rows) { return (rows * 2 + 63) & ~(size_t)63; }

}  // namespace

// hi / lo halves of every layer's weight rows: [layers][qkv 384 | proj 128 | fc1 128 | fc2 128][128] fp32, layers in the order
// 4 table-token, depth - 4 temporal, 4 second-stage
int ttk_uplift3_prepare(ttk_uplift* h) {
  const int n_layers = h->depth + 4;
  const size_t elems = (size_t)n_layers * LAYER_ROWS * D;
  if (!h->w3_hi) TTK_CUDA(cudaMalloc((void**)&h->w3_hi, elems * sizeof(float)));
  if (!h->w3_lo) TTK_CUDA(cudaMalloc((void**)&h->w3_lo, elems * sizeof(float)));
  const char* names[4] = {"attn.qkv.weight", "attn.proj.weight", "mlp1.fc1.weight", "mlp1.fc2.weight"};
  const int rows[4] = {384, 128, 128, 128};
  int l = 0;
  for (int stage = 0; stage < 3; ++stage) {
    const int n = stage == 1 ? h->depth - 4 : 4;
    for (int i = 0; i < n; ++i, ++l) {
      size_t off = (size_t)l * LAYER_ROWS * D;
      for (int m = 0; m < 4; ++m) {
        const int cnt = rows[m] * D;
        split_weights_kernel<<<ttk_cdiv(cnt, 256), 256>>>(h->dev(lname(stage, i, names[m])), h->w3_hi + off, h->w3_lo + off, cnt);
        TTK_LAUNCH_CHECK();
        off += cnt;
      }
    }
  }
  TTK_CUDA(cudaDeviceSynchronize());
  h->w3_ready = true;
  return TTK_OK;
}

// x [rows][128] + stats + qkv [rows][384] + o / a [rows][128] for the largest stage (table tokens: batch T 14 rows)
size_t ttk_uplift3_workspace_bytes(const ttk_uplift* h, int batch, int T) {
  (void)h;
  const size_t rows = (size_t)batch * T * (NTAB + 1);
  return (rows * (D + 3 * D + D) + stats_floats(rows)) * sizeof(float) + 4096;
}

// One stage.  POS: io.X (ball embeddings [batch T][128]) and io.table_emb -> io.X (ball tokens after the table-token layers);
// TEMPORAL: io.X in place; SECOND: cls + (io.X or io.second_emb) -> io.table_emb[0 .. batch) (the cls rows, input of the rotation head).
int ttk_uplift3_stage(ttk_uplift* h, int mode, const UpliftIO& io, void* ws, cudaStream_t st) {
  const int T = io.T, batch = io.batch;
  const long long ntok = (long long)batch * T;
  const int S = mode == MODE_POS ? NTAB + 1 : (mode == MODE_TEMPORAL ? T : T + 1);
  const long long n_seq = mode == MODE_POS ? ntok : batch;
  const long long rows = n_seq * S;
  TTK_CHECK_ARG(rows < 2147483647LL && S <= ATT_ROWS, "uplift (tf32x3): batch too large for one call (%lld rows)", rows);
  float* wsf = (float*)ws;
  float* x = mode == MODE_TEMPORAL ? io.X : wsf;                     // the temporal stage updates X in place
  float* stats = wsf + (size_t)batch * T * (NTAB + 1) * D;
  float* qkv = stats + stats_floats((size_t)batch * T * (NTAB + 1));
  float* oa = qkv + (size_t)batch * T * (NTAB + 1) * 3 * D;
  const float* second_in = h->skip ? io.X : io.second_emb;
  const int blocks = ttk_cdiv(rows, 8);
  if (mode == MODE_POS)
    assemble_kernel<MODE_POS><<<blocks, 256, 0, st>>>(io.X, io.table_emb, nullptr, x, stats, rows, T);
  else if (mode == MODE_TEMPORAL)
    assemble_kernel<MODE_TEMPORAL><<<blocks, 256, 0, st>>>(io.X, nullptr, nullptr, x, stats, rows, T);
  else
    assemble_kernel<MODE_SECOND><<<blocks, 256, 0, st>>>(second_in, nullptr, h->dev("cls_token"), x, stats, rows, T);
  TTK_LAUNCH_CHECK();
  h->launches++;
  const int first = mode == MODE_POS ? 0 : (mode == MODE_TEMPORAL ? 4 : h->depth);
  const int n_layers = mode == MODE_TEMPORAL ? h->depth - 4 : 4;
  for (int i = 0; i < n_layers; ++i) {
    const size_t woff = (size_t)(first + i) * LAYER_ROWS * D;
    const float *whi = h->w3_hi + woff, *wlo = h->w3_lo + woff;
    Gemm3Args g;
    // qkv = LN1(x) Wqkv^T + b
    g = Gemm3Args{x, whi, wlo, h->dev(lname(mode, i, "attn.qkv.bias")), nullptr, qkv, (int)rows, 3 * D, 0, stats,
                  h->dev(lname(mode, i, "norm1.weight")), h->dev(lname(mode, i, "norm1.bias")), nullptr};
    int rc = ttk_gemm3(g, st);
    if (rc) return rc;
    const float* invf = h->dev(lname(mode, i, "attn.rotary_emb.inv_freq"));
    // Last table-token layer: only the ball token (row 0 of every sequence) is used afterwards, so its attention has one query per
    // sequence and projection + MLP run on those rows alone (1/14 of the rows), straight on io.X.
    const bool ball_only = mode == MODE_POS && i + 1 == n_layers;
    if (ball_only) {
      rc = launch_attention3(mode, true, qkv, oa, io.table, io.mask, io.times, invf, batch, T, io.mask_additive, st);
      if (rc) return rc;
      gather_rows_kernel<<<ttk_cdiv(ntok, 8), 256, 0, st>>>(x, io.X, ntok, NTAB + 1);
      TTK_LAUNCH_CHECK();
      float* bstats = qkv;                              // q | k | v are dead once the attention has run
      float* ba = oa + (size_t)ntok * D;
      g = Gemm3Args{oa, whi + 384 * D, wlo + 384 * D, nullptr, io.X, io.X, (int)ntok, D, 0, nullptr, nullptr, nullptr, bstats};
      rc = ttk_gemm3(g, st);
      if (rc) return rc;
      g = Gemm3Args{io.X, whi + 512 * D, wlo + 512 * D, h->dev(lname(mode, i, "mlp1.fc1.bias")), nullptr, ba, (int)ntok, D, 1, bstats,
                    h->dev(lname(mode, i, "norm2.weight")), h->dev(lname(mode, i, "norm2.bias")), nullptr};
      rc = ttk_gemm3(g, st);
      if (rc) return rc;
      g = Gemm3Args{ba, whi + 640 * D, wlo + 640 * D, h->dev(lname(mode, i, "mlp1.fc2.bias")), io.X, io.X, (int)ntok, D, 0, nullptr, nullptr, nullptr, nullptr};
      rc = ttk_gemm3(g, st);
      if (rc) return rc;
      h->launches += 6;
      return TTK_OK;
    }
    rc = launch_attention3(mode, false, qkv, oa, io.table, io.mask, io.times, invf, batch, T, io.mask_additive, st);
    if (rc) return rc;
    // x += o Wproj^T (no bias: model.py:268 passes attn_drop_rate into the proj_bias slot); statistics for LN2
    g = Gemm3Args{oa, whi + 384 * D, wlo + 384 * D, nullptr, x, x, (int)rows, D, 0, nullptr, nullptr, nullptr, stats};
    rc = ttk_gemm3(g, st);
    if (rc) return rc;
    // a = ReLU(LN2(x) W1^T + b1)
    g = Gemm3Args{x, whi + 512 * D, wlo + 512 * D, h->dev(lname(mode, i, "mlp1.fc1.bias")), nullptr, oa, (int)rows, D, 1, stats,
                  h->dev(lname(mode, i, "norm2.weight")), h->dev(lname(mode, i, "norm2.bias")), nullptr};
    rc = ttk_gemm3(g, st);
    if (rc) return rc;
    // x += a W2^T + b2; statistics for the next layer's LN1
    g = Gemm3Args{oa, whi + 640 * D, wlo + 640 * D, h->dev(lname(mode, i, "mlp1.fc2.bias")), x, x, (int)rows, D, 0, nullptr, nullptr, nullptr, stats};
    rc = ttk_gemm3(g, st);
    if (rc) return rc;
    h->launches += 5;
  }
  if (mode == MODE_POS) {
    gather_rows_kernel<<<ttk_cdiv(ntok, 8), 256, 0, st>>>(x, io.X, ntok, NTAB + 1);
    TTK_LAUNCH_CHECK();
    h->launches++;
  } else if (mode == MODE_SECOND) {
    gather_rows_kernel<<<ttk_cdiv(batch, 8), 256, 0, st>>>(x, io.table_emb, batch, T + 1);
    TTK_LAUNCH_CHECK();
    h->launches++;
  }
  return TTK_OK;
}

extern "C" int ttk_uplift_debug_attention3(int mode, int first_only, const float* qkv_dev, float* o_dev, const float* table_dev,
                                           const float* mask_dev, const float* times_dev, const float* inv_freq_dev, int batch, int seq_len,
                                           int mask_additive, void* stream) {
  TTK_CHECK_ARG(mode >= MODE_POS && mode <= MODE_SECOND && (!first_only || mode == MODE_POS), "ttk_uplift_debug_attention3: bad mode %d / first_only %d",
                mode, first_only);
  TTK_CHECK_ARG(batch > 0 && seq_len >= 2 && seq_len + 1 <= ATT_ROWS, "ttk_uplift_debug_attention3: seq_len must be in [2, %d] (got %d)",
                ATT_ROWS - 1, seq_len);
  TTK_CHECK_ARG(qkv_dev && o_dev && table_dev && mask_dev && times_dev && inv_freq_dev, "ttk_uplift_debug_attention3: null pointer");
  return launch_attention3(mode, first_only != 0, qkv_dev, o_dev, table_dev, mask_dev, times_dev, inv_freq_dev, batch, seq_len, mask_additive,
                           (cudaStream_t)stream);
}
