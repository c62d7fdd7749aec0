// HRNet-W18-small (WASB ball detector / HRNet table detector) executor.
// Reference: balldetection/models/wasb.py:445-486 (HRNet.forward), :35-105 (blocks), :108-245
// (HighResolutionModule), :383-416 (transitions), :596-608 (WASBNet.forward);
// tabledetection/models/hrnet.py:510-590.
//
// The network is a static plan (ops over NHWC tensors) built once per handle.  Eval-mode batch
// norm is folded into the conv weights by the host; ReLU, the residual add of a block and the
// multi-resolution fuse sums (nearest up-sampling = index shift) run in the conv epilogues.
// The arithmetic paths share the plan:
//   TTK_F32    - fp32 SIMT direct convolution (parity with the CPU reference),
//   TTK_TF32   - fp32 storage, tcgen05 implicit GEMM with TF32 operands (conv_umma.cu),
//   TTK_TF32X3 - fp32 storage, tcgen05 implicit GEMM with three TF32 products of split operands per product (fp32-level results),
//   TTK_BF16   - bf16 storage, fp32 accumulate, tcgen05 implicit GEMM,
//   TTK_F16    - the same with IEEE fp16 storage and operands (umma_prims.h: Fmt16 holds what differs between the two 16-bit formats).
#include <algorithm>
#include <map>
#include <type_traits>

#include "hrnet.h"
#include "umma_prims.h"

namespace {

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
const int kBranchCh[4] = {16, 32, 64, 128};

int pad16(int c) { return (c + 15) / 16 * 16; }

struct Builder {
  ttk_hrnet* h;
  std::map<std::string, int> by_name;

  void add_conv(const std::string& name, const std::string& bn, int cin, int cout, int k, int stride) {
    TtkConv c;
    c.name = "model." + name;
    c.bn = bn.empty() ? "" : "model." + bn;
    c.cin = cin;
    c.cout = cout;
    c.k = k;
    c.stride = stride;
    c.cin_p = pad16(cin);
    c.cout_p = pad16(cout);
    by_name[name] = (int)h->convs.size();
    h->convs.push_back(c);
  }

  int tensor(int c, int shift) {
    TtkTensor t;
    t.c = c;
    t.shift = shift;
    t.first = -1;
    t.last = -1;
    t.offset = 0;
    h->tensors.push_back(t);
    return (int)h->tensors.size() - 1;
  }

  // conv op: out = act(conv(in) + bias + sum(res))
  int conv(const std::string& name, int in, bool relu, std::vector<int> res = {}) {
    const int ci = by_name.at(name);
    const TtkConv& c = h->convs[ci];
    const TtkTensor& ti = h->tensors[in];
    const int out = tensor(c.cout_p, ti.shift + (c.stride == 2 ? 1 : 0));
    TtkOp op;
    op.type = OP_CONV;
    op.conv = ci;
    op.in = in;
    op.out = out;
    op.relu = relu;
    op.nres = (int)res.size();
    for (int i = 0; i < op.nres; ++i) op.res[i] = res[i];
    h->ops.push_back(op);
    return out;
  }

  int sum(int in, std::vector<int> res, bool relu) {
    const TtkTensor ti = h->tensors[in];
    const int out = tensor(ti.c, ti.shift);
    TtkOp op;
    op.type = OP_SUM;
    op.in = in;
    op.out = out;
    op.relu = relu;
    op.nres = (int)res.size();
    for (int i = 0; i < op.nres; ++i) op.res[i] = res[i];
    h->ops.push_back(op);
    return out;
  }
};

std::string fmt(const char* f, int a = 0, int b = 0, int c = 0) {
  char buf[128];
  snprintf(buf, sizeof(buf), f, a, b, c);
  return buf;
}

// Conv list in the order of oracle/hrnet.py:conv_specs (checked name by name in tests/test_abi.py).
void build_convs(Builder& B, int in_ch, int out_ch) {
  B.add_conv("conv1", "bn1", in_ch, 64, 3, 1);
  B.add_conv("conv2", "bn2", 64, 64, 3, 1);
  B.add_conv("layer1.0.conv1", "layer1.0.bn1", 64, 32, 1, 1);
  B.add_conv("layer1.0.conv2", "layer1.0.bn2", 32, 32, 3, 1);
  B.add_conv("layer1.0.conv3", "layer1.0.bn3", 32, 128, 1, 1);
  B.add_conv("layer1.0.downsample.0", "layer1.0.downsample.1", 64, 128, 1, 1);
  std::vector<int> pre = {128};
  for (int stage = 2; stage <= 4; ++stage) {
    const int nb = stage;
    for (int i = 0; i < nb; ++i) {
      if (i < (int)pre.size()) {
        if (kBranchCh[i] != pre[i])
          B.add_conv(fmt("transition%d.%d.0", stage - 1, i), fmt("transition%d.%d.1", stage - 1, i), pre[i], kBranchCh[i], 3, 1);
      } else {
        B.add_conv(fmt("transition%d.%d.0.0", stage - 1, i), fmt("transition%d.%d.0.1", stage - 1, i), pre.back(), kBranchCh[i], 3, 2);
      }
    }
    for (int b = 0; b < nb; ++b)
      for (int blk = 0; blk < 2; ++blk) {
        const std::string p = fmt("stage%d.0.branches.%d.%d", stage, b, blk);
        B.add_conv(p + ".conv1", p + ".bn1", kBranchCh[b], kBranchCh[b], 3, 1);
        B.add_conv(p + ".conv2", p + ".bn2", kBranchCh[b], kBranchCh[b], 3, 1);
      }
    for (int i = 0; i < nb; ++i)
      for (int j = 0; j < nb; ++j) {
        const std::string p = fmt("stage%d.0.fuse_layers.%d.%d", stage, i, j);
        if (j > i) {
          B.add_conv(p + ".0", p + ".1", kBranchCh[j], kBranchCh[i], 1, 1);
        } else if (j < i) {
          for (int k = 0; k < i - j; ++k) {
            const int cout = (k == i - j - 1) ? kBranchCh[i] : kBranchCh[j];
            B.add_conv(p + fmt(".%d.0", k), p + fmt(".%d.1", k), kBranchCh[j], cout, 3, 2);
          }
        }
      }
    pre.assign(kBranchCh, kBranchCh + nb);
  }
  B.add_conv("final_layers.0", "", 16, out_ch, 1, 1);
}

void build_ops(Builder& B) {
  ttk_hrnet* h = B.h;
  h->input_tensor = B.tensor(16, 0);
  int x = B.conv("conv1", h->input_tensor, true);
  x = B.conv("conv2", x, true);
  // Bottleneck (wasb.py:86-105): projection shortcut first so conv3's epilogue can add it
  int a = B.conv("layer1.0.conv1", x, true);
  a = B.conv("layer1.0.conv2", a, true);
  const int sc = B.conv("layer1.0.downsample.0", x, false);
  x = B.conv("layer1.0.conv3", a, true, {sc});
  std::vector<int> ys = {x};
  std::vector<int> pre = {128};
  for (int stage = 2; stage <= 4; ++stage) {
    const int nb = stage;
    std::vector<int> xs;
    for (int i = 0; i < nb; ++i) {
      if (i < (int)pre.size()) {
        if (kBranchCh[i] != pre[i])
          xs.push_back(B.conv(fmt("transition%d.%d.0", stage - 1, i), ys[i], true));
        else
          xs.push_back(ys[i]);
      } else {
        xs.push_back(B.conv(fmt("transition%d.%d.0.0", stage - 1, i), ys.back(), true));
      }
    }
    // branches: two BasicBlocks each (wasb.py:48-64); low resolutions first so that their
    // tensors are ready when the full-resolution fuse needs them
    for (int b = nb - 1; b >= 0; --b)
      for (int blk = 0; blk < 2; ++blk) {
        const std::string p = fmt("stage%d.0.branches.%d.%d", stage, b, blk);
        const int t = B.conv(p + ".conv1", xs[b], true);
        xs[b] = B.conv(p + ".conv2", t, true, {xs[b]});
      }
    // fuse (wasb.py:231-243): y_i = relu(sum_j f_ij(x_j))
    std::vector<int> out(nb);
    for (int i = 0; i < nb; ++i) {
      std::vector<int> others;
      for (int j = 0; j < nb; ++j) {
        const std::string p = fmt("stage%d.0.fuse_layers.%d.%d", stage, i, j);
        if (j == i) {
          if (i == 0) continue;           // x_0 is the main input of the sum op below
          others.push_back(xs[j]);
        } else if (j > i) {
          others.push_back(B.conv(p + ".0", xs[j], false));   // 1x1 at low resolution; up-sampling = index shift
        } else if (j < i - 1) {
          int t = xs[j];
          for (int k = 0; k < i - j; ++k) t = B.conv(p + fmt(".%d.0", k), t, k != i - j - 1);
          others.push_back(t);
        }
      }
      if (i == 0) {
        out[0] = B.sum(xs[0], others, true);
      } else {
        // the single stride-2 conv from branch i-1 hosts the sum of all other terms in its epilogue
        const std::string p = fmt("stage%d.0.fuse_layers.%d.%d", stage, i, i - 1);
        out[i] = B.conv(p + ".0.0", xs[i - 1], true, others);
      }
    }
    ys = out;
    pre.assign(kBranchCh, kBranchCh + nb);
  }
  TtkOp fin;
  fin.type = OP_FINAL;
  fin.in = ys[0];
  fin.conv = B.by_name.at("final_layers.0");
  h->ops.push_back(fin);
  // Dead-code elimination: only branch 0 of the last stage feeds the final layer (out_scales = [0], wasb.py:479-485), so the other
  // fuse outputs of stage 4 -- thirteen convolutions, 12 GFLOP of the reference's 344 per stack but ~8 % of the trunk's time, the
  // reference computes them and drops them -- are never read.  An op is kept only if a kept op reads its output.
  {
    std::vector<char> live_t(h->tensors.size(), 0), keep(h->ops.size(), 0);
    live_t[fin.in] = 1;
    keep.back() = 1;
    for (int o = (int)h->ops.size() - 2; o >= 0; --o) {
      const TtkOp& op = h->ops[o];
      if (op.out < 0 || !live_t[op.out]) continue;
      keep[o] = 1;
      live_t[op.in] = 1;
      for (int i = 0; i < op.nres; ++i) live_t[op.res[i]] = 1;
    }
    std::vector<TtkOp> kept;
    for (size_t o = 0; o < h->ops.size(); ++o)
      if (keep[o]) kept.push_back(h->ops[o]);
    h->dead_ops = (int)(h->ops.size() - kept.size());
    h->ops.swap(kept);
  }
  for (int o = 0; o + 1 < (int)h->ops.size(); ++o) {
    const TtkOp& ds = h->ops[o];
    const TtkOp& c3 = h->ops[o + 1];
    if (ds.type == OP_CONV && c3.type == OP_CONV && ds.conv == B.by_name.at("layer1.0.downsample.0") &&
        c3.conv == B.by_name.at("layer1.0.conv3") && c3.nres == 1 && c3.res[0] == ds.out) {
      h->dual_ds_op = o;
      h->dual_c3_op = o + 1;
    }
  }
  // liveness
  for (int o = 0; o < (int)h->ops.size(); ++o) {
    const TtkOp& op = h->ops[o];
    auto touch = [&](int t) {
      if (t < 0) return;
      if (h->tensors[t].first < 0) h->tensors[t].first = o;
      h->tensors[t].last = o;
    };
    touch(op.in);
    for (int i = 0; i < op.nres; ++i) touch(op.res[i]);
    touch(op.out);
  }
}

// First-fit offset assignment over tensor lifetimes; returns the peak size in bytes.
size_t plan_memory(ttk_hrnet* h, int bs, int H, int W, size_t elem) {
  struct Block {
    size_t off, size;
    int last;
  };
  std::vector<Block> live;
  size_t peak = 0;
  for (int o = 0; o < (int)h->ops.size(); ++o) {
    live.erase(std::remove_if(live.begin(), live.end(), [&](const Block& b) { return b.last < o; }), live.end());
    const int t = h->ops[o].out;
    if (t < 0) continue;
    TtkTensor& tt = h->tensors[t];
    size_t size = (size_t)bs * (H >> tt.shift) * (W >> tt.shift) * tt.c * elem;
    size = (size + 1023) & ~(size_t)1023;
    std::sort(live.begin(), live.end(), [](const Block& a, const Block& b) { return a.off < b.off; });
    size_t off = 0;
    for (const Block& b : live) {
      if (off + size <= b.off) break;
      off = std::max(off, b.off + b.size);
    }
    tt.offset = off;
    live.push_back({off, size, tt.last});
    peak = std::max(peak, off + size);
  }
  return peak;
}

// ------------------------------------------------------------------------------------------
// fp32-accumulate SIMT direct convolution on NHWC tensors (T = float, bf16 or fp16 storage)
// ------------------------------------------------------------------------------------------
template <typename T>
struct Io;
template <>
struct Io<float> {
  static __device__ __forceinline__ void load4(const float* p, float* v) {
    const float4 q = *reinterpret_cast<const float4*>(p);
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  }
  static __device__ __forceinline__ void store4(float* p, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <>
struct Io<__nv_bfloat16> {
  static __device__ __forceinline__ void load4(const __nv_bfloat16* p, float* v) {
    const uint2 q = *reinterpret_cast<const uint2*>(p);
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&q.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&q.y);
    v[0] = __low2float(a); v[1] = __high2float(a); v[2] = __low2float(b); v[3] = __high2float(b);
  }
  static __device__ __forceinline__ void store4(__nv_bfloat16* p, const float* v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 q;
    q.x = *reinterpret_cast<uint32_t*>(&a);
    q.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = q;
  }
};

template <>
struct Io<__half> {
  static __device__ __forceinline__ void load4(const __half* p, float* v) {
    const uint2 q = *reinterpret_cast<const uint2*>(p);
    v[0] = umma::Fmt16<1>::lo(q.x); v[1] = umma::Fmt16<1>::hi(q.x); v[2] = umma::Fmt16<1>::lo(q.y); v[3] = umma::Fmt16<1>::hi(q.y);
  }
  static __device__ __forceinline__ void store4(__half* p, const float* v) {
    *reinterpret_cast<uint2*>(p) = make_uint2(umma::Fmt16<1>::pack(v[0], v[1]), umma::Fmt16<1>::pack(v[2], v[3]));
  }
};

constexpr int CK = 8;        // input channels staged per step
constexpr int COT = 16;      // output channels per thread
constexpr int TH = 16;       // output rows per block

template <int K, int S>
struct Tile {
  static constexpr int PIX = S == 1 ? 4 : 2;            // output pixels per thread, 8 columns apart
  static constexpr int TW = 8 * PIX;                    // output columns per block
  static constexpr int IH = (TH - 1) * S + K;           // staged input rows
  static constexpr int IW = (TW - 1) * S + K;           // staged input columns
  static constexpr int PLANE_RAW = IH * IW;
  static constexpr int PLANE = PLANE_RAW + ((34 - PLANE_RAW % 32) % 32);   // PLANE % 32 == 2: conflict-free transposed fill
};

template <typename T, int K, int S>
__global__ void __launch_bounds__(128) conv_simt_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                        const float* __restrict__ w, const float* __restrict__ bias,
                                                        const T* __restrict__ res0, const T* __restrict__ res1,
                                                        const T* __restrict__ res2, int rs0, int rs1, int rs2, int nres,
                                                        int hin, int win, int hout, int wout, int cin, int cout, int relu) {
  using TL = Tile<K, S>;
  constexpr int PAD = K / 2;
  __shared__ float s_in[CK * TL::PLANE];
  __shared__ __align__(16) float s_w[K * K * CK * COT];
  const int tid = threadIdx.x;
  const int lane8 = tid & 7, row = tid >> 3;
  const int cog = cout / COT;
  const int n = blockIdx.z / cog, co0 = (blockIdx.z % cog) * COT;
  const int oy0 = blockIdx.y * TH, ox0 = blockIdx.x * TL::TW;
  const int iy0 = oy0 * S - PAD, ix0 = ox0 * S - PAD;
  const T* in_n = in + (size_t)n * hin * win * cin;

  float acc[TL::PIX][COT];
#pragma unroll
  for (int p = 0; p < TL::PIX; ++p)
#pragma unroll
    for (int c = 0; c < COT; ++c) acc[p][c] = 0.f;

  for (int c0 = 0; c0 < cin; c0 += CK) {
    // stage the input tile transposed to [channel][row][col]; lane -> (channel group fastest, pixel)
    for (int e = tid; e < TL::PLANE_RAW * (CK / 4); e += 128) {
      const int g = e % (CK / 4), pix = e / (CK / 4);
      const int r = pix / TL::IW, c = pix - r * TL::IW;
      const int iy = iy0 + r, ix = ix0 + c;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (iy >= 0 && iy < hin && ix >= 0 && ix < win) Io<T>::load4(in_n + ((size_t)iy * win + ix) * cin + c0 + 4 * g, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) s_in[(4 * g + j) * TL::PLANE + pix] = v[j];
    }
    for (int e = tid; e < K * K * CK * COT / 4; e += 128) {
      const int q = e % (COT / 4), ck = (e / (COT / 4)) % CK, tap = e / (COT / 4 * CK);
      reinterpret_cast<float4*>(s_w)[e] =
          *reinterpret_cast<const float4*>(w + ((size_t)tap * cin + c0 + ck) * cout + co0 + 4 * q);
    }
    __syncthreads();
#pragma unroll 2
    for (int ck = 0; ck < CK; ++ck) {
#pragma unroll
      for (int ky = 0; ky < K; ++ky) {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
          float wv[COT];
#pragma unroll
          for (int q = 0; q < COT / 4; ++q) {
            const float4 t = reinterpret_cast<const float4*>(s_w)[((ky * K + kx) * CK + ck) * (COT / 4) + q];
            wv[4 * q] = t.x; wv[4 * q + 1] = t.y; wv[4 * q + 2] = t.z; wv[4 * q + 3] = t.w;
          }
#pragma unroll
          for (int p = 0; p < TL::PIX; ++p) {
            const float v = s_in[ck * TL::PLANE + (row * S + ky) * TL::IW + (lane8 + 8 * p) * S + kx];
#pragma unroll
            for (int c = 0; c < COT; ++c) acc[p][c] = fmaf(v, wv[c], acc[p][c]);
          }
        }
      }
    }
    __syncthreads();
  }

  const int oy = oy0 + row;
  if (oy >= hout) return;
  float b[COT];
#pragma unroll
  for (int c = 0; c < COT; ++c) b[c] = bias[co0 + c];
  const T* rp[3] = {res0, res1, res2};
  const int rsh[3] = {rs0, rs1, rs2};
#pragma unroll
  for (int p = 0; p < TL::PIX; ++p) {
    const int ox = ox0 + lane8 + 8 * p;
    if (ox >= wout) continue;
    float v[COT];
#pragma unroll
    for (int c = 0; c < COT; ++c) v[c] = acc[p][c] + b[c];
    for (int r = 0; r < nres; ++r) {
      const int sh = rsh[r];
      const T* q = rp[r] + (((size_t)n * (hout >> sh) + (oy >> sh)) * (wout >> sh) + (ox >> sh)) * cout + co0;
#pragma unroll
      for (int c4 = 0; c4 < COT / 4; ++c4) {
        float t[4];
        Io<T>::load4(q + 4 * c4, t);
#pragma unroll
        for (int j = 0; j < 4; ++j) v[4 * c4 + j] += t[j];
      }
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < COT; ++c) v[c] = fmaxf(v[c], 0.f);
    }
    T* o = out + (((size_t)n * hout + oy) * wout + ox) * cout + co0;
#pragma unroll
    for (int c4 = 0; c4 < COT / 4; ++c4) Io<T>::store4(o + 4 * c4, v + 4 * c4);
  }
}

// rounded_weights: the weights rounded to the 16-bit storage format T
template <typename T>
int launch_conv_simt(const TtkConv& cv, const ConvLaunch& a, bool rounded_weights, cudaStream_t st) {
  const float* w = !rounded_weights ? cv.w_f32 : std::is_same<T, __half>::value ? cv.w_hfr : cv.w_bfr;
  const int cog = a.cout / COT;
#define TTK_SIMT(K_, S_)                                                                                              \
  {                                                                                                                   \
    dim3 grid(ttk_cdiv(a.wout, Tile<K_, S_>::TW), ttk_cdiv(a.hout, TH), a.n* cog);                                    \
    conv_simt_kernel<T, K_, S_><<<grid, 128, 0, st>>>((const T*)a.in, (T*)a.out, w, cv.bias, (const T*)a.res[0],      \
                                                      (const T*)a.res[1], (const T*)a.res[2], a.res_shift[0],         \
                                                      a.res_shift[1], a.res_shift[2], a.nres, a.hin, a.win, a.hout,   \
                                                      a.wout, a.cin, a.cout, a.relu);                                 \
  }
  if (cv.k == 3 && cv.stride == 1) TTK_SIMT(3, 1)
  else if (cv.k == 3 && cv.stride == 2) TTK_SIMT(3, 2)
  else if (cv.k == 1 && cv.stride == 1) TTK_SIMT(1, 1)
  else {
    ttk_set_error("conv %s: unsupported k=%d stride=%d", cv.name.c_str(), cv.k, cv.stride);
    return TTK_ERR_UNSUPPORTED;
  }
#undef TTK_SIMT
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

// out = act(in + sum_r res_r[y >> s_r, x >> s_r])   (full-resolution fuse of a HighResolutionModule)
// 32 bytes per thread per access (16 bf16 / 8 fp32 channels, 256-bit loads and stores), two independent items in flight per thread.
// One grid row per image row and shifts for the channel-vector split (c / V is a power of two), so no thread divides: the first
// version decomposed a flat 64-bit index with three divisions per item and ran at half the HBM rate because of them.
__device__ __forceinline__ void sum_ld256(const void* p, uint32_t* w) {
  asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7])
               : "l"(p));
}
template <typename T>
__global__ void __launch_bounds__(256) sum_kernel(const T* __restrict__ in, T* __restrict__ out, const T* __restrict__ res0,
                                                  const T* __restrict__ res1, const T* __restrict__ res2, int rs0, int rs1,
                                                  int rs2, int nres, int h, int w, int c, int cv_shift, int relu) {
  constexpr int V = 32 / sizeof(T);                 // channels per 32-byte item
  const T* rp[3] = {res0, res1, res2};
  const int rsh[3] = {rs0, rs1, rs2};
  const int y = blockIdx.y, b = blockIdx.z;
  const int row_items = w << cv_shift;
  const size_t row0 = ((size_t)b * h + y) * (size_t)row_items;      // in 32-byte items
  const int e0 = blockIdx.x * 512 + threadIdx.x;
  float v[2][V];
  uint32_t raw[2][8];
  bool live[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int e = e0 + u * 256;
    live[u] = e < row_items;
    if (live[u]) sum_ld256(in + (row0 + e) * V, raw[u]);
  }
  using F16 = umma::Fmt16Of<T>;                     // 16-bit storage: bf16 or fp16
  auto widen = [](const uint32_t* q, float* f, bool add) {
    if (sizeof(T) == 2) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float lo = F16::lo(q[j]), hi = F16::hi(q[j]);
        f[2 * j % V] = add ? f[2 * j % V] + lo : lo;
        f[(2 * j + 1) % V] = add ? f[(2 * j + 1) % V] + hi : hi;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j % V] = add ? f[j % V] + __uint_as_float(q[j]) : __uint_as_float(q[j]);
    }
  };
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    if (!live[u]) continue;
    const int e = e0 + u * 256;
    widen(raw[u], v[u], false);
    const int x = e >> cv_shift, ci = e & ((1 << cv_shift) - 1);
    for (int r = 0; r < nres; ++r) {
      const int sh = rsh[r];
      uint32_t q[8];
      sum_ld256(rp[r] + (((size_t)b * (h >> sh) + (y >> sh)) * (w >> sh) + (x >> sh)) * c + ci * V, q);
      widen(q, v[u], true);
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < V; ++j) v[u][j] = fmaxf(v[u][j], 0.f);
    }
    uint32_t o[8];
    if (sizeof(T) == 2) {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = F16::pack(v[u][2 * j % V], v[u][(2 * j + 1) % V]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __float_as_uint(v[u][j % V]);
    }
    T* op = out + (row0 + e) * V;
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(op), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]),
                 "r"(o[6]), "r"(o[7])
                 : "memory");
  }
}

// final 1x1 conv 16 -> out_count channels, NHWC16 in, planar float32 out (wasb.py:332, :606-608)
template <typename T>
__global__ void __launch_bounds__(256) final_kernel(const T* __restrict__ in, float* __restrict__ out,
                                                    const float* __restrict__ w, const float* __restrict__ b, int n, int hw,
                                                    int out_count) {
  extern __shared__ float s_wb[];   // [out_count][16] + [out_count]
  for (int i = threadIdx.x; i < out_count * 17; i += blockDim.x) s_wb[i] = i < out_count * 16 ? w[i] : b[i - out_count * 16];
  __syncthreads();
  const long long total = (long long)n * hw;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (long long)gridDim.x * blockDim.x) {
    float v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) Io<T>::load4(in + p * 16 + 4 * q, v + 4 * q);
    const long long img = p / hw, pix = p - img * hw;
    for (int o = 0; o < out_count; ++o) {
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < 16; ++c) acc = fmaf(v[c], s_wb[o * 16 + c], acc);
      out[(img * out_count + o) * hw + pix] = acc + s_wb[out_count * 16 + o];
    }
  }
}

// Record an event before launch #recs.size() and describe the launch (algorithmic flops, compulsory bytes).
int profile_mark(ttk_hrnet* h, int oi, int bs, int H, int W, size_t elem, cudaStream_t st) {
  const size_t i = h->recs.size();
  while (h->events.size() <= i + 1) {
    cudaEvent_t e;
    TTK_CUDA(cudaEventCreate(&e));
    h->events.push_back(e);
  }
  TTK_CUDA(cudaEventRecord(h->events[i], st));
  const TtkOp& op = h->ops[oi];
  ttk_hrnet::Rec r;
  r.op = oi;
  r.n = bs;
  auto numel = [&](int t) { const TtkTensor& tt = h->tensors[t]; return (double)bs * (H >> tt.shift) * (W >> tt.shift) * tt.c; };
  if (op.type == OP_CONV) {
    const TtkConv& c = h->convs[op.conv];
    const TtkTensor& to = h->tensors[op.out];
    const double opix = (double)bs * (H >> to.shift) * (W >> to.shift);
    r.flops = 2.0 * opix * c.cin * c.cout * c.k * c.k;
    r.bytes = (numel(op.in) + numel(op.out)) * elem + (double)c.cin_p * c.cout_p * c.k * c.k * elem;
    for (int k = 0; k < op.nres; ++k) r.bytes += numel(op.res[k]) * elem;
    if (h->cur_esz && !h->cur_x3 && h->dual_ready && h->use_dual && oi == h->dual_c3_op) {
      // fused bottleneck tail: the projection shortcut's GEMM rides along and its output tensor never exists
      const TtkOp& ds = h->ops[h->dual_ds_op];
      const TtkConv& dc = h->convs[ds.conv];
      r.flops += 2.0 * opix * dc.cin * dc.cout;
      r.bytes += numel(ds.in) * elem + (double)dc.cin_p * dc.cout_p * elem - numel(op.res[0]) * elem;
    }
  } else if (op.type == OP_SUM) {
    r.flops = numel(op.out) * op.nres;
    r.bytes = (numel(op.in) + numel(op.out)) * elem;
    for (int k = 0; k < op.nres; ++k) r.bytes += numel(op.res[k]) * elem;
  } else {
    r.flops = 2.0 * bs * H * W * 16 * h->out_count;
    r.bytes = numel(op.in) * elem + (double)bs * H * W * h->out_count * 4;
  }
  h->recs.push_back(r);
  return TTK_OK;
}

// B operands of the fused bottleneck tail (conv3 and the projection shortcut K-concatenated), bf16, fp16 and TF32 images
int prepare_dual(ttk_hrnet* h) {
  if (h->dual_ds_op < 0) return TTK_OK;
  const TtkConv& ds = h->convs[h->ops[h->dual_ds_op].conv];
  const TtkConv& c3 = h->convs[h->ops[h->dual_c3_op].conv];
  if (ds.w_host.empty() || c3.w_host.empty()) return TTK_OK;
  std::vector<float> b(128);
  for (int co = 0; co < 128; ++co) b[co] = c3.b_host[co] + ds.b_host[co];
  for (int mode = 0; mode < 3; ++mode) {
    const int esz = mode == 1 ? 4 : 2;
    const bool f16 = mode == 2;
    std::vector<uint8_t> w;
    ttk_conv_umma_pack_dual(c3.w_host.data(), ds.w_host.data(), esz, w, f16);
    void** dst = f16 ? &h->w_dual_f16 : esz == 2 ? &h->w_dual : &h->w_dual32;
    if (!*dst) TTK_CUDA(cudaMalloc(dst, w.size()));
    TTK_CUDA(cudaMemcpy(*dst, w.data(), w.size(), cudaMemcpyHostToDevice));
  }
  if (!h->bias_dual) TTK_CUDA(cudaMalloc((void**)&h->bias_dual, 128 * sizeof(float)));
  TTK_CUDA(cudaMemcpy(h->bias_dual, b.data(), 128 * sizeof(float), cudaMemcpyHostToDevice));
  h->dual_ready = true;
  return TTK_OK;
}

// op oi is conv1 of a BasicBlock whose conv2 (op oi + 1) adds the block input: candidates for block_umma.cu
bool is_basic_block(const ttk_hrnet* h, size_t oi) {
  if (oi + 1 >= h->ops.size()) return false;
  const TtkOp &a = h->ops[oi], &b = h->ops[oi + 1];
  if (a.type != OP_CONV || b.type != OP_CONV || a.nres != 0 || !a.relu || !b.relu || b.in != a.out || b.nres != 1 || b.res[0] != a.in) return false;
  const TtkConv &c1 = h->convs[a.conv], &c2 = h->convs[b.conv];
  if (c1.k != 3 || c2.k != 3 || c1.stride != 1 || c2.stride != 1) return false;
  if (c1.cin_p != c1.cout_p || c2.cin_p != c1.cin_p || c2.cout_p != c1.cin_p) return false;
  if (c1.cin_p != 16 && c1.cin_p != 32) return false;
  if (h->tensors[a.out].last != (int)oi + 1) return false;          // the intermediate tensor has no other reader
  return true;
}

// esz: 0 = SIMT kernels on T storage, 2 = 16-bit tcgen05 path (bf16 or fp16, as T), 4 = TF32 tcgen05 path on fp32 storage (x3:
// 3xTF32; convolutions only -- the fused BasicBlock and bottleneck kernels have no x3 variant, so those convolutions run one by one)
template <typename T>
int run_plan(ttk_hrnet* h, const void* x, int bs, int H, int W, float* heat, char* ws, int esz, bool x3, cudaStream_t st) {
  const bool umma = esz != 0;
  constexpr bool f16 = std::is_same<T, __half>::value;
  h->cur_esz = esz;
  h->cur_x3 = x3;
  bool dual_skipped = false;
  for (size_t oi = 0; oi < h->ops.size(); ++oi) {
    const TtkOp& op = h->ops[oi];
    // TF32: the fused kernels exist (16 channels) and are parity-green, but the thin MMAs of a 16-channel convolution keep them at or
    // above the time of the two HBM-bound convolutions (DESIGN.md section 4.2), so they run only when asked for (use_block_fusion 2 / 3)
    if (umma && !x3 && is_basic_block(h, oi) && ((esz == 2 && h->use_block_fusion) || (esz == 4 && h->use_block_fusion >= 2 && h->convs[op.conv].cin_p == 16))) {
      const TtkOp& op2 = h->ops[oi + 1];
      const TtkTensor& ti = h->tensors[op.in];
      auto p2 = [&](int t) -> void* { return t == h->input_tensor ? const_cast<void*>(x) : (void*)(ws + h->tensors[t].offset); };
      if (h->profile) {
        int rc = profile_mark(h, (int)oi, bs, H, W, sizeof(T), st);
        if (rc) return rc;
        // one launch does both convolutions: x in, y out, the intermediate tensor and the residual read never touch HBM
        ttk_hrnet::Rec& r = h->recs.back();
        const TtkConv& c2 = h->convs[op2.conv];
        const double opix = (double)bs * (H >> ti.shift) * (W >> ti.shift);
        r.flops += 2.0 * opix * c2.cin * c2.cout * 9;
        r.bytes = 2.0 * opix * ti.c * sizeof(T) + 2.0 * 9 * ti.c * ti.c * sizeof(T);
      }
      // TF32: mode 2 = two 3-row tiles in flight (fp32 residual from global memory), mode 3 = one 4-row tile (residual from the staged tile)
      const int rc = ttk_block_umma_launch(h->convs[op.conv], h->convs[op2.conv], p2(op.in), p2(op2.out), bs, H >> ti.shift, W >> ti.shift, st,
                                           esz == 4 && h->use_block_fusion == 3 ? 5 : esz, f16);
      if (rc == TTK_OK) {
        h->launches++;
        ++oi;                                      // conv2 is done as well
        continue;
      }
      if (rc != TTK_ERR_UNSUPPORTED) return rc;
      if (h->profile) h->recs.pop_back();
    }
    // bottleneck fusion (tensor-core path): the projection shortcut is folded into conv3's GEMM
    if (umma && !x3 && h->dual_ready && h->use_dual && (int)oi == h->dual_ds_op) {
      dual_skipped = true;
      continue;
    }
    if (h->profile) {
      int rc = profile_mark(h, (int)oi, bs, H, W, sizeof(T), st);
      if (rc) return rc;
    }
    auto ptr = [&](int t) -> void* {
      if (t == h->input_tensor) return const_cast<void*>(x);
      return ws + h->tensors[t].offset;
    };
    if (op.type == OP_CONV) {
      const TtkConv& cv = h->convs[op.conv];
      const TtkTensor& ti = h->tensors[op.in];
      const TtkTensor& to = h->tensors[op.out];
      ConvLaunch a;
      a.in = ptr(op.in);
      a.out = ptr(op.out);
      a.nres = op.nres;
      for (int r = 0; r < 3; ++r) {
        a.res[r] = r < op.nres ? ptr(op.res[r]) : nullptr;
        a.res_shift[r] = r < op.nres ? h->tensors[op.res[r]].shift - to.shift : 0;
      }
      a.n = bs;
      a.hin = H >> ti.shift;
      a.win = W >> ti.shift;
      a.hout = H >> to.shift;
      a.wout = W >> to.shift;
      a.cin = cv.cin_p;
      a.cout = cv.cout_p;
      a.relu = op.relu ? 1 : 0;
      int rc = TTK_ERR_UNSUPPORTED;
      if (dual_skipped && (int)oi == h->dual_c3_op) {
        const TtkOp& ds = h->ops[h->dual_ds_op];
        ConvLaunch d = a;
        d.nres = 0;
        d.in2 = ptr(ds.in);
        d.cin2 = h->convs[ds.conv].cin_p;
        rc = ttk_conv_umma_launch_dual(esz == 2 ? (f16 ? h->w_dual_f16 : h->w_dual) : h->w_dual32, h->bias_dual, d, st, esz, f16);
        if (rc == TTK_ERR_UNSUPPORTED) {      // driver refused the maps: run the two convolutions separately from now on
          h->use_dual = 0;
          ConvLaunch s0;
          const TtkConv& dcv = h->convs[ds.conv];
          const TtkTensor& dti = h->tensors[ds.in];
          const TtkTensor& dto = h->tensors[ds.out];
          s0.in = ptr(ds.in);
          s0.out = ptr(ds.out);
          s0.nres = 0;
          for (int r = 0; r < 3; ++r) { s0.res[r] = nullptr; s0.res_shift[r] = 0; }
          s0.n = bs; s0.hin = H >> dti.shift; s0.win = W >> dti.shift; s0.hout = H >> dto.shift; s0.wout = W >> dto.shift;
          s0.cin = dcv.cin_p; s0.cout = dcv.cout_p; s0.relu = 0;
          rc = ttk_conv_umma_launch(dcv, s0, st, esz, false, f16);
          if (rc == TTK_ERR_UNSUPPORTED) rc = launch_conv_simt<T>(dcv, s0, sizeof(T) == 2, st);
          if (rc != TTK_OK) return rc;
          h->launches++;
          rc = ttk_conv_umma_launch(cv, a, st, esz, false, f16);
        }
      } else if (umma) {
        rc = ttk_conv_umma_launch(cv, a, st, esz, x3, f16);
      }
      if (rc == TTK_ERR_UNSUPPORTED) {
        // no tensor-core kernel for this shape: the SIMT kernel on the same storage (fp32-level on fp32 tensors)
        if (umma && h->profile) h->recs.back().simt_fallback = true;
        rc = launch_conv_simt<T>(cv, a, sizeof(T) == 2, st);
      }
      if (rc != TTK_OK) return rc;
      h->launches++;
    } else if (op.type == OP_SUM) {
      const TtkTensor& to = h->tensors[op.out];
      const int hh = H >> to.shift, ww = W >> to.shift;
      const int cv = to.c / (32 / (int)sizeof(T));          // 32-byte items per pixel
      int cv_shift = 0;
      while ((1 << cv_shift) < cv) ++cv_shift;
      if ((1 << cv_shift) != cv || bs > 65535 || hh > 65535) {
        ttk_set_error("fuse sum: %d channels / batch %d / height %d not supported", to.c, bs, hh);
        return TTK_ERR_UNSUPPORTED;
      }
      const dim3 blocks(ttk_cdiv(ww << cv_shift, 512), hh, bs);
      int sh[3] = {0, 0, 0};
      const void* rp[3] = {nullptr, nullptr, nullptr};
      for (int r = 0; r < op.nres; ++r) {
        rp[r] = ptr(op.res[r]);
        sh[r] = h->tensors[op.res[r]].shift - to.shift;
      }
      sum_kernel<T><<<blocks, 256, 0, st>>>((const T*)ptr(op.in), (T*)ptr(op.out), (const T*)rp[0], (const T*)rp[1],
                                           (const T*)rp[2], sh[0], sh[1], sh[2], op.nres, hh, ww, to.c, cv_shift, op.relu ? 1 : 0);
      TTK_LAUNCH_CHECK();
      h->launches++;
    } else {
      const long long total = (long long)bs * H * W;
      const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ttk_num_sms() * 16);
      final_kernel<T><<<blocks, 256, h->out_count * 17 * sizeof(float), st>>>((const T*)ptr(op.in), heat, h->final_w, h->final_b,
                                                                            bs, H * W, h->out_count);
      TTK_LAUNCH_CHECK();
      h->launches++;
    }
  }
  return TTK_OK;
}

}  // namespace
namespace {
int upload(float** dst, const std::vector<float>& src) {
  if (!*dst) TTK_CUDA(cudaMalloc((void**)dst, src.size() * sizeof(float)));
  TTK_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(float), cudaMemcpyHostToDevice));
  return TTK_OK;
}

float bf16_round(float v) { return __bfloat162float(umma::Fmt16<0>::round(v)); }
float f16_round(float v) { return __half2float(umma::Fmt16<1>::round(v)); }

}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" int ttk_hrnet_create(int in_ch, int out_ch, int out_first, int out_count, ttk_hrnet** out) {
  TTK_CHECK_ARG(out, "ttk_hrnet_create: null out");
  TTK_CHECK_ARG(in_ch >= 1 && in_ch <= 16, "ttk_hrnet_create: in_ch must be 1..16 (got %d)", in_ch);
  TTK_CHECK_ARG(out_ch >= 1 && out_ch <= 16, "ttk_hrnet_create: out_ch must be 1..16 (got %d)", out_ch);
  TTK_CHECK_ARG(out_first >= 0 && out_count >= 1 && out_first + out_count <= out_ch, "ttk_hrnet_create: bad output slice");
  ttk_hrnet* h = new ttk_hrnet();
  h->in_ch = in_ch;
  h->out_ch = out_ch;
  h->out_first = out_first;
  h->out_count = out_count;
  Builder B;
  B.h = h;
  build_convs(B, in_ch, out_ch);
  build_ops(B);
  const char* env = getenv("TTK_HRNET_SUBBATCH");
  if (env && atoi(env) > 0) h->subbatch = atoi(env);
  env = getenv("TTK_FORCE_SIMT");
  if (env && atoi(env) > 0) h->force_simt = 1;
  *out = h;
  return TTK_OK;
}

extern "C" void ttk_hrnet_destroy(ttk_hrnet* h) {
  if (!h) return;
  for (cudaEvent_t e : h->events) cudaEventDestroy(e);
  for (TtkConv& c : h->convs) {
    cudaFree(c.w_f32);
    cudaFree(c.w_bfr);
    cudaFree(c.w_hfr);
    cudaFree(c.bias);
    cudaFree(c.w_umma);
    cudaFree(c.w_umma_f16);
    cudaFree(c.w_umma32);
    cudaFree(c.w_x3);
  }
  cudaFree(h->w_dual);
  cudaFree(h->w_dual_f16);
  cudaFree(h->w_dual32);
  cudaFree(h->bias_dual);
  cudaFree(h->final_w);
  cudaFree(h->final_b);
  delete h;
}

extern "C" int ttk_hrnet_num_convs(const ttk_hrnet* h) { return h ? (int)h->convs.size() : 0; }

extern "C" int ttk_hrnet_conv_info(const ttk_hrnet* h, int i, char* name, char* bn, int* cin, int* cout, int* k, int* stride) {
  TTK_CHECK_ARG(h && i >= 0 && i < (int)h->convs.size(), "ttk_hrnet_conv_info: bad index %d", i);
  const TtkConv& c = h->convs[i];
  if (name) snprintf(name, 128, "%s", c.name.c_str());
  if (bn) snprintf(bn, 128, "%s", c.bn.c_str());
  if (cin) *cin = c.cin;
  if (cout) *cout = c.cout;
  if (k) *k = c.k;
  if (stride) *stride = c.stride;
  return TTK_OK;
}

extern "C" int ttk_hrnet_set_conv(ttk_hrnet* h, int i, const float* w_host, const float* b_host) {
  TTK_CHECK_ARG(h && i >= 0 && i < (int)h->convs.size(), "ttk_hrnet_set_conv: bad index %d", i);
  TTK_CHECK_ARG(w_host && b_host, "ttk_hrnet_set_conv: null pointer");
  if (int rc = ttk_bind_device(&h->device, "ttk_hrnet_set_conv")) return rc;
  TtkConv& c = h->convs[i];
  const int kk = c.k * c.k;
  if (i == (int)h->convs.size() - 1) {
    // final 1x1 conv: only the materialised output slice
    std::vector<float> w((size_t)h->out_count * 16, 0.f), b(h->out_count);
    for (int o = 0; o < h->out_count; ++o) {
      for (int ci = 0; ci < c.cin; ++ci) w[o * 16 + ci] = w_host[(size_t)(h->out_first + o) * c.cin + ci];
      b[o] = b_host[h->out_first + o];
    }
    int rc = upload(&h->final_w, w);
    if (rc) return rc;
    rc = upload(&h->final_b, b);
    if (rc) return rc;
    c.set = true;
    return TTK_OK;
  }
  // [cout][cin][k][k] -> [tap][cin_p][cout_p], zero padded
  std::vector<float> w((size_t)kk * c.cin_p * c.cout_p, 0.f), wr(w.size(), 0.f), wh(w.size(), 0.f), b(c.cout_p, 0.f);
  for (int co = 0; co < c.cout; ++co) {
    b[co] = b_host[co];
    for (int ci = 0; ci < c.cin; ++ci)
      for (int t = 0; t < kk; ++t) {
        const float v = w_host[((size_t)co * c.cin + ci) * kk + t];
        w[((size_t)t * c.cin_p + ci) * c.cout_p + co] = v;
        wr[((size_t)t * c.cin_p + ci) * c.cout_p + co] = bf16_round(v);
        wh[((size_t)t * c.cin_p + ci) * c.cout_p + co] = f16_round(v);
      }
  }
  c.w_host.assign(w_host, w_host + (size_t)c.cout * c.cin * kk);
  c.b_host.assign(b_host, b_host + c.cout);
  h->dual_ready = false;
  int rc = upload(&c.w_f32, w);
  if (rc) return rc;
  rc = upload(&c.w_bfr, wr);
  if (rc) return rc;
  rc = upload(&c.w_hfr, wh);
  if (rc) return rc;
  rc = upload(&c.bias, b);
  if (rc) return rc;
  rc = ttk_conv_umma_pack(c, w_host);
  if (rc) return rc;
  c.set = true;
  return TTK_OK;
}

extern "C" size_t ttk_hrnet_workspace_bytes(const ttk_hrnet* h, int batch, int height, int width, int dtype) {
  if (!h || batch <= 0 || height <= 0 || width <= 0) return 0;
  const int bs = std::min(batch, h->subbatch);
  return plan_memory(const_cast<ttk_hrnet*>(h), bs, height, width, dtype == TTK_BF16 || dtype == TTK_F16 ? 2 : 4);      // TTK_TF32 stores fp32
}

extern "C" int ttk_hrnet_forward(ttk_hrnet* h, const void* x_dev, int batch, int height, int width, int dtype,
                                 float* heatmaps_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
  TTK_CHECK_ARG(h, "ttk_hrnet_forward: null handle");
  if (int rc = ttk_bind_device(&h->device, "ttk_hrnet_forward")) return rc;
  TTK_CHECK_ARG(dtype == TTK_F32 || dtype == TTK_BF16 || dtype == TTK_TF32 || dtype == TTK_TF32X3 || dtype == TTK_F16,
                "ttk_hrnet_forward: bad dtype %d", dtype);
  TTK_CHECK_ARG(batch >= 0 && height > 0 && width > 0 && height % 8 == 0 && width % 8 == 0,
                "ttk_hrnet_forward: height and width must be positive multiples of 8 (got %dx%d)", height, width);
  for (const TtkConv& c : h->convs)
    if (!c.set) {
      ttk_set_error("ttk_hrnet_forward: weights of %s were never set", c.name.c_str());
      return TTK_ERR_STATE;
    }
  h->launches = 0;
  h->recs.clear();
  if (!h->dual_ready && dtype != TTK_F32) {
    int rc = prepare_dual(h);
    if (rc) return rc;
  }
  if (batch == 0) return TTK_OK;
  TTK_CHECK_ARG(x_dev && heatmaps_dev && workspace_dev, "ttk_hrnet_forward: null pointer");
  const size_t elem = dtype == TTK_BF16 || dtype == TTK_F16 ? 2 : 4;
  const int bs = std::min(batch, h->subbatch);
  const size_t need = plan_memory(h, bs, height, width, elem);
  TTK_CHECK_ARG(workspace_bytes >= need, "ttk_hrnet_forward: workspace too small (%zu < %zu)", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  for (int b0 = 0; b0 < batch; b0 += bs) {
    const int nb = std::min(bs, batch - b0);
    const char* x = (const char*)x_dev + (size_t)b0 * height * width * 16 * elem;
    float* heat = heatmaps_dev + (size_t)b0 * h->out_count * height * width;
    int rc;
    if (dtype == TTK_F32)
      rc = run_plan<float>(h, x, nb, height, width, heat, (char*)workspace_dev, 0, false, st);
    else if (dtype == TTK_TF32 || dtype == TTK_TF32X3)
      rc = run_plan<float>(h, x, nb, height, width, heat, (char*)workspace_dev, h->force_simt ? 0 : 4, dtype == TTK_TF32X3, st);
    else if (dtype == TTK_F16)
      rc = run_plan<__half>(h, x, nb, height, width, heat, (char*)workspace_dev, h->force_simt ? 0 : 2, false, st);
    else
      rc = run_plan<__nv_bfloat16>(h, x, nb, height, width, heat, (char*)workspace_dev, h->force_simt ? 0 : 2, false, st);
    if (rc != TTK_OK) return rc;
  }
  if (h->profile && !h->recs.empty()) TTK_CUDA(cudaEventRecord(h->events[h->recs.size()], st));
  return TTK_OK;
}

extern "C" int ttk_hrnet_set_profile(ttk_hrnet* h, int enable) {
  TTK_CHECK_ARG(h, "ttk_hrnet_set_profile: null handle");
  h->profile = enable ? 1 : 0;
  h->recs.clear();
  return TTK_OK;
}

extern "C" int ttk_hrnet_profile_count(const ttk_hrnet* h) { return h ? (int)h->recs.size() : 0; }

extern "C" int ttk_hrnet_profile_read(ttk_hrnet* h, int i, int* op_type, int* conv_index, float* ms, double* flops, double* bytes) {
  TTK_CHECK_ARG(h && i >= 0 && i < (int)h->recs.size(), "ttk_hrnet_profile_read: bad index %d", i);
  const ttk_hrnet::Rec& r = h->recs[i];
  float t = 0.f;
  TTK_CUDA(cudaEventElapsedTime(&t, h->events[i], h->events[i + 1]));   // caller synchronised the stream
  if (op_type) *op_type = r.simt_fallback ? 3 : h->ops[r.op].type;
  if (conv_index) *conv_index = h->ops[r.op].conv;
  if (ms) *ms = t;
  if (flops) *flops = r.flops;
  if (bytes) *bytes = r.bytes;
  return TTK_OK;
}

extern "C" int ttk_hrnet_set_subbatch(ttk_hrnet* h, int images) {
  TTK_CHECK_ARG(h && images >= 1, "ttk_hrnet_set_subbatch: need images >= 1");
  h->subbatch = images;
  return TTK_OK;
}

extern "C" int ttk_hrnet_set_force_simt(ttk_hrnet* h, int enable) {
  TTK_CHECK_ARG(h, "ttk_hrnet_set_force_simt: null handle");
  h->force_simt = enable ? 1 : 0;
  return TTK_OK;
}

// Test hook: run ONE convolution of the plan (bias + optional same-shape residual + optional ReLU) on caller buffers.
// path: 0 = fp32 SIMT (float tensors), 1 = bf16 SIMT, 2 = bf16 tcgen05, 3 = TF32 tcgen05 on float tensors, 4 = 3xTF32 tcgen05 on
// float tensors (2 to 4 return TTK_ERR_UNSUPPORTED if the shape has no kernel).
namespace {
ConvLaunch debug_launch(const TtkConv& cv, const void* in_dev, int n, int hin, int win, const void* res_dev, int relu, void* out_dev) {
  ConvLaunch a;
  a.in = in_dev;
  a.out = out_dev;
  a.nres = res_dev ? 1 : 0;
  for (int r = 0; r < 3; ++r) {
    a.res[r] = r == 0 ? res_dev : nullptr;
    a.res_shift[r] = 0;
  }
  a.n = n;
  a.hin = hin;
  a.win = win;
  a.hout = cv.stride == 2 ? (hin + 1) / 2 : hin;
  a.wout = cv.stride == 2 ? (win + 1) / 2 : win;
  a.cin = cv.cin_p;
  a.cout = cv.cout_p;
  a.relu = relu;
  return a;
}
}  // namespace

extern "C" int ttk_hrnet_debug_conv(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, const void* res_dev,
                                    int relu, int path, void* out_dev, void* stream) {
  TTK_CHECK_ARG(h && conv_index >= 0 && conv_index < (int)h->convs.size() - 1, "ttk_hrnet_debug_conv: bad conv index %d", conv_index);
  const TtkConv& cv = h->convs[conv_index];
  TTK_CHECK_ARG(cv.set, "ttk_hrnet_debug_conv: weights not set");
  TTK_CHECK_ARG(path >= 0 && path <= 4, "ttk_hrnet_debug_conv: bad path %d", path);
  const ConvLaunch a = debug_launch(cv, in_dev, n, hin, win, res_dev, relu, out_dev);
  cudaStream_t st = (cudaStream_t)stream;
  if (path == 0) return launch_conv_simt<float>(cv, a, false, st);
  if (path == 1) return launch_conv_simt<__nv_bfloat16>(cv, a, true, st);
  return ttk_conv_umma_launch(cv, a, st, path == 2 ? 2 : 4, path == 4);
}

// Test hook: the same for fp16 tensors: simt 1 = fp16 SIMT, 0 = fp16 tcgen05 (TTK_ERR_UNSUPPORTED if the shape has no kernel).
extern "C" int ttk_hrnet_debug_conv_f16(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, const void* res_dev,
                                        int relu, int simt, void* out_dev, void* stream) {
  TTK_CHECK_ARG(h && conv_index >= 0 && conv_index < (int)h->convs.size() - 1, "ttk_hrnet_debug_conv_f16: bad conv index %d", conv_index);
  const TtkConv& cv = h->convs[conv_index];
  TTK_CHECK_ARG(cv.set, "ttk_hrnet_debug_conv_f16: weights not set");
  const ConvLaunch a = debug_launch(cv, in_dev, n, hin, win, res_dev, relu, out_dev);
  if (simt) return launch_conv_simt<__half>(cv, a, true, (cudaStream_t)stream);
  return ttk_conv_umma_launch(cv, a, (cudaStream_t)stream, 2, false, true);
}

// Test hook: one BasicBlock (conv_index = its conv1, conv_index + 1 = its conv2) through the fused tcgen05 kernel on caller buffers:
// out = relu(conv2(relu(conv1(in))) + in), NHWC bf16.
extern "C" int ttk_hrnet_debug_block(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, void* out_dev, void* stream) {
  TTK_CHECK_ARG(h && conv_index >= 0 && conv_index + 1 < (int)h->convs.size() - 1, "ttk_hrnet_debug_block: bad conv index %d", conv_index);
  const TtkConv &c1 = h->convs[conv_index], &c2 = h->convs[conv_index + 1];
  TTK_CHECK_ARG(c1.set && c2.set, "ttk_hrnet_debug_block: weights not set");
  return ttk_block_umma_launch(c1, c2, in_dev, out_dev, n, hin, win, (cudaStream_t)stream, 2);
}

extern "C" int ttk_hrnet_set_block_fusion(ttk_hrnet* h, int enable) {
  TTK_CHECK_ARG(h, "ttk_hrnet_set_block_fusion: null handle");
  h->use_block_fusion = enable;          // 0 off, 1 bf16 blocks (default), 2 / 3 also the TF32 16-channel blocks (two 3-row tiles / one 4-row tile)
  return TTK_OK;
}

extern "C" int ttk_hrnet_last_launches(const ttk_hrnet* h) { return h ? h->launches : 0; }
