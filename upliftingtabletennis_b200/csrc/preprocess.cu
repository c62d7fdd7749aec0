// Fused frame pre-processing: bit-exact cv2.resize (uint8 INTER_LINEAR, 11-bit fixed point)
// + LUT normalise + [prev,cur,next] stack + layout change, one pass, uint8 in.
// Reference: balldetection/transforms.py:17-52, :379-402; interface.py:110-112.
//
// HBM-bound: per stack 3 source frames are read once (later taps hit L1/L2) and the stack is
// written once with 128-bit stores.  One thread produces one output pixel (all 3*F channels).
#include <algorithm>

#include "ttk_internal.h"
#include "umma_prims.h"

namespace {

struct AxisTap {
  int s0, s1, a0, a1;
};

// OpenCV resize tap for destination index d (see oracle/preprocess.py: axis_taps).
// __dmul_rn/__dadd_rn/__fsub_rn keep the compiler from contracting into FMAs, which would
// change the rounding of the float32 coordinate.
__device__ __forceinline__ AxisTap axis_tap(int d, int n_src, double scale) {
  const double fd = __dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5);
  float f = (float)fd;
  int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  if (s < 0) {
    s = 0;
    f = 0.f;
  }
  if (s >= n_src - 1) {
    s = n_src - 1;
    f = 0.f;
  }
  AxisTap t;
  t.s0 = s;
  t.s1 = min(s + 1, n_src - 1);
  t.a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  t.a1 = __float2int_rn(__fmul_rn(f, 2048.f));
  return t;
}

// F frames per stack; MODE 0: NCHW f32, 1: NHWC16 f32, 2: NHWC16 bf16, 3: NHWC16 fp16.  IDX: stack s starts at frame first_frame[s]
// instead of s * stack_stride (first_frame is the last parameter, so the strided instantiations keep their parameter offsets).
template <int F, int MODE, bool IDX>
__global__ void __launch_bounds__(256) preprocess_kernel(const uint8_t* __restrict__ frames, int src_h, int src_w,
                                                         int stack_stride, int dst_h, int dst_w, double scale_x,
                                                         double scale_y, const float* __restrict__ lut,
                                                         void* __restrict__ out, const int32_t* __restrict__ first_frame) {
  __shared__ float s_lut[768];
  for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = lut[i];
  __syncthreads();
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int s = blockIdx.z;
  if (x >= dst_w) return;
  const bool same = (src_h == dst_h && src_w == dst_w);
  const AxisTap tx = axis_tap(x, src_w, scale_x);
  const AxisTap ty = axis_tap(y, src_h, scale_y);
  float v[3 * F];
#pragma unroll
  for (int f = 0; f < F; ++f) {
    const uint8_t* img = frames + (size_t)((IDX ? __ldg(first_frame + s) : s * stack_stride) + f) * src_h * src_w * 3;
    const uint8_t* r0 = img + ((size_t)ty.s0 * src_w) * 3;
    const uint8_t* r1 = img + ((size_t)ty.s1 * src_w) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int u8;
      if (same) {
        u8 = __ldg(img + ((size_t)y * src_w + x) * 3 + c);
      } else {
        const int h0 = __ldg(r0 + tx.s0 * 3 + c) * tx.a0 + __ldg(r0 + tx.s1 * 3 + c) * tx.a1;
        const int h1 = __ldg(r1 + tx.s0 * 3 + c) * tx.a0 + __ldg(r1 + tx.s1 * 3 + c) * tx.a1;
        const int acc = ((ty.a0 * (h0 >> 4)) >> 16) + ((ty.a1 * (h1 >> 4)) >> 16);
        u8 = min(255, max(0, (acc + 2) >> 2));
      }
      v[f * 3 + c] = s_lut[c * 256 + u8];
    }
  }
  if (MODE == 0) {
    float* o = (float*)out + (size_t)s * (3 * F) * dst_h * dst_w + (size_t)y * dst_w + x;
#pragma unroll
    for (int c = 0; c < 3 * F; ++c) o[(size_t)c * dst_h * dst_w] = v[c];
  } else if (MODE == 1) {
    float4* o = (float4*)((float*)out + ((size_t)(s * dst_h + y) * dst_w + x) * 16);
    float w[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) w[c] = c < 3 * F ? v[c] : 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = make_float4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
  } else {
    uint4* o = (uint4*)((uint16_t*)out + ((size_t)(s * dst_h + y) * dst_w + x) * 16);
    uint32_t w[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float lo = 2 * c < 3 * F ? v[2 * c] : 0.f;
      const float hi = 2 * c + 1 < 3 * F ? v[2 * c + 1] : 0.f;
      w[c] = umma::Fmt16<MODE == 3>::pack(lo, hi);
    }
    o[0] = make_uint4(w[0], w[1], w[2], w[3]);
    o[1] = make_uint4(w[4], w[5], w[6], w[7]);
  }
}

// Same arithmetic as a persistent tile kernel (the measured path for 1080p sources).
//   * A block owns one 256-pixel column block and walks (stack, output row) tiles with a grid stride, so the horizontal
//     taps, the byte offsets and the replicated normalisation table are set up once per block, not once per row.
//   * The two source rows of each frame are staged in shared memory with coalesced 128-bit loads (the per-pixel taps
//     overlap heavily: 1.5 source pixels per output pixel at 1080p -> 704p); the loads of tile t+1 are issued before
//     tile t is computed and land in the other half of a double buffer: one __syncthreads per tile.
//   * The 6 bytes a pixel needs per source row (2 taps x BGR) come from three 32-bit shared loads aligned by a funnel
//     shift; PRMT pairs (tap0, tap1) bytes and DP2A forms tap0*a0 + tap1*a1 -- 10 instructions per row instead of 12 byte
//     loads + 6 multiply-adds, and half the shared-memory wavefronts.
//   * (a * x) >> 16 is one multiply-high with a pre-shifted weight.
// Needs 16-byte aligned source rows.
constexpr int PRE_ROW_BYTES = 1536;      // >= (256 outputs * max scale 1.6 + 3) * 3 bytes + alignment slack
constexpr int PRE_STAGE = 3;             // 128-bit staging loads per thread and tile (3 frames x 2 rows x <= 96 vectors / 256 threads)
constexpr int LUT_COPIES = 8;            // normalisation table replicated so that random look-ups spread over the banks
template <int F, int MODE, bool IDX>
__global__ void __launch_bounds__(256) preprocess_tile_kernel(const uint8_t* __restrict__ frames, int src_h, int src_w,
                                                              int stack_stride, int n_stacks, int dst_h, int dst_w, int nxb,
                                                              double scale_x, double scale_y, const float* __restrict__ lut,
                                                              void* __restrict__ out, const int32_t* __restrict__ first_frame) {
  __shared__ float s_lut[768 * LUT_COPIES];                    // [entry][copy]
  __shared__ __align__(16) uint8_t s_rows[2][F * 2 * PRE_ROW_BYTES];
  for (int i = threadIdx.x; i < 768 * LUT_COPIES; i += blockDim.x) s_lut[i] = lut[i / LUT_COPIES];
  const int xb = blockIdx.x % nxb, t_first = blockIdx.x / nxb, t_step = gridDim.x / nxb;
  const int n_tiles = n_stacks * dst_h;
  const int x0 = xb * 256;
  const int x = x0 + threadIdx.x;
  const int x_last = min(x0 + 256, dst_w) - 1;
  const AxisTap tx_first = axis_tap(x0, src_w, scale_x), tx_last = axis_tap(x_last, src_w, scale_x);
  const AxisTap tx = axis_tap(min(x, dst_w - 1), src_w, scale_x);
  const int byte_lo = (tx_first.s0 * 3) & ~15;                // 16-byte aligned start within the source row
  const int byte_hi = (tx_last.s1 + 1) * 3;                    // exclusive
  const int nvec = (byte_hi - byte_lo + 15) >> 4;
  const size_t row_bytes = (size_t)src_w * 3, frame_bytes = row_bytes * src_h;
  // the second tap is read 3 bytes after the first: wherever that is not source pixel s1 (clamped borders) its weight is zero
  const int o0 = tx.s0 * 3 - byte_lo;
  const int word0 = o0 >> 2, shift = (o0 & 3) * 8;
  const uint32_t wx = (uint32_t)tx.a0 | ((uint32_t)tx.a1 << 16);
  const float* my_lut = s_lut + (threadIdx.x & (LUT_COPIES - 1));
  // staging slots of this thread: vector v of source row r (0: upper, 1: lower) of frame f
  int st_dst[PRE_STAGE], st_col[PRE_STAGE];                    // shared offset (< 0: none), byte offset within the source row
  size_t st_src[PRE_STAGE];                                    // byte offset from the stack's first frame, without the row term
  bool st_low[PRE_STAGE], st_ragged[PRE_STAGE];
#pragma unroll
  for (int j = 0; j < PRE_STAGE; ++j) {
    const int i = threadIdx.x + 256 * j;
    const int v = i % nvec, r = (i / nvec) & 1, f = i / (2 * nvec);
    st_dst[j] = i < F * 2 * nvec ? (f * 2 + r) * PRE_ROW_BYTES + 16 * v : -1;
    st_col[j] = byte_lo + 16 * v;
    st_src[j] = (size_t)f * frame_bytes + st_col[j];
    st_low[j] = r != 0;
    st_ragged[j] = st_col[j] + 16 > (int)row_bytes;
  }
  uint4 q[PRE_STAGE];
  auto fetch = [&](int s, const AxisTap& ty) {                 // global -> registers
    const uint8_t* base = frames + (IDX ? (size_t)__ldg(first_frame + s) * frame_bytes : (size_t)s * stack_stride * frame_bytes);
    const uint8_t* up = base + (size_t)ty.s0 * row_bytes;
    const uint8_t* low = base + (size_t)ty.s1 * row_bytes;
#pragma unroll
    for (int j = 0; j < PRE_STAGE; ++j) {
      if (st_dst[j] < 0) continue;
      const uint8_t* src = (st_low[j] ? low : up) + st_src[j];
      if (!st_ragged[j]) {
        q[j] = __ldg(reinterpret_cast<const uint4*>(src));
      } else {                                                  // ragged end of the row
        uint8_t tmp[16];
        for (int b = 0; b < 16; ++b) tmp[b] = (st_col[j] + b < (int)row_bytes) ? __ldg(src + b) : 0;
        q[j] = *reinterpret_cast<uint4*>(tmp);
      }
    }
  };
  auto stash = [&](int buf) {                                  // registers -> shared
#pragma unroll
    for (int j = 0; j < PRE_STAGE; ++j)
      if (st_dst[j] >= 0) *reinterpret_cast<uint4*>(s_rows[buf] + st_dst[j]) = q[j];
  };
  int t = t_first, buf = 0;
  int s = t / dst_h, y = t - s * dst_h;                          // (stack, row) of tile t, advanced without divisions
  const int s_step = t_step / dst_h, y_step = t_step - s_step * dst_h;
  AxisTap ty = axis_tap(min(y, dst_h - 1), src_h, scale_y);
  if (t < n_tiles) {
    fetch(s, ty);
    stash(0);
  }
  __syncthreads();
  for (; t < n_tiles; t += t_step, buf ^= 1) {
    const bool more = t + t_step < n_tiles;
    int s_next = s + s_step, y_next = y + y_step;
    if (y_next >= dst_h) y_next -= dst_h, ++s_next;
    const AxisTap ty_next = axis_tap(y_next, src_h, scale_y);
    if (more) fetch(s_next, ty_next);
    if (x < dst_w) {
      const uint32_t wy0 = (uint32_t)ty.a0 << 16, wy1 = (uint32_t)ty.a1 << 16;
      float v[3 * F];
#pragma unroll
      for (int f = 0; f < F; ++f) {
        uint32_t h[2][3];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const uint32_t* w = reinterpret_cast<const uint32_t*>(s_rows[buf] + (f * 2 + r) * PRE_ROW_BYTES) + word0;
          const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
          const uint32_t lo = __funnelshift_r(w0, w1, shift), hi = __funnelshift_r(w1, w2, shift);   // bytes 0..3, 4..7 from the first tap
          const uint32_t p01 = __byte_perm(lo, hi, 0x4130), p2 = __byte_perm(lo, hi, 0x0052);       // (B0,B1,G0,G1), (R0,R1,-,-)
          h[r][0] = __dp2a_lo(wx, p01, 0u);
          h[r][1] = __dp2a_hi(wx, p01, 0u);
          h[r][2] = __dp2a_lo(wx, p2, 0u);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const uint32_t acc = __umulhi(wy0, h[0][c] >> 4) + __umulhi(wy1, h[1][c] >> 4);           // ((a * (h >> 4)) >> 16, twice
          // the weights of an axis sum to at most 2049, so acc <= 1020 and the result needs no saturation (cv2 saturates here)
          const uint32_t u8 = (acc + 2u) >> 2;
          v[f * 3 + c] = my_lut[(c * 256 + u8) * LUT_COPIES];
        }
      }
      if (MODE == 0) {
        float* o = (float*)out + (size_t)s * (3 * F) * dst_h * dst_w + (size_t)y * dst_w + x;
#pragma unroll
        for (int c = 0; c < 3 * F; ++c) o[(size_t)c * dst_h * dst_w] = v[c];
      } else if (MODE == 1) {
        float4* o = (float4*)((float*)out + ((size_t)(s * dst_h + y) * dst_w + x) * 16);
        float w[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) w[c] = c < 3 * F ? v[c] : 0.f;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) o[q4] = make_float4(w[4 * q4], w[4 * q4 + 1], w[4 * q4 + 2], w[4 * q4 + 3]);
      } else {
        uint4* o = (uint4*)((uint16_t*)out + ((size_t)(s * dst_h + y) * dst_w + x) * 16);
        uint32_t w[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float lo = 2 * c < 3 * F ? v[2 * c] : 0.f;
          const float hi = 2 * c + 1 < 3 * F ? v[2 * c + 1] : 0.f;
          w[c] = umma::Fmt16<MODE == 3>::pack(lo, hi);
        }
        o[0] = make_uint4(w[0], w[1], w[2], w[3]);
        o[1] = make_uint4(w[4], w[5], w[6], w[7]);
      }
    }
    if (more) stash(buf ^ 1);
    s = s_next, y = y_next, ty = ty_next;
    __syncthreads();
  }
}

template <int F, bool IDX>
int launch(int mode, dim3 grid, cudaStream_t st, const uint8_t* frames, int src_h, int src_w, int stack_stride, int dst_h,
           int dst_w, const float* lut, void* out, const int32_t* first) {
  const double sx = (double)src_w / (double)dst_w, sy = (double)src_h / (double)dst_h;
  const bool staged = !(src_h == dst_h && src_w == dst_w) && ((size_t)src_w * 3) % 16 == 0 && ((uintptr_t)frames & 15) == 0 &&
                      (256.0 * sx + 4.0) * 3.0 + 32.0 <= PRE_ROW_BYTES;
  if (staged) {
    static int n_sm = 0;
    if (!n_sm) {
      int dev = 0;
      TTK_CUDA(cudaGetDevice(&dev));
      TTK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    }
    const int n_stacks = grid.z, nxb = grid.x;
    const long long n_tiles = (long long)n_stacks * dst_h;
    // 5 resident blocks per SM (42 KB of shared memory each); every column block gets the same number of row walkers
    const int walkers = (int)std::max(1LL, std::min<long long>(n_tiles, (n_sm * 5) / nxb));
    const dim3 g(nxb * walkers);
    if (mode == 0)
      preprocess_tile_kernel<F, 0, IDX><<<g, 256, 0, st>>>(frames, src_h, src_w, stack_stride, n_stacks, dst_h, dst_w, nxb, sx, sy, lut, out,
                                                          first);
    else if (mode == 1)
      preprocess_tile_kernel<F, 1, IDX><<<g, 256, 0, st>>>(frames, src_h, src_w, stack_stride, n_stacks, dst_h, dst_w, nxb, sx, sy, lut, out,
                                                          first);
    else if (mode == 2)
      preprocess_tile_kernel<F, 2, IDX><<<g, 256, 0, st>>>(frames, src_h, src_w, stack_stride, n_stacks, dst_h, dst_w, nxb, sx, sy, lut, out,
                                                          first);
    else
      preprocess_tile_kernel<F, 3, IDX><<<g, 256, 0, st>>>(frames, src_h, src_w, stack_stride, n_stacks, dst_h, dst_w, nxb, sx, sy, lut, out,
                                                          first);
    TTK_LAUNCH_CHECK();
    return TTK_OK;
  }
  if (mode == 0)
    preprocess_kernel<F, 0, IDX><<<grid, 256, 0, st>>>(frames, src_h, src_w, stack_stride, dst_h, dst_w, sx, sy, lut, out, first);
  else if (mode == 1)
    preprocess_kernel<F, 1, IDX><<<grid, 256, 0, st>>>(frames, src_h, src_w, stack_stride, dst_h, dst_w, sx, sy, lut, out, first);
  else if (mode == 2)
    preprocess_kernel<F, 2, IDX><<<grid, 256, 0, st>>>(frames, src_h, src_w, stack_stride, dst_h, dst_w, sx, sy, lut, out, first);
  else
    preprocess_kernel<F, 3, IDX><<<grid, 256, 0, st>>>(frames, src_h, src_w, stack_stride, dst_h, dst_w, sx, sy, lut, out, first);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

}  // namespace

// layout / dtype -> kernel MODE, or -1 (the error is set)
static int preprocess_mode(const char* fn, int layout, int dtype) {
  if (layout == TTK_LAYOUT_NCHW_F32) {
    if (dtype == TTK_F32) return 0;
    ttk_set_error("%s: NCHW output is float32 only", fn);
    return -1;
  }
  if (layout == TTK_LAYOUT_NHWC16) {
    if (dtype == TTK_F32 || dtype == TTK_BF16 || dtype == TTK_F16) return dtype == TTK_F32 ? 1 : dtype == TTK_BF16 ? 2 : 3;
    ttk_set_error("%s: bad dtype", fn);
    return -1;
  }
  ttk_set_error("%s: bad layout %d", fn, layout);
  return -1;
}

extern "C" int ttk_preprocess_stacks(const uint8_t* frames_dev, int n_frames, int src_h, int src_w, int frames_per_stack,
                                     int stack_stride, int n_stacks, int dst_h, int dst_w, const float* lut_dev,
                                     void* out_dev, int layout, int dtype, void* stream) {
  TTK_CHECK_ARG(frames_dev && lut_dev && out_dev, "ttk_preprocess_stacks: null pointer");
  TTK_CHECK_ARG(frames_per_stack == 1 || frames_per_stack == 3, "ttk_preprocess_stacks: frames_per_stack must be 1 or 3");
  TTK_CHECK_ARG(n_stacks >= 0 && stack_stride >= 1 && src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0,
                "ttk_preprocess_stacks: bad sizes");
  TTK_CHECK_ARG(n_stacks == 0 || (n_stacks - 1) * stack_stride + frames_per_stack <= n_frames,
                "ttk_preprocess_stacks: stacks read past the last frame (%d stacks, stride %d, %d frames)", n_stacks,
                stack_stride, n_frames);
  TTK_CHECK_ARG(n_stacks <= 65535 && dst_h <= 65535, "ttk_preprocess_stacks: grid too large");
  const int mode = preprocess_mode("ttk_preprocess_stacks", layout, dtype);
  if (mode < 0) return TTK_ERR_ARG;
  if (n_stacks == 0) return TTK_OK;
  dim3 grid(ttk_cdiv(dst_w, 256), dst_h, n_stacks);
  cudaStream_t st = (cudaStream_t)stream;
  if (frames_per_stack == 3)
    return launch<3, false>(mode, grid, st, frames_dev, src_h, src_w, stack_stride, dst_h, dst_w, lut_dev, out_dev, nullptr);
  return launch<1, false>(mode, grid, st, frames_dev, src_h, src_w, stack_stride, dst_h, dst_w, lut_dev, out_dev, nullptr);
}

extern "C" int ttk_preprocess_stacks_indexed(const uint8_t* frames_dev, int n_frames, int src_h, int src_w, int frames_per_stack,
                                             const int32_t* first_frame_dev, int n_stacks, int dst_h, int dst_w,
                                             const float* lut_dev, void* out_dev, int layout, int dtype, void* stream) {
  TTK_CHECK_ARG(frames_dev && lut_dev && out_dev && first_frame_dev, "ttk_preprocess_stacks_indexed: null pointer");
  TTK_CHECK_ARG(frames_per_stack == 1 || frames_per_stack == 3, "ttk_preprocess_stacks_indexed: frames_per_stack must be 1 or 3");
  TTK_CHECK_ARG(n_stacks >= 0 && n_frames >= frames_per_stack && src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0,
                "ttk_preprocess_stacks_indexed: bad sizes");
  TTK_CHECK_ARG(n_stacks <= 65535 && dst_h <= 65535, "ttk_preprocess_stacks_indexed: grid too large");
  const int mode = preprocess_mode("ttk_preprocess_stacks_indexed", layout, dtype);
  if (mode < 0) return TTK_ERR_ARG;
  if (n_stacks == 0) return TTK_OK;
  dim3 grid(ttk_cdiv(dst_w, 256), dst_h, n_stacks);
  cudaStream_t st = (cudaStream_t)stream;
  if (frames_per_stack == 3)
    return launch<3, true>(mode, grid, st, frames_dev, src_h, src_w, 1, dst_h, dst_w, lut_dev, out_dev, first_frame_dev);
  return launch<1, true>(mode, grid, st, frames_dev, src_h, src_w, 1, dst_h, dst_w, lut_dev, out_dev, first_frame_dev);
}
