// Small bandwidth-bound kernels either side of the networks:
//   ttk_trajectory_pack : inference/utils.py:268-309 (_uplifting_transform), batched over clips
//   ttk_rotation_local  : uplifting/helper.py:394-420 (transform_rotationaxes)
//   ttk_project         : uplifting/helper.py:137-204 (world2cam, cam2img), interface.py:301-312
//   ttk_reproject_clips : ttk_project over many clips of different lengths, each with its own camera, plus the reprojection error
#include "ttk_internal.h"

namespace {

// one block per clip
__global__ void trajectory_pack_kernel(const double* __restrict__ ball, const double* __restrict__ times,
                                       const int32_t* __restrict__ offsets, const double* __restrict__ table, int seq_len,
                                       double img_w, double img_h, float* __restrict__ ball_out, float* __restrict__ table_out,
                                       float* __restrict__ times_out, float* __restrict__ mask_out) {
  const int clip = blockIdx.x;
  const int begin = offsets[clip];
  const int n = min(offsets[clip + 1] - begin, seq_len);
  for (int t = threadIdx.x; t < seq_len; t += blockDim.x) {
    float bx = 0.f, by = 0.f, tm = 0.f, mk = 0.f;
    if (t < n) {
      bx = (float)(ball[(size_t)(begin + t) * 2] / img_w);        // float64 divide, then the float32 cast of torch.tensor(...)
      by = (float)(ball[(size_t)(begin + t) * 2 + 1] / img_h);
      tm = (float)times[begin + t];
      mk = 1.f;
    }
    ball_out[((size_t)clip * seq_len + t) * 2] = bx;
    ball_out[((size_t)clip * seq_len + t) * 2 + 1] = by;
    times_out[(size_t)clip * seq_len + t] = tm;
    mask_out[(size_t)clip * seq_len + t] = mk;
  }
  for (int k = threadIdx.x; k < 13; k += blockDim.x) {
    const double* p = table + ((size_t)clip * 13 + k) * 3;
    float* o = table_out + ((size_t)clip * 13 + k) * 3;
    o[0] = (float)(p[0] / img_w);
    o[1] = (float)(p[1] / img_h);
    o[2] = (float)p[2];
  }
}

__global__ void rotation_local_kernel(const float* __restrict__ rot, const float* __restrict__ pos, int batch, int seq_len,
                                      float* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  const float* p = pos + (size_t)b * seq_len * 3;
  const float vx = __fsub_rn(p[3], p[0]), vy = __fsub_rn(p[4], p[1]);
  const float nrm = sqrtf(__fadd_rn(__fmul_rn(vx, vx), __fmul_rn(vy, vy)));
  const float ex = vx / nrm, ey = vy / nrm;              // e_x = v0 / |v0| (z component 0)
  // e_y = e_z x e_x = (-ex.y, ex.x, 0)
  const float r0 = rot[b * 3], r1 = rot[b * 3 + 1], r2 = rot[b * 3 + 2];
  out[b * 3 + 0] = __fadd_rn(__fmul_rn(r0, ex), __fmul_rn(r1, ey));
  out[b * 3 + 1] = __fadd_rn(__fmul_rn(r0, -ey), __fmul_rn(r1, ex));
  out[b * 3 + 2] = r2;
}

// cam2img(world2cam(p)) of one point with the matrices in shared memory: s_e the 4x4 Mext, s_i the leading 3x3 of Mint, both row
// major.  project_kernel and reproject_clips_kernel both call it, so a point comes out with the same bits from either.
template <typename T>
__device__ __forceinline__ void project_point(const T* s_e, const T* s_i, T x, T y, T z, T& u, T& v) {
  T c[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) c[r] = s_e[r * 4] * x + s_e[r * 4 + 1] * y + s_e[r * 4 + 2] * z + s_e[r * 4 + 3];
  const T cx = c[0] / c[3], cy = c[1] / c[3], cz = c[2] / c[3];
  T q[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) q[r] = s_i[r * 3] * cx + s_i[r * 3 + 1] * cy + s_i[r * 3 + 2] * cz;
  u = q[0] / q[2];
  v = q[1] / q[2];
}

template <typename T>
__global__ void project_kernel(const T* __restrict__ pts, const T* __restrict__ mext, const T* __restrict__ mint, int n,
                               T* __restrict__ out) {
  __shared__ T s_e[16], s_i[9];
  if (threadIdx.x < 16) s_e[threadIdx.x] = mext[threadIdx.x];
  if (threadIdx.x < 9) s_i[threadIdx.x] = mint[threadIdx.x];
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  T u, v;
  project_point(s_e, s_i, pts[(size_t)i * 3], pts[(size_t)i * 3 + 1], pts[(size_t)i * 3 + 2], u, v);
  out[(size_t)i * 2] = u;
  out[(size_t)i * 2 + 1] = v;
}

constexpr int RC_THREADS = 128;

// one CTA per clip: its points offs[c] .. offs[c+1]-1 through project_point with the clip's Mext and the leading 3x3 of its (3, 4) Mint,
// and the Euclidean distance of each to the detection of the same row.  Thread 0 sums the distances in row order (sequential float64
// adds) and keeps the largest, so that a host loop over the rows gives the same bits; a NaN distance makes both NaN.  A clip with
// valid[c] == 0 writes NaN for its points and errors.
__global__ void __launch_bounds__(RC_THREADS) reproject_clips_kernel(const double* __restrict__ pts, const int32_t* __restrict__ offs,
                                                                     const double* __restrict__ mint, const double* __restrict__ mext,
                                                                     const int32_t* __restrict__ valid, const double* __restrict__ det,
                                                                     double* __restrict__ out, double* __restrict__ err) {
  __shared__ double s_e[16], s_i[9], s_d[RC_THREADS];
  const int clip = blockIdx.x;
  const int begin = offs[clip], n = offs[clip + 1] - begin;
  const bool ok = valid[clip] != 0;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  if (threadIdx.x < 16) s_e[threadIdx.x] = mext[(size_t)clip * 16 + threadIdx.x];
  if (threadIdx.x < 9) s_i[threadIdx.x] = mint[(size_t)clip * 12 + (threadIdx.x / 3) * 4 + threadIdx.x % 3];
  __syncthreads();
  double sum = 0.0, worst = nan;
  for (int t0 = 0; t0 < n; t0 += RC_THREADS) {
    const int t = t0 + threadIdx.x;
    if (t < n) {
      const size_t r = (size_t)begin + t;
      double u = nan, v = nan;
      if (ok) project_point(s_e, s_i, pts[r * 3], pts[r * 3 + 1], pts[r * 3 + 2], u, v);
      out[r * 2] = u;
      out[r * 2 + 1] = v;
      const double dx = __dsub_rn(u, det[r * 2]), dy = __dsub_rn(v, det[r * 2 + 1]);
      s_d[threadIdx.x] = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const int m = min(RC_THREADS, n - t0);
      for (int i = 0; i < m; ++i) {
        const double d = s_d[i];
        sum = __dadd_rn(sum, d);
        if (t0 + i == 0 || d > worst || isnan(d)) worst = d;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    err[(size_t)clip * 2] = ok ? sum / (double)n : nan;         // n == 0: 0 / 0, NaN
    err[(size_t)clip * 2 + 1] = ok ? worst : nan;
  }
}

}  // namespace

extern "C" int ttk_trajectory_pack(const double* ball_xy_dev, const double* times_dev, const int32_t* offsets_dev,
                                   const double* table_dev, int n_clips, int seq_len, double img_w, double img_h,
                                   float* ball_out, float* table_out, float* times_out, float* mask_out, void* stream) {
  TTK_CHECK_ARG(n_clips >= 0 && seq_len > 0, "ttk_trajectory_pack: bad sizes");
  if (n_clips == 0) return TTK_OK;
  TTK_CHECK_ARG(ball_xy_dev && times_dev && offsets_dev && table_dev && ball_out && table_out && times_out && mask_out,
                "ttk_trajectory_pack: null pointer");
  trajectory_pack_kernel<<<n_clips, 64, 0, (cudaStream_t)stream>>>(ball_xy_dev, times_dev, offsets_dev, table_dev, seq_len, img_w,
                                                                  img_h, ball_out, table_out, times_out, mask_out);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_rotation_local(const float* rot_dev, const float* pos_dev, int batch, int seq_len, float* out_dev,
                                  void* stream) {
  TTK_CHECK_ARG(batch >= 0 && seq_len >= 2, "ttk_rotation_local: need at least two positions per trajectory");
  if (batch == 0) return TTK_OK;
  TTK_CHECK_ARG(rot_dev && pos_dev && out_dev, "ttk_rotation_local: null pointer");
  rotation_local_kernel<<<ttk_cdiv(batch, 128), 128, 0, (cudaStream_t)stream>>>(rot_dev, pos_dev, batch, seq_len, out_dev);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_project(const void* points_dev, const void* mext_dev, const void* mint_dev, int n, int dtype_f64,
                           void* out_dev, void* stream) {
  TTK_CHECK_ARG(n >= 0, "ttk_project: bad n");
  if (n == 0) return TTK_OK;
  TTK_CHECK_ARG(points_dev && mext_dev && mint_dev && out_dev, "ttk_project: null pointer");
  if (dtype_f64)
    project_kernel<double><<<ttk_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((const double*)points_dev, (const double*)mext_dev,
                                                                              (const double*)mint_dev, n, (double*)out_dev);
  else
    project_kernel<float><<<ttk_cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((const float*)points_dev, (const float*)mext_dev,
                                                                            (const float*)mint_dev, n, (float*)out_dev);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_reproject_clips(const double* points_dev, int n_points, const int32_t* offsets_dev, int n_clips, const double* mint_dev,
                                   const double* mext_dev, const int32_t* valid_dev, const double* det_xy_dev, double* out_xy_dev,
                                   double* out_err_dev, void* stream) {
  TTK_CHECK_ARG(n_clips >= 0 && n_points >= 0, "ttk_reproject_clips: bad sizes");
  if (n_clips == 0) return TTK_OK;
  TTK_CHECK_ARG(offsets_dev && mint_dev && mext_dev && valid_dev && out_err_dev, "ttk_reproject_clips: null pointer");
  TTK_CHECK_ARG(n_points == 0 || (points_dev && det_xy_dev && out_xy_dev), "ttk_reproject_clips: null pointer");
  reproject_clips_kernel<<<n_clips, RC_THREADS, 0, (cudaStream_t)stream>>>(points_dev, offsets_dev, mint_dev, mext_dev, valid_dev,
                                                                           det_xy_dev, out_xy_dev, out_err_dev);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}
