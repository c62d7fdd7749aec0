// Trajectory filters between decode and uplift, on the device (SURVEY.md section 8f row 2):
//   ttk_filter_ball  : inference/utils.py:70-102 (filter_trajectory_ball): two-detector agreement, ordered compaction
//   ttk_filter_table : inference/utils.py:137-169 (filter_trajectory_table) + :172-232 (_filter_keypoints_with_dbscan):
//                      two-detector agreement per keypoint, DBSCAN(eps, min_samples), centroid of the largest cluster.
// DBSCAN follows scikit-learn's semantics exactly (sklearn/cluster/_dbscan.py, _dbscan_inner.pyx): a point is a core
// point when at least min_samples points (itself included) lie within eps (inclusive, compared on squared distances
// like the KD-tree's reduced distance); clusters are numbered by their lowest-index core point; a border point joins
// the lowest-numbered cluster that has a core point in its neighbourhood (clusters are grown one after the other);
// Counter.most_common(1) returns, among equally large clusters, the one that appears first in point order.
// ttk_filter_ball_clips and ttk_filter_table_clips run the same per-clip arithmetic over n clips of different lengths in one launch.
// All arithmetic is float64 without contraction, sums run in point order like numpy's axis-0 reduction.
#include <limits.h>

#include "ttk_internal.h"

namespace {

constexpr int FB_THREADS = 1024;

// ---- ball: one CTA, ordered stream compaction -------------------------------------------------------------------
__global__ void __launch_bounds__(FB_THREADS) filter_ball_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                 int T, double fps, double threshold, double visible,
                                                                 double* __restrict__ out_xy, int64_t* __restrict__ out_idx,
                                                                 double* __restrict__ out_times, int32_t* __restrict__ out_offsets) {
  __shared__ int s_warp[FB_THREADS / 32];
  __shared__ int s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int t0 = 0; t0 < T; t0 += FB_THREADS) {
    const int t = t0 + threadIdx.x;
    bool keep = false;
    double x = 0, y = 0;
    if (t < T) {
      x = p1[(size_t)t * 3];
      y = p1[(size_t)t * 3 + 1];
      const double dx = __dsub_rn(x, p2[(size_t)t * 3]), dy = __dsub_rn(y, p2[(size_t)t * 3 + 1]);
      const double d = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));      // np.linalg.norm(., axis=1)
      keep = !(d > threshold || p1[(size_t)t * 3 + 2] != visible || p2[(size_t)t * 3 + 2] != visible);
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (keep) {
      const int o = before + __popc(m & ((1u << lane) - 1u));
      out_xy[(size_t)o * 2] = x;
      out_xy[(size_t)o * 2 + 1] = y;
      out_idx[o] = t;
      out_times[o] = (double)t / fps;             // float(t / fps)
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < FB_THREADS / 32; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out_offsets[0] = 0;
    out_offsets[1] = s_base;
  }
}

// ---- ball over n clips: one CTA, ordered compaction of the concatenation --------------------------------------------------
// Compacting the concatenated clips in frame order packs each clip's rows contiguously in clip order, so the per-clip
// result of filter_ball_kernel is this kernel's rows out_offsets[c] .. out_offsets[c+1]-1 once idx and times count from
// the clip's first frame.  out_offsets[c] is the number of kept frames before frame offs[c].
__global__ void __launch_bounds__(FB_THREADS) filter_ball_clips_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                       const int32_t* __restrict__ offs, int n_clips, int T,
                                                                       double fps, double threshold, double visible,
                                                                       double* __restrict__ out_xy, int64_t* __restrict__ out_idx,
                                                                       double* __restrict__ out_times,
                                                                       int32_t* __restrict__ out_offsets) {
  __shared__ int s_warp[FB_THREADS / 32];
  __shared__ int s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int t0 = 0; t0 < T; t0 += FB_THREADS) {
    const int t = t0 + threadIdx.x;
    bool keep = false;
    double x = 0, y = 0;
    int c_first = 0, c_last = -1;            // clips [c_first, c_last] start at frame t; c_last is the clip frame t belongs to
    if (t < T) {
      x = p1[(size_t)t * 3];
      y = p1[(size_t)t * 3 + 1];
      const double dx = __dsub_rn(x, p2[(size_t)t * 3]), dy = __dsub_rn(y, p2[(size_t)t * 3 + 1]);
      const double d = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
      keep = !(d > threshold || p1[(size_t)t * 3 + 2] != visible || p2[(size_t)t * 3 + 2] != visible);
      int lo = 0, hi = n_clips + 1;          // first c with offs[c] >= t
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (offs[mid] < t) lo = mid + 1; else hi = mid;
      }
      c_first = lo;
      c_last = lo - 1;
      while (c_last + 1 < n_clips && offs[c_last + 1] == t) ++c_last;     // the empty clips at t, then the clip holding t
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    const int o = before + __popc(m & ((1u << lane) - 1u));
    for (int c = c_first; c <= c_last; ++c) out_offsets[c] = o;
    if (keep) {
      const int local = t - offs[c_last];
      out_xy[(size_t)o * 2] = x;
      out_xy[(size_t)o * 2 + 1] = y;
      out_idx[o] = local;
      out_times[o] = (double)local / fps;     // float(t / fps) of the clip's own frame index
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < FB_THREADS / 32; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
  }
  for (int c = threadIdx.x; c <= n_clips; c += FB_THREADS)      // clips that end the concatenation (and out_offsets[n_clips])
    if (offs[c] >= T) out_offsets[c] = s_base;
}

// ---- table: one CTA per (clip, keypoint) --------------------------------------------------------------------------
constexpr int FT_THREADS = 256;

struct TableWs {          // per (clip, keypoint) slices of the workspace, T entries each
  double* xs;
  double* ys;
  int* comp;              // cluster id = lowest core index of the component (INT_MAX: not core)
  int* label;             // final label per point (-1 noise)
  int* count;             // members per cluster id
  int* first;             // lowest member index per cluster id
};

__device__ __forceinline__ bool within(double ax, double ay, double bx, double by, double eps2) {
  const double dx = __dsub_rn(ax, bx), dy = __dsub_rn(ay, by);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)) <= eps2;
}

__device__ __forceinline__ TableWs table_ws(double* ws_d, int* ws_i, size_t entry, int T) {     // T entries from `entry` on
  TableWs w;
  w.xs = ws_d + entry * 2;
  w.ys = w.xs + T;
  w.comp = ws_i + entry * 4;
  w.label = w.comp + T;
  w.count = w.label + T;
  w.first = w.count + T;
  return w;
}

// keypoint kp of one clip: a, b = its T x K x 3 detections, o = its (x, y, v) output
__device__ __forceinline__ void table_keypoint(const double* __restrict__ a, const double* __restrict__ b, int T, int K, int kp,
                                               double agree, double eps, int min_samples, int min_points, double visible,
                                               double* __restrict__ o, const TableWs& w) {
  __shared__ int s_warp[FT_THREADS / 32];
  __shared__ int s_n, s_changed, s_best;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  // 1. frames where both detectors see the keypoint and agree (strictly) within `agree` px, in frame order
  for (int t0 = 0; t0 < T; t0 += FT_THREADS) {
    const int t = t0 + threadIdx.x;
    bool keep = false;
    double x = 0, y = 0;
    if (t < T) {
      const double* q1 = a + ((size_t)t * K + kp) * 3;
      const double* q2 = b + ((size_t)t * K + kp) * 3;
      x = q1[0];
      y = q1[1];
      if (q1[2] == visible && q2[2] == visible) {
        const double dx = __dsub_rn(x, q2[0]), dy = __dsub_rn(y, q2[1]);
        keep = sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))) < agree;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = s_n;
    for (int i = 0; i < warp; ++i) before += s_warp[i];
    if (keep) {
      const int p = before + __popc(m & ((1u << lane) - 1u));
      w.xs[p] = x;
      w.ys[p] = y;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int i = 0; i < FT_THREADS / 32; ++i) tot += s_warp[i];
      s_n += tot;
    }
    __syncthreads();
  }
  const int n = s_n;
  if (n < min_points) {                         // "if len(valids_x) < 3" -> invisible
    if (threadIdx.x == 0) o[0] = -1.0, o[1] = -1.0, o[2] = 0.0;
    return;
  }
  const double eps2 = __dmul_rn(eps, eps);
  int best = -2;                                // -2: mean of all points
  if (n >= min_samples) {
    // 2. core points
    for (int i = threadIdx.x; i < n; i += FT_THREADS) {
      const double xi = w.xs[i], yi = w.ys[i];
      int c = 0;
      for (int j = 0; j < n; ++j) c += within(xi, yi, w.xs[j], w.ys[j], eps2) ? 1 : 0;
      w.comp[i] = c >= min_samples ? i : INT_MAX;
      w.count[i] = 0;
      w.first[i] = INT_MAX;
    }
    __syncthreads();
    // 3. connected components of the core graph: min-label propagation with pointer jumping
    for (;;) {
      if (threadIdx.x == 0) s_changed = 0;
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += FT_THREADS) {
        const int ci = w.comp[i];
        if (ci == INT_MAX) continue;
        const double xi = w.xs[i], yi = w.ys[i];
        int m = ci;
        for (int j = 0; j < n; ++j) {
          const int cj = w.comp[j];
          if (cj < m && within(xi, yi, w.xs[j], w.ys[j], eps2)) m = cj;
        }
        const int r = w.comp[m];                // labels only decrease and always name a core point of the same component
        if (r < m) m = r;
        if (m < ci) {
          atomicMin(&w.comp[i], m);
          s_changed = 1;
        }
      }
      __syncthreads();
      const int ch = s_changed;
      __syncthreads();
      if (!ch) break;
    }
    // 4. labels (border points: lowest-numbered adjacent cluster), cluster sizes, first member
    for (int i = threadIdx.x; i < n; i += FT_THREADS) {
      int l = w.comp[i];
      if (l == INT_MAX) {
        const double xi = w.xs[i], yi = w.ys[i];
        for (int j = 0; j < n; ++j) {
          const int cj = w.comp[j];
          if (cj < l && within(xi, yi, w.xs[j], w.ys[j], eps2)) l = cj;
        }
      }
      w.label[i] = l == INT_MAX ? -1 : l;
      if (l != INT_MAX) {
        atomicAdd(&w.count[l], 1);
        atomicMin(&w.first[l], i);
      }
    }
    __syncthreads();
    // 5. largest cluster, ties -> earliest first member (Counter insertion order + max())
    if (threadIdx.x == 0) {
      int bc = 0, bf = INT_MAX, bl = -2;
      for (int l = 0; l < n; ++l) {
        const int c = w.count[l];
        if (c > bc || (c == bc && c > 0 && w.first[l] < bf)) bc = c, bf = w.first[l], bl = l;
      }
      s_best = bl;
    }
    __syncthreads();
    best = s_best;
  }
  // 6. centroid: sequential sums in point order (numpy add.reduce over axis 0), then / count
  if (threadIdx.x == 0) {
    double sx = 0.0, sy = 0.0;
    int c = 0;
    for (int i = 0; i < n; ++i) {
      if (best == -2 || w.label[i] == best) {
        sx = __dadd_rn(sx, w.xs[i]);
        sy = __dadd_rn(sy, w.ys[i]);
        ++c;
      }
    }
    o[0] = sx / (double)c;
    o[1] = sy / (double)c;
    o[2] = visible;
  }
}

__global__ void __launch_bounds__(FT_THREADS) filter_table_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                  int T, int K, double agree, double eps, int min_samples,
                                                                  int min_points, double visible, double* __restrict__ out,
                                                                  double* __restrict__ ws_d, int* __restrict__ ws_i) {
  const int kp = blockIdx.x, clip = blockIdx.y;
  const size_t slice = (size_t)clip * K + kp;
  table_keypoint(p1 + (size_t)clip * T * K * 3, p2 + (size_t)clip * T * K * 3, T, K, kp, agree, eps, min_samples, min_points, visible,
                 out + slice * 3, table_ws(ws_d, ws_i, slice * T, T));
}

// clips of different lengths: clip c holds frames offs[c] .. offs[c+1]-1 of the concatenation; its workspace is the K x T_c entries
// from offs[c] * K on, so the workspace scales with the total frame count
__global__ void __launch_bounds__(FT_THREADS) filter_table_clips_kernel(const double* __restrict__ p1, const double* __restrict__ p2,
                                                                        const int32_t* __restrict__ offs, int K, double agree,
                                                                        double eps, int min_samples, int min_points, double visible,
                                                                        double* __restrict__ out, double* __restrict__ ws_d,
                                                                        int* __restrict__ ws_i) {
  const int kp = blockIdx.x, clip = blockIdx.y;
  const int f0 = offs[clip], T = offs[clip + 1] - f0;
  table_keypoint(p1 + (size_t)f0 * K * 3, p2 + (size_t)f0 * K * 3, T, K, kp, agree, eps, min_samples, min_points, visible,
                 out + ((size_t)clip * K + kp) * 3, table_ws(ws_d, ws_i, (size_t)f0 * K + (size_t)kp * T, T));
}

}  // namespace

extern "C" int ttk_filter_ball(const double* pos1_dev, const double* pos2_dev, int n_frames, double fps, double threshold_px,
                               double* out_xy_dev, int64_t* out_idx_dev, double* out_times_dev, int32_t* out_offsets_dev,
                               void* stream) {
  TTK_CHECK_ARG(n_frames >= 0, "ttk_filter_ball: bad n_frames");
  TTK_CHECK_ARG(out_offsets_dev, "ttk_filter_ball: null pointer");
  TTK_CHECK_ARG(n_frames == 0 || (pos1_dev && pos2_dev && out_xy_dev && out_idx_dev && out_times_dev), "ttk_filter_ball: null pointer");
  filter_ball_kernel<<<1, FB_THREADS, 0, (cudaStream_t)stream>>>(pos1_dev, pos2_dev, n_frames, fps, threshold_px, 1.0, out_xy_dev,
                                                                out_idx_dev, out_times_dev, out_offsets_dev);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" size_t ttk_filter_table_workspace_bytes(int n_clips, int n_frames, int n_keypoints) {
  if (n_clips <= 0 || n_frames <= 0 || n_keypoints <= 0) return 0;
  return (size_t)n_clips * n_keypoints * n_frames * (2 * sizeof(double) + 4 * sizeof(int));
}

extern "C" int ttk_filter_table(const double* pos1_dev, const double* pos2_dev, int n_clips, int n_frames, int n_keypoints,
                                double agree_px, double eps, int min_samples, double* out_dev, void* workspace_dev,
                                size_t workspace_bytes, void* stream) {
  TTK_CHECK_ARG(n_clips >= 0 && n_frames >= 0 && n_keypoints > 0 && n_keypoints <= 65535 && n_clips <= 65535 && min_samples >= 1,
                "ttk_filter_table: bad sizes");
  if (n_clips == 0) return TTK_OK;
  TTK_CHECK_ARG(out_dev, "ttk_filter_table: null pointer");
  TTK_CHECK_ARG(n_frames == 0 || (pos1_dev && pos2_dev && workspace_dev), "ttk_filter_table: null pointer");
  TTK_CHECK_ARG(workspace_bytes >= ttk_filter_table_workspace_bytes(n_clips, n_frames, n_keypoints), "ttk_filter_table: workspace too small");
  double* ws_d = (double*)workspace_dev;
  int* ws_i = (int*)(ws_d + (size_t)n_clips * n_keypoints * n_frames * 2);
  filter_table_kernel<<<dim3(n_keypoints, n_clips), FT_THREADS, 0, (cudaStream_t)stream>>>(
      pos1_dev, pos2_dev, n_frames, n_keypoints, agree_px, eps, min_samples, 3, 1.0, out_dev, ws_d, ws_i);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_filter_ball_clips(const double* pos1_dev, const double* pos2_dev, int n_clips, const int32_t* frame_offsets_dev,
                                     int n_frames, double fps, double threshold_px, double* out_xy_dev, int64_t* out_idx_dev,
                                     double* out_times_dev, int32_t* out_offsets_dev, void* stream) {
  TTK_CHECK_ARG(n_clips >= 0 && n_frames >= 0, "ttk_filter_ball_clips: bad sizes");
  TTK_CHECK_ARG(frame_offsets_dev && out_offsets_dev, "ttk_filter_ball_clips: null pointer");
  TTK_CHECK_ARG(n_frames == 0 || (pos1_dev && pos2_dev && out_xy_dev && out_idx_dev && out_times_dev), "ttk_filter_ball_clips: null pointer");
  filter_ball_clips_kernel<<<1, FB_THREADS, 0, (cudaStream_t)stream>>>(pos1_dev, pos2_dev, frame_offsets_dev, n_clips, n_frames, fps,
                                                                      threshold_px, 1.0, out_xy_dev, out_idx_dev, out_times_dev,
                                                                      out_offsets_dev);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}

extern "C" int ttk_filter_table_clips(const double* pos1_dev, const double* pos2_dev, int n_clips, const int32_t* frame_offsets_dev,
                                      int n_frames, int n_keypoints, double agree_px, double eps, int min_samples, double* out_dev,
                                      void* workspace_dev, size_t workspace_bytes, void* stream) {
  TTK_CHECK_ARG(n_clips >= 0 && n_frames >= 0 && n_keypoints > 0 && n_keypoints <= 65535 && n_clips <= 65535 && min_samples >= 1,
                "ttk_filter_table_clips: bad sizes");
  if (n_clips == 0) return TTK_OK;
  TTK_CHECK_ARG(out_dev && frame_offsets_dev, "ttk_filter_table_clips: null pointer");
  TTK_CHECK_ARG(n_frames == 0 || (pos1_dev && pos2_dev && workspace_dev), "ttk_filter_table_clips: null pointer");
  TTK_CHECK_ARG(workspace_bytes >= ttk_filter_table_workspace_bytes(1, n_frames, n_keypoints), "ttk_filter_table_clips: workspace too small");
  double* ws_d = (double*)workspace_dev;
  int* ws_i = (int*)(ws_d + (size_t)n_keypoints * n_frames * 2);
  filter_table_clips_kernel<<<dim3(n_keypoints, n_clips), FT_THREADS, 0, (cudaStream_t)stream>>>(
      pos1_dev, pos2_dev, frame_offsets_dev, n_keypoints, agree_px, eps, min_samples, 3, 1.0, out_dev, ws_d, ws_i);
  TTK_LAUNCH_CHECK();
  return TTK_OK;
}
