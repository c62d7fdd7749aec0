/* libttk -- B200 (sm_100a) kernels for the UpliftingTableTennis inference hot path.
 *
 * C ABI.  The reference (KieDani/UpliftingTableTennis) is pure Python/PyTorch and has no
 * FFI of its own (SURVEY.md section 8b); each entry point below therefore replaces one
 * Python call seam of the reference and cites it.  Host code (Python, ctypes) owns every
 * activation/input/output buffer and passes raw device pointers plus the CUDA stream to
 * launch on; the library never synchronises the device and never allocates on the forward
 * path.  Handles own only their pre-packed weights.
 *
 * Conventions
 *   - return value: 0 = ok, negative = error; ttk_last_error() gives the message of the last
 *     failing call on the calling thread.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - pointers named *_dev are device pointers, *_host host pointers.
 *   - activations are NHWC ("pixels x channels"), C padded to a multiple of 16.
 */
#ifndef TTK_H
#define TTK_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTK_VERSION 100          /* 0.1.0 */
#define TTK_API __attribute__((visibility("default")))

enum { TTK_OK = 0, TTK_ERR_ARG = -1, TTK_ERR_CUDA = -2, TTK_ERR_STATE = -3, TTK_ERR_UNSUPPORTED = -4 };
/* Arithmetic / storage type of a path.  TTK_TF32: fp32 storage, tensor-core products with TF32 operands (inputs rounded to
 * nearest-even TF32 by TMA, fp32 accumulate) -- the class cuDNN uses for the reference's convolutions on a GPU.
 * TTK_TF32X3 (uplifting transformer, ViTPose, HRNet): fp32 storage, every product as three TF32 tensor-core products of split operands
 * (a_hi b_hi + a_lo b_hi + a_hi b_lo) -- fp32-level results, the class of the reference's fp32 Linear layers.
 * TTK_F16 (HRNet and pre-processing only): IEEE fp16 storage and tensor-core operands, fp32 accumulate -- the tiles and kernels of
 * TTK_BF16 with 10 mantissa bits instead of 7, the class of torch.autocast('cuda') / model.half().  Its range is +-65504: an activation
 * past it becomes inf, as under autocast; the library does not rescale. */
enum { TTK_F32 = 0, TTK_BF16 = 1, TTK_TF32 = 2, TTK_TF32X3 = 3, TTK_F16 = 4 };
enum { TTK_DECODE_TABLE = 0, TTK_DECODE_BALL = 1 }; /* the two live sub-pixel variants */
enum { TTK_LAYOUT_NCHW_F32 = 0, TTK_LAYOUT_NHWC16 = 1 };

TTK_API int ttk_version(void);
TTK_API const char* ttk_last_error(void);
/* Host helper of the plugin side (interface.py: numpy frames -> pinned staging ring): memcpy with non-temporal stores. */
TTK_API int ttk_host_copy_stream(void* dst, const void* src, size_t bytes);
/* Host threads waiting for `device` sleep instead of spin (cudaDeviceScheduleBlockingSync; process-global for that device): for hosts
 * that run one rank per GPU with few cores per GPU.  old_flags (may be NULL) receives the previous device flags. */
TTK_API int ttk_host_blocking_sync(int device, unsigned* old_flags);
/* 1 when a CUDA device with compute capability 10.x is present, else 0 (never raises). */
TTK_API int ttk_device_ok(void);

/* ---------------------------------------------------------------------------------------
 * Frame pre-processing: cv2.resize (uint8, INTER_LINEAR, bit exact) + ImageNet normalise
 * (3x256 LUT) + stack [prev, cur, next] + HWC->CHW.
 * Replaces balldetection/transforms.py:17-52 (Resize), :379-402 (NormalizeImage) and
 * interface.py:110-112 (concat / rearrange / astype / H2D); tabledetection/transforms.py:9-40.
 *
 * frames_dev : n_frames x src_h x src_w x 3 uint8 (HWC, channel order as stored: BGR from the
 *              hub API).  Stack s reads frames s*stack_stride + {0..frames_per_stack-1}.
 * lut_dev    : 3 x 256 float32, lut[c][v] = float32((v/255 - mean[c]) / std[c]) (host float64).
 * out_dev    : layout NCHW_F32: n_stacks x (3*fps) x dst_h x dst_w float32 (the reference tensor)
 *              layout NHWC16  : n_stacks x dst_h x dst_w x 16, dtype f32, bf16 or f16 (the float32
 *              value rounded to nearest-even), channels 3*fps..15 zero -- the detector input.
 */
TTK_API int ttk_preprocess_stacks(const uint8_t* frames_dev, int n_frames, int src_h, int src_w,
                          int frames_per_stack, int stack_stride, int n_stacks,
                          int dst_h, int dst_w, const float* lut_dev,
                          void* out_dev, int layout, int dtype, void* stream);
/* The same output, with stack s reading frames first_frame_dev[s] + {0..frames_per_stack-1} (int32, device): stacks of several clips
 * in one pass, no window crossing a clip.  Bytes are identical to ttk_preprocess_stacks for the same frames.  The caller guarantees
 * 0 <= first_frame_dev[s] <= n_frames - frames_per_stack (the table is device memory and is not read on the host). */
TTK_API int ttk_preprocess_stacks_indexed(const uint8_t* frames_dev, int n_frames, int src_h, int src_w,
                          int frames_per_stack, const int32_t* first_frame_dev, int n_stacks,
                          int dst_h, int dst_w, const float* lut_dev,
                          void* out_dev, int layout, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------
 * HRNet-W18-small heatmap network (WASB ball detector / HRNet table detector).
 * Replaces WASBNet.forward (balldetection/models/wasb.py:596-608), HRNet.forward (:445-486)
 * and MyHRNet.forward (tabledetection/models/hrnet.py:588-590); weights come from the
 * reference checkpoint through load_model (inference/inference_balldetection.py:40-61).
 */
typedef struct ttk_hrnet ttk_hrnet;

/* in_ch: 9 (WASB, 3 stacked frames) or 3 (table); out_ch: 3 or 13 = channels of the final
 * 1x1 conv; out_first/out_count: the slice of them that is materialised (WASB returns
 * channel 1 only: out_first=1, out_count=1). */
TTK_API int ttk_hrnet_create(int in_ch, int out_ch, int out_first, int out_count, ttk_hrnet** out);
TTK_API void ttk_hrnet_destroy(ttk_hrnet* h);
TTK_API int ttk_hrnet_num_convs(const ttk_hrnet* h);
/* name: state-dict key of the conv weight without ".weight"; bn: state-dict prefix of its
 * batch norm ("" = none, the conv has a bias).  Buffers must hold 128 chars. */
TTK_API int ttk_hrnet_conv_info(const ttk_hrnet* h, int i, char* name, char* bn, int* cin, int* cout,
                        int* k, int* stride);
/* BN-folded weights of conv i: w_host[cout][cin][k][k] float32, b_host[cout] float32.
 * The library re-packs them for both arithmetic paths and uploads them. */
TTK_API int ttk_hrnet_set_conv(ttk_hrnet* h, int i, const float* w_host, const float* b_host);
TTK_API size_t ttk_hrnet_workspace_bytes(const ttk_hrnet* h, int batch, int height, int width, int dtype);
/* x_dev: batch x H x W x 16 (NHWC16, dtype); heatmaps_dev: batch x out_count x H x W float32.
 * H and W must be multiples of 8.  dtype TTK_F32: fp32 SIMT path (parity with the CPU
 * reference at 1e-4); TTK_TF32: x and the activations are float32, the convolutions run on the
 * tcgen05 tensor cores with TF32 operands (the reference-on-GPU class, balldetection/models/wasb.py:29-105
 * through cuDNN's default TF32); TTK_TF32X3: float32 tensors as for TTK_TF32, every product as three TF32 tensor-core products of
 * split operands (fp32-level results: the reference on a CPU, or on a GPU with cudnn.allow_tf32 off; no fused BasicBlock or bottleneck
 * kernels); TTK_BF16: tcgen05 path with bf16 storage, fp32 accumulate; TTK_F16: the same kernels with fp16 storage and operands (x and
 * every activation fp16, heatmaps float32).  A convolution without a tensor-core kernel for its shape runs on the SIMT kernel of the same
 * storage type. */
TTK_API int ttk_hrnet_forward(ttk_hrnet* h, const void* x_dev, int batch, int height, int width, int dtype,
                      float* heatmaps_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* kernels launched by the last ttk_hrnet_forward on this handle (for bench accounting) */
TTK_API int ttk_hrnet_last_launches(const ttk_hrnet* h);
/* Images processed per pass through the layer plan (default 16; measured 760 / 877 / 962 / 1002 frames/s at
 * 2 / 4 / 8 / 16: per-launch fixed costs outweigh L2 residency of thin layers).  Bounds the activation workspace. */
TTK_API int ttk_hrnet_set_subbatch(ttk_hrnet* h, int images);
/* Measurement aid (bench.py): when enabled, ttk_hrnet_forward brackets every kernel launch with CUDA
 * events on `stream`.  After the caller synchronised the stream, ttk_hrnet_profile_read returns, per
 * launch: op type (0 conv, 1 fuse-sum, 2 final conv, 3 conv of a tensor-core path that ran on the SIMT kernel because its shape has
 * no tensor-core kernel), conv index (-1 if none), duration in ms,
 * algorithmic flops (2*MAC on the reference's logical channel counts) and compulsory bytes
 * (inputs + outputs + weights once). */
TTK_API int ttk_hrnet_set_force_simt(ttk_hrnet* h, int enable);   /* tensor-core paths through the SIMT kernels of their storage type (cross-check) */
/* Test hook: run one convolution of the plan on caller buffers (NHWC, channels padded to 16): out = act(conv(in) + bias [+ res]).
 * path 0: fp32 SIMT (float32 tensors), 1: bf16 SIMT, 2: bf16 tcgen05, 3: TF32 tcgen05 on float32 tensors, 4: 3xTF32 tcgen05 on
 * float32 tensors (2 to 4 return TTK_ERR_UNSUPPORTED when the shape has no tensor-core kernel; any other path is TTK_ERR_ARG). */
TTK_API int ttk_hrnet_debug_conv(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, const void* res_dev,
                         int relu, int path, void* out_dev, void* stream);
/* Test hook: the same on fp16 tensors (fp16-rounded weights): simt 1 = fp16 SIMT kernel, 0 = fp16 tcgen05 kernel
 * (TTK_ERR_UNSUPPORTED when the shape has none). */
TTK_API int ttk_hrnet_debug_conv_f16(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, const void* res_dev,
                             int relu, int simt, void* out_dev, void* stream);
/* Test hook: one BasicBlock (convs conv_index and conv_index + 1, 16 or 32 padded channels) through the fused tcgen05 kernel:
 * out = relu(conv2(relu(conv1(in))) + in), NHWC bf16.  ttk_hrnet_set_block_fusion: 0 runs the blocks conv by conv (A/B, cross-check),
 * 1 (default) fuses the bf16 blocks of the 16- and 32-channel branches, 2 / 3 also the TF32 16-channel blocks (two 3-row tiles in flight
 * with the fp32 residual from global memory / one 4-row tile with the residual from the staged tile; measured no faster than conv by
 * conv, DESIGN.md 4.2). */
TTK_API int ttk_hrnet_debug_block(ttk_hrnet* h, int conv_index, const void* in_dev, int n, int hin, int win, void* out_dev, void* stream);
TTK_API int ttk_hrnet_set_block_fusion(ttk_hrnet* h, int enable);
TTK_API int ttk_hrnet_set_profile(ttk_hrnet* h, int enable);
TTK_API int ttk_hrnet_profile_count(const ttk_hrnet* h);
TTK_API int ttk_hrnet_profile_read(ttk_hrnet* h, int i, int* op_type, int* conv_index, float* ms, double* flops, double* bytes);

/* ---------------------------------------------------------------------------------------
 * ViTPose-small heatmap detector (SURVEY.md section 8 row a4' / 8f row 4): ViT backbone
 * (patch 16, dim 384, depth 12, 12 heads) + two transposed convolutions + 1x1 conv.
 * Replaces VitPose.forward (balldetection/models/vitpose.py:92-103, tabledetection/models/vitpose.py),
 * ViT.forward (vit_pose/vit_models/backbone/vit.py:375-389) and TopdownHeatmapSimpleHead.forward
 * (vit_pose/vit_models/head/topdown_heatmap_simple_head.py:188-193); weights from load_model
 * (inference/inference_balldetection.py:40-61).
 */
typedef struct ttk_vit ttk_vit;
/* in_ch 9 (ball: 3 stacked frames) or 3 (table); out_ch 1 or 13; height x width: the fixed input
 * resolution (the position embedding is tied to it: 640 x 1152 for balldetection/config.py:82-83). */
TTK_API int ttk_vit_create(int in_ch, int out_ch, int height, int width, ttk_vit** out);
TTK_API void ttk_vit_destroy(ttk_vit* h);
TTK_API int ttk_vit_num_params(const ttk_vit* h);
/* name: state-dict key of the reference module; numel: element count (row-major, as stored by torch). */
TTK_API int ttk_vit_param_info(const ttk_vit* h, int i, char* name, int* numel);
TTK_API int ttk_vit_set_param(ttk_vit* h, int i, const float* data_host, int numel);
/* returns the token count; hp/wp (may be NULL) receive the token grid.  Heatmaps are 4hp x 4wp. */
TTK_API int ttk_vit_tokens(const ttk_vit* h, int* hp, int* wp);
TTK_API int ttk_vit_set_subbatch(ttk_vit* h, int images);
TTK_API size_t ttk_vit_workspace_bytes(const ttk_vit* h, int batch, int dtype);
/* x_dev: batch x in_ch x height x width float32 (NCHW, the reference's input tensor);
 * heatmaps_dev: batch x out_ch x 4hp x 4wp float32.  dtype TTK_TF32X3: float32 tensors, every product as three
 * TF32 tensor-core products of split operands (float32-class results: the arithmetic class of the reference's
 * Linear layers and attention); TTK_F32: float32 SIMT kernels (strict parity with the CPU reference);
 * TTK_BF16: bf16 operands on tcgen05 tensor cores, float32 accumulate/residual. */
TTK_API int ttk_vit_forward(ttk_vit* h, const float* x_dev, int batch, int dtype, float* heatmaps_dev,
                    void* workspace_dev, size_t workspace_bytes, void* stream);
TTK_API int ttk_vit_last_launches(const ttk_vit* h);
/* Test hooks: the detector's two building blocks on caller buffers (dtype TTK_F32: float32 SIMT kernels, TTK_BF16: tcgen05,
 * TTK_TF32X3: tcgen05 with split float32 operands -- A, W, qkv (and C when c_bf16 == 2, and out) are then pairs of float32
 * planes [2][rows][cols]: plane 0 = tf32(x), plane 1 = x - plane 0).
 * GEMM: C[m][n] = act(sum_k A[m][k] W[n][k] + bias[n]) (+ R[m][n]); act 0 none, 1 GELU (erf), 2 ReLU; A, W in `dtype`;
 * C bf16 when c_bf16 else float32; up_w > 0 scatters row (img, y, x) of an up_h x up_w grid to (img, 2y+py, 2x+px) of the 2x grid.
 * Attention: qkv [images*tokens][1152] in `dtype` -> out [images*tokens][384] (12 heads of 32), scratch for the bf16 path. */
TTK_API int ttk_vit_debug_gemm(const void* a_dev, const void* w_dev, const float* bias_dev, const float* res_dev, void* c_dev, int m, int n,
                       int k, int act, int c_bf16, int up_h, int up_w, int py, int px, int dtype, void* stream);
TTK_API int ttk_vit_debug_attention(const void* qkv_dev, void* out_dev, void* scratch_dev, size_t scratch_bytes, int images, int tokens,
                            int dtype, void* stream);

/* ---------------------------------------------------------------------------------------
 * Heatmap decode: first-max argmax + 3x3 zero-padded window + bounded Gaussian fit +
 * heatmap->image rescale.  Replaces extract_position_torch_gaussian,
 * tabledetection/helper_tabledetection.py:50-156 (variant TABLE; interface.py:116,169) and
 * balldetection/helper_balldetection.py:29-110 (variant BALL; inference/utils.py:59).
 *
 * heatmaps_dev : n_maps x H x W float32 (any (B,C) flattening)
 * out_xyv_dev  : n_maps x 3 float64  [x_img, y_img, 1.0]
 * out_idx_dev  : n_maps int32 flat argmax index            (may be NULL)
 * out_win_dev  : n_maps x 9 float32 window, row major      (may be NULL)
 * workspace    : ttk_decode_workspace_bytes(n_maps, H, W)
 */
TTK_API size_t ttk_decode_workspace_bytes(int n_maps, int height, int width);
TTK_API int ttk_heatmap_decode(const float* heatmaps_dev, int n_maps, int height, int width, int variant,
                       int image_width, int image_height, double* out_xyv_dev, int32_t* out_idx_dev,
                       float* out_win_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* Measurement aid (bench.py): with profiling on, ttk_heatmap_decode brackets its two kernels with CUDA events on `stream`;
 * after the caller synchronised the stream, ttk_decode_profile_read returns the durations in ms of the argmax pass (the
 * HBM-bound kernel: one read of every heatmap value) and of the per-map fit.  Process-wide state: not for concurrent callers. */
TTK_API int ttk_decode_set_profile(int enable);
TTK_API int ttk_decode_profile_read(float* argmax_ms, float* fit_ms);

/* ---------------------------------------------------------------------------------------
 * Trajectory filters between decode and uplift (device versions, SURVEY.md section 8f row 2).
 *
 * ttk_filter_ball replaces filter_trajectory_ball (inference/utils.py:70-102): keep frame t when both
 * detectors report the ball visible (== 1) and their positions differ by at most threshold_px
 * (NaN distances are kept, like `diff > 20` in the reference).  pos*_dev: n_frames x 3 float64 (x, y, v).
 * Outputs are compacted in frame order: out_xy n x 2 float64, out_idx n int64, out_times n float64
 * (= t / fps); capacity n_frames each.  out_offsets_dev[2] int32 = {0, n}: the prefix-sum format
 * ttk_trajectory_pack consumes, so the count never has to visit the host.
 */
TTK_API int ttk_filter_ball(const double* pos1_dev, const double* pos2_dev, int n_frames, double fps, double threshold_px,
                    double* out_xy_dev, int64_t* out_idx_dev, double* out_times_dev, int32_t* out_offsets_dev,
                    void* stream);
/* ttk_filter_ball over n_clips clips in one launch.  pos*_dev: the clips' n_frames x 3 detections concatenated;
 * frame_offsets_dev[n_clips+1] int32 (device): clip c is frames [offs[c], offs[c+1]), offs[0] = 0, non-decreasing, offs[n_clips] =
 * n_frames (empty clips allowed).  Each clip is filtered exactly like ttk_filter_ball: out_idx and out_times (= idx / fps) count from
 * the clip's first frame.  The kept rows are packed in clip order; out_offsets_dev[n_clips+1] receives the per-clip prefix sums on the
 * device, in the format ttk_trajectory_pack reads.  Capacity n_frames rows per output. */
TTK_API int ttk_filter_ball_clips(const double* pos1_dev, const double* pos2_dev, int n_clips, const int32_t* frame_offsets_dev,
                    int n_frames, double fps, double threshold_px, double* out_xy_dev, int64_t* out_idx_dev,
                    double* out_times_dev, int32_t* out_offsets_dev, void* stream);

/* ttk_filter_table replaces filter_trajectory_table (inference/utils.py:137-169) and
 * _filter_keypoints_with_dbscan (:172-232; scikit-learn DBSCAN semantics, see csrc/filters.cu):
 * per keypoint, frames where both detectors see it and agree within (<) agree_px are clustered with
 * DBSCAN(eps, min_samples); the centroid of the largest cluster is returned as (x, y, 1), or
 * (-1, -1, 0) when fewer than 3 frames qualify.  pos*_dev: n_clips x n_frames x n_keypoints x 3
 * float64; out_dev: n_clips x n_keypoints x 3 float64.  The reference calls it with
 * agree_px = 10, eps = 10, min_samples = 3.
 */
TTK_API size_t ttk_filter_table_workspace_bytes(int n_clips, int n_frames, int n_keypoints);
TTK_API int ttk_filter_table(const double* pos1_dev, const double* pos2_dev, int n_clips, int n_frames, int n_keypoints,
                     double agree_px, double eps, int min_samples, double* out_dev, void* workspace_dev,
                     size_t workspace_bytes, void* stream);
/* ttk_filter_table over n_clips clips of different lengths: pos*_dev hold the clips' frames concatenated (n_frames x n_keypoints x 3),
 * frame_offsets_dev as for ttk_filter_ball_clips.  out_dev: n_clips x n_keypoints x 3, each clip bit-identical to ttk_filter_table on
 * that clip alone.  workspace: ttk_filter_table_workspace_bytes(1, n_frames, n_keypoints). */
TTK_API int ttk_filter_table_clips(const double* pos1_dev, const double* pos2_dev, int n_clips, const int32_t* frame_offsets_dev,
                     int n_frames, int n_keypoints, double agree_px, double eps, int min_samples, double* out_dev,
                     void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Trajectory packing: pixel -> [0,1] normalisation, pad/crop to seq_len, mask.
 * Replaces _uplifting_transform (inference/utils.py:268-309), batched over clips.
 * ball_xy_dev: sum(lengths) x 2 float64 (concatenated clips), times_dev: sum(lengths) float64,
 * offsets_dev: n_clips+1 int32 prefix sums, table_dev: n_clips x 13 x 3 float64.
 * Outputs float32: ball n x seq x 2, table n x 13 x 3, times n x seq, mask n x seq.
 */
TTK_API int ttk_trajectory_pack(const double* ball_xy_dev, const double* times_dev, const int32_t* offsets_dev,
                        const double* table_dev, int n_clips, int seq_len, double img_w, double img_h,
                        float* ball_out, float* table_out, float* times_out, float* mask_out, void* stream);

/* ---------------------------------------------------------------------------------------
 * Camera calibration from the 13 table keypoints (SURVEY.md section 8f row 3).
 * Replaces calibrate_camera (inference/utils.py:312-329) = calc_cameramatrices(use_ransac=True)
 * (dataprocessing/regress_cameramatrices.py:119-231) with the DLT start of dataprocessing/my_dlt.py:
 * DLT on the visible keypoints, n_hypotheses BFGS fits of (fx, fy, t, euler xyz) on keys 10, 11 + the
 * sampled keys, inlier count at inlier_threshold_px, refit on the inliers of the first best hypothesis.
 * The optimiser is SciPy's BFGS restated (csrc/calib.h).
 *
 * keypoints_dev    : n_clips x 13 x 3 float64 (x, y, v); v == 1 marks a visible keypoint (>= 6 needed)
 * world_points_dev : 13 x 3 float64 table model (uplifting/helper.py:36-50)
 * samples_dev      : n_clips x n_hypotheses x n_sample int32, 1-based keypoint ids per hypothesis --
 *                    the reference draws them with numpy's Generator(42).choice (:138-143), the host
 *                    computes the same table
 * mint_out_dev     : n_clips x 3 x 4, mext_out_dev: n_clips x 4 x 4 float64 (what the reference returns)
 * info_out_dev     : n_clips x 4 int32: inlier count, best hypothesis, BFGS status of the refit
 *                    (0 converged, 1 maxiter, 2 precision loss, 3 nan), DLT ok
 */
TTK_API size_t ttk_calibrate_workspace_bytes(int n_clips, int n_hypotheses);
TTK_API int ttk_calibrate_camera(const double* keypoints_dev, const double* world_points_dev, const int32_t* samples_dev,
                         int n_clips, int n_hypotheses, int n_sample, int image_width, int image_height,
                         double inlier_threshold_px, double* mint_out_dev, double* mext_out_dev, int32_t* info_out_dev,
                         void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Uplifting transformer (MultiStageModel 'multistage' / 'connectstage', size 'large',
 * tabletoken_mode 'dynamic', time_rotation 'new').
 * Replaces MultiStageModel.forward (uplifting/model.py:529-571) incl. FirstStage (:335-390),
 * SimpleStaticLayer (:278-300), rotary attention (:186-229, :56-102), embeddings, heads; weights
 * from inference/inference_uplifting.py:33-58.
 */
typedef struct ttk_uplift ttk_uplift;
TTK_API int ttk_uplift_create(int dim, int heads, int depth, int use_skipconnection, ttk_uplift** out);
TTK_API void ttk_uplift_destroy(ttk_uplift* h);
TTK_API int ttk_uplift_num_params(const ttk_uplift* h);
/* name: state-dict key; numel: element count (row-major, as stored by torch). */
TTK_API int ttk_uplift_param_info(const ttk_uplift* h, int i, char* name, int* numel);
TTK_API int ttk_uplift_set_param(ttk_uplift* h, int i, const float* data_host, int numel);
TTK_API size_t ttk_uplift_workspace_bytes(const ttk_uplift* h, int batch, int seq_len, int dtype);
/* ball B x T x 2, table B x 13 x 3 (x, y, visibility), mask B x T, times B x T (s);
 * rot_out B x 3 (global axes), pos_out B x T x 3.  All float32 device pointers.  seq_len in [2, 63].
 * mask_additive 0: mask in {0, 1} (0 = padding, never attended); 1: mask holds the additive values themselves ({-1e9, 0}), which
 * the reference keeps as they are (model.py:541-546): a padded query row then attends uniformly over the valid keys.
 * The caller validates the mask (the reference raises ValueError on an all-ones mask). */
TTK_API int ttk_uplift_forward(ttk_uplift* h, const float* ball_dev, const float* table_dev, const float* mask_dev,
                       const float* times_dev, int batch, int seq_len, int mask_additive, int dtype, float* rot_out_dev,
                       float* pos_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* kernels launched by the last ttk_uplift_forward on this handle (0 when it failed its argument checks) */
TTK_API int ttk_uplift_last_launches(const ttk_uplift* h);
/* Test hooks: the two kernels of the tf32x3 path on caller buffers.
 * GEMM (one-to-one with the library's Gemm3Args): c[m][n] = act(A' W^T + bias) (+ res), K = 128, n a multiple of 128, W = w_hi + w_lo
 * with w_hi = tf32(W) rounded to nearest, ties away; A' = LayerNorm(a) with the given float32 (mean, rstd) rows, gamma and beta when
 * ln_stats is not NULL; res may alias c; out_stats [m][2] receives mean / rstd (eps 1e-5) of c's rows (n = 128 only, else
 * TTK_ERR_UNSUPPORTED).
 * Attention: mode 0 table-token stage (batch * seq_len sequences of 14 rows; first_only: only token 0 is a query and o has one row per
 * sequence), 1 temporal stage (batch sequences of seq_len rows), 2 second stage (batch sequences of seq_len + 1 rows, token 0 the cls
 * token); qkv [rows][384] with bias, o [rows][128]; table, mask, times, mask_additive as for ttk_uplift_forward; inv_freq [16]. */
TTK_API int ttk_uplift_debug_gemm3(const float* a_dev, const float* w_hi_dev, const float* w_lo_dev, const float* bias_dev,
                           const float* res_dev, float* c_dev, int m, int n, int relu, const float* ln_stats_dev,
                           const float* ln_gamma_dev, const float* ln_beta_dev, float* out_stats_dev, void* stream);
TTK_API int ttk_uplift_debug_attention3(int mode, int first_only, const float* qkv_dev, float* o_dev, const float* table_dev,
                                const float* mask_dev, const float* times_dev, const float* inv_freq_dev, int batch, int seq_len,
                                int mask_additive, void* stream);

/* Spin global -> local axes.  Replaces transform_rotationaxes (uplifting/helper.py:394-420).
 * rot B x 3, pos B x T x 3 -> out B x 3, float32. */
TTK_API int ttk_rotation_local(const float* rot_dev, const float* pos_dev, int batch, int seq_len,
                       float* out_dev, void* stream);

/* Camera projection cam2img(world2cam(p)).  Replaces uplifting/helper.py:137-204 and
 * TableTennisPipeline.reproject (interface.py:301-312).  points n x 3, mext 4x4 row major,
 * mint 3x3 row major (the leading 3x3 of Mint), out n x 2.  dtype_f64 != 0: float64 (the numpy
 * path of the reference), else float32 (its torch path). */
TTK_API int ttk_project(const void* points_dev, const void* mext_dev, const void* mint_dev, int n,
                int dtype_f64, void* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TTK_H */
