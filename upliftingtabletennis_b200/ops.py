"""Python-side wrappers of the stateless libttk entry points (include/ttk.h).  Device memory,
streams and tensors are torch's; arithmetic happens in the CUDA library only."""
import numpy as np
import torch

from . import _lib
from ._lib import lib, check, ptr, stream_ptr

MEAN = (0.485, 0.456, 0.406)     # balldetection/transforms.py:507
STD = (0.229, 0.224, 0.225)
_lut_cache = {}


def normalize_lut(device):
    """3x256 float32 table of float32((v/255 - mean[c]) / std[c]), computed in float64 on the host
    exactly as NormalizeImage does per pixel (balldetection/transforms.py:388-390)."""
    key = str(device)
    if key not in _lut_cache:
        v = np.arange(256, dtype=np.float64) / 255.0
        lut = np.stack([(v - MEAN[c]) / STD[c] for c in range(3)]).astype(np.float32)
        _lut_cache[key] = torch.from_numpy(lut).to(device)
    return _lut_cache[key]


def preprocess_stacks(frames, frames_per_stack, stack_stride, n_stacks, dst_w, dst_h, layout='nhwc16', dtype=torch.float32,
                      out=None):
    """frames: (n, H, W, 3) uint8 CUDA tensor.  Returns (n_stacks, 3*fps, h, w) float32 for layout
    'nchw' (the reference's tensor, interface.py:110-112) or (n_stacks, h, w, 16) for 'nhwc16'."""
    _lib.require_device()
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    frames = frames.contiguous()
    n, sh, sw, _ = frames.shape
    if layout == 'nchw':
        assert dtype == torch.float32
        shape, lay = (n_stacks, 3 * frames_per_stack, dst_h, dst_w), _lib.LAYOUT_NCHW_F32
    else:
        shape, lay = (n_stacks, dst_h, dst_w, 16), _lib.LAYOUT_NHWC16
    dts = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
    if dtype not in dts:
        raise ValueError('preprocess_stacks: dtype must be torch.float32, torch.bfloat16 or torch.float16, got %r' % (dtype,))
    if out is None:
        out = torch.empty(shape, dtype=dtype, device=frames.device)
    assert tuple(out.shape) == shape and out.dtype == dtype and out.is_contiguous()
    dt = dts[dtype]
    check(lib.ttk_preprocess_stacks(ptr(frames), n, sh, sw, frames_per_stack, stack_stride, n_stacks, dst_h, dst_w,
                                    ptr(normalize_lut(frames.device)), ptr(out), lay, dt, stream_ptr()))
    return out


def preprocess_stacks_indexed(frames, frames_per_stack, first_frame, dst_w, dst_h, layout='nhwc16', dtype=torch.float32):
    """preprocess_stacks with stack s reading frames first_frame[s] + {0..frames_per_stack-1}: first_frame is an (n_stacks,) int32
    CUDA tensor whose entries the caller has checked against len(frames) (it is not read on the host).  Same bytes per stack."""
    _lib.require_device()
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 3
    assert first_frame.is_cuda and first_frame.dtype == torch.int32 and first_frame.dim() == 1
    frames, first_frame = frames.contiguous(), first_frame.contiguous()
    n, sh, sw, _ = frames.shape
    n_stacks = first_frame.shape[0]
    if layout == 'nchw':
        assert dtype == torch.float32
        shape, lay = (n_stacks, 3 * frames_per_stack, dst_h, dst_w), _lib.LAYOUT_NCHW_F32
    else:
        shape, lay = (n_stacks, dst_h, dst_w, 16), _lib.LAYOUT_NHWC16
    dts = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}
    if dtype not in dts:
        raise ValueError('preprocess_stacks_indexed: dtype must be torch.float32, torch.bfloat16 or torch.float16, got %r' % (dtype,))
    out = torch.empty(shape, dtype=dtype, device=frames.device)
    check(lib.ttk_preprocess_stacks_indexed(ptr(frames), n, sh, sw, frames_per_stack, ptr(first_frame), n_stacks, dst_h, dst_w,
                                            ptr(normalize_lut(frames.device)), ptr(out), lay, dts[dtype], stream_ptr()))
    return out


def decode_heatmaps(heatmaps, image_width, image_height, variant='table', return_debug=False):
    """heatmaps: (..., H, W) float32 CUDA tensor -> (..., 3) float64 CUDA tensor [x_img, y_img, 1].
    variant 'table': tabledetection/helper_tabledetection.py:50-156; 'ball': balldetection/helper_balldetection.py:29-110."""
    _lib.require_device()
    assert heatmaps.is_cuda and heatmaps.dtype == torch.float32 and heatmaps.dim() >= 2
    hm = heatmaps.contiguous()
    H, W = hm.shape[-2:]
    lead = hm.shape[:-2]
    n = int(np.prod(lead)) if len(lead) else 1
    out = torch.empty((n, 3), dtype=torch.float64, device=hm.device)
    idx = torch.empty((n,), dtype=torch.int32, device=hm.device)
    win = torch.empty((n, 9), dtype=torch.float32, device=hm.device)
    v = {'table': _lib.DECODE_TABLE, 'ball': _lib.DECODE_BALL}[variant]
    for b0 in range(0, n, 65535):
        nb = min(65535, n - b0)
        ws_bytes = lib.ttk_decode_workspace_bytes(nb, H, W)
        ws = torch.empty((max(ws_bytes, 8),), dtype=torch.uint8, device=hm.device)
        check(lib.ttk_heatmap_decode(ptr(hm.view(n, H, W)[b0:b0 + nb]), nb, H, W, v, int(image_width), int(image_height),
                                     ptr(out[b0:b0 + nb]), ptr(idx[b0:b0 + nb]), ptr(win[b0:b0 + nb]), ptr(ws), ws_bytes,
                                     stream_ptr()))
    out = out.view(*lead, 3)
    if return_debug:
        return out, idx.view(*lead), win.view(*lead, 3, 3)
    return out


def trajectory_pack(ball_xy, times, offsets, table, seq_len=50, img_w=1920.0, img_h=1080.0):
    """Batched _uplifting_transform (inference/utils.py:268-309).  ball_xy (sum T', 2) f64, times (sum T',) f64,
    offsets (n+1,) int32 prefix sums, table (n, 13, 3) f64 -- all CUDA.  Returns float32 ball, table, times, mask."""
    _lib.require_device()
    n = table.shape[0]
    dev = table.device
    ball_o = torch.empty((n, seq_len, 2), dtype=torch.float32, device=dev)
    table_o = torch.empty((n, 13, 3), dtype=torch.float32, device=dev)
    times_o = torch.empty((n, seq_len), dtype=torch.float32, device=dev)
    mask_o = torch.empty((n, seq_len), dtype=torch.float32, device=dev)
    ball_xy, times, offsets, table = ball_xy.contiguous(), times.contiguous(), offsets.contiguous(), table.contiguous()     # held until the call returns
    check(lib.ttk_trajectory_pack(ptr(ball_xy), ptr(times), ptr(offsets), ptr(table), n, seq_len, float(img_w), float(img_h), ptr(ball_o),
                                  ptr(table_o), ptr(times_o), ptr(mask_o), stream_ptr()))
    return ball_o, table_o, times_o, mask_o


def rotation_local(rot, pos):
    """transform_rotationaxes (uplifting/helper.py:394-420): rot (B,3), pos (B,T,3) float32 CUDA -> (B,3)."""
    _lib.require_device()
    rot, pos = rot.contiguous(), pos.contiguous()
    out = torch.empty_like(rot)
    check(lib.ttk_rotation_local(ptr(rot), ptr(pos), rot.shape[0], pos.shape[1], ptr(out), stream_ptr()))
    return out


def project(points, mext, mint):
    """cam2img(world2cam(points, Mext), Mint) (uplifting/helper.py:137-204).  points (N,3), Mext (4,4), Mint (3,3|3,4);
    float64 or float32 CUDA tensors -> (N,2)."""
    _lib.require_device()
    f64 = points.dtype == torch.float64
    dt = points.dtype
    pts = points.contiguous()
    me = mext.to(dt).contiguous()
    mi = mint[:3, :3].to(dt).contiguous()
    out = torch.empty((pts.shape[0], 2), dtype=dt, device=pts.device)
    check(lib.ttk_project(ptr(pts), ptr(me), ptr(mi), pts.shape[0], 1 if f64 else 0, ptr(out), stream_ptr()))
    return out


def reproject_clips(points, offsets, mint, mext, valid, det_xy):
    """`project` (float64) over n clips of different lengths in one launch.  points (sum T', 3) float64 CUDA, the clips concatenated;
    offsets (n+1,) int32 CUDA prefix sums (filter_ball_clips' format); mint (n, 3, 4), mext (n, 4, 4) float64 CUDA; valid (n,) int32
    CUDA; det_xy (sum T', 2) float64 CUDA, each row's 2D detection.  Returns xy (sum T', 2), each clip bit-identical to `project` on it
    alone, and err (n, 2): mean (summed in row order) and max Euclidean distance between xy and det_xy.  A clip with valid == 0 gets
    NaN points and errors."""
    _lib.require_device()
    assert points.is_cuda and points.dtype == torch.float64 and points.dim() == 2 and points.shape[1] == 3
    assert det_xy.is_cuda and det_xy.dtype == torch.float64 and tuple(det_xy.shape) == (points.shape[0], 2)
    assert offsets.is_cuda and offsets.dtype == torch.int32 and offsets.dim() == 1
    n = offsets.shape[0] - 1
    assert mint.is_cuda and mext.is_cuda and valid.is_cuda
    assert mint.dtype == mext.dtype == torch.float64 and tuple(mint.shape) == (n, 3, 4) and tuple(mext.shape) == (n, 4, 4)
    assert valid.dtype == torch.int32 and tuple(valid.shape) == (n,)
    pts, offs, mi, me, ok, det = (t.contiguous() for t in (points, offsets, mint, mext, valid, det_xy))
    xy = torch.empty((pts.shape[0], 2), dtype=torch.float64, device=pts.device)
    err = torch.empty((n, 2), dtype=torch.float64, device=pts.device)
    check(lib.ttk_reproject_clips(ptr(pts), pts.shape[0], ptr(offs), n, ptr(mi), ptr(me), ptr(ok), ptr(det), ptr(xy), ptr(err),
                                  stream_ptr()))
    return xy, err


def filter_ball(pos1, pos2, fps, threshold=20.0):
    """filter_trajectory_ball (inference/utils.py:70-102) on the device.  pos1/pos2: (T, 3) float64 CUDA (x, y, v).
    Returns compacted xy (T, 2) f64, idx (T,) int64, times (T,) f64 (the first n rows are valid) and offsets (2,) int32
    = [0, n] -- n stays on the device; `trajectory_pack` takes `offsets` directly."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() == 2 and pos1.shape[1] == 3
    pos1, pos2 = pos1.contiguous(), pos2.contiguous()
    T, dev = pos1.shape[0], pos1.device
    xy = torch.empty((T, 2), dtype=torch.float64, device=dev)
    idx = torch.empty((T,), dtype=torch.int64, device=dev)
    times = torch.empty((T,), dtype=torch.float64, device=dev)
    offs = torch.empty((2,), dtype=torch.int32, device=dev)
    check(lib.ttk_filter_ball(ptr(pos1), ptr(pos2), T, float(fps), float(threshold), ptr(xy), ptr(idx), ptr(times), ptr(offs),
                              stream_ptr()))
    return xy, idx, times, offs


def filter_ball_clips(pos1, pos2, frame_offsets, fps, threshold=20.0):
    """filter_ball over n clips in one launch.  pos1/pos2: (sum T, 3) float64 CUDA, the clips concatenated; frame_offsets: (n+1,)
    int32 CUDA prefix sums of the clip lengths.  Returns xy (sum T, 2), idx (sum T,) int64 and times (sum T,) counted from each
    clip's first frame, and offsets (n+1,) int32: clip c's kept rows are offsets[c]:offsets[c+1] -- `trajectory_pack`'s format."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() == 2 and pos1.shape[1] == 3
    assert frame_offsets.is_cuda and frame_offsets.dtype == torch.int32 and frame_offsets.dim() == 1
    pos1, pos2, frame_offsets = pos1.contiguous(), pos2.contiguous(), frame_offsets.contiguous()
    T, dev, n = pos1.shape[0], pos1.device, frame_offsets.shape[0] - 1
    xy = torch.empty((T, 2), dtype=torch.float64, device=dev)
    idx = torch.empty((T,), dtype=torch.int64, device=dev)
    times = torch.empty((T,), dtype=torch.float64, device=dev)
    offs = torch.empty((n + 1,), dtype=torch.int32, device=dev)
    check(lib.ttk_filter_ball_clips(ptr(pos1), ptr(pos2), n, ptr(frame_offsets), T, float(fps), float(threshold), ptr(xy), ptr(idx),
                                    ptr(times), ptr(offs), stream_ptr()))
    return xy, idx, times, offs


def filter_ball_timed(pos1, pos2, stamps, threshold=20.0):
    """filter_ball with each row's capture time instead of fps: stamps (T,) float64 CUDA, one per row of pos1.  A kept row t gets
    time stamps[t] - stamps[0]; xy, idx and offsets are filter_ball's."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() == 2 and pos1.shape[1] == 3
    assert stamps.is_cuda and stamps.dtype == torch.float64 and tuple(stamps.shape) == (pos1.shape[0],)
    pos1, pos2, stamps = pos1.contiguous(), pos2.contiguous(), stamps.contiguous()
    T, dev = pos1.shape[0], pos1.device
    xy = torch.empty((T, 2), dtype=torch.float64, device=dev)
    idx = torch.empty((T,), dtype=torch.int64, device=dev)
    times = torch.empty((T,), dtype=torch.float64, device=dev)
    offs = torch.empty((2,), dtype=torch.int32, device=dev)
    check(lib.ttk_filter_ball_timed(ptr(pos1), ptr(pos2), T, ptr(stamps), float(threshold), ptr(xy), ptr(idx), ptr(times), ptr(offs),
                                    stream_ptr()))
    return xy, idx, times, offs


def filter_ball_clips_timed(pos1, pos2, frame_offsets, stamps, threshold=20.0):
    """filter_ball_clips with each row's capture time instead of fps: stamps (sum T,) float64 CUDA in the layout of pos1.  A kept row
    gets its stamp minus the stamp of its clip's first row; xy, idx and offsets are filter_ball_clips'."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() == 2 and pos1.shape[1] == 3
    assert frame_offsets.is_cuda and frame_offsets.dtype == torch.int32 and frame_offsets.dim() == 1
    assert stamps.is_cuda and stamps.dtype == torch.float64 and tuple(stamps.shape) == (pos1.shape[0],)
    pos1, pos2, frame_offsets, stamps = pos1.contiguous(), pos2.contiguous(), frame_offsets.contiguous(), stamps.contiguous()
    T, dev, n = pos1.shape[0], pos1.device, frame_offsets.shape[0] - 1
    xy = torch.empty((T, 2), dtype=torch.float64, device=dev)
    idx = torch.empty((T,), dtype=torch.int64, device=dev)
    times = torch.empty((T,), dtype=torch.float64, device=dev)
    offs = torch.empty((n + 1,), dtype=torch.int32, device=dev)
    check(lib.ttk_filter_ball_clips_timed(ptr(pos1), ptr(pos2), n, ptr(frame_offsets), T, ptr(stamps), float(threshold), ptr(xy),
                                          ptr(idx), ptr(times), ptr(offs), stream_ptr()))
    return xy, idx, times, offs


def filter_table_clips(pos1, pos2, frame_offsets, agree=10.0, eps=10.0, min_samples=3):
    """filter_table over n clips of different lengths: pos1/pos2 (sum T, K, 3) float64 CUDA, the clips concatenated; frame_offsets
    (n+1,) int32 CUDA prefix sums.  Returns (n, K, 3) float64, each clip bit-identical to filter_table on that clip alone."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() == 3 and pos1.shape[-1] == 3
    assert frame_offsets.is_cuda and frame_offsets.dtype == torch.int32 and frame_offsets.dim() == 1
    a, b, frame_offsets = pos1.contiguous(), pos2.contiguous(), frame_offsets.contiguous()
    T, K, _ = a.shape
    n = frame_offsets.shape[0] - 1
    out = torch.empty((n, K, 3), dtype=torch.float64, device=a.device)
    ws_bytes = lib.ttk_filter_table_workspace_bytes(1, T, K)
    ws = torch.empty((max(ws_bytes, 8),), dtype=torch.uint8, device=a.device)
    check(lib.ttk_filter_table_clips(ptr(a), ptr(b), n, ptr(frame_offsets), T, K, float(agree), float(eps), int(min_samples), ptr(out),
                                     ptr(ws), ws_bytes, stream_ptr()))
    return out


def filter_table(pos1, pos2, agree=10.0, eps=10.0, min_samples=3):
    """filter_trajectory_table + DBSCAN (inference/utils.py:137-232) on the device.  pos1/pos2: (T, K, 3) or
    (clips, T, K, 3) float64 CUDA -> (K, 3) / (clips, K, 3) float64 CUDA."""
    _lib.require_device()
    assert pos1.is_cuda and pos1.dtype == torch.float64 and pos1.shape == pos2.shape and pos1.dim() in (3, 4) and pos1.shape[-1] == 3
    single = pos1.dim() == 3
    a, b = (p.contiguous().view((1,) + tuple(p.shape)) if single else p.contiguous() for p in (pos1, pos2))
    n, T, K, _ = a.shape
    out = torch.empty((n, K, 3), dtype=torch.float64, device=a.device)
    ws_bytes = lib.ttk_filter_table_workspace_bytes(n, T, K)
    ws = torch.empty((max(ws_bytes, 8),), dtype=torch.uint8, device=a.device)
    check(lib.ttk_filter_table(ptr(a), ptr(b), n, T, K, float(agree), float(eps), int(min_samples), ptr(out), ptr(ws), ws_bytes,
                               stream_ptr()))
    return out[0] if single else out


TABLE_HEIGHT, TABLE_WIDTH, TABLE_LENGTH = 0.76, 1.525, 2.74          # uplifting/helper.py:32-34
TABLE_POINTS = np.array([                                           # uplifting/helper.py:36-50
    [-TABLE_LENGTH / 2, TABLE_WIDTH / 2, TABLE_HEIGHT], [-TABLE_LENGTH / 2, -TABLE_WIDTH / 2, TABLE_HEIGHT],
    [0.0, TABLE_WIDTH / 2, TABLE_HEIGHT], [0.0, -TABLE_WIDTH / 2, TABLE_HEIGHT],
    [TABLE_LENGTH / 2, TABLE_WIDTH / 2, TABLE_HEIGHT], [TABLE_LENGTH / 2, -TABLE_WIDTH / 2, TABLE_HEIGHT],
    [0.0, TABLE_WIDTH / 2 + 0.1525, TABLE_HEIGHT], [0.0, -(TABLE_WIDTH / 2 + 0.1525), TABLE_HEIGHT],
    [0.0, 0.0, TABLE_HEIGHT], [0.0, TABLE_WIDTH / 2 + 0.1525, TABLE_HEIGHT + 0.1525],
    [0.0, -(TABLE_WIDTH / 2 + 0.1525), TABLE_HEIGHT + 0.1525], [-TABLE_LENGTH / 2, 0, TABLE_HEIGHT],
    [TABLE_LENGTH / 2, 0, TABLE_HEIGHT]], dtype=np.float64)
RANSAC_ITERATIONS, RANSAC_POINTS, RANSAC_FIXED_KEYS, RANSAC_THRESHOLD = 100, 6, (10, 11), 3.5     # regress_cameramatrices.py:129-136
TOO_FEW_POINTS = 'not enough points for DLT'                       # the reference's AssertionError (:211)


def ransac_sample_table(keypoints_host):
    """Hypothesis table of regress_cameramatrices_ransac (:138-143) for (n, 13, 3) host keypoints: (n, 100, 4) int32
    1-based ids, drawn like the reference (numpy Generator(seed=42).choice over the visible non-fixed keys, per clip).
    Data independent host logic; raises like the reference when fewer than 6 keypoints are visible."""
    tables = []
    for kp in keypoints_host:
        keys = [i + 1 for i in range(len(kp)) if kp[i][2] == 1]
        assert len(keys) >= RANSAC_POINTS, TOO_FEW_POINTS
        rnd = np.random.default_rng(seed=42)
        pool = [k for k in keys if k not in RANSAC_FIXED_KEYS]
        tables.append([[int(s) for s in rnd.choice(pool, size=RANSAC_POINTS - len(RANSAC_FIXED_KEYS), replace=False)]
                       for _ in range(RANSAC_ITERATIONS)])
    return np.asarray(tables, dtype=np.int32)


_SAMPLE_TABLES = {}     # 13-bit visibility pattern -> (100, 4) int32 table


def ransac_sample_table_cached(keypoints_host):
    """ransac_sample_table with each clip's table looked up by its visibility pattern: the table depends on which keypoints are visible
    and on nothing else (Generator(42).choice over the visible non-fixed keys), so each pattern is drawn once per process.  Returns
    identical tables; raises the same AssertionError for fewer than 6 visible keypoints."""
    tables = []
    for kp in keypoints_host:
        bits = sum(1 << i for i in range(len(kp)) if kp[i][2] == 1)
        t = _SAMPLE_TABLES.get(bits)
        if t is None:
            t = _SAMPLE_TABLES[bits] = ransac_sample_table(np.asarray(kp)[None])[0]
            t.flags.writeable = False
        tables.append(t)
    return np.asarray(tables, dtype=np.int32)


def calibrate_camera(keypoints, samples, width=1920, height=1080, threshold=RANSAC_THRESHOLD):
    """calibrate_camera (inference/utils.py:312-329) for a batch of clips.  keypoints (n, 13, 3) float64 CUDA,
    samples (n, H, S) int32 CUDA from `ransac_sample_table`.  Returns Mint (n, 3, 4), Mext (n, 4, 4) float64 and
    info (n, 4) int32 [inliers, best hypothesis, BFGS status of the refit, DLT ok], all CUDA."""
    _lib.require_device()
    assert keypoints.is_cuda and keypoints.dtype == torch.float64 and keypoints.dim() == 3 and keypoints.shape[1:] == (13, 3)
    assert samples.is_cuda and samples.dtype == torch.int32 and samples.dim() == 3 and samples.shape[0] == keypoints.shape[0]
    kp, smp = keypoints.contiguous(), samples.contiguous()
    n, dev = kp.shape[0], kp.device
    world = torch.from_numpy(TABLE_POINTS).to(dev)
    mint = torch.empty((n, 3, 4), dtype=torch.float64, device=dev)
    mext = torch.empty((n, 4, 4), dtype=torch.float64, device=dev)
    info = torch.empty((n, 4), dtype=torch.int32, device=dev)
    ws_bytes = lib.ttk_calibrate_workspace_bytes(n, smp.shape[1])
    ws = torch.empty((max(ws_bytes, 8),), dtype=torch.uint8, device=dev)
    check(lib.ttk_calibrate_camera(ptr(kp), ptr(world), ptr(smp), n, smp.shape[1], smp.shape[2], int(width), int(height),
                                   float(threshold), ptr(mint), ptr(mext), ptr(info), ptr(ws), ws_bytes, stream_ptr()))
    return mint, mext, info
