"""Host logic of the rally cameras (predict_clips / LiveSession.end_rally with cameras=True): the cached RANSAC sample tables, the
calibration messages, the RallyCamera records assembled from the device results, and that cameras=False runs none of it.  The device
steps are replaced by CPU models here (tests/test_gpu_rally_cameras.py runs them on the GPU).  No GPU needed."""
import numpy as np
import pytest
import torch

from upliftingtabletennis_b200 import interface, ops
from upliftingtabletennis_b200.interface import RallyCamera, TableTennisPipeline, calibration_error
from upliftingtabletennis_b200.live import BALL, LiveSession


def _pattern_keypoints(visible):
    kp = np.zeros((13, 3))
    kp[:, :2] = np.arange(26).reshape(13, 2)
    kp[:, 2] = [1.0 if i in visible else 0.0 for i in range(13)]
    return kp


EDGE_PATTERNS = [
    range(13),                                  # all 13
    [0, 1, 2, 3, 9, 10],                        # exactly 6, keys 10 and 11 among them
    [0, 2, 4, 6, 8, 12],                        # exactly 6, keys 10 and 11 absent: 6 free keys to draw 4 from
    [1, 3, 5, 7, 9, 11],                        # exactly 6, key 10 present, key 11 absent
    [i for i in range(13) if i not in (9, 10)],     # all but keys 10 and 11
    [9, 10, 0, 1, 2, 3, 4],
]


@pytest.mark.parametrize('visible', EDGE_PATTERNS)
def test_cached_sample_table_equals_the_draw(visible):
    kp = _pattern_keypoints(list(visible))[None]
    want = ops.ransac_sample_table(kp)
    assert want.shape == (1, ops.RANSAC_ITERATIONS, 4)
    for _ in range(2):                                  # a draw, then a cache hit
        got = ops.ransac_sample_table_cached(kp)
        assert got.dtype == want.dtype and np.array_equal(got, want)


def test_cached_sample_table_random_patterns():
    rng = np.random.default_rng(5)
    kps = []
    while len(kps) < 200:
        vis = rng.uniform(0, 1, 13) < rng.uniform(0.4, 1.0)
        if vis.sum() >= ops.RANSAC_POINTS:
            kps.append(_pattern_keypoints(np.flatnonzero(vis).tolist()))
    kps = np.stack(kps)
    assert np.array_equal(ops.ransac_sample_table_cached(kps), ops.ransac_sample_table(kps))
    assert np.array_equal(ops.ransac_sample_table_cached(kps[::-1]), ops.ransac_sample_table(kps[::-1]))


def test_too_few_visible_keypoints_raise_the_same_assertion():
    kp = _pattern_keypoints([0, 1, 2, 9, 10])[None]
    for fn in (ops.ransac_sample_table, ops.ransac_sample_table_cached):
        with pytest.raises(AssertionError) as e:
            fn(kp)
        assert str(e.value) == ops.TOO_FEW_POINTS == 'not enough points for DLT'


def test_calibration_messages_are_the_references():
    assert calibration_error([13, 4, 0, 1]) is None
    assert calibration_error(np.array([7, 0, 2, 1], np.int32)) is None
    assert calibration_error([13, 4, 0, 0]) == 'Intrinsic matrix K has K[2,2] close to zero, indicating a degenerate camera.'
    assert calibration_error([0, 4, 0, 0]).startswith('Intrinsic matrix K has K[2,2] close to zero')       # the DLT check comes first
    assert calibration_error([0, 0, 0, 1]) == 'RANSAC failed to find a valid model.'


# ---- the records, with the two device steps modelled on the CPU ------------------------------------------------------------------
def _fake_calibrate(info_rows):
    def calibrate(kp, samples, width, height):
        assert kp.shape[0] == samples.shape[0] and samples.shape[1:] == (ops.RANSAC_ITERATIONS, 4) and (width, height) == (1920, 1080)
        n = kp.shape[0]
        mint = torch.zeros((n, 3, 4), dtype=torch.float64)
        mint[:, 0, 0] = mint[:, 1, 1] = 1000.0
        mint[:, 0, 2], mint[:, 1, 2], mint[:, 2, 2] = 960.0, 540.0, 1.0
        mext = torch.eye(4, dtype=torch.float64).repeat(n, 1, 1)
        mext[:, 2, 3] = 5.0 + kp[:, 0, 0]                     # a camera per clip
        info = torch.tensor([info_rows[int(k)] for k in kp[:, 0, 0]], dtype=torch.int32)
        return mint, mext, info
    return calibrate


def _fake_reproject(points, offsets, mint, mext, valid, det_xy):
    """The kernel's contract in numpy: projection, then mean (in row order) and max of the pixel distances; NaN for invalid clips."""
    pts, offs, det = points.numpy(), offsets.numpy(), det_xy.numpy()
    xy = np.full((len(pts), 2), np.nan)
    err = np.full((len(offs) - 1, 2), np.nan)
    for c in range(len(offs) - 1):
        a, b = offs[c], offs[c + 1]
        if not valid[c]:
            continue
        cam = np.c_[pts[a:b], np.ones(b - a)] @ mext[c].numpy().T
        q = (cam[:, :3] / cam[:, 3:]) @ mint[c, :, :3].numpy().T
        xy[a:b] = q[:, :2] / q[:, 2:]
        d = np.sqrt(((xy[a:b] - det[a:b]) ** 2).sum(axis=1))
        err[c] = d.mean(), d.max()
    return torch.from_numpy(xy), torch.from_numpy(err)


@pytest.fixture
def camera_ops(monkeypatch):
    """Calibration info per clip (keyed by the clip's first keypoint x): success, degenerate DLT, RANSAC failure."""
    rows = {0: [13, 3, 0, 1], 1: [0, 0, 0, 0], 2: [0, 5, 0, 1]}
    monkeypatch.setattr(ops, 'calibrate_camera', _fake_calibrate(rows))
    monkeypatch.setattr(ops, 'reproject_clips', _fake_reproject)


@pytest.fixture
def no_camera_ops(monkeypatch):
    def called(*args, **kw):
        raise AssertionError('a camera step ran with cameras=False')
    for name in ('calibrate_camera', 'reproject_clips', 'ransac_sample_table', 'ransac_sample_table_cached'):
        monkeypatch.setattr(ops, name, called)
    monkeypatch.setattr(interface, '_rally_cameras', called)


def _keypoints(tag, visible=13):
    kp = _pattern_keypoints(list(range(visible)))
    kp[0, 0] = tag
    return kp


def _check_record(cam, kp, det, pos):
    assert isinstance(cam, RallyCamera) and RallyCamera._fields == (
        'keypoints', 'Mint', 'Mext', 'ball_2d', 'detections_2d', 'error_px', 'error')
    assert isinstance(cam.keypoints, np.ndarray) and cam.keypoints.dtype == np.float64 and np.array_equal(cam.keypoints, kp)
    assert isinstance(cam.detections_2d, np.ndarray) and cam.detections_2d.shape == (len(pos), 2) and np.array_equal(cam.detections_2d, det)
    tag, visible = int(kp[0, 0]), int(kp[:, 2].sum())
    if visible < 6:
        want = 'not enough points for DLT'
    else:
        want = {0: None, 1: 'Intrinsic matrix K has K[2,2] close to zero, indicating a degenerate camera.',
                2: 'RANSAC failed to find a valid model.'}[tag]
    assert cam.error == want
    if want is not None:
        assert cam.Mint is None and cam.Mext is None and cam.ball_2d is None and cam.error_px is None
        return
    assert cam.Mint.shape == (3, 4) and cam.Mext.shape == (4, 4) and cam.Mint.dtype == cam.Mext.dtype == np.float64
    assert cam.ball_2d.shape == (len(pos), 2) and cam.ball_2d.dtype == np.float64 and np.isfinite(cam.ball_2d).all()
    assert isinstance(cam.error_px, tuple) and all(isinstance(v, float) for v in cam.error_px)
    d = np.sqrt(((cam.ball_2d - det) ** 2).sum(axis=1))
    assert cam.error_px == (d.mean(), d.max())


def test_rally_cameras_records(camera_ops):
    kps = [_keypoints(0), _keypoints(2), _keypoints(0, 5), _keypoints(1), _keypoints(0, 6)]
    counts = [3, 1, 4, 2, 5]
    rng = np.random.default_rng(1)
    det = rng.uniform(0, 1000, (sum(counts), 2))
    pos = [rng.uniform(-1, 1, (c, 3)).astype(np.float32) for c in counts]
    cams = interface._rally_cameras(torch.from_numpy(np.stack(kps)), torch.from_numpy(det), counts, pos)
    offs = np.concatenate([[0], np.cumsum(counts)])
    for i, cam in enumerate(cams):
        _check_record(cam, kps[i], det[offs[i]:offs[i + 1]], pos[i])
    # no clip with 6 visible keypoints: no calibration at all, every record says why
    cams = interface._rally_cameras(torch.from_numpy(np.stack(kps[2:3])), torch.from_numpy(det[:4]), [4], pos[2:3])
    assert cams[0].error == 'not enough points for DLT'


# ---- predict_clips and end_rally, device work replaced ------------------------------------------------------------------------
class _Up:
    """The uplifting model: T' = the mask's sum; pos3d a function of the packed ball rows."""
    transform_mode = 'global'

    def __init__(self):
        self.model = torch.nn.Linear(2, 2)
        self.model.compute_dtype = 'tf32x3'

    def predict_without_normalization(self, ball, table, mask, times):
        n = int(mask.sum().item())
        return torch.zeros(3), np.repeat(ball[0, :n, :1].numpy(), 3, axis=1)


class _Part:
    def __init__(self):
        self.model = torch.nn.Linear(2, 2)
        self.model.compute_dtype = 'tf32'


def _fake_pipe(monkeypatch, clip_keypoints):
    """A TableTennisPipeline whose detectors, filters and uplift run on the CPU: clip i has i + 2 agreeing ball detections at
    x = 100 i + t and the filtered table keypoints clip_keypoints[i]."""
    pipe = TableTennisPipeline.__new__(TableTennisPipeline)
    pipe.uplifting_model = _Up()
    parts = [_Part() for _ in range(4)] + [pipe.uplifting_model]
    pipe._parts = lambda: parts
    pipe._replica_parts = lambda slot, device_index: parts
    pipe._home_device = lambda: torch.device('cpu')
    pipe.device = torch.device('cpu')

    def detections(i):
        c = i + 2
        return torch.stack([100.0 * i + torch.arange(c, dtype=torch.float64), torch.full((c,), 7.0, dtype=torch.float64)], dim=1)

    def detect(parts_, clips, fps):
        ids = [int(c[0]) for c in clips]                        # a clip is [its index] * frames
        counts = [i + 2 for i in ids]
        n = len(ids)
        ball = torch.zeros((n, 50, 2))
        mask = torch.zeros((n, 50))
        for j, (i, c) in enumerate(zip(ids, counts)):
            ball[j, :c] = detections(i).float()
            mask[j, :c] = 1
        xy = torch.cat([detections(i) for i in ids] + [torch.full((5, 2), -1.0, dtype=torch.float64)])      # unused capacity
        tab = torch.from_numpy(np.stack([clip_keypoints[i] for i in ids]))
        return (ball, None, None, mask), torch.tensor(counts, dtype=torch.int32), [(tab, xy)]

    def uplift(parts_, packed, counts):
        ball = packed[0]
        return torch.zeros((len(counts), 3)), np.repeat(ball[:, :, :1].numpy(), 3, axis=2)

    pipe._detect_clips, pipe._uplift_clips = detect, uplift
    # the single-clip tail (live sessions), from the ball positions (x, y, v) of each stack
    monkeypatch.setattr(ops, 'filter_ball', lambda p1, p2, fps: (p1[:, :2].clone(), None, None, torch.tensor([0, p1.shape[0]])))
    monkeypatch.setattr(ops, 'filter_table', lambda t1, t2: torch.from_numpy(clip_keypoints[int(t1[0, 0, 0])]))

    def pack(ball_xy, times, offsets, table, *args):
        n = int(offsets[1])
        ball = torch.zeros((1, 50, 2))
        mask = torch.zeros((1, 50))
        ball[0, :n], mask[0, :n] = ball_xy[:n].float(), 1
        return ball, table, None, mask
    monkeypatch.setattr(ops, 'trajectory_pack', pack)
    return pipe, detections


CLIP_KEYPOINTS = [_keypoints(0), _keypoints(2), _keypoints(0, 4), _keypoints(1)]


@pytest.fixture
def gpus(monkeypatch):
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 2)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: None)


@pytest.mark.parametrize('devices', [None, [0, 0], [0, 1, 1]])
def test_predict_clips_without_cameras_runs_no_camera_step(monkeypatch, gpus, no_camera_ops, devices):
    pipe, _ = _fake_pipe(monkeypatch, CLIP_KEYPOINTS)
    clips = [[i] * 5 for i in range(len(CLIP_KEYPOINTS))]
    out = pipe.predict_clips(clips, 50.0, devices=devices)
    assert [len(r) for r in out] == [2] * len(clips)
    assert [r[1].shape[0] for r in out] == [i + 2 for i in range(len(clips))]
    assert pipe.predict_clips(clips, 50.0, devices=devices, cameras=False)[3][1].shape == (5, 3)


@pytest.mark.parametrize('devices', [None, [0, 0], [0, 1, 1]])
def test_predict_clips_cameras_extend_each_result(monkeypatch, gpus, camera_ops, devices):
    pipe, detections = _fake_pipe(monkeypatch, CLIP_KEYPOINTS)
    clips = [[i] * 5 for i in range(len(CLIP_KEYPOINTS))]
    plain = pipe.predict_clips(clips, 50.0, devices=devices)
    out = pipe.predict_clips(clips, 50.0, devices=devices, cameras=True)
    for i, ((spin, pos), (spin2, pos2, cam)) in enumerate(zip(plain, out)):
        assert torch.equal(spin, spin2) and np.array_equal(pos, pos2)
        _check_record(cam, CLIP_KEYPOINTS[i], detections(i).numpy(), pos)


class _Session(LiveSession):
    """LiveSession with its pool and detector passes on the CPU: a ball stack's positions are (clip id, 7, 1) rows, a table stack's
    the clip id; end_rally runs the real _finish and TableTennisPipeline._tail."""

    def _alloc_pool(self, shape):
        return [None]

    def _device_write(self, frames, p0):
        pass

    def _device_wrap(self, src, dst, m):
        pass

    def _device_pass(self, fps, first, runs):
        e = self._entries[0]
        for st, idx in runs:
            clip = float(self.clip[st])
            for d in ((0, 1) if fps == BALL else (2, 3)):
                if fps == BALL:
                    p = torch.tensor([[[100.0 * clip + j, 7.0, 1.0]] for j in idx], dtype=torch.float64)
                else:
                    p = torch.full((len(idx), 13, 3), clip, dtype=torch.float64)
                self._store(e, st, d, idx[0], p)


def test_end_rally_without_cameras_runs_no_camera_step(monkeypatch, no_camera_ops):
    pipe, _ = _fake_pipe(monkeypatch, CLIP_KEYPOINTS)
    live = _Session(pipe, 50.0, 2, 4, 64)
    live.clip = [1, 3]
    frame = np.zeros((4, 4, 3), np.uint8)
    for _ in range(6):
        live.push(0, frame)
        live.push(1, [frame, frame])
    spin, pos = live.end_rally(0)
    assert pos.shape == (4, 3)
    spin, pos = live.end_rally(1, cameras=False)
    assert pos.shape == (10, 3)


def test_end_rally_cameras(monkeypatch, camera_ops):
    pipe, _ = _fake_pipe(monkeypatch, CLIP_KEYPOINTS)
    live = _Session(pipe, 50.0, 2, 4, 64)
    frame = np.zeros((4, 4, 3), np.uint8)
    for clip in range(len(CLIP_KEYPOINTS)):
        live.clip = [clip, 0]
        live.push(0, [frame] * (clip + 4))
        spin, pos, cam = live.end_rally(0, cameras=True)
        assert pos.shape == (clip + 2, 3)
        det = np.stack([100.0 * clip + np.arange(clip + 2), np.full(clip + 2, 7.0)], axis=1)
        _check_record(cam, CLIP_KEYPOINTS[clip], det, pos)
