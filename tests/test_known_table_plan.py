"""Host logic of known tables (predict / predict_clips with table_keypoints=, LiveSession.set_table): the checks, all raised before any
device step; that a known table runs neither table detector nor table filter; the table stack plan of predict_clips over the clips
whose table is detected, across block boundaries, and the rows the known tables land in; the live bookkeeping of streams with a table
across pool wraps; and one calibration per distinct keypoint array with cameras=True.  The device steps are replaced by CPU models
(tests/test_gpu_known_table.py runs them on the GPU).  No GPU needed."""
import random

import numpy as np
import pytest
import torch

from upliftingtabletennis_b200 import interface, ops
from upliftingtabletennis_b200 import live as live_module
from upliftingtabletennis_b200.interface import (TableTennisPipeline, check_table_keypoints, clip_blocks, clip_stack_plan,
                                                 select_stacks)
from upliftingtabletennis_b200.live import BALL, TABLE, LiveSession

FPS = 50.0


def _device_step(*args, **kw):
    raise AssertionError('a device step ran')


class _NoDevice:
    """A detector or model whose every use is a device step."""

    def __getattr__(self, name):
        _device_step()


def _table(tag, visible=13):
    """A valid known table: keypoint k at (tag + k, 2 k), the first `visible` keypoints visible, the others (-1, -1, 0)."""
    kp = np.stack([tag + np.arange(13.0), 2.0 * np.arange(13), np.ones(13)], axis=1)
    kp[visible:] = (-1.0, -1.0, 0.0)
    return kp


def _detected(frame):
    """The table keypoints the modelled table detectors find on a frame: 13 visible keypoints at (frame id, 0)."""
    return np.tile([float(frame), 0.0, 1.0], (13, 1))


# ---- the checks ---------------------------------------------------------------------------------------------------------------------
def _with(i, j, value):
    kp = _table(0.0)
    kp[i, j] = value
    return kp


BAD = [
    (np.zeros((12, 3)), 'shape'),
    (np.zeros((13, 2)), 'shape'),
    (np.zeros((13, 3, 1)), 'shape'),
    (np.zeros(39), 'shape'),
    ([[1.0, 2.0, 1.0]] * 12 + [[1.0, 2.0]], 'numbers'),         # ragged
    ([['a', 'b', 'c']] * 13, 'numbers'),
    (_with(4, 0, np.nan), 'finite'),
    (_with(12, 1, np.inf), 'finite'),
    (_with(0, 2, -np.inf), 'finite'),
    (_with(3, 2, 0.5), 'visibility'),
    (_with(7, 2, 2.0), 'visibility'),
    (_with(7, 2, -1.0), 'visibility'),
]


def test_check_table_keypoints():
    kp = _table(3.0, visible=9)
    for given in (kp, kp.tolist(), torch.from_numpy(kp), torch.from_numpy(kp).float(), kp.astype(np.float32), kp.astype(np.int64)):
        got = check_table_keypoints(given, 'clip 0')
        assert got.dtype == np.float64 and got.shape == (13, 3) and got.flags['C_CONTIGUOUS']
        assert np.array_equal(got, np.asarray(given, dtype=np.float64) if not isinstance(given, torch.Tensor) else given.double().numpy())
    assert check_table_keypoints(kp, 'x') is not kp                 # a copy: the caller may change its array afterwards
    for bad, words in BAD:
        with pytest.raises(ValueError, match=words) as e:
            check_table_keypoints(bad, 'stream 3')
        assert str(e.value).startswith('stream 3: ')


def _blocked_pipe(monkeypatch):
    """A pipeline in which every detector, model and device step raises."""
    pipe = TableTennisPipeline.__new__(TableTennisPipeline)
    pipe.ball_detector = pipe.ball_detector_aux = pipe.table_detector = pipe.table_detector_aux = _NoDevice()
    pipe.uplifting_model = _NoDevice()
    pipe.device = torch.device('cpu')
    for name in ('_parts', '_detect_clips', '_uplift_clips', '_tail'):
        monkeypatch.setattr(pipe, name, _device_step, raising=False)
    for name in ('filter_ball', 'filter_ball_timed', 'filter_ball_clips', 'filter_ball_clips_timed', 'filter_table', 'filter_table_clips',
                 'trajectory_pack'):
        monkeypatch.setattr(ops, name, _device_step)
    monkeypatch.setattr(interface, '_upload_tables', _device_step)
    monkeypatch.setattr(live_module, '_upload_tables', _device_step)
    monkeypatch.setattr(torch.cuda, 'device_count', _device_step)
    return pipe


@pytest.mark.parametrize('bad,words', BAD)
def test_predict_refuses_bad_keypoints_before_any_device_step(monkeypatch, bad, words):
    pipe = _blocked_pipe(monkeypatch)
    with pytest.raises(ValueError, match='table_keypoints: .*' + words):
        pipe.predict([0, 1, 2, 3], FPS, table_keypoints=bad)
    with pytest.raises(ValueError, match=words):
        pipe.predict([0, 1, 2, 3], None, timestamps=[0.0, 0.1, 0.2, 0.3], table_keypoints=bad)


@pytest.mark.parametrize('bad,words', BAD)
@pytest.mark.parametrize('devices', [None, [0, 1]])
def test_predict_clips_refuses_bad_keypoints_naming_the_clip(monkeypatch, bad, words, devices):
    pipe = _blocked_pipe(monkeypatch)
    clips = [[0, 1, 2], [3, 4, 5, 6], [7, 8, 9, 10]]
    with pytest.raises(ValueError, match='clip 2: .*' + words):
        pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=[_table(0), None, bad])
    with pytest.raises(ValueError, match='clip 1: .*' + words):
        pipe.predict_clips(clips, FPS, devices=devices, cameras=True, table_keypoints=[None, bad, None])


@pytest.mark.parametrize('devices', [None, [0, 1]])
def test_predict_clips_refuses_a_list_of_another_length(monkeypatch, devices):
    pipe = _blocked_pipe(monkeypatch)
    clips = [[0, 1, 2], [3, 4, 5, 6], [7, 8, 9, 10]]
    for tables in ([_table(0)] * 2, [None] * 4, []):
        with pytest.raises(ValueError, match='table_keypoints: %d entries for 3 clips' % len(tables)):
            pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=tables)


# ---- predict and predict_clips with their device steps modelled ------------------------------------------------------------------
class _Model(torch.nn.Linear):
    def __init__(self, dtype='tf32'):
        super().__init__(2, 2)
        self.compute_dtype = dtype


class _Det:
    """A detector over frames that are their own ids (ints): a ball stack's position is (its centre frame, 7, 1), a table stack's
    keypoints are _detected(its frame).  Records the frames of every table pass."""
    segment = 512

    def __init__(self, frames_per_stack):
        self.frames_per_stack = frames_per_stack
        self.model = _Model()
        self.passes = []

    def _upload(self, images, dev, out=None):
        return torch.tensor(images, dtype=torch.float64), list(range(len(images))), None

    def _run(self, frames, stride, n_stacks, return_heatmaps, ready, heatmaps_to_host=False, first=None):
        f0 = first[0] if first is not None else [s * stride for s in range(n_stacks)]
        assert len(f0) == n_stacks
        if self.frames_per_stack == 3:
            pos = torch.stack([torch.tensor([[frames[f + 1], 7.0, 1.0]], dtype=torch.float64) for f in f0])
        else:
            self.passes.append([int(frames[f]) for f in f0])
            pos = torch.stack([torch.from_numpy(_detected(frames[f])) for f in f0])
        return pos, None


class _Up:
    """pos3d row t = (ball x, time, first table keypoint x); spin = the first table keypoint."""
    transform_mode = 'global'

    def __init__(self):
        self.model = _Model('tf32x3')

    def predict_without_normalization(self, ball, table, mask, times):
        n = int(mask.sum().item())
        pos = np.stack([ball[0, :n, 0].numpy(), times[0, :n].numpy(), np.full(n, float(table[0, 0, 0]), np.float32)], axis=1)
        return table[0, 0].clone(), pos


class _Filters:
    """CPU models of the ball filters (every row kept), the table filters (the keypoints of the clip's first frame, whose x is the
    frame id) and the packing; records the table filters' calls."""

    def __init__(self, monkeypatch):
        self.table_calls = []
        for name in ('filter_ball', 'filter_ball_clips', 'filter_ball_timed', 'filter_ball_clips_timed', 'filter_table',
                     'filter_table_clips', 'trajectory_pack'):
            monkeypatch.setattr(ops, name, getattr(self, name))

    def filter_ball(self, p1, p2, fps):
        T = p1.shape[0]
        return p1[:, :2].clone(), torch.arange(T), torch.arange(T, dtype=torch.float64) / fps, torch.tensor([0, T], dtype=torch.int32)

    def filter_ball_timed(self, p1, p2, stamps):
        T = p1.shape[0]
        return p1[:, :2].clone(), torch.arange(T), stamps - stamps[0], torch.tensor([0, T], dtype=torch.int32)

    def filter_ball_clips(self, p1, p2, offs, fps):
        local = torch.cat([torch.arange(int(offs[c + 1] - offs[c])) for c in range(len(offs) - 1)])
        return p1[:, :2].clone(), local, local.double() / fps, offs.clone()

    def filter_ball_clips_timed(self, p1, p2, offs, stamps):
        first = torch.cat([stamps[offs[c]].repeat(int(offs[c + 1] - offs[c])) for c in range(len(offs) - 1)])
        return p1[:, :2].clone(), None, stamps - first, offs.clone()

    def filter_table(self, t1, t2):
        self.table_calls.append(('filter_table', t1.shape[0]))
        return t1[0].clone()

    def filter_table_clips(self, t1, t2, offs):
        self.table_calls.append(('filter_table_clips', offs.tolist()))
        return torch.stack([t1[int(offs[c])] for c in range(len(offs) - 1)])

    def trajectory_pack(self, ball_xy, times, offsets, table, *args):
        n = len(offsets) - 1
        assert table.shape == (n, 13, 3) and table.dtype == torch.float64
        ball, tms, mask = torch.zeros((n, 50, 2)), torch.zeros((n, 50)), torch.zeros((n, 50))
        for c in range(n):
            a, b = int(offsets[c]), int(offsets[c + 1])
            ball[c, :b - a], tms[c, :b - a], mask[c, :b - a] = ball_xy[a:b].float(), times[a:b].float(), 1
        return ball, table.clone(), tms, mask


def _pipe(monkeypatch):
    pipe = TableTennisPipeline.__new__(TableTennisPipeline)
    pipe.ball_detector, pipe.ball_detector_aux = _Det(3), _Det(3)
    pipe.table_detector, pipe.table_detector_aux = _Det(1), _Det(1)
    pipe.uplifting_model = _Up()
    pipe.device = torch.device('cpu')
    pipe._home_device = lambda: torch.device('cpu')
    pipe._replica_parts = lambda slot, device_index: pipe._parts()
    pipe.uplifted_tables = []

    def uplift(parts, packed, counts):
        ball, table, times, mask = packed
        pipe.uplifted_tables.append(table.clone())
        pos = np.stack([ball[:, :, 0].numpy(), times.numpy(), np.repeat(table[:, :1, 0].float().numpy(), 50, axis=1)], axis=2)
        return table[:, 0].clone(), pos

    pipe._uplift_clips = uplift
    monkeypatch.setattr(torch.cuda, 'current_device', lambda: 0)
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 2)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: None)
    monkeypatch.setattr(interface, '_upload_stamps', lambda stamps, dev: torch.from_numpy(np.array(stamps, np.float64)))
    for module in (interface, live_module):
        monkeypatch.setattr(module, '_upload_tables', lambda kp, dev: torch.from_numpy(np.array(kp, np.float64)))
    monkeypatch.setattr(interface, '_upload_plan', lambda plan, stamps, dev: (
        torch.tensor(plan, dtype=torch.int32), None if stamps is None else torch.from_numpy(np.asarray(stamps, np.float64))))
    return pipe


def _no_table_detection(monkeypatch, pipe):
    for det in (pipe.table_detector, pipe.table_detector_aux):
        monkeypatch.setattr(det, '_run', _device_step)
    monkeypatch.setattr(ops, 'filter_table', _device_step)
    monkeypatch.setattr(ops, 'filter_table_clips', _device_step)


def _same(got, want):
    assert torch.equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_predict_with_keypoints_runs_no_table_detector(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    clip = list(range(100, 109))
    own = pipe.predict(clip, FPS)
    assert own[1][0, 2] == 100.0                            # detected: the table of the clip's first frame
    _no_table_detection(monkeypatch, pipe)
    K = _table(42.0, visible=10)
    spin, pos = pipe.predict(clip, FPS, table_keypoints=K.tolist())
    assert torch.equal(spin, torch.from_numpy(K[0])) and np.all(pos[:, 2] == 42.0)
    assert np.array_equal(pos[:, :2], own[1][:, :2])         # the ball path is the same
    # the clip's own filtered keypoints give predict's result
    _same(pipe.predict(clip, FPS, table_keypoints=_detected(100)), own)
    # with timestamps
    ts = 1.7e9 + np.cumsum(np.full(9, 0.02))
    spin, pos = pipe.predict(clip, None, timestamps=ts, table_keypoints=torch.from_numpy(K))
    assert np.all(pos[:, 2] == 42.0) and np.array_equal(pos[:, 1], (ts[1:8] - ts[1]).astype(np.float32))


@pytest.mark.parametrize('devices', [None, [0, 1, 1]])
def test_predict_clips_with_every_table_known_runs_no_table_detector(monkeypatch, devices):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    _no_table_detection(monkeypatch, pipe)
    clips = [list(range(f, f + n)) for f, n in ((0, 5), (10, 3), (20, 50), (80, 7))]
    tables = [_table(t) for t in (1.0, 2.0, 1.0, 3.0)]
    out = pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=tables)
    for (spin, pos), c, K in zip(out, clips, tables):
        assert torch.equal(spin, torch.from_numpy(K[0])) and np.all(pos[:, 2] == K[0, 0])
        _same((spin, pos), pipe.predict(c, FPS, table_keypoints=K))


@pytest.mark.parametrize('segment', [512, 60, 8])
@pytest.mark.parametrize('pattern', ['mixed', 'none', 'first', 'last'])
def test_predict_clips_table_plan_covers_the_detected_clips_only(monkeypatch, segment, pattern):
    rng = np.random.default_rng(segment)
    pipe = _pipe(monkeypatch)
    filters = _Filters(monkeypatch)
    pipe.ball_detector.segment = segment                    # several blocks when the clips are long
    lengths = [17, 3, 3, 29, 4, 50, 8, 12, 5, 40]
    clips, f = [], 0
    for n in lengths:
        clips.append(list(range(f, f + n)))
        f += n
    known = {'mixed': [i % 3 != 1 for i in range(len(clips))], 'none': [False] * len(clips),
             'first': [i == 0 for i in range(len(clips))], 'last': [i == len(clips) - 1 for i in range(len(clips))]}[pattern]
    tables = [_table(1000.0 + i, visible=int(rng.integers(0, 14))) if k else None for i, k in enumerate(known)]
    out = pipe.predict_clips(clips, FPS, table_keypoints=tables)
    # per block, the table passes and the table filter cover the block's clips whose entry is None, in clip order
    blocks = clip_blocks(lengths, segment)
    detected = [[i for i in range(a, b) if tables[i] is None] for a, b in blocks]
    want_calls = [('filter_table_clips', clip_stack_plan([lengths[i] for i in d], 1)[1]) for d in detected if d]
    assert filters.table_calls == want_calls
    assert pipe.table_detector.passes == pipe.table_detector_aux.passes
    assert [f for p in pipe.table_detector.passes for f in p] == [f for i in range(len(clips)) if tables[i] is None for f in clips[i]]
    # the supplied arrays land in their clips' rows, the filtered keypoints in the others
    rows = torch.cat(pipe.uplifted_tables)
    for i, (c, K) in enumerate(zip(clips, tables)):
        assert torch.equal(rows[i], torch.from_numpy(_detected(c[0]) if K is None else K)), i
    # each result is predict with the same arguments
    for (spin, pos), c, K in zip(out, clips, tables):
        _same((spin, pos), pipe.predict(c, FPS, table_keypoints=K))


@pytest.mark.parametrize('lengths,keep', [([5, 3, 4], [1]), ([5, 3, 4], []), ([5, 3, 4], [0, 1, 2]), ([1, 6, 2, 9], [0, 3])])
@pytest.mark.parametrize('frames_per_stack', [1, 3])
def test_select_stacks(lengths, keep, frames_per_stack):
    first, offs = clip_stack_plan(lengths, frames_per_stack)
    sel, sel_offs = select_stacks(first, offs, keep)
    sub_first, sub_offs = clip_stack_plan([lengths[i] for i in keep], frames_per_stack)
    assert sel_offs == sub_offs and len(sel) == len(sub_first)
    starts = np.concatenate([[0], np.cumsum(lengths)])
    # the same stacks as the plan over the kept clips alone, in the frames of all clips
    shift = [starts[i] - s for i, s in zip(keep, np.concatenate([[0], np.cumsum([lengths[i] for i in keep])]))]
    assert sel == [f + shift[c] for c in range(len(keep)) for f in sub_first[sub_offs[c]:sub_offs[c + 1]]]
    assert select_stacks(first, offs, range(len(lengths))) == (first, offs)


@pytest.mark.parametrize('devices', [None, [0, 0], [0, 1, 1]])
def test_predict_clips_mixed_with_stamps_and_devices(monkeypatch, devices):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    lengths = [9, 4, 30, 3, 12]
    clips = [list(range(100 * i, 100 * i + n)) for i, n in enumerate(lengths)]
    tables = [None, _table(5.0), _table(6.0, 4), None, _table(5.0)]
    stamps = [1.7e9 + np.cumsum(np.full(n, 0.02 + 0.01 * i)) for i, n in enumerate(lengths)]
    got = pipe.predict_clips(clips, None, devices=devices, timestamps=stamps, table_keypoints=tables)
    for g, c, ts, K in zip(got, clips, stamps, tables):
        _same(g, pipe.predict(c, None, timestamps=ts, table_keypoints=K))


# ---- cameras=True: one calibration per distinct array ----------------------------------------------------------------------------
@pytest.fixture
def calibrations(monkeypatch):
    rows = []

    def calibrate(kp, samples, width, height):
        assert kp.shape[0] == samples.shape[0]
        rows.append(kp.clone())
        n = kp.shape[0]
        mint = torch.zeros((n, 3, 4), dtype=torch.float64)
        mint[:, 0, 0] = kp[:, 0, 0]
        mext = torch.eye(4, dtype=torch.float64).repeat(n, 1, 1)
        return mint, mext, torch.tensor([[13, 3, 0, 1]] * n, dtype=torch.int32)

    def reproject(points, offsets, mint, mext, valid, det_xy):
        return torch.zeros((points.shape[0], 2), dtype=torch.float64), torch.zeros((len(offsets) - 1, 2), dtype=torch.float64)

    monkeypatch.setattr(ops, 'calibrate_camera', calibrate)
    monkeypatch.setattr(ops, 'reproject_clips', reproject)
    return rows


@pytest.mark.parametrize('devices', [None, [0, 0]])
def test_cameras_calibrate_each_distinct_array_once(monkeypatch, calibrations, devices):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    A, B = _table(7.0), _table(8.0, visible=8)
    few = _table(9.0, visible=5)                             # too few visible keypoints: not calibrated at all
    clips = [list(range(100 * i, 100 * i + 6)) for i in range(8)]
    tables = [A, A, None, B, few, A, B, A]
    out = pipe.predict_clips(clips, FPS, devices=devices, cameras=True, table_keypoints=tables)
    got = [tuple(r[:, 0, 0].tolist()) for r in calibrations]
    if devices is None:
        assert got == [(7.0, 200.0, 8.0)]                   # A, the detected table of clip 2, B: in the order of first use
    else:                                                   # per device: clips 0-3, then clips 4-7
        assert sorted(got) == sorted([(7.0, 200.0, 8.0), (7.0, 8.0)])
    for (spin, pos, cam), K, c in zip(out, tables, clips):
        want = _detected(c[0]) if K is None else K
        assert np.array_equal(cam.keypoints, want)
        if K is few:
            assert cam.error == ops.TOO_FEW_POINTS and cam.Mint is None
        else:
            assert cam.error is None and cam.Mint[0, 0] == want[0, 0]


# ---- live sessions -------------------------------------------------------------------------------------------------------------
class _Session(LiveSession):
    """LiveSession with its pool modelled on the CPU (each slot holds a frame id) and the passes run by the _Det models on the slots'
    frames; records every pass; end_rally runs the real _finish and TableTennisPipeline._tail."""

    def _alloc_pool(self, shape):
        self.slot = [None] * (self.streams * self.slots)
        self.passes = []
        return [None]

    def _check_frames(self, frames):
        if self._pool is None:
            self._pool = self._alloc_pool(None)

    def _device_write(self, frames, p0):
        self.slot[p0:p0 + len(frames)] = frames

    def _hand_off(self, e, frames, p0):                     # devices=[...]: the write runs on the entry's launcher
        e.submit(self._device_write, list(frames), p0)

    def _device_wrap(self, src, dst, m):
        self.slot[dst:dst + m] = self.slot[src:src + m]

    def _device_pass(self, fps, first, runs):
        self.passes.append((fps, list(first), [(st, list(idx)) for st, idx in runs]))
        e = self._entry[runs[0][0]]
        parts = self.pipe._parts()
        frames = [-1 if f is None else f for f in self.slot]
        a = 0
        for st, idx in runs:
            for d in ((0, 1) if fps == BALL else (2, 3)):
                pos = parts[d]._run(frames, 1, len(idx), False, None, first=(first[a:a + len(idx)], None))[0]
                self._store(e, st, d, idx[0], pos)
            a += len(idx)


def test_set_table_refusals(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, FPS, 2, 4, 8)
    for bad, words in BAD:
        with pytest.raises(ValueError, match='stream 1: .*' + words):
            live.set_table(1, bad)
    assert live._pool is None and live._tables == [None, None]
    live.push(1, [10, 11])
    with pytest.raises(ValueError, match='stream 1: set_table with a rally of 2 frames open'):
        live.set_table(1, _table(0))
    with pytest.raises(ValueError, match='stream 1: set_table with a rally'):
        live.set_table(1, None)
    live.set_table(0, _table(0))                            # the other stream has no open rally
    with pytest.raises(ValueError, match='stream must be'):
        live.set_table(2, _table(0))
    assert live._tables[1] is None and np.array_equal(live._tables[0], _table(0))


def test_end_rally_with_a_table_runs_no_table_detector(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    _no_table_detection(monkeypatch, pipe)
    K = _table(4.0, visible=7)
    for devices in (None, [0]):
        live = _Session(pipe, FPS, 1, 4, 8, devices=devices)
        live.set_table(0, K)
        frames = list(range(500, 521))                     # 21 frames through an 8-slot region: wraps
        for f in frames:
            live.push(0, [f])
            assert not live._pending[TABLE]
        _same(live.end_rally(0), pipe.predict(frames, FPS, table_keypoints=K))
        assert all(p[0] == BALL for p in live.passes)
        live.close()


@pytest.mark.parametrize('devices', [None, [0]])
def test_live_tables_across_wraps_and_streams(monkeypatch, devices):
    rng = random.Random(5)
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    k = 4
    live = _Session(pipe, FPS, 3, k, 8, devices=devices)
    A, B = _table(70.0), _table(80.0, visible=6)
    # per stream: its rallies' lengths and the table set before each (None: detected); stream 1 switches between the two
    plan = {0: [(23, A), (9, A), (41, A)], 1: [(12, None), (30, B), (3, None), (17, B)], 2: [(49, None), (5, None)]}
    ids = iter(range(10 ** 6))
    done, left = [0, 0, 0], [plan[s][0][0] for s in range(3)]
    rally = {s: [] for s in range(3)}
    for s in range(3):
        live.set_table(s, plan[s][0][1])
    checked = 0
    while any(done[s] < len(plan[s]) for s in range(3)):
        s = rng.choice([i for i in range(3) if done[i] < len(plan[i])])
        c = min(rng.choice([1, 1, 2, 5, 9]), left[s])
        frames = [next(ids) for _ in range(c)]
        live.push(s, frames)
        rally[s].extend(frames)
        left[s] -= c
        tabled = {i for i in range(3) if live._tables[i] is not None}
        # no table stack pending for a stream with a table, and the k rule on the stacks that exist
        assert not [x for x in live._pending[TABLE] if x[0] in tabled]
        assert len(live._pending[BALL]) < k and len(live._pending[TABLE]) < k
        if left[s] == 0:
            K = plan[s][done[s]][1]
            got = live.end_rally(s)
            _same(got, pipe.predict(rally[s], FPS, table_keypoints=K))
            assert got[1][0, 2] == (rally[s][0] if K is None else K[0, 0])
            checked += 1
            rally[s] = []
            done[s] += 1
            if done[s] < len(plan[s]):
                left[s] = plan[s][done[s]][0]
                live.set_table(s, plan[s][done[s]][1])      # applies from this next rally; None restores detection
    assert checked == sum(len(p) for p in plan.values())
    # no table pass ever held a stack of a stream while its table was set: table passes hold streams 1 (its detected rallies) and 2
    table_streams = {st for fps, _, runs in live.passes if fps == TABLE for st, _ in runs}
    assert table_streams == {1, 2}
    live.close()


def test_table_applies_from_the_next_rally(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, FPS, 1, 4, 64)
    live.push(0, [1, 2, 3, 4])
    with pytest.raises(ValueError, match='rally of 4 frames open'):
        live.set_table(0, _table(9.0))
    assert live.end_rally(0)[1][0, 2] == 1.0                # still detected
    live.set_table(0, _table(9.0))
    live.push(0, [5, 6, 7, 8])
    assert not live._pending[TABLE]
    assert live.end_rally(0)[1][0, 2] == 9.0
    live.push(0, [9, 10, 11])                               # stays in force
    assert live.end_rally(0)[1][0, 2] == 9.0
    live.set_table(0, None)
    live.push(0, [12, 13, 14])
    assert [x[1] for x in live._pending[TABLE]] == [0, 1, 2]
    assert live.end_rally(0)[1][0, 2] == 12.0
    # a failed end_rally ends the rally too: the table can be set after it
    live.push(0, [15, 16])
    with pytest.raises(ValueError, match='at least 3'):
        live.end_rally(0)
    live.set_table(0, _table(3.0))
    live.push(0, [17, 18, 19])
    assert live.end_rally(0)[1][0, 2] == 3.0


def test_timestamped_session_with_a_table(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, None, 2, 4, 8)
    K = _table(11.0)
    live.set_table(1, K)
    ts = 1.7e9 + np.cumsum(np.full(13, 0.04))
    frames = list(range(300, 313))
    live.push(1, frames[:6], timestamps=ts[:6])
    live.push(0, [1, 2, 3], timestamps=[0.0, 0.1, 0.2])
    live.push(1, frames[6:], timestamps=ts[6:])
    _same(live.end_rally(1), pipe.predict(frames, None, timestamps=ts, table_keypoints=K))
    _same(live.end_rally(0), pipe.predict([1, 2, 3], None, timestamps=[0.0, 0.1, 0.2]))


def test_end_rally_cameras_with_a_table(monkeypatch, calibrations):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, FPS, 1, 4, 8)
    live.push(0, list(range(40, 50)))
    spin, pos, cam = live.end_rally(0, cameras=True)
    assert np.array_equal(cam.keypoints, _detected(40))
    live.set_table(0, cam.keypoints)                        # the typical use: the first rally's camera for the ones after it
    first = len(live.passes)
    live.push(0, list(range(60, 70)))
    spin, pos, cam2 = live.end_rally(0, cameras=True)
    assert np.array_equal(cam2.keypoints, cam.keypoints) and cam2.Mint[0, 0] == 40.0
    assert live.passes[first:] and all(p[0] == BALL for p in live.passes[first:])
