"""Host logic of per-frame capture timestamps (predict / predict_clips / live sessions with fps=None): the checks, all raised before
any device step; the ball-row layout of the stamps predict_clips uploads and the one host-to-device copy that carries them with the
stack plan; the stamps a live session keeps per stream across pool wraps and resets at end_rally; and that a call with fps never
reaches the timed filters.  The device steps are replaced by CPU models (tests/test_gpu_timestamps.py runs them on the GPU).  No GPU
needed."""
import random

import numpy as np
import pytest
import torch

from upliftingtabletennis_b200 import interface, ops
from upliftingtabletennis_b200.interface import TableTennisPipeline, ball_row_stamps, check_timestamps, clip_stack_plan
from upliftingtabletennis_b200.live import BALL, TABLE, LiveSession

FPS = 50.0


def _device_step(*args, **kw):
    raise AssertionError('a device step ran')


class _NoDevice:
    """A detector or model whose every use is a device step."""

    def __getattr__(self, name):
        _device_step()


# ---- the checks ---------------------------------------------------------------------------------------------------------------------
BAD = [
    ([0.0, 0.1], 'shape'),                                      # too few
    ([0.0, 0.1, 0.2, 0.3, 0.4], 'shape'),                       # too many
    ([[0.0, 0.1, 0.2, 0.3]], 'shape'),                          # not one per frame
    ([0.0, np.nan, 0.2, 0.3], 'finite'),
    ([0.0, 0.1, np.inf, 0.3], 'finite'),
    ([-np.inf, 0.1, 0.2, 0.3], 'finite'),
    ([0.0, 0.1, 0.1, 0.3], 'increase'),                         # a repeated stamp
    ([0.0, 0.2, 0.1, 0.3], 'increase'),
    (['a', 'b', 'c', 'd'], 'seconds'),
    (None, 'timestamps with fps=None'),                         # no time source at all
]


def test_check_timestamps():
    ts = check_timestamps([1.7e9, 1.7e9 + 0.02, 1.7e9 + 0.06], 3, 'clip 0')
    assert ts.dtype == np.float64 and ts.shape == (3,)
    assert check_timestamps(np.arange(4, dtype=np.int64), 4, 'x').dtype == np.float64
    assert check_timestamps(torch.arange(4, dtype=torch.float32), 4, 'x').dtype == np.float64
    assert check_timestamps([], 0, 'x').shape == (0,)
    for bad, words in BAD[:-1]:
        with pytest.raises(ValueError, match=words) as e:
            check_timestamps(bad, 4, 'stream 3')
        assert str(e.value).startswith('stream 3: ')


def _blocked_pipe(monkeypatch):
    """A pipeline in which every detector, model and device step raises."""
    pipe = TableTennisPipeline.__new__(TableTennisPipeline)
    pipe.ball_detector = pipe.ball_detector_aux = pipe.table_detector = pipe.table_detector_aux = _NoDevice()
    pipe.uplifting_model = _NoDevice()
    pipe.device = torch.device('cpu')
    for name in ('_parts', '_detect_clips', '_uplift_clips', '_tail'):
        monkeypatch.setattr(pipe, name, _device_step, raising=False)
    for name in ('filter_ball', 'filter_ball_timed', 'filter_ball_clips', 'filter_ball_clips_timed', 'trajectory_pack'):
        monkeypatch.setattr(ops, name, _device_step)
    monkeypatch.setattr(torch.cuda, 'device_count', _device_step)
    return pipe


@pytest.mark.parametrize('bad,words', BAD)
def test_predict_refuses_bad_stamps_before_any_device_step(monkeypatch, bad, words):
    pipe = _blocked_pipe(monkeypatch)
    with pytest.raises(ValueError, match=words):
        pipe.predict([0, 1, 2, 3], None, timestamps=bad)


def test_predict_needs_exactly_one_time_source(monkeypatch):
    pipe = _blocked_pipe(monkeypatch)
    for fps, ts in ((FPS, [0.0, 0.1, 0.2]), (None, None), (0.0, [0.0, 0.1, 0.2])):
        with pytest.raises(ValueError, match='either fps'):
            pipe.predict([0, 1, 2], fps, timestamps=ts)
        with pytest.raises(ValueError, match='either fps'):
            pipe.predict_clips([[0, 1, 2]], fps, timestamps=None if ts is None else [ts])


@pytest.mark.parametrize('bad,words', BAD[:-1])
@pytest.mark.parametrize('devices', [None, [0, 1]])
def test_predict_clips_refuses_bad_stamps_naming_the_clip(monkeypatch, bad, words, devices):
    pipe = _blocked_pipe(monkeypatch)
    clips = [[0, 1, 2], [3, 4, 5, 6], [7, 8, 9, 10]]
    good = [[0.0, 0.1, 0.2], [5.0, 5.1, 5.2, 5.3]]
    with pytest.raises(ValueError, match='clip 2: .*' + words):
        pipe.predict_clips(clips, None, devices=devices, timestamps=good + [bad])
    with pytest.raises(ValueError, match='timestamps: 2 entries for 3 clips'):
        pipe.predict_clips(clips, None, devices=devices, timestamps=good)
    with pytest.raises(ValueError, match='timestamps: 4 entries for 3 clips'):
        pipe.predict_clips(clips, None, devices=devices, timestamps=good + [[0, 1, 2, 3]] * 2)


# ---- predict and predict_clips with their device steps modelled ------------------------------------------------------------------
class _Model(torch.nn.Linear):
    def __init__(self, dtype='tf32'):
        super().__init__(2, 2)
        self.compute_dtype = dtype


class _Det:
    """A detector over frames that are their own ids (ints): a ball stack's position is (its centre frame, 7, 1), a table stack's 13
    keypoints are its frame."""
    segment = 512

    def __init__(self, frames_per_stack):
        self.frames_per_stack = frames_per_stack
        self.model = _Model()

    def _upload(self, images, dev, out=None):
        return torch.tensor(images, dtype=torch.float64), list(range(len(images))), None

    def _run(self, frames, stride, n_stacks, return_heatmaps, ready, heatmaps_to_host=False, first=None):
        f0 = first[0] if first is not None else [s * stride for s in range(n_stacks)]
        if self.frames_per_stack == 3:
            pos = torch.stack([torch.tensor([[frames[f + 1], 7.0, 1.0]], dtype=torch.float64) for f in f0])
        else:
            pos = torch.stack([torch.full((13, 3), float(frames[f]), dtype=torch.float64) for f in f0])
        return pos, None


class _Up:
    transform_mode = 'global'

    def __init__(self):
        self.model = _Model('tf32x3')

    def predict_without_normalization(self, ball, table, mask, times):
        n = int(mask.sum().item())
        return torch.zeros(3), np.stack([ball[0, :n, 0].numpy(), times[0, :n].numpy(), np.zeros(n)], axis=1)


class _Filters:
    """CPU models of the ball filters (every row kept), the table filter and the packing; records each call."""

    def __init__(self, monkeypatch, timed_allowed=True):
        self.calls = []
        for name in ('filter_ball', 'filter_ball_clips', 'filter_ball_timed', 'filter_ball_clips_timed', 'filter_table',
                     'filter_table_clips', 'trajectory_pack'):
            monkeypatch.setattr(ops, name, getattr(self, name))
        self.timed_allowed = timed_allowed

    def _timed(self):
        if not self.timed_allowed:
            raise AssertionError('a timed filter ran for a call with fps')

    def filter_ball(self, p1, p2, fps):
        self.calls.append(('filter_ball', fps))
        T = p1.shape[0]
        return p1[:, :2].clone(), torch.arange(T), torch.arange(T, dtype=torch.float64) / fps, torch.tensor([0, T], dtype=torch.int32)

    def filter_ball_timed(self, p1, p2, stamps):
        self._timed()
        self.calls.append(('filter_ball_timed', stamps.clone()))
        T = p1.shape[0]
        return p1[:, :2].clone(), torch.arange(T), stamps - stamps[0], torch.tensor([0, T], dtype=torch.int32)

    def filter_ball_clips(self, p1, p2, offs, fps):
        self.calls.append(('filter_ball_clips', fps, offs.clone()))
        local = torch.cat([torch.arange(int(offs[c + 1] - offs[c])) for c in range(len(offs) - 1)])
        return p1[:, :2].clone(), local, local.double() / fps, offs.clone()

    def filter_ball_clips_timed(self, p1, p2, offs, stamps):
        self._timed()
        self.calls.append(('filter_ball_clips_timed', stamps.clone(), offs.clone(), p1[:, 0].long().tolist()))
        first = torch.cat([stamps[offs[c]].repeat(int(offs[c + 1] - offs[c])) for c in range(len(offs) - 1)])
        return p1[:, :2].clone(), None, stamps - first, offs.clone()

    def filter_table(self, t1, t2):
        return t1[0]

    def filter_table_clips(self, t1, t2, offs):
        return torch.stack([t1[int(offs[c])] for c in range(len(offs) - 1)])

    def trajectory_pack(self, ball_xy, times, offsets, table, *args):
        n = len(offsets) - 1
        ball, tms, mask = torch.zeros((n, 50, 2)), torch.zeros((n, 50)), torch.zeros((n, 50))
        for c in range(n):
            a, b = int(offsets[c]), int(offsets[c + 1])
            ball[c, :b - a], tms[c, :b - a], mask[c, :b - a] = ball_xy[a:b].float(), times[a:b].float(), 1
        return ball, table, tms, mask


def _pipe(monkeypatch):
    pipe = TableTennisPipeline.__new__(TableTennisPipeline)
    pipe.ball_detector, pipe.ball_detector_aux = _Det(3), _Det(3)
    pipe.table_detector, pipe.table_detector_aux = _Det(1), _Det(1)
    pipe.uplifting_model = _Up()
    pipe.device = torch.device('cpu')
    pipe._home_device = lambda: torch.device('cpu')
    pipe._replica_parts = lambda slot, device_index: pipe._parts()

    def uplift(parts, packed, counts):
        ball, _, times, mask = packed
        return torch.zeros((len(counts), 3)), np.stack([ball[:, :, 0].numpy(), times.numpy(), np.zeros(times.shape)], axis=2)

    pipe._uplift_clips = uplift
    monkeypatch.setattr(torch.cuda, 'current_device', lambda: 0)
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: 2)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: None)
    monkeypatch.setattr(interface, '_upload_stamps', lambda stamps, dev: torch.from_numpy(np.array(stamps, np.float64)))
    # the real host packing of _upload_plan, with the pinned buffer and the copy modelled on the CPU
    real = interface._upload_plan

    def upload_plan(plan, stamps, dev):
        with monkeypatch.context() as m:
            m.setattr(torch.Tensor, 'pin_memory', lambda self: self)
            return real(plan, stamps, torch.device('cpu'))

    monkeypatch.setattr(interface, '_upload_plan', upload_plan)
    return pipe


def _epoch_stamps(rng, n):
    return 1.7e9 + np.cumsum(rng.choice([0.02, 0.04, 0.06], n) + rng.uniform(-1e-3, 1e-3, n))


@pytest.mark.parametrize('lengths', [[3], [4], [50], [3, 4, 50], [17, 3, 3, 29, 4, 50, 8], [50] * 12])
@pytest.mark.parametrize('devices', [None, [0, 1, 1]])
def test_predict_clips_stamp_layout(monkeypatch, lengths, devices):
    rng = np.random.default_rng(len(lengths))
    pipe = _pipe(monkeypatch)
    filters = _Filters(monkeypatch)
    pipe.ball_detector.segment = 60                         # several blocks when the clips are long
    ids, clips, stamps = 0, [], []
    for n in lengths:
        clips.append(list(range(ids, ids + n)))
        stamps.append(_epoch_stamps(rng, n))
        ids += n
    out = pipe.predict_clips(clips, None, devices=devices, timestamps=stamps)
    # every block's filter got its clips' centre-frame stamps, row by row in the ball stacks' order
    calls = [c for c in filters.calls if c[0] == 'filter_ball_clips_timed']
    assert calls and not [c for c in filters.calls if c[0] == 'filter_ball_clips']
    frame_stamp = dict(zip(range(ids), np.concatenate(stamps)))
    rows = []                                               # (centre frame, stamp) of every ball row (blocks may run on threads)
    for _, st, offs, centre in calls:
        assert st.dtype == torch.float64 and offs.dtype == torch.int32 and offs[0] == 0 and offs[-1] == st.shape[0] == len(centre)
        rows += list(zip(centre, st.numpy().tolist()))
    centre = [f for c in clips for f in c[1:-1]]
    assert sorted(f for f, _ in rows) == centre and len(centre) == sum(n - 2 for n in lengths)
    assert all(t == frame_stamp[f] for f, t in rows)
    if devices is None:                                     # one thread: the blocks in clip order
        assert np.array_equal(torch.cat([c[1] for c in calls]).numpy(), ball_row_stamps(stamps))
    # the plan that came with them is clip_stack_plan's
    first, offs = clip_stack_plan(lengths, 3)
    assert len(first) == len(centre) and offs[-1] == len(centre)
    # each result: the positions of its clip's centre frames and the times of predict(c, None, timestamps=t)
    for (spin, pos), c, ts in zip(out, clips, stamps):
        assert np.array_equal(pos[:, 0], np.array(c[1:-1], np.float32))
        assert np.array_equal(pos[:, 1], (ts[1:-1] - ts[1]).astype(np.float32))
    want = [pipe.predict(c, None, timestamps=t) for c, t in zip(clips, stamps)]
    for (s, p), (s2, p2) in zip(out, want):
        assert torch.equal(s, s2) and np.array_equal(p, p2)


def test_ball_row_stamps_layout():
    assert ball_row_stamps([]).shape == (0,)
    assert ball_row_stamps([np.array([1.0, 2.0, 3.0])]).tolist() == [2.0]
    assert ball_row_stamps([np.array([1.0, 2.0, 3.0, 4.0])]).tolist() == [2.0, 3.0]
    ts = np.arange(50, dtype=np.float64) * 0.02 + 1.7e9
    assert np.array_equal(ball_row_stamps([ts]), ts[1:49])
    got = ball_row_stamps([np.array([0.0, 1.0, 2.0]), np.array([10.0, 11.0, 12.0, 13.0]), ts])
    assert np.array_equal(got, np.concatenate([[1.0], [11.0, 12.0], ts[1:49]]))


@pytest.mark.parametrize('n_stamps', [0, 5, 300])
def test_upload_plan_packs_stamps_and_plan_in_one_buffer(monkeypatch, n_stamps):
    monkeypatch.setattr(torch.Tensor, 'pin_memory', lambda self: self)
    rng = np.random.default_rng(n_stamps)
    plan = rng.integers(-5, 1 << 30, 2 * n_stamps + 7).tolist()
    stamps = _epoch_stamps(rng, n_stamps)
    p, s = interface._upload_plan(plan, stamps, torch.device('cpu'))
    assert p.dtype == torch.int32 and p.tolist() == plan
    assert s.dtype == torch.float64 and np.array_equal(s.numpy().view(np.int64), stamps.view(np.int64))
    assert p.untyped_storage().data_ptr() == s.untyped_storage().data_ptr()        # one buffer, so one copy
    p, s = interface._upload_plan(plan, None, torch.device('cpu'))
    assert p.tolist() == plan and s is None


def test_predict_passes_the_centre_frame_stamps(monkeypatch):
    pipe = _pipe(monkeypatch)
    filters = _Filters(monkeypatch)
    ts = _epoch_stamps(np.random.default_rng(2), 9)
    spin, pos = pipe.predict(list(range(9)), None, timestamps=ts)
    (name, st), = [c for c in filters.calls if c[0].startswith('filter_ball')]
    assert name == 'filter_ball_timed' and np.array_equal(st.numpy(), ts[1:8])
    assert np.array_equal(pos[:, 1], (ts[1:8] - ts[1]).astype(np.float32))
    # timestamps (k - 1) / fps: the times of the fps path
    ts = (np.arange(9, dtype=np.float64) - 1) / FPS
    assert np.array_equal(pipe.predict(list(range(9)), None, timestamps=ts)[1], pipe.predict(list(range(9)), FPS)[1])


@pytest.mark.parametrize('devices', [None, [0, 1]])
def test_calls_with_fps_never_reach_the_timed_filters(monkeypatch, devices):
    pipe = _pipe(monkeypatch)
    filters = _Filters(monkeypatch, timed_allowed=False)
    monkeypatch.setattr(interface, '_upload_stamps', _device_step)
    clips = [list(range(0, 5)), list(range(5, 12))]
    pipe.predict(clips[0], FPS)
    pipe.predict_clips(clips, FPS, devices=devices)
    live = _Session(pipe, FPS, 2, 4, 8, devices=None)
    for s in (0, 1):
        live.push(s, clips[s])
    live.end_rally(0)
    live.end_rally(1)
    names = {c[0] for c in filters.calls}
    assert names == {'filter_ball', 'filter_ball_clips'}


# ---- live sessions ---------------------------------------------------------------------------------------------------------------
class _Session(LiveSession):
    """LiveSession with its pool modelled on the CPU (each slot holds a frame id) and the passes run by the _Det models on the slots'
    frames; end_rally runs the real _finish and TableTennisPipeline._tail."""

    def _alloc_pool(self, shape):
        self.slot = [None] * (self.streams * self.slots)
        self.writes = 0
        return [None]

    def _check_frames(self, frames):
        if self._pool is None:
            self._pool = self._alloc_pool(None)

    def _device_write(self, frames, p0):
        self.writes += 1
        self.slot[p0:p0 + len(frames)] = frames

    def _hand_off(self, e, frames, p0):                     # devices=[...]: the write runs on the entry's launcher
        e.submit(self._device_write, list(frames), p0)

    def _device_wrap(self, src, dst, m):
        self.slot[dst:dst + m] = self.slot[src:src + m]

    def _device_pass(self, fps, first, runs):
        e = self._entries[0]
        parts = self.pipe._parts()
        frames = [-1 if f is None else f for f in self.slot]
        a = 0
        for st, idx in runs:
            for d in ((0, 1) if fps == BALL else (2, 3)):
                pos = parts[d]._run(frames, 1, len(idx), False, None, first=(first[a:a + len(idx)], None))[0]
                self._store(e, st, d, idx[0], pos)
            a += len(idx)


def test_live_push_refuses_bad_stamps_before_any_device_step(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, None, 2, 4, 8)
    for bad, words in BAD[:-1]:
        with pytest.raises(ValueError, match='stream 1: .*' + words):
            live.push(1, [10, 11, 12, 13], timestamps=bad)
    with pytest.raises(ValueError, match='needs timestamps'):
        live.push(1, [10, 11, 12, 13])
    with pytest.raises(ValueError, match='needs timestamps'):
        live.push(1, [])
    assert live._pool is None                                # nothing was allocated, written or launched
    live.push(1, [10, 11], timestamps=[5.0, 5.5])
    writes = live.writes
    for bad in ([5.5, 6.0], [5.4, 6.0], [6.0, 5.9]):        # not after the rally's previous frame, or not increasing
        with pytest.raises(ValueError, match='stream 1: '):
            live.push(1, [12, 13], timestamps=bad)
    with pytest.raises(ValueError, match='stream 1: '):
        live.push(1, [12], timestamps=5.5)
    assert live.writes == writes and live._n[1] == 2 and live._stamps[1] == [5.0, 5.5]
    live.push(1, [12], timestamps=5.6)                      # a single frame takes a single stamp
    assert live._stamps[1] == [5.0, 5.5, 5.6]
    # the other stream's clock is its own
    live.push(0, [20, 21, 22], timestamps=[1.0, 2.0, 3.0])
    # a session with fps takes no stamps
    live = _Session(pipe, FPS, 1, 4, 8)
    with pytest.raises(ValueError, match='takes no timestamps'):
        live.push(0, [1, 2, 3], timestamps=[0.0, 0.1, 0.2])
    assert live._pool is None


@pytest.mark.parametrize('devices', [None, [0]])
def test_live_stamps_across_wraps_and_streams(monkeypatch, devices):
    rng = random.Random(3)
    nrng = np.random.default_rng(3)
    pipe = _pipe(monkeypatch)
    filters = _Filters(monkeypatch)
    live = _Session(pipe, None, 3, 4, 8, devices=devices)
    targets = [[23, 9, 41], [12, 30, 3, 17], [49, 5]]        # rally lengths per stream; an 8-slot pool wraps inside them
    ids = iter(range(10 ** 6))
    done, left = [0, 0, 0], [t[0] for t in targets]
    rally = {s: ([], []) for s in range(3)}                 # per stream: the open rally's frames and stamps
    clock = [1.7e9, 1.7e9 + 3.0, 100.0]
    checked = 0
    while any(d < len(t) for d, t in zip(done, targets)):
        s = rng.choice([i for i in range(3) if done[i] < len(targets[i])])
        c = min(rng.choice([1, 1, 2, 5, 9]), left[s])
        frames = [next(ids) for _ in range(c)]
        stamps = [clock[s] + 0.02 * k + float(nrng.integers(0, 3)) * 0.02 for k in range(1, c + 1)]
        stamps = list(np.maximum.accumulate(stamps) + np.arange(c) * 1e-6)
        clock[s] = stamps[-1] if stamps else clock[s]
        if c == 1:
            live.push(s, frames, timestamps=stamps[0])          # one frame, one number
        else:
            live.push(s, frames, timestamps=np.array(stamps))
        rally[s][0].extend(frames)
        rally[s][1].extend(stamps)
        assert live._stamps[s] == rally[s][1]               # kept on the host, untouched by wraps
        left[s] -= c
        if left[s] == 0:
            frames, stamps = rally[s]
            filters.calls.clear()
            spin, pos = live.end_rally(s)
            (name, st), = [x for x in filters.calls if x[0].startswith('filter_ball')]
            assert name == 'filter_ball_timed' and st.numpy().tolist() == stamps[1:-1]
            assert np.array_equal(pos[:, 0], np.array(frames[1:-1], np.float32))     # the pool held the rally's frames
            want = pipe.predict(frames, None, timestamps=stamps)
            assert torch.equal(spin, want[0]) and np.array_equal(pos, want[1])
            assert live._stamps[s] == [] and live._n[s] == 0  # reset with the rally
            checked += 1
            rally[s] = ([], [])
            clock[s] -= 5.0                                 # a new rally may restart the clock
            done[s] += 1
            left[s] = targets[s][done[s]] if done[s] < len(targets[s]) else 0
    assert checked == sum(len(t) for t in targets)
    live.close()


def test_live_stamps_reset_when_end_rally_raises(monkeypatch):
    pipe = _pipe(monkeypatch)
    _Filters(monkeypatch)
    live = _Session(pipe, None, 1, 4, 8)
    live.push(0, [1, 2], timestamps=[10.0, 11.0])
    with pytest.raises(ValueError, match='at least 3'):
        live.end_rally(0)
    assert live._stamps[0] == []
    live.push(0, [3, 4, 5], timestamps=[0.0, 0.5, 0.7])        # an earlier clock is fine in a new rally
    spin, pos = live.end_rally(0)
    assert np.array_equal(pos[:, 1], np.array([0.0], np.float32))
