"""Known tables on the GPU, bit for bit (predict / predict_clips with table_keypoints=, LiveSession.set_table): predict with a clip's own
filtered keypoints against predict; predict with another clip's keypoints, and with some of them invisible, against the reference
workflow with filter_trajectory_table replaced by them; predict_clips with a mixed list against the predict loop, on one device, on
replicas, with cameras and with timestamps; live sessions with tables set on some of three interleaved streams against predict; and
that the table detectors launch nothing when every table is known.  WASB + HRNet, and ViTPose as all four detectors, in the default
arithmetic and in bf16.  Needs a B200: run with `-m gpu`."""
import random

import numpy as np
import pytest
import torch

from test_gpu_live import _assert_same, _write_weights

pytestmark = pytest.mark.gpu

FPS = 50.0
# main and auxiliary detector of each kind share their weights, so that the ball detections and the table keypoints of a clip agree
COMPOSITIONS = {'wasb-hrnet': ('wasb', 'wasb', 'hrnet', 'hrnet'), 'vitpose': ('vitpose', 'vitpose', 'vitpose', 'vitpose')}
CASES = [('wasb-hrnet', None), ('wasb-hrnet', 'bf16'), ('vitpose', None), ('vitpose', 'bf16')]


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


@pytest.fixture(scope='module')
def hub(tmp_path_factory):
    d = str(tmp_path_factory.mktemp('hub'))
    _write_weights(d)
    return d


@pytest.fixture(scope='module')
def frames():
    from upliftingtabletennis_b200 import synthetic
    return synthetic.frames_1080p(200, seed=9)


def _pipeline(composition, dtype=None):
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    b, ba, t, ta = COMPOSITIONS[composition]
    return TableTennisPipeline(ball_model=b, ball_model_aux=ba, table_model=t, table_model_aux=ta, dtype=dtype)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


class _TableRuns:
    """Counts the passes of the pipeline's two table detectors (a pass is one _run call)."""

    def __init__(self, monkeypatch, pipe):
        self.calls = 0
        for det in (pipe.table_detector, pipe.table_detector_aux):
            run = det._run

            def counted(*args, _run=run, **kw):
                self.calls += 1
                return _run(*args, **kw)
            monkeypatch.setattr(det, '_run', counted)


def _own_keypoints(pipe, clip):
    return pipe.predict_clips([clip], FPS, cameras=True)[0][2].keypoints


def _hidden(kp, keys=(0, 5, 11)):
    out = kp.copy()
    out[list(keys)] = (-1.0, -1.0, 0.0)
    return out


def _reference(pipe, clip, K):
    """The reference workflow with a known table: both ball detectors on the triples, filter_trajectory_ball, _uplifting_transform with
    K, the uplifting model (and its rotation to local axes)."""
    from upliftingtabletennis_b200.interface import _uplifting_transform, filter_trajectory_ball
    triples = [(clip[i], clip[i + 1], clip[i + 2]) for i in range(len(clip) - 2)]
    bp, _ = pipe.ball_detector.predict(triples, return_heatmaps=False)
    bp_aux, _ = pipe.ball_detector_aux.predict(triples, return_heatmaps=False)
    det, _, times = filter_trajectory_ball(bp, bp_aux, FPS)
    b, t, ti, m = _uplifting_transform(det, K, times)
    return pipe.uplifting_model.predict_without_normalization(b, t, m, ti)


@pytest.mark.parametrize('composition,dtype', CASES)
def test_predict_with_known_tables(dev, hub, frames, monkeypatch, composition, dtype):
    pipe = _pipeline(composition, dtype)
    clip, other = list(frames[:40]), list(frames[100:130])
    want = pipe.predict(clip, FPS)
    own = _own_keypoints(pipe, clip)
    foreign = _own_keypoints(pipe, other)
    assert not np.array_equal(own, foreign) and foreign[:, 2].sum() >= 6
    runs = _TableRuns(monkeypatch, pipe)
    # the clip's own keypoints (numpy, a list, a CUDA tensor): predict's bits, and no table pass
    for K in (own, own.tolist(), torch.from_numpy(own).to(dev)):
        _assert_same(pipe.predict(clip, FPS, table_keypoints=K), want)
    assert runs.calls == 0
    # another clip's keypoints, and a copy with three of them invisible: the reference workflow with that K
    for K in (foreign, _hidden(foreign)):
        got = pipe.predict(clip, FPS, table_keypoints=K)
        _assert_same(got, _reference(pipe, clip, K))
        assert not np.array_equal(got[1], want[1])
    # with timestamps
    stamps = 1.7e9 + (np.arange(len(clip), dtype=np.float64) - 1) / FPS * 1.5
    got = pipe.predict(clip, None, timestamps=stamps, table_keypoints=own)
    assert runs.calls == 0
    _assert_same(got, pipe.predict(clip, None, timestamps=stamps))


CLIP_LENGTHS = [3, 12, 50, 5, 27, 4, 17, 9]


def _clips(frames, lengths):
    out, f0 = [], 0
    for n in lengths:
        out.append(list(frames[f0:f0 + n]))
        f0 += n
    return out


def _mixed_tables(pipe, frames):
    own = _own_keypoints(pipe, list(frames[150:190]))
    return [None, own, _hidden(own), None, own, own, None, _hidden(own, (2, 3))]


def _same_cameras(got, K, pipe):
    """A RallyCamera of a clip with the known table K: keypoints K, Mint / Mext calibrate_camera(K), ball_2d reproject."""
    spin, pos, cam = got
    assert np.array_equal(_bits(cam.keypoints), _bits(K))
    try:
        mint, mext = pipe.calibrate_camera(K)
    except (AssertionError, ValueError) as e:
        assert cam.error == str(e) and cam.Mint is None
        return
    assert cam.error is None
    assert np.array_equal(_bits(cam.Mint), _bits(mint)) and np.array_equal(_bits(cam.Mext), _bits(mext))
    assert np.array_equal(_bits(cam.ball_2d), _bits(pipe.reproject(pos, mint, mext)))


@pytest.mark.parametrize('composition,dtype', CASES)
def test_predict_clips_mixed_equal_the_predict_loop(dev, hub, frames, composition, dtype):
    pipe = _pipeline(composition, dtype)
    clips = _clips(frames, CLIP_LENGTHS)
    tables = _mixed_tables(pipe, frames)
    want = [pipe.predict(c, FPS, table_keypoints=K) for c, K in zip(clips, tables)]
    for devices in (None, [0, 0]):
        got = pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=tables)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            _assert_same(g, w)
    # a block of clips at a time
    pipe.ball_detector.segment = 64
    try:
        for g, w in zip(pipe.predict_clips(clips, FPS, table_keypoints=tables), want):
            _assert_same(g, w)
    finally:
        del pipe.ball_detector.segment
    # cameras: the same pairs, and the camera of the known table (or of the detected one, as predict_clips computes it alone)
    for devices in (None, [0, 0]):
        cams = pipe.predict_clips(clips, FPS, devices=devices, cameras=True, table_keypoints=tables)
        for i, (g, w, K) in enumerate(zip(cams, want, tables)):
            _assert_same(g[:2], w)
            _same_cameras(g, _own_keypoints(pipe, clips[i]) if K is None else K, pipe)
    # timestamps
    stamps = [1.7e9 + 10.0 * i + np.cumsum(np.full(len(c), 0.02 + 0.005 * (i % 3))) for i, c in enumerate(clips)]
    want = [pipe.predict(c, None, timestamps=ts, table_keypoints=K) for c, ts, K in zip(clips, stamps, tables)]
    for devices in (None, [0, 0]):
        for g, w in zip(pipe.predict_clips(clips, None, devices=devices, timestamps=stamps, table_keypoints=tables), want):
            _assert_same(g, w)


def test_predict_clips_every_table_known_launches_no_table_pass(dev, hub, frames, monkeypatch):
    pipe = _pipeline('wasb-hrnet')
    clips = _clips(frames, CLIP_LENGTHS)
    own = _own_keypoints(pipe, clips[2])
    tables = [own] * len(clips)
    want = [pipe.predict(c, FPS, table_keypoints=own) for c in clips]
    runs = _TableRuns(monkeypatch, pipe)
    for devices in (None, [0]):                 # ([0]: the pipeline's own models on a launcher thread)
        for g, w in zip(pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=tables), want):
            _assert_same(g, w)
    assert runs.calls == 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_predict_clips_mixed_two_gpus(dev, hub, frames):
    pipe = _pipeline('wasb-hrnet')
    clips = _clips(frames, CLIP_LENGTHS)
    tables = _mixed_tables(pipe, frames)
    want = [pipe.predict(c, FPS, table_keypoints=K) for c, K in zip(clips, tables)]
    for devices in ([0, 1], [1]):
        for g, w in zip(pipe.predict_clips(clips, FPS, devices=devices, table_keypoints=tables), want):
            _assert_same(g, w)


RALLIES = [[(0, 31), (31, 40), (60, 75)], [(40, 52), (75, 99)], [(99, 150), (150, 155)]]     # per stream: frame ranges of its rallies


@pytest.mark.parametrize('devices', [None, [0, 0]])
@pytest.mark.parametrize('composition,dtype', CASES)
def test_live_sessions_with_tables_equal_predict(dev, hub, frames, devices, composition, dtype):
    pipe = _pipeline(composition, dtype)
    own = _own_keypoints(pipe, list(frames[160:200]))
    # per stream and rally: the table set before it.  Stream 0 keeps one; stream 1 has none, then one; stream 2 one, then None again
    tables = [[own, own, own], [None, _hidden(own)], [own, None]]
    rng = random.Random(11)
    for cameras in (False, True):
        with pipe.live(FPS, streams=3, k=4, slots=8, devices=devices) as live:
            pos = [[0, rs[0][0]] for rs in RALLIES]
            for s in range(3):
                live.set_table(s, tables[s][0])
            while any(pos[s][0] < len(RALLIES[s]) for s in range(3)):
                s = rng.choice([i for i in range(3) if pos[i][0] < len(RALLIES[i])])
                r, a = pos[s]
                b = RALLIES[s][r][1]
                c = min(rng.choice([1, 1, 2, 3, 6]), b - a)
                live.push(s, list(frames[a:a + c]))
                pos[s][1] = a + c
                if a + c < b:
                    continue
                K = tables[s][r]
                clip = list(frames[RALLIES[s][r][0]:b])
                got = live.end_rally(s, cameras=cameras)
                _assert_same(got[:2], pipe.predict(clip, FPS, table_keypoints=K))
                if cameras:
                    _same_cameras(got, _own_keypoints(pipe, clip) if K is None else K, pipe)
                if r + 1 < len(RALLIES[s]):
                    live.set_table(s, tables[s][r + 1])
                    pos[s] = [r + 1, RALLIES[s][r + 1][0]]
                else:
                    pos[s] = [r + 1, b]


def test_live_stream_with_a_table_launches_no_table_pass(dev, hub, frames, monkeypatch):
    pipe = _pipeline('wasb-hrnet')
    clip = list(frames[:45])
    own = _own_keypoints(pipe, clip)
    want = pipe.predict(clip, FPS)
    runs = _TableRuns(monkeypatch, pipe)
    with pipe.live(FPS, streams=2, k=4, slots=8) as live:
        live.set_table(1, own)
        for f in clip:
            live.push(1, f)
        _assert_same(live.end_rally(1), want)
    assert runs.calls == 0
