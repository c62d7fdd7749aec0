"""Per-frame capture timestamps on the GPU, bit for bit: ttk_filter_ball_timed / ttk_filter_ball_clips_timed against a float64 numpy
restatement and, with stamps (k - 1) / fps, against the untimed kernels; predict with such stamps against predict with fps; a clip with
dropped frames against the reference workflow with its times shifted on the host; predict_clips and live sessions with stamps against
the predict loop.  Needs a B200: run with `-m gpu`."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RES = (192, 128)                      # detector input (W, H); frames are 1080p
FPS = 50.0


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _tbits(t):
    return t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t


# ---- the kernels -------------------------------------------------------------------------------------------------------------------
def _filter_numpy(p1, p2, offs, stamps, threshold=20.0):
    """The timed filters' contract in float64 numpy: keep row t unless the distance exceeds threshold (NaN is kept) or a detector does
    not see the ball; time = stamps[t] - stamps[first row of the clip]."""
    xy, idx, times, out_offs = [], [], [], [0]
    for c in range(len(offs) - 1):
        a, b = offs[c], offs[c + 1]
        for t in range(a, b):
            d = np.sqrt((p1[t, 0] - p2[t, 0]) * (p1[t, 0] - p2[t, 0]) + (p1[t, 1] - p2[t, 1]) * (p1[t, 1] - p2[t, 1]))
            if d > threshold or p1[t, 2] != 1.0 or p2[t, 2] != 1.0:
                continue
            xy.append(p1[t, :2])
            idx.append(t - a)
            times.append(stamps[t] - stamps[a])
        out_offs.append(len(idx))
    return np.array(xy, np.float64).reshape(-1, 2), np.array(idx, np.int64), np.array(times, np.float64), np.array(out_offs, np.int32)


def _detections(rng, n):
    """Two detectors' (x, y, v) rows: agreeing, disagreeing, invisible, NaN and exactly-20-px rows."""
    p1 = np.c_[rng.uniform(0, 1920, n), rng.uniform(0, 1080, n), np.ones(n)]
    p2 = p1.copy()
    kind = rng.integers(0, 6, n)
    p2[kind == 1, :2] += rng.uniform(-15, 15, (int((kind == 1).sum()), 2))
    p2[kind == 2, 0] += 30.0                                # 30 px apart: dropped
    p1[kind == 3, 2] = 0.0                                  # one detector does not see it
    p1[kind == 4, 0] = np.nan                               # NaN distance: kept, like `diff > 20` in the reference
    p2[kind == 5, 0] += 12.0                                # 12, 16: exactly 20 px, kept
    p2[kind == 5, 1] += 16.0
    return p1, p2


def _stamps(rng, lengths, origin):
    """Strictly increasing stamps per clip: frame gaps of 1, 2 or 3 frame times at ~50 fps with jitter, from `origin` on."""
    out = []
    for n in lengths:
        gaps = rng.choice([0.02, 0.04, 0.06], n) + rng.uniform(-1e-3, 1e-3, n)
        out.append(origin + rng.uniform(0, 100) + np.cumsum(gaps))
    return np.concatenate(out + [np.zeros(0)])


CLIP_ROWS = [0, 1, 37, 0, 1, 1500, 2, 0, 64, 1025]          # empty clips, one-row clips, several CTA passes


@pytest.mark.parametrize('origin', [0.0, 1.7e9])
def test_timed_filters_equal_numpy(dev, origin):
    from upliftingtabletennis_b200 import ops
    rng = np.random.default_rng(3)
    T = sum(CLIP_ROWS)
    p1, p2 = _detections(rng, T)
    stamps = _stamps(rng, CLIP_ROWS, origin)
    assert stamps.shape == (T,) and np.isfinite(p1[:, 0]).sum() < T
    offs = np.concatenate([[0], np.cumsum(CLIP_ROWS)]).astype(np.int32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    xy, idx, times, out_offs = ops.filter_ball_clips_timed(t(p1), t(p2), t(offs), t(stamps))
    want = _filter_numpy(p1, p2, offs, stamps)
    n = want[3][-1]
    assert np.array_equal(out_offs.cpu().numpy(), want[3])
    assert np.array_equal(_bits(xy[:n].cpu().numpy()), _bits(want[0]))
    assert np.array_equal(idx[:n].cpu().numpy(), want[1])
    assert np.array_equal(_bits(times[:n].cpu().numpy()), _bits(want[2]))
    # the one-clip kernel on each clip alone
    for c in range(len(CLIP_ROWS)):
        a, b = offs[c], offs[c + 1]
        xy1, idx1, times1, offs1 = ops.filter_ball_timed(t(p1[a:b]), t(p2[a:b]), t(stamps[a:b]))
        k0, k1 = want[3][c], want[3][c + 1]
        assert offs1.cpu().tolist() == [0, k1 - k0], c
        assert np.array_equal(_bits(xy1[:k1 - k0].cpu().numpy()), _bits(want[0][k0:k1])), c
        assert np.array_equal(idx1[:k1 - k0].cpu().numpy(), want[1][k0:k1]), c
        assert np.array_equal(_bits(times1[:k1 - k0].cpu().numpy()), _bits(want[2][k0:k1])), c


def test_timed_filters_equal_untimed_with_fps_stamps(dev):
    from upliftingtabletennis_b200 import ops
    rng = np.random.default_rng(4)
    T = sum(CLIP_ROWS)
    p1, p2 = _detections(rng, T)
    offs = np.concatenate([[0], np.cumsum(CLIP_ROWS)]).astype(np.int32)
    for fps in (50.0, 59.94, 30.0):
        # the stamps predict derives from timestamps[k] = (k - 1) / fps: ball row t is frame t + 1, stamp t / fps
        stamps = np.concatenate([np.arange(n) / fps for n in CLIP_ROWS])
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        got = ops.filter_ball_clips_timed(t(p1), t(p2), t(offs), t(stamps))
        want = ops.filter_ball_clips(t(p1), t(p2), t(offs), fps)
        n = int(want[3][-1])
        for g, w in zip(got, want):                       # bits: the xy of NaN-distance rows hold NaN
            assert g.dtype == w.dtype and torch.equal(_tbits(g[:n]), _tbits(w[:n]))
        assert torch.equal(got[3], want[3])
        a, b = offs[5], offs[6]
        got = ops.filter_ball_timed(t(p1[a:b]), t(p2[a:b]), t(stamps[a:b]))
        want = ops.filter_ball(t(p1[a:b]), t(p2[a:b]), fps)
        n = int(want[3][1])
        for g, w in zip(got, want):
            assert torch.equal(_tbits(g[:n]), _tbits(w[:n]))


# ---- the pipeline ------------------------------------------------------------------------------------------------------------------
def _write_weights(hub):
    """WASB, HRNet and uplifting checkpoints, written where _get_weights_path looks."""
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    from upliftingtabletennis_b200.uplift import get_model
    torch.hub.set_dir(hub)
    w = os.path.join(hub, 'checkpoints', 'tt_uplifting_extracted', 'weights')
    up = get_model('connectstage', 'large', 'dynamic', 'new')
    for sub, sd, info in (
            ('inference_balldetection/wasb', synthetic.hrnet_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=1),
             {'model_name': 'wasb', 'image_resolution': RES, 'in_frames': 3, 'lr': 0.0}),
            ('inference_tabledetection/hrnet', synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=2),
             {'model_name': 'hrnet', 'image_resolution': RES}),
            ('inference_uplifting/ours', synthetic.uplift_state_dict(up, seed=3),
             {'name': 'connectstage', 'size': 'large', 'tabletoken_mode': 'dynamic', 'time_rotation': 'new', 'transform_mode': 'global',
              'randdet_prob': 0.0, 'randmiss_prob': 0.0, 'tablemiss_prob': 0.0})):
        os.makedirs(os.path.join(w, sub), exist_ok=True)
        torch.save({'model_state_dict': sd, 'identifier': 'synthetic', 'additional_info': info}, os.path.join(w, sub, 'model.pt'))


@pytest.fixture(scope='module')
def hub(tmp_path_factory):
    d = str(tmp_path_factory.mktemp('hub'))
    _write_weights(d)
    return d


@pytest.fixture(scope='module')
def frames():
    from upliftingtabletennis_b200 import synthetic
    return synthetic.frames_1080p(200, seed=9)


def _pipeline(dtype=None):
    # main and auxiliary detector of each kind share their weights, so every ball stack agrees
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    return TableTennisPipeline(ball_model='wasb', ball_model_aux='wasb', table_model='hrnet', table_model_aux='hrnet', dtype=dtype)


def _skipping(frames, first, n, skip=3):
    """n frames from frames[first:] with every `skip`-th one dropped, and their capture times on a Unix-epoch clock at FPS."""
    keep = [k for k in range(first, first + n * skip) if (k - first) % skip != skip - 1][:n]
    return [frames[k] for k in keep], 1.7e9 + np.array(keep, np.float64) / FPS


def _assert_same(got, want):
    (s, p), (s2, p2) = got[:2], want[:2]
    assert isinstance(s, torch.Tensor) and s.device == s2.device and s.dtype == s2.dtype and torch.equal(s, s2)
    assert isinstance(p, np.ndarray) and p.dtype == p2.dtype and np.array_equal(p, p2)


@pytest.mark.parametrize('dtype', [None, 'bf16'])
def test_predict_with_fps_stamps_equals_predict(dev, hub, frames, dtype):
    pipe = _pipeline(dtype)
    clip = list(frames[:40])
    want = pipe.predict(clip, FPS)
    assert want[1].shape == (38, 3)
    stamps = (np.arange(len(clip), dtype=np.float64) - 1) / FPS
    _assert_same(pipe.predict(clip, None, timestamps=stamps), want)
    _assert_same(pipe.predict(clip, None, timestamps=list(stamps)), want)
    # shifted stamps change the times, and with them the trajectory
    got = pipe.predict(clip, None, timestamps=stamps * 2.0)
    assert got[1].shape == want[1].shape and not np.array_equal(got[1], want[1])


def test_dropped_frames_equal_the_reference_workflow(dev, hub, frames):
    from upliftingtabletennis_b200.interface import _uplifting_transform, filter_trajectory_ball, filter_trajectory_table
    pipe = _pipeline()
    clip, ts = _skipping(frames, 0, 45)
    spin, pos = pipe.predict(clip, None, timestamps=ts)
    assert pos.shape == (43, 3)
    # the reference's stages one by one, with the fps times replaced on the host by the capture times of the kept stacks' centre frames
    triples = [(clip[i], clip[i + 1], clip[i + 2]) for i in range(len(clip) - 2)]
    bp, _ = pipe.ball_detector.predict(triples, return_heatmaps=False)
    bp_aux, _ = pipe.ball_detector_aux.predict(triples, return_heatmaps=False)
    det, idx, _ = filter_trajectory_ball(bp, bp_aux, FPS)
    times = ts[idx + 1] - ts[1]
    tk, _ = pipe.table_detector.predict(clip, return_heatmaps=False)
    tk_aux, _ = pipe.table_detector_aux.predict(clip, return_heatmaps=False)
    kp = filter_trajectory_table(tk, tk_aux)
    b, t, ti, m = _uplifting_transform(det, kp, times)
    spin2, pos2 = pipe.uplifting_model.predict_without_normalization(b, t, m, ti)
    assert spin.device == spin2.device and torch.equal(spin, spin2)
    assert pos.dtype == pos2.dtype and np.array_equal(pos, pos2)
    # and it is not the constant-rate result
    assert not np.array_equal(pos, pipe.predict(clip, FPS)[1])


CLIP_LENGTHS = [3, 12, 40, 5, 27, 4, 17, 9]


def _clips_with_stamps(frames, lengths):
    clips, stamps, f0 = [], [], 0
    for i, n in enumerate(lengths):
        c, ts = _skipping(frames, f0, n, skip=2 + i % 3)
        clips.append(c)
        stamps.append(ts + 17.0 * i)
        f0 += n
    return clips, stamps


def test_predict_clips_with_stamps_equals_the_predict_loop(dev, hub, frames):
    pipe = _pipeline()
    clips, stamps = _clips_with_stamps(frames, CLIP_LENGTHS)
    want = [pipe.predict(c, None, timestamps=t) for c, t in zip(clips, stamps)]
    got = pipe.predict_clips(clips, None, timestamps=stamps)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        _assert_same(g, w)
    cur = torch.cuda.current_device()
    for g, w in zip(pipe.predict_clips(clips, None, devices=[0, 0], timestamps=stamps), want):
        _assert_same(g, w)
    assert torch.cuda.current_device() == cur
    # a block of clips at a time
    pipe.ball_detector.segment = 64
    try:
        for g, w in zip(pipe.predict_clips(clips, None, timestamps=stamps), want):
            _assert_same(g, w)
    finally:
        del pipe.ball_detector.segment
    # cameras: the same (spin, pos3d), and the camera of predict_clips on the clip alone
    cams = pipe.predict_clips(clips, None, cameras=True, timestamps=stamps)
    cams2 = pipe.predict_clips(clips, None, devices=[0, 0], cameras=True, timestamps=stamps)
    for i, (g, g2, w) in enumerate(zip(cams, cams2, want)):
        _assert_same(g, w)
        _assert_same(g2, w)
        alone = pipe.predict_clips([clips[i]], None, cameras=True, timestamps=[stamps[i]])[0][2]
        for f in alone._fields:
            a, b, c = getattr(g[2], f), getattr(g2[2], f), getattr(alone, f)
            if isinstance(c, np.ndarray):
                assert np.array_equal(_bits(a), _bits(c)) and np.array_equal(_bits(b), _bits(c)), (i, f)
            else:
                assert a == b == c, (i, f)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_predict_clips_with_stamps_two_gpus(dev, hub, frames):
    pipe = _pipeline()
    clips, stamps = _clips_with_stamps(frames, CLIP_LENGTHS)
    want = [pipe.predict(c, None, timestamps=t) for c, t in zip(clips, stamps)]
    for devices in ([0, 1], [1]):
        for g, w in zip(pipe.predict_clips(clips, None, devices=devices, timestamps=stamps), want):
            _assert_same(g, w)


@pytest.mark.parametrize('devices', [None, [0]])
def test_live_session_with_stamps_equals_predict(dev, hub, frames, devices):
    import random
    rng = random.Random(7)
    pipe = _pipeline()
    # per stream, rallies of frames with dropped ones (a caller that skips frames to keep up) and their camera times
    rallies = [[_skipping(frames, 0, 23), _skipping(frames, 60, 9, 2)],
               [_skipping(frames, 30, 31, 4), _skipping(frames, 100, 3)],
               [_skipping(frames, 120, 17, 2)]]
    want = {(s, r): pipe.predict(c, None, timestamps=ts) for s in range(3) for r, (c, ts) in enumerate(rallies[s])}
    with pipe.live(None, streams=3, k=4, slots=8, devices=devices) as live:
        pos = {s: [0, 0] for s in range(3)}          # per stream: rally, next frame
        while any(pos[s][0] < len(rallies[s]) for s in range(3)):
            s = rng.choice([i for i in range(3) if pos[i][0] < len(rallies[i])])
            r, a = pos[s]
            clip, ts = rallies[s][r]
            c = min(rng.choice([1, 1, 2, 5, 9]), len(clip) - a)
            if c == 1 and rng.random() < 0.5:
                live.push(s, clip[a], timestamps=float(ts[a]))          # one frame, one stamp
            else:
                live.push(s, clip[a:a + c], timestamps=ts[a:a + c])
            pos[s][1] = a + c
            if pos[s][1] == len(clip):
                _assert_same(live.end_rally(s), want[(s, r)])
                pos[s] = [r + 1, 0]
