"""The rally cameras on the GPU: ttk_reproject_clips bit for bit against ttk_project per clip and its errors against a float64 numpy
loop; predict_clips(..., cameras=True) against the reference's overlay workflow (predict, both table detectors, filter_trajectory,
calibrate_camera, reproject) clip by clip, bit for bit, on one device, on two replicas of one device and on two GPUs; and
LiveSession.end_rally(..., cameras=True) against predict_clips.  Needs a B200: run with `-m gpu`."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


# ---- the kernel ---------------------------------------------------------------------------------------------
def _cameras(golden):
    g = golden('calibration')
    return [(g['Mint%d' % i], g['Mext%d' % i]) for i in range(int(g['n']))]


def _clip_inputs(cams, lengths, seed):
    """World points around the table, each clip's detections its true projection plus pixel noise."""
    from oracle import tails as otl
    rng = np.random.default_rng(seed)
    pts, det = [], []
    for c, n in enumerate(lengths):
        p = np.stack([rng.uniform(-1.5, 1.5, n), rng.uniform(-0.8, 0.8, n), rng.uniform(0.7, 2.0, n)], axis=1)
        mint, mext = cams[c % len(cams)]
        pts.append(p)
        det.append((otl.reproject(p, mint, mext) if n else np.zeros((0, 2))) + rng.normal(0, 2.0, (n, 2)))
    mint = np.stack([cams[c % len(cams)][0] for c in range(len(lengths))])
    mext = np.stack([cams[c % len(cams)][1] for c in range(len(lengths))])
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    return np.concatenate(pts), offs, mint, mext, np.concatenate(det)


def _reproject(dev, pts, offs, mint, mext, valid, det):
    from upliftingtabletennis_b200 import ops
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)     # noqa: E731
    xy, err = ops.reproject_clips(t(pts), t(offs), t(mint), t(mext), t(np.asarray(valid, np.int32)), t(det))
    return xy.cpu().numpy(), err.cpu().numpy()


def _error_loop(xy, det):
    """Mean (summed in row order) and max of the Euclidean pixel distances, in float64 on the host."""
    s, worst = 0.0, float('nan')
    for t in range(len(xy)):
        dx, dy = xy[t, 0] - det[t, 0], xy[t, 1] - det[t, 1]
        d = float(np.sqrt(dx * dx + dy * dy))
        s += d
        worst = d if t == 0 or d > worst else worst
    return (s / len(xy) if len(xy) else float('nan')), worst


LENGTHS = [1, 2, 49, 0, 17, 300]


def test_reproject_clips_equals_project_per_clip(dev, golden):
    from upliftingtabletennis_b200 import ops
    cams = _cameras(golden)
    pts, offs, mint, mext, det = _clip_inputs(cams, LENGTHS, 3)
    xy, err = _reproject(dev, pts, offs, mint, mext, [1] * len(LENGTHS), det)
    assert xy.shape == (len(pts), 2) and err.shape == (len(LENGTHS), 2)
    for c in range(len(LENGTHS)):
        a, b = offs[c], offs[c + 1]
        ref = ops.project(torch.from_numpy(pts[a:b]).to(dev), torch.from_numpy(mext[c]).to(dev), torch.from_numpy(mint[c]).to(dev))
        assert np.array_equal(_bits(xy[a:b]), _bits(ref.cpu().numpy())), c
        mean, worst = _error_loop(xy[a:b], det[a:b])
        if b == a:
            assert np.isnan(err[c]).all(), c
        else:
            assert np.array_equal(_bits(err[c]), _bits([mean, worst])), c
            assert 0.0 < mean <= worst < 20.0, c            # the detections are 2 px noise around the truth


def test_reproject_clips_invalid_clips_are_nan(dev, golden):
    cams = _cameras(golden)
    pts, offs, mint, mext, det = _clip_inputs(cams, LENGTHS, 4)
    xy, err = _reproject(dev, pts, offs, mint, mext, [1] * len(LENGTHS), det)
    valid = [1, 0, 1, 1, 0, 1]
    mint[1] = np.nan                                    # an invalid clip's matrices are not read
    xy2, err2 = _reproject(dev, pts, offs, mint, mext, valid, det)
    for c, ok in enumerate(valid):
        a, b = offs[c], offs[c + 1]
        if ok:
            assert np.array_equal(_bits(xy2[a:b]), _bits(xy[a:b])) and np.array_equal(_bits(err2[c]), _bits(err[c])), c
        else:
            assert np.isnan(xy2[a:b]).all() and np.isnan(err2[c]).all(), c
    # and nothing for no clips
    xy3, err3 = _reproject(dev, np.zeros((0, 3)), np.zeros(1, np.int32), np.zeros((0, 3, 4)), np.zeros((0, 4, 4)), [], np.zeros((0, 2)))
    assert xy3.shape == (0, 2) and err3.shape == (0, 2)


# ---- the pipeline ------------------------------------------------------------------------------------------------
RES = (192, 128)                      # detector input (W, H); frames are 1080p


def _write_weights(hub):
    """WASB, HRNet and uplifting checkpoints, written where _get_weights_path looks (as tests/test_gpu_pipeline_clips.py does)."""
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


# main and auxiliary detector of each kind share their weights: every ball stack agrees, and every table keypoint of a clip is visible
CLIP_LENGTHS = [3, 12, 50, 5, 27, 4, 51, 17, 9, 6]


def _clips(frames, lengths):
    out, f0 = [], 0
    for n in lengths:
        out.append(list(frames[f0:f0 + n]))
        f0 += n
    assert f0 <= len(frames)
    return out


def _pipeline(ball, table, dtype=None):
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    return TableTennisPipeline(ball_model=ball, ball_model_aux=ball, table_model=table, table_model_aux=table, dtype=dtype)


def _reference_workflow(pipe, clip, fps):
    """What a user of the reference runs to draw the trajectory: predict, both table detectors, filter_trajectory, calibrate_camera,
    reproject; plus the filtered ball detections of the two ball detectors."""
    spin, pos = pipe.predict(clip, fps)
    tk, _ = pipe.table_detector.predict(clip, return_heatmaps=False)
    tk_aux, _ = pipe.table_detector_aux.predict(clip, return_heatmaps=False)
    kp = pipe.table_detector.filter_trajectory(tk, tk_aux)
    triples = [(clip[i], clip[i + 1], clip[i + 2]) for i in range(len(clip) - 2)]
    bp, _ = pipe.ball_detector.predict(triples, return_heatmaps=False)
    bp_aux, _ = pipe.ball_detector_aux.predict(triples, return_heatmaps=False)
    det, _, _ = pipe.ball_detector.filter_trajectory(bp, bp_aux, fps)
    try:
        mint, mext = pipe.calibrate_camera(kp)
    except (AssertionError, ValueError) as e:
        return spin, pos, kp, det, None, None, None, str(e)
    return spin, pos, kp, det, mint, mext, pipe.reproject(pos, mint, mext), None


def _check_against_reference(got, want):
    spin, pos, cam = got
    rspin, rpos, kp, det, mint, mext, ball_2d, error = want
    assert spin.device == rspin.device and torch.equal(spin, rspin)
    assert pos.dtype == rpos.dtype and np.array_equal(pos, rpos)
    assert np.array_equal(_bits(cam.keypoints), _bits(kp))
    assert np.array_equal(_bits(cam.detections_2d), _bits(det)) and len(det) == len(pos)
    assert cam.error == error
    if error is not None:
        assert cam.Mint is None and cam.Mext is None and cam.ball_2d is None and cam.error_px is None
        return False
    assert np.array_equal(_bits(cam.Mint), _bits(mint)) and np.array_equal(_bits(cam.Mext), _bits(mext))
    assert np.array_equal(_bits(cam.ball_2d), _bits(ball_2d))
    assert cam.error_px == _error_loop(ball_2d, det)
    return True


def _assert_same(got, want):
    """Two lists of (spin, pos3d, RallyCamera), bit for bit."""
    assert len(got) == len(want)
    for i, ((s, p, c), (s2, p2, c2)) in enumerate(zip(got, want)):
        assert s.device == s2.device and torch.equal(s, s2) and np.array_equal(p, p2), i
        for f in c._fields:
            a, b = getattr(c, f), getattr(c2, f)
            if isinstance(a, np.ndarray):
                assert isinstance(b, np.ndarray) and a.shape == b.shape and np.array_equal(_bits(a), _bits(b)), (i, f)
            else:
                assert a == b, (i, f)


@pytest.mark.parametrize('dtype', [None, 'bf16'])
def test_predict_clips_cameras_equal_the_reference_workflow(dev, hub, frames, dtype):
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    pipe = _pipeline('wasb', 'hrnet', dtype=dtype)
    clips = _clips(frames, CLIP_LENGTHS)
    plain = pipe.predict_clips(clips, 50.0)
    got = pipe.predict_clips(clips, 50.0, cameras=True)
    assert [len(r) for r in got] == [3] * len(clips)
    calibrated = 0
    for i, c in enumerate(clips):
        assert torch.equal(got[i][0], plain[i][0]) and np.array_equal(got[i][1], plain[i][1])
        calibrated += _check_against_reference(got[i], _reference_workflow(pipe, c, 50.0))
    assert calibrated >= 1, [g[2].error for g in got]
    # a block of clips at a time: the same records
    pipe.ball_detector.segment = 64
    try:
        _assert_same(pipe.predict_clips(clips, 50.0, cameras=True), got)
    finally:
        del pipe.ball_detector.segment
    # an auxiliary table detector that disagrees: keypoints go invisible and calibrations fail; the other results still come back
    pipe.table_detector_aux.model.load_state_dict(synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=8))
    got = pipe.predict_clips(clips[:4], 50.0, cameras=True)
    failed = 0
    for i, c in enumerate(clips[:4]):
        failed += not _check_against_reference(got[i], _reference_workflow(pipe, c, 50.0))
    assert failed >= 1, [g[2].error for g in got]


def test_predict_clips_cameras_on_replicas(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    clips = _clips(frames, CLIP_LENGTHS)
    want = pipe.predict_clips(clips, 50.0, cameras=True)
    cur = torch.cuda.current_device()
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 0], cameras=True), want)
    assert torch.cuda.current_device() == cur
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 0, 0], cameras=True), want)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_predict_clips_cameras_two_gpus(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    clips = _clips(frames, CLIP_LENGTHS)
    want = pipe.predict_clips(clips, 50.0, cameras=True)
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 1], cameras=True), want)
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[1], cameras=True), want)


@pytest.mark.parametrize('devices', [None, [0]])
def test_end_rally_cameras_equal_predict_clips(dev, hub, frames, devices):
    pipe = _pipeline('wasb', 'hrnet')
    rallies = _clips(frames, [20, 3, 33])
    want = [pipe.predict_clips([r], 50.0, cameras=True)[0] for r in rallies]
    with pipe.live(50.0, streams=2, k=4, slots=16, devices=devices) as live:
        for r, rally in enumerate(rallies):
            for f in rally:
                live.push(r % 2, f)
            _assert_same([live.end_rally(r % 2, cameras=True)], [want[r]])
        for f in rallies[0]:
            live.push(1, f)
        spin, pos = live.end_rally(1)                   # cameras=False: predict's pair
        assert torch.equal(spin, want[0][0]) and np.array_equal(pos, want[0][1])
