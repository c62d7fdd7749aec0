"""TableTennisPipeline.predict_clips on the GPU: its three kernels (indexed pre-processing, the ball filter over several clips, the
table filter over clips of different lengths) bit for bit against the per-clip entry points, and the method against the per-clip
predict loop, bit for bit, on one device, on two replicas of one device and on two GPUs.  Needs a B200: run with `-m gpu`."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


# ---- kernels ------------------------------------------------------------------------------------------------
# (src h, w) -> (dst w, h): a downscale on the staged tile kernel (rows of 16-byte multiples), one on the per-pixel kernel (ragged
# rows) and the same-size copy
SIZES = [((96, 160), (96, 64)), ((70, 90), (48, 40)), ((64, 96), (96, 64))]
MODES = [('nchw', torch.float32), ('nhwc16', torch.float32), ('nhwc16', torch.bfloat16), ('nhwc16', torch.float16)]


@pytest.mark.parametrize('fps', [1, 3])
@pytest.mark.parametrize('size', SIZES)
@pytest.mark.parametrize('layout,dtype', MODES)
def test_preprocess_indexed_equals_per_stack(dev, fps, size, layout, dtype):
    from upliftingtabletennis_b200 import ops
    (sh, sw), (dw, dh) = size
    g = torch.Generator().manual_seed(7)
    frames = torch.randint(0, 256, (23, sh, sw, 3), dtype=torch.uint8, generator=g).to(dev)
    first = [0, 5, 5, 20, 1, 23 - fps, 11, 3, 12, 0, 17, 9, 2, 14, 6, 8, 19, 4, 10]      # repeats, out of order, both ends
    x = ops.preprocess_stacks_indexed(frames, fps, torch.tensor(first, dtype=torch.int32, device=dev), dw, dh, layout=layout, dtype=dtype)
    for s, f in enumerate(first):
        ref = ops.preprocess_stacks(frames[f:f + fps], fps, 1, 1, dw, dh, layout=layout, dtype=dtype)
        assert torch.equal(x[s:s + 1].view(torch.uint8), ref.view(torch.uint8)), (s, f)


def _ball_detections(lengths, seed):
    rng = np.random.default_rng(seed)
    n = sum(lengths)
    p1 = np.stack([rng.uniform(0, 1920, n), rng.uniform(0, 1080, n), (rng.uniform(0, 1, n) > 0.1).astype(np.float64)], axis=1)
    p2 = p1.copy()
    p2[:, 2] = (rng.uniform(0, 1, n) > 0.1).astype(np.float64)
    kind = rng.integers(0, 5, n)
    p2[kind == 0, :2] += rng.uniform(-30, 30, (int((kind == 0).sum()), 2))          # some agree within 20 px, some do not
    p2[kind == 1, 0] += 12.0                                                        # distance exactly 20: kept (`diff > 20` drops)
    p2[kind == 1, 1] += 16.0
    p1[kind == 2, 0] = np.nan                                                       # NaN distances are kept
    p2[kind == 3, :2] += 40.0
    return p1, p2


def test_filter_ball_clips_equals_per_clip(dev):
    from upliftingtabletennis_b200 import ops
    lengths = [0, 1, 5, 0, 1100, 37, 1, 0, 2048, 0]          # empty clips (also first and last), one frame, several CTA-wide loops
    p1, p2 = _ball_detections(lengths, 3)
    # exact ties where p1 already holds integers: move to integer coordinates so that the 12 / 16 offsets give exactly 20
    p1[:, :2] = np.round(p1[:, :2])
    p2[:, :2] = np.where(np.isnan(p2[:, :2]), p2[:, :2], np.round(p2[:, :2]))
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    t1, t2 = torch.from_numpy(p1).to(dev), torch.from_numpy(p2).to(dev)
    xy, idx, times, out_offs = ops.filter_ball_clips(t1, t2, torch.from_numpy(offs).to(dev), 50.0)
    out_offs = out_offs.cpu().numpy()
    assert out_offs[0] == 0 and np.all(np.diff(out_offs) >= 0)
    seen_nan = seen_tie = False
    for c in range(len(lengths)):
        a, b = offs[c], offs[c + 1]
        rxy, ridx, rtimes, roffs = ops.filter_ball(t1[a:b], t2[a:b], 50.0)
        n = int(roffs[1])
        assert out_offs[c + 1] - out_offs[c] == n, c
        lo, hi = out_offs[c], out_offs[c + 1]
        assert torch.equal(xy[lo:hi].view(torch.int64), rxy[:n].view(torch.int64)), c         # bitwise, NaN included
        assert torch.equal(idx[lo:hi], ridx[:n]) and torch.equal(times[lo:hi], rtimes[:n]), c
        seen_nan |= bool(torch.isnan(rxy[:n]).any())
        d = np.hypot(p1[a:b, 0] - p2[a:b, 0], p1[a:b, 1] - p2[a:b, 1])
        seen_tie |= bool(np.any((d == 20.0) & (p1[a:b, 2] == 1) & (p2[a:b, 2] == 1)))
    assert seen_nan and seen_tie
    assert out_offs[-1] == sum(int(out_offs[c + 1] - out_offs[c]) for c in range(len(lengths)))


def test_filter_table_clips_equals_per_clip(dev):
    from upliftingtabletennis_b200 import ops
    lengths = [0, 1, 2, 3, 7, 50, 300, 0, 64]
    rng = np.random.default_rng(11)
    n, K = sum(lengths), 13
    # integer grid coordinates: distances of exactly eps (10) between points and of exactly 10 between the two detectors occur
    base = rng.integers(100, 1800, (1, K, 2)).astype(np.float64)
    p1 = np.concatenate([base + 5 * rng.integers(0, 6, (n, K, 2)), (rng.uniform(0, 1, (n, K, 1)) > 0.1).astype(np.float64)], axis=2)
    p2 = p1.copy()
    p2[..., :2] += rng.choice([0.0, 3.0, 6.0, 8.0, 10.0, 30.0], (n, K, 2), p=[0.3, 0.2, 0.2, 0.1, 0.1, 0.1])
    p2[..., 2] = (rng.uniform(0, 1, (n, K)) > 0.1).astype(np.float64)
    p1[rng.uniform(0, 1, (n, K)) < 0.1, 0] += 200.0                           # outliers: noise points and second clusters
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    t1, t2 = torch.from_numpy(p1).to(dev), torch.from_numpy(p2).to(dev)
    out = ops.filter_table_clips(t1, t2, torch.from_numpy(offs).to(dev))
    assert out.shape == (len(lengths), K, 3)
    for c in range(len(lengths)):
        a, b = offs[c], offs[c + 1]
        ref = ops.filter_table(t1[a:b], t2[a:b])
        assert torch.equal(out[c].view(torch.int64), ref.view(torch.int64)), c
    # the uniform batched entry point agrees too, on clips of one length
    same = torch.stack([t1[offs[5]:offs[6]], t1[offs[8]:offs[8] + 50]]), torch.stack([t2[offs[5]:offs[6]], t2[offs[8]:offs[8] + 50]])
    offs2 = torch.tensor([0, 50, 100], dtype=torch.int32, device=dev)
    assert torch.equal(ops.filter_table(*same), ops.filter_table_clips(same[0].reshape(100, K, 3), same[1].reshape(100, K, 3), offs2))


# ---- the method ---------------------------------------------------------------------------------------------
RES = (192, 128)                      # detector input (W, H): small, so that the fp32 SIMT paths stay quick; frames are 1080p


def _write_weights(hub):
    """Checkpoints for every architecture, written where _get_weights_path looks (like test_full_pipeline_1080p_rally)."""
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    from upliftingtabletennis_b200.uplift import get_model
    from upliftingtabletennis_b200.vitpose import state_dict_layout
    torch.hub.set_dir(hub)
    w = os.path.join(hub, 'checkpoints', 'tt_uplifting_extracted', 'weights')
    tokens = (RES[0] // 16) * (RES[1] // 16)
    up = get_model('connectstage', 'large', 'dynamic', 'new')
    for sub, sd, info in (
            ('inference_balldetection/wasb', synthetic.hrnet_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=1),
             {'model_name': 'wasb', 'image_resolution': RES, 'in_frames': 3, 'lr': 0.0}),
            ('inference_balldetection/vitpose', synthetic.vit_state_dict(state_dict_layout(9, tokens, 1), seed=4),
             {'model_name': 'vitpose', 'image_resolution': RES, 'in_frames': 3, 'lr': 0.0}),
            ('inference_tabledetection/hrnet', synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=2),
             {'model_name': 'hrnet', 'image_resolution': RES}),
            ('inference_tabledetection/vitpose', synthetic.vit_state_dict(state_dict_layout(3, tokens, 13), seed=5),
             {'model_name': 'vitpose', 'image_resolution': RES}),
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
    return synthetic.frames_1080p(300, seed=9)


# main and auxiliary detector of each kind share their weights, so every ball stack agrees: a clip of n frames has n - 2 detections
LENGTHS = [3, 12, 50, 5, 27, 4, 51, 17, 40, 9, 33, 6]           # 1 to 49 detections
ARCHS = [('vitpose', 'hrnet'), ('wasb', 'vitpose')]


def _clips(frames, lengths):
    out, f0 = [], 0
    for n in lengths:
        out.append(list(frames[f0:f0 + n]))
        f0 += n
    assert f0 <= len(frames)
    return out


def _assert_same(got, want):
    assert len(got) == len(want)
    for i, ((s, p), (s2, p2)) in enumerate(zip(got, want)):
        assert isinstance(s, torch.Tensor) and s.device == s2.device and s.shape == s2.shape and s.dtype == s2.dtype, i
        assert isinstance(p, np.ndarray) and p.shape == p2.shape and p.dtype == p2.dtype, i
        assert torch.equal(s, s2) and np.array_equal(p, p2), i


def _pipeline(ball, table, dtype=None):
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    return TableTennisPipeline(ball_model=ball, ball_model_aux=ball, table_model=table, table_model_aux=table, dtype=dtype)


@pytest.mark.parametrize('dtype', [None, 'bf16', 'fp32'])
@pytest.mark.parametrize('archs', ARCHS)
def test_predict_clips_equals_predict(dev, hub, frames, archs, dtype):
    pipe = _pipeline(*archs, dtype=dtype)
    clips = _clips(frames, LENGTHS)
    want = [pipe.predict(c, 50.0) for c in clips]
    assert [p.shape[0] for _, p in want] == [n - 2 for n in LENGTHS]
    cur = torch.cuda.current_device()
    _assert_same(pipe.predict_clips(clips, 50.0), want)
    assert torch.cuda.current_device() == cur
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 0]), want)        # two replicas on one GPU
    assert torch.cuda.current_device() == cur
    # a block of clips at a time: the same results when the blocks hold a few clips each
    pipe.ball_detector.segment = 64
    try:
        _assert_same(pipe.predict_clips(clips, 50.0), want)
    finally:
        del pipe.ball_detector.segment
    assert pipe.predict_clips([], 50.0) == []


def test_predict_clips_errors_match_predict(dev, hub, frames):
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    pipe = _pipeline('wasb', 'hrnet')
    # 52 and 60 frames: 50 and 58 agreeing detections -> the all-ones mask predict rejects; clip 3 is the first such clip
    clips = _clips(frames, [10, 4, 20, 52, 7, 60, 12])
    for i in (3, 5):
        with pytest.raises(ValueError):
            pipe.predict(clips[i], 50.0)
    for devices in (None, [0, 0]):
        with pytest.raises(ValueError, match=r'clip 3 \(50 agreeing'):
            pipe.predict_clips(clips, 50.0, devices=devices)
    # another auxiliary ball detector: the two now disagree on most frames, and a clip with no agreeing detection fails in predict
    pipe.ball_detector_aux.model.load_state_dict(synthetic.hrnet_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=8))
    clips = _clips(frames, [10, 4, 20, 7, 30, 12, 3])
    first_bad = None
    for i, c in enumerate(clips):
        try:
            pipe.predict(c, 50.0)
        except ValueError:
            first_bad = i if first_bad is None else first_bad
    assert first_bad is not None
    for devices in (None, [0, 0]):                # [0, 0]: the replicas follow the changed weights
        with pytest.raises(ValueError, match=r'clip %d \(0 agreeing' % first_bad):
            pipe.predict_clips(clips, 50.0, devices=devices)
    with pytest.raises(ValueError, match='clip 1'):
        pipe.predict_clips([clips[0], clips[1][:2]], 50.0)


def test_predict_clips_replicas_follow_the_pipeline(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    clips = _clips(frames, [9, 14, 30, 6, 21])
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 'cuda:0', torch.device('cuda', 0)]),
                 [pipe.predict(c, 50.0) for c in clips])
    pipe.table_detector_aux.model.compute_dtype = 'bf16'
    pipe.table_detector.model.compute_dtype = 'bf16'
    pipe.uplifting_model.model.compute_dtype = 'fp32'
    _assert_same(pipe.predict_clips(clips, 50.0, devices=[0, 0, 0]), [pipe.predict(c, 50.0) for c in clips])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_predict_clips_two_gpus(dev, hub, frames):
    pipe = _pipeline('vitpose', 'hrnet')
    clips = _clips(frames, LENGTHS)
    want = [pipe.predict(c, 50.0) for c in clips]
    cur = torch.cuda.current_device()
    got = pipe.predict_clips(clips, 50.0, devices=[0, 1])
    assert torch.cuda.current_device() == cur
    _assert_same(got, want)
