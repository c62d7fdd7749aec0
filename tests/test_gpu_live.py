"""TableTennisPipeline.live on the GPU: every rally's end_rally against predict on the same frames, bit for bit -- one stream with
frames pushed one at a time, in ragged chunks and as one list; a small frame pool that wraps mid-rally and across rallies; three
interleaved streams; the errors predict raises, and the stream's next rally after each; frame shape and model changes; the pool's
memory after close().  Needs a B200: run with `-m gpu`."""
import os
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RES = (192, 128)                      # detector input (W, H): small, so that the fp32 SIMT paths stay quick; frames are 1080p
ARCHS = [('wasb', 'hrnet'), ('vitpose', 'hrnet'), ('wasb', 'vitpose')]


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available()
    return torch.device('cuda:0')


def _write_weights(hub):
    """Checkpoints for every architecture, written where _get_weights_path looks (as in test_gpu_pipeline_clips.py)."""
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


def _pipeline(ball, table, dtype=None):
    # main and auxiliary detector of each kind share their weights, so every ball stack agrees: a rally of n frames has n - 2
    # agreeing detections
    from upliftingtabletennis_b200.interface import TableTennisPipeline
    return TableTennisPipeline(ball_model=ball, ball_model_aux=ball, table_model=table, table_model_aux=table, dtype=dtype)


def _assert_same(got, want):
    (s, p), (s2, p2) = got, want
    assert isinstance(s, torch.Tensor) and s.device == s2.device and s.shape == s2.shape and s.dtype == s2.dtype
    assert isinstance(p, np.ndarray) and p.shape == p2.shape and p.dtype == p2.dtype
    assert torch.equal(s, s2) and np.array_equal(p, p2)


def _push_chunks(session, stream, frames, chunks):
    a = 0
    for c in chunks:
        session.push(stream, frames[a:a + c] if c > 1 else frames[a])
        a += c
    assert a == len(frames)


def _ragged(n, pattern=(1, 5, 2, 17)):
    out, i = [], 0
    while sum(out) < n:
        out.append(min(pattern[i % len(pattern)], n - sum(out)))
        i += 1
    return out


@pytest.mark.parametrize('dtype', [None, 'bf16', 'fp32'])
@pytest.mark.parametrize('archs', ARCHS)
def test_one_stream_equals_predict(dev, hub, frames, archs, dtype):
    pipe = _pipeline(*archs, dtype=dtype)
    rally = list(frames[:40])
    want = pipe.predict(rally, 50.0)
    assert want[1].shape[0] == 38
    with pipe.live(50.0) as live:
        for chunks in ([1] * 40, _ragged(40), [40]):
            _push_chunks(live, 0, rally, chunks)
            _assert_same(live.end_rally(0), want)
        if dtype is None:               # torch CPU and CUDA frames as well as numpy arrays
            _push_chunks(live, 0, [torch.from_numpy(f) for f in rally], _ragged(40, (3, 1, 7)))
            _assert_same(live.end_rally(0), want)
            live.push(0, torch.from_numpy(frames[:40]).to(dev))
            _assert_same(live.end_rally(0), want)


def test_pushed_frames_can_be_reused_at_once(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    rally = list(frames[:30])
    want = pipe.predict(rally, 50.0)
    shape = tuple(frames.shape[1:])
    with pipe.live(50.0) as live:
        # CUDA frames overwritten on the current stream and freed right after push; the freed block may be handed out again at once
        buf = torch.from_numpy(frames[:30]).to(dev)
        live.push(0, buf)
        buf.fill_(255)
        del buf
        junk = torch.zeros((30,) + shape, dtype=torch.uint8, device=dev)
        _assert_same(live.end_rally(0), want)
        del junk
        # one CUDA frame buffer that every frame is decoded into, as a GPU decoder does
        f = torch.empty(shape, dtype=torch.uint8, device=dev)
        for im in rally:
            f.copy_(torch.from_numpy(im).to(dev))
            live.push(0, f)
        _assert_same(live.end_rally(0), want)
        # one pinned host buffer, refilled after every push
        h = torch.empty(shape, dtype=torch.uint8).pin_memory()
        for im in rally:
            h.copy_(torch.from_numpy(im))
            live.push(0, h)
        _assert_same(live.end_rally(0), want)
        with pytest.raises(ValueError):
            live.push(0, [h, f])                # host and CUDA frames in one push


def test_wrap_mid_rally_and_across_rallies(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    lengths = [23, 3, 17, 30, 9]        # back to back in an 8-slot region: wraps inside rallies and right after rally ends
    clips, f0 = [], 0
    for n in lengths:
        clips.append(list(frames[f0:f0 + n]))
        f0 += n
    want = [pipe.predict(c, 50.0) for c in clips]
    for k in (16, 3):
        with pipe.live(50.0, slots=8, k=k) as live:
            for c, w in zip(clips, want):
                _push_chunks(live, 0, c, _ragged(len(c), (1, 5, 2, 17, 1)))
                _assert_same(live.end_rally(0), w)
            live.push(0, clips[3])      # one push longer than the region
            _assert_same(live.end_rally(0), want[3])


def test_three_streams_interleaved(dev, hub, frames):
    pipe = _pipeline('vitpose', 'hrnet')
    # frame ranges of each stream's rallies, ended one by one
    rallies = [[(0, 31), (31, 40)], [(40, 52), (52, 95), (95, 99)], [(99, 150), (150, 155)]]
    want = {(s, i): pipe.predict(list(frames[a:b]), 50.0) for s in range(3) for i, (a, b) in enumerate(rallies[s])}
    rng = random.Random(4)
    for k, slots in ((4, 8), (16, None)):
        with pipe.live(50.0, streams=3, k=k, slots=slots) as live:
            pos = [[r, a] for r, a in zip([0, 0, 0], [rs[0][0] for rs in rallies])]       # per stream: rally, next frame
            ended = 0
            while ended < sum(len(r) for r in rallies):
                s = rng.choice([i for i in range(3) if pos[i][0] < len(rallies[i])])
                r, a = pos[s]
                b = rallies[s][r][1]
                c = min(rng.choice([1, 1, 2, 3, 6]), b - a)
                live.push(s, list(frames[a:a + c]) if c > 1 else frames[a])
                pos[s][1] = a + c
                if a + c == b:
                    _assert_same(live.end_rally(s), want[(s, r)])
                    ended += 1
                    pos[s] = [r + 1, rallies[s][r + 1][0] if r + 1 < len(rallies[s]) else b]


def test_errors_leave_the_stream_usable(dev, hub, frames):
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    pipe = _pipeline('wasb', 'hrnet')
    good = list(frames[200:230])
    want = pipe.predict(good, 50.0)
    with pipe.live(50.0, slots=8) as live:
        for n in (0, 1, 2):             # fewer than 3 frames: no ball stack
            if n:
                live.push(0, list(frames[:n]))
            with pytest.raises(ValueError):
                live.end_rally(0)
            _push_chunks(live, 0, good, _ragged(len(good)))
            _assert_same(live.end_rally(0), want)
        # 52 frames: 50 agreeing detections, the all-ones mask predict rejects
        with pytest.raises(ValueError):
            pipe.predict(list(frames[:52]), 50.0)
        _push_chunks(live, 0, list(frames[:52]), _ragged(52))
        with pytest.raises(ValueError):
            live.end_rally(0)
        _push_chunks(live, 0, good, _ragged(len(good)))
        _assert_same(live.end_rally(0), want)
        # a frame of another shape is refused and the rally goes on
        live.push(0, good[:10])
        with pytest.raises(ValueError):
            live.push(0, np.zeros((720, 1280, 3), np.uint8))
        with pytest.raises(ValueError):
            live.push(0, good[10].astype(np.float32))
        live.push(0, good[10:])
        _assert_same(live.end_rally(0), want)
        # a compute_dtype changed while a rally is open
        live.push(0, good[:7])
        old = pipe.table_detector_aux.model.compute_dtype
        pipe.table_detector_aux.model.compute_dtype = 'bf16'
        with pytest.raises(RuntimeError):
            live.push(0, good[7])
        want_bf16 = pipe.predict(good, 50.0)
        _push_chunks(live, 0, good, _ragged(len(good)))
        _assert_same(live.end_rally(0), want_bf16)
        live.push(0, good[:7])
        pipe.table_detector_aux.model.compute_dtype = old
        with pytest.raises(RuntimeError):
            live.end_rally(0)
        # another auxiliary ball detector: the two disagree on most frames, and a rally with no agreeing detection fails in predict
        sd = {k: v.clone() for k, v in pipe.ball_detector_aux.model.state_dict().items()}
        pipe.ball_detector_aux.model.load_state_dict(synthetic.hrnet_state_dict(HRNetEngine(9, 3, 1, 1).state_dict_layout(), seed=8))
        failed = 0
        f0 = 0
        for n in (10, 4, 20, 7, 30, 12, 3):
            clip = list(frames[f0:f0 + n])
            f0 += n
            try:
                w = pipe.predict(clip, 50.0)
            except ValueError:
                failed += 1
                _push_chunks(live, 0, clip, _ragged(n))
                with pytest.raises(ValueError):
                    live.end_rally(0)
            else:
                _push_chunks(live, 0, clip, _ragged(n))
                _assert_same(live.end_rally(0), w)
        assert failed
        pipe.ball_detector_aux.model.load_state_dict(sd)
        _push_chunks(live, 0, good, _ragged(len(good)))
        _assert_same(live.end_rally(0), want)
    with pytest.raises(RuntimeError):
        live.push(0, good[0])           # closed


def test_close_releases_the_pool(dev, hub, frames):
    pipe = _pipeline('wasb', 'hrnet')
    rally = list(frames[:20])
    want = pipe.predict(rally, 50.0)
    for _ in range(2):                  # the first round warms every workspace a session uses
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        live = pipe.live(50.0, streams=2)
        live.push(0, rally)
        live.push(1, rally[:5])
        assert torch.cuda.memory_allocated() >= before + 2 * 64 * rally[0].nbytes
        got = live.end_rally(0)
        live.close()
        _assert_same(got, want)
        del got
        torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before
