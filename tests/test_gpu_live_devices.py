"""TableTennisPipeline.live(..., devices=[...]) on the GPU: every rally's end_rally against predict on the same frames, bit for bit, with
the streams spread over entries that each run on a launcher thread with their own replicas -- three interleaved streams pushed singly
and in ragged chunks through an 8-slot pool that wraps; WASB + HRNet in every arithmetic class (and with fp16 auxiliary detectors),
ViTPose main detectors and the default composition; frames reused right after push; predict called while rallies are open; a model
change mid-rally; and, where two GPUs are visible, entries on both, one entry off the pipeline's device, and CUDA frames pushed from
the other GPU.  Needs a B200: run with `-m gpu`."""
import random
import threading

import numpy as np
import pytest
import torch

from test_gpu_live import _assert_same, _push_chunks, _ragged, _write_weights

pytestmark = pytest.mark.gpu

RALLIES = [[(0, 31), (31, 40)], [(40, 52), (52, 95)], [(99, 150), (150, 155)]]     # per stream: frame ranges of its rallies
COMPOSITIONS = {'wasb-hrnet': ('wasb', 'wasb', 'hrnet', 'hrnet'), 'vitpose': ('vitpose', 'vitpose', 'vitpose', 'hrnet'),
                'default': ('vitpose', 'wasb', 'vitpose', 'hrnet')}


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


def _predict(pipe, clip):
    """predict's result, or the ValueError class it raises (the default composition's main and auxiliary ball detectors disagree)."""
    try:
        return pipe.predict(clip, 50.0)
    except ValueError:
        return ValueError


def _check(live, s, want):
    device = torch.cuda.current_device()
    if want is ValueError:
        with pytest.raises(ValueError):
            live.end_rally(s)
    else:
        _assert_same(live.end_rally(s), want)
    assert torch.cuda.current_device() == device


def _interleaved(live, frames, want, seed, as_frame=lambda f: f):
    """Three streams, their rallies pushed in random interleaved chunks (singly and ragged), each ended when its last frame is in."""
    rng = random.Random(seed)
    pos = [[0, rs[0][0]] for rs in RALLIES]                 # per stream: rally, next frame
    ended = 0
    while ended < sum(len(r) for r in RALLIES):
        s = rng.choice([i for i in range(3) if pos[i][0] < len(RALLIES[i])])
        r, a = pos[s]
        b = RALLIES[s][r][1]
        c = min(rng.choice([1, 1, 2, 3, 6]), b - a)
        live.push(s, [as_frame(f) for f in frames[a:a + c]] if c > 1 else as_frame(frames[a]))
        pos[s][1] = a + c
        if a + c == b:
            _check(live, s, want[(s, r)])
            ended += 1
            pos[s] = [r + 1, RALLIES[s][r + 1][0] if r + 1 < len(RALLIES[s]) else b]


def _want(pipe, frames):
    return {(s, i): _predict(pipe, list(frames[a:b])) for s in range(3) for i, (a, b) in enumerate(RALLIES[s])}


@pytest.mark.parametrize('devices', [[0, 0], [0]])
@pytest.mark.parametrize('composition,dtype', [('wasb-hrnet', None), ('wasb-hrnet', 'bf16'), ('wasb-hrnet', 'fp32'),
                                               ('wasb-hrnet', 'fp16-aux'), ('vitpose', None), ('default', None)])
def test_interleaved_streams_equal_predict(hub, frames, devices, composition, dtype):
    pipe = _pipeline(composition, None if dtype == 'fp16-aux' else dtype)
    if dtype == 'fp16-aux':
        pipe.ball_detector_aux.model.compute_dtype = 'fp16'
        pipe.table_detector_aux.model.compute_dtype = 'fp16'
    want = _want(pipe, frames)
    if composition != 'default':
        assert ValueError not in want.values()
    for k, slots in ((4, 8), (16, None)):
        with pipe.live(50.0, streams=3, k=k, slots=slots, devices=devices) as live:
            _interleaved(live, frames, want, seed=k)


@pytest.mark.parametrize('devices', [[0, 0], [0]])
def test_pushed_frames_can_be_reused_at_once(hub, frames, devices):
    dev = torch.device('cuda:0')
    pipe = _pipeline('wasb-hrnet')
    rally = list(frames[:30])
    other = list(frames[100:120])
    want, want_other = pipe.predict(rally, 50.0), pipe.predict(other, 50.0)
    shape = tuple(frames.shape[1:])
    with pipe.live(50.0, streams=2, slots=8, devices=devices) as live:
        # one numpy buffer refilled after every push; predict runs on the pipeline's own models while both rallies are open
        buf = np.empty(shape, np.uint8)
        for i, im in enumerate(rally):
            buf[...] = im
            live.push(0, buf)
            if i < len(other):
                live.push(1, other[i])
            if i == 10:
                _assert_same(pipe.predict(rally, 50.0), want)
        _assert_same(live.end_rally(0), want)
        _assert_same(live.end_rally(1), want_other)
        # one pinned host buffer, refilled after every push
        h = torch.empty(shape, dtype=torch.uint8).pin_memory()
        for im in rally:
            h.copy_(torch.from_numpy(im))
            live.push(0, h)
        _assert_same(live.end_rally(0), want)
        # CUDA frames overwritten on the current stream and freed right after push; the freed block may be handed out again at once
        cuda = torch.from_numpy(frames[:30]).to(dev)
        live.push(0, cuda)
        cuda.fill_(255)
        del cuda
        junk = torch.zeros((30,) + shape, dtype=torch.uint8, device=dev)
        _assert_same(live.end_rally(0), want)
        del junk
        # one CUDA frame buffer that every frame is decoded into, as a GPU decoder does
        f = torch.empty(shape, dtype=torch.uint8, device=dev)
        for im in other:
            f.copy_(torch.from_numpy(im).to(dev))
            live.push(1, f)
        _assert_same(live.end_rally(1), want_other)


@pytest.mark.parametrize('devices', [[0, 0], [0]])
def test_cuda_pushes_do_not_wait_for_queued_passes(hub, frames, devices):
    dev = torch.device('cuda:0')
    pipe = _pipeline('wasb-hrnet')
    rally = list(frames[:12])
    want = pipe.predict(rally, 50.0)
    cuda = [torch.from_numpy(f).to(dev) for f in rally]
    with pipe.live(50.0, streams=len(devices), k=2, devices=devices) as live:
        live.push(0, cuda[:4])                          # passes queued on the launcher
        gate = threading.Event()
        live._entries[0].launcher.submit(gate.wait)     # and the launcher busy, as with a long pass
        t = threading.Thread(target=live.push, args=(0, cuda[4:]))
        t.start()
        t.join(60)
        returned = not t.is_alive()
        gate.set()
        t.join()
        assert returned                                 # 8 frames fit the staging ring: push did not wait for the launcher
        for f in cuda:
            f.fill_(7)                                  # overwritten right after push, on the stream the copies ran on
        _assert_same(live.end_rally(0), want)


@pytest.mark.parametrize('devices', [[0, 0], [0]])
def test_a_model_change_mid_rally_raises(hub, frames, devices):
    from upliftingtabletennis_b200 import synthetic
    from upliftingtabletennis_b200.detector import HRNetEngine
    pipe = _pipeline('wasb-hrnet')
    good = list(frames[:25])
    want = pipe.predict(good, 50.0)
    with pipe.live(50.0, streams=2, slots=8, devices=devices) as live:
        live.push(0, good[:9])
        live.push(1, good[:4])
        sd = {k: v.clone() for k, v in pipe.table_detector_aux.model.state_dict().items()}
        pipe.table_detector_aux.model.load_state_dict(synthetic.hrnet_state_dict(HRNetEngine(3, 13, 0, 13).state_dict_layout(), seed=6))
        for s in (0, 1):
            with pytest.raises(RuntimeError):
                live.push(s, good[9])
        want_new = pipe.predict(good, 50.0)
        for s in (0, 1):
            _push_chunks(live, s, good, _ragged(len(good)))
            _check(live, s, want_new)
        pipe.table_detector_aux.model.load_state_dict(sd)
        _push_chunks(live, 1, good, _ragged(len(good)))
        _check(live, 1, want)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
@pytest.mark.parametrize('devices', [[0, 1], [1], ['cuda:1', 'cuda:0']])
def test_two_gpus(hub, frames, devices):
    pipe = _pipeline('wasb-hrnet')
    want = _want(pipe, frames)
    with pipe.live(50.0, streams=3, slots=8, k=4, devices=devices) as live:
        _interleaved(live, frames, want, seed=1)
        # CUDA frames on the other GPU than their stream's entry (and on the entry's own), freed right after push
        for on in (0, 1):
            cuda = torch.device('cuda', on)
            _interleaved(live, frames, want, seed=2 + on, as_frame=lambda f: torch.from_numpy(f).to(cuda))
    with pipe.live(50.0, streams=3, devices=devices) as live:
        _interleaved(live, frames, want, seed=5)
