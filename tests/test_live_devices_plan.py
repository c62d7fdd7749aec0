"""Host logic of TableTennisPipeline.live(..., devices=[...]): streams in contiguous blocks over the entries, each entry's device work
on a launcher thread of its own in push order, replicas rebuilt when the models change, launcher errors, and the `devices` argument.
LiveSession runs with its device work replaced by a model of each entry's pool, run where the real work runs (the entry's launcher,
or the caller's thread for devices=None): every pass must read frames of its own entry's streams, inside their regions and not yet
overwritten, and each rally must be covered by exactly predict's stacks, all detected with one replica of the weights it opened
under, by the time its tail runs.  No GPU needed."""
import random
import threading

import numpy as np
import pytest
import torch

from upliftingtabletennis_b200 import sharding
from upliftingtabletennis_b200.interface import _fingerprint
from upliftingtabletennis_b200.live import BALL, TABLE, LiveSession

GPUS = 4


@pytest.fixture(autouse=True)
def fake_gpus(monkeypatch):
    monkeypatch.setattr(torch.cuda, 'device_count', lambda: GPUS)
    monkeypatch.setattr(torch.cuda, 'set_device', lambda d: None)


class FakePipe:
    def __init__(self):
        self.models = []
        for _ in range(5):
            m = torch.nn.Linear(2, 2)
            m.compute_dtype = 'tf32'
            self.models.append(m)
        self.builds = []                # (replica cache key, device) of every replica build

    def _parts(self):
        return [type('Part', (), {'model': m})() for m in self.models]

    def key(self):
        return tuple(_fingerprint(m) for m in self.models)

    def _replica_parts(self, slot, device_index):
        self.builds.append((slot, device_index))
        return ('replica', len(self.builds), self.key())


class FakeSession(LiveSession):
    """LiveSession whose device work is a model of each entry's pool (each slot holds a frame's (stream, rally, index) label)."""

    def __init__(self, streams, slots, k, devices):
        super().__init__(FakePipe(), 50.0, streams, k, slots, devices)
        self.rally = [0] * streams
        self.labels = {}                # id(frame) -> (stream, rally, index)
        self.keep = []
        self.launched = {}              # (stream, rally, frames per stack) -> stack indices, in launch order
        self.used = {}                  # (stream, rally) -> replicas its stacks were detected with
        self.threads = {}               # entry -> threads its device work ran on
        self.fail = None                # entry whose next pass raises

    def frames(self, s, count):
        out = []
        for _ in range(count):
            f = np.zeros((2, 2, 3), np.uint8)
            self.labels[id(f)] = (s, self.rally[s], self._n[s] + len(out))
            out.append(f)
        self.keep += out
        return out

    def _reset(self, s):
        super()._reset(s)
        self.rally[s] += 1

    def _on_thread(self, e):
        t = threading.current_thread()
        if e.launcher is None:
            assert t is threading.main_thread()
        else:
            assert t.name.startswith('ttk-live%d' % e.device.index)
        self.threads.setdefault(id(e), set()).add(t)

    def _alloc_pool(self, shape):
        for e in self._entries:
            e.pool = [None] * (len(e.streams) * self.slots)
        return [e.pool for e in self._entries]

    RING = 3                            # staging ring slots: small, so that pushes refill slots the launcher may still read

    def _alloc_ring(self, e, cuda):
        return [{} for _ in range(self.RING)]

    def _stage(self, e, slot, f, done):
        assert not threading.current_thread().name.startswith('ttk-live')      # on the caller's thread
        slot['label'] = self.labels[id(f)]

    def _device_write(self, frames, p0, staged=None):
        e = self._entry[p0 // self.slots]
        self._on_thread(e)
        assert e.base <= p0 and p0 - e.base + len(frames) <= len(e.pool)
        labels = [f['label'] if isinstance(f, dict) else self.labels[id(f)] for f in frames]     # a ring slot, or the frame itself
        e.pool[p0 - e.base:p0 - e.base + len(frames)] = labels

    def _device_wrap(self, src, dst, m):
        e = self._entry[dst // self.slots]
        self._on_thread(e)
        src, dst = src - e.base, dst - e.base
        assert dst + m <= src or m == 0
        e.pool[dst:dst + m] = e.pool[src:src + m]

    def _device_pass(self, fps, first, runs):
        e = self._entry[runs[0][0]]
        self._on_thread(e)
        if self.fail is e:
            raise OSError('launcher failure')
        stacks = [(st, j) for st, idx in runs for j in idx]
        assert len(stacks) == len(first)
        for (st, j), p in zip(stacks, first):
            assert st in e.streams                                                  # the entry's own streams
            assert st * self.slots <= p and p + fps <= (st + 1) * self.slots          # inside the stream's region
            got = e.pool[p - e.base:p - e.base + fps]
            r = got[0][1]
            assert got == [(st, r, j + i) for i in range(fps)]                      # its frames, none overwritten
            self.launched.setdefault((st, r, fps), []).append(j)
            self.used.setdefault((st, r), set()).add(e.parts)

    def _finish(self, s, n):
        e = self._entry[s]
        self._on_thread(e)
        r = self.rally[s]
        # every stack of the rally has been detected before its tail runs, with the replica of the weights the rally opened under
        assert self.launched.get((s, r, BALL), []) == list(range(n - 2))
        assert self.launched.get((s, r, TABLE), []) == list(range(n))
        if e.launcher is not None:
            assert self.used[(s, r)] == {e.parts} and e.parts[2] == self.pipe.key()
        return s, r, n


def _push(session, s, count):
    session.push(s, session.frames(s, count))
    for e in session._entries:                  # the k rule, per entry
        assert len(e.pending[BALL]) < session.k and len(e.pending[TABLE]) < session.k


def _builds(session):
    """The entries whose replicas were built, in order, once every launcher has run what it was given."""
    for e in session._entries:
        e.launcher.submit(lambda: None).result()
    return [slot[2] for slot, _ in session.pipe.builds]


def _close(session):
    session.close()
    # no rally, ended or dropped, had stacks detected with two replicas: no pass mixed rallies opened under different weights
    assert all(len(used) == 1 for used in session.used.values())
    assert not [t for t in threading.enumerate() if t.name.startswith('ttk-live')]


DEVICES = [None, [0], [0, 0], [1, 3], [2, 0, 1]]


@pytest.mark.parametrize('streams,devices', [(5, [0, 1, 2]), (4, [3, 3]), (3, [0, 1, 2]), (7, [1, 0]), (2, None)])
def test_streams_map_to_entries_by_shard_range(streams, devices):
    live = FakeSession(streams, 8, 4, devices)
    n = 1 if devices is None else len(devices)
    for r in range(n):
        a, b = sharding.shard_range(streams, r, n)
        e = live._entries[r]
        assert e.streams == range(a, b) and all(live._entry[s] is e for s in range(a, b))
        assert (e.device, e.launcher) == (None, None) if devices is None else e.device == torch.device('cuda', devices[r])
    _close(live)


@pytest.mark.parametrize('devices', DEVICES)
@pytest.mark.parametrize('slots,k', [(8, 16), (8, 1), (5, 100), (64, 16)])
def test_ragged_pushes_and_back_to_back_rallies(devices, slots, k):
    live = FakeSession(1 if devices is None else len(devices), slots, k, devices)
    for chunks in ([1, 5, 2, 17, 1, 1, 9], [3], [20], [7, 7, 7, 1, 20], [60]):
        for s in range(live.streams):
            for c in chunks:
                _push(live, s, c)
            r = live.rally[s]
            assert live.end_rally(s) == (s, r, sum(chunks))
    _close(live)


@pytest.mark.parametrize('devices', DEVICES)
@pytest.mark.parametrize('slots,k', [(8, 16), (8, 4), (6, 2), (64, 16)])
def test_interleaved_streams(devices, slots, k):
    rng = random.Random(slots * 31 + k + len(devices or []))
    targets = [[23, 9, 41], [12, 30, 3, 17], [49, 5], [8, 8, 27], [33]]     # rally lengths per stream, ending at different times
    live = FakeSession(len(targets), slots, k, devices)
    done, left, ended = [0] * len(targets), [t[0] for t in targets], []
    while any(d < len(t) for d, t in zip(done, targets)):
        s = rng.choice([i for i in range(len(targets)) if done[i] < len(targets[i])])
        c = min(rng.choice([1, 1, 2, 5, 9]), left[s])
        if c:
            _push(live, s, c)
            left[s] -= c
        if left[s] == 0:
            e = live._entry[s]
            others = [x for x in e.pending[TABLE] if x[0] != s]
            r = live.rally[s]
            assert live.end_rally(s) == (s, r, targets[s][done[s]])
            ended.append(targets[s][done[s]])
            assert e.pending[TABLE] == others           # end_rally flushes its own stream's stacks only
            done[s] += 1
            left[s] = targets[s][done[s]] if done[s] < len(targets[s]) else 0
    assert sorted(ended) == sorted(n for t in targets for n in t)
    for e in live._entries:                             # one thread per entry: the launcher, or the caller's
        assert len(live.threads.get(id(e), ())) == 1
    _close(live)


def test_devices_argument_errors():
    for devices in ('cuda:0', 0, torch.device('cuda', 0), [], [GPUS], [-1], ['cpu'], ['cuda'], [True], [1.0], ['cuda:x']):
        with pytest.raises(ValueError):
            FakeSession(4, 8, 4, devices)
    with pytest.raises(ValueError):
        FakeSession(2, 8, 4, [0, 1, 2])                 # more entries than streams
    with pytest.raises(ValueError):
        FakeSession(2, 8, 4, [0, 0, 0])
    # a repeated device is one entry per item; torch.device and 'cuda:N' name a device too
    live = FakeSession(3, 8, 4, [torch.device('cuda', 2), 'cuda:2', 1])
    assert [e.device.index for e in live._entries] == [2, 2, 1]
    assert len({id(e.launcher) for e in live._entries}) == 3
    _close(live)
    with pytest.raises(ValueError):                     # the other arguments are checked first, as without devices
        LiveSession(None, 50.0, streams=0, devices=[0])


@pytest.mark.parametrize('change', ['compute_dtype', 'in_place', 'load_state_dict', 'replaced'])
def test_a_model_change_drops_the_open_rallies_of_an_entry(change):
    live = FakeSession(4, 8, 3, [0, 1])                 # entry 0: streams 0, 1; entry 1: streams 2, 3
    for s in (0, 1, 2):
        _push(live, s, 5)
    _push(live, 1, 1)                                   # stream 1 has a ball and a table stack pending
    assert _builds(live) == [0, 1]
    m = live.pipe.models[2]
    if change == 'compute_dtype':
        m.compute_dtype = 'bf16'
    elif change == 'in_place':
        with torch.no_grad():
            m.weight.add_(1.0)
    elif change == 'load_state_dict':
        m.load_state_dict({k: v + 1 for k, v in m.state_dict().items()})
    else:
        m.weight = torch.nn.Parameter(m.weight.detach().clone())
    with pytest.raises(RuntimeError):
        if change == 'replaced':                        # a push compares version counters only; end_rally the whole fingerprint
            live.end_rally(0)
        else:
            live.push(0, live.frames(0, 1))
    assert live._n[0] == 0
    # a new rally on entry 0 rebuilds its replicas; stream 1's open rally, detected with the old ones, is dropped at once ...
    _push(live, 0, 7)
    assert _builds(live) == [0, 1, 0]
    assert not [x for x in live._entries[0].pending[BALL] if x[0] == 1]
    with pytest.raises(RuntimeError):
        live.push(1, live.frames(1, 1))
    # ... and every new rally runs on the rebuilt replica (_finish checks it); entry 1 rebuilds at its next rally
    _push(live, 1, 6)
    for s, n in ((0, 7), (1, 6)):
        r = live.rally[s]
        assert live.end_rally(s) == (s, r, n)
    with pytest.raises(RuntimeError):
        live.end_rally(2)
    _push(live, 2, 4)
    r = live.rally[2]
    assert live.end_rally(2) == (2, r, 4)
    assert _builds(live) == [0, 1, 0, 1]
    _close(live)


def test_a_launcher_error_surfaces_on_its_entry_and_at_close():
    live = FakeSession(4, 8, 2, [0, 1])
    for s in range(4):
        _push(live, s, 3)
    bad = live._entries[1]
    live.fail = bad
    try:                                                # queues a pass that raises on entry 1's launcher; the push itself meets
        live.push(2, live.frames(2, 4))                 # the error already when it waits for a ring slot written after the pass
    except OSError:
        pass
    bad.launcher.submit(lambda: None).result()          # (the launcher has run it)
    for call in (lambda: live.push(3, live.frames(3, 1)), lambda: live.end_rally(2), lambda: live.push(2, live.frames(2, 1))):
        with pytest.raises(OSError, match='launcher failure'):
            call()
    # entry 0 goes on
    _push(live, 0, 5)
    r = live.rally[0]
    assert live.end_rally(0) == (0, r, 8)
    with pytest.raises(OSError, match='launcher failure'):
        live.close()
    assert not [t for t in threading.enumerate() if t.name.startswith('ttk-live')]
    assert live._entries[0].pool is None and live._entries[1].pool is None
    with pytest.raises(RuntimeError):
        live.push(0, live.frames(0, 1))                 # closed


def test_the_staging_ring_bounds_what_a_launcher_has_queued():
    live = FakeSession(2, 8, 100, [0])
    _push(live, 0, 2)
    gate = threading.Event()
    live._entries[0].launcher.submit(gate.wait)         # the launcher is busy (a long pass)
    _push(live, 1, live.RING)                           # fills the ring without waiting for the launcher
    t = threading.Thread(target=live.push, args=(0, live.frames(0, 1)))
    t.start()
    t.join(0.5)
    assert t.is_alive()                                 # one frame more waits for a slot the launcher has written out
    gate.set()
    t.join(10)
    assert not t.is_alive()
    for s, n in ((0, 3), (1, live.RING)):
        r = live.rally[s]
        assert live.end_rally(s) == (s, r, n)
    _close(live)


def test_a_failed_write_reaches_the_push_that_waits_for_its_slot():
    live = FakeSession(1, 8, 100, [0])
    _push(live, 0, 4)
    live._entries[0].launcher.submit(lambda: None).result()
    gate = threading.Event()
    live._entries[0].launcher.submit(gate.wait)

    def fail(*args):
        raise OSError('copy failure')
    live._device_write = fail
    live.push(0, live.frames(0, live.RING))             # queued behind the gate, each write fails
    gate.set()
    with pytest.raises(OSError, match='copy failure'):
        live.push(0, live.frames(0, 1))
    with pytest.raises(OSError, match='copy failure'):
        live.close()


def test_leaving_a_with_block_keeps_its_own_exception():
    live = FakeSession(2, 8, 2, [0, 1])
    live.fail = live._entries[1]
    with pytest.raises(KeyError):
        with live:
            _push(live, 1, 4)
            live._entries[1].launcher.submit(lambda: None).result()
            raise KeyError('the caller')
    assert not [t for t in threading.enumerate() if t.name.startswith('ttk-live')]


def test_end_rally_errors_leave_the_entry_usable():
    live = FakeSession(2, 8, 4, [0, 1])
    for n in (0, 1, 2):
        if n:
            _push(live, 1, n)
        with pytest.raises(ValueError):
            live.end_rally(1)
    _push(live, 1, 9)
    r = live.rally[1]
    assert live.end_rally(1) == (1, r, 9)
    assert live._entries[1].error is None
    _close(live)
