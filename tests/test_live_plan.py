"""Host logic of TableTennisPipeline.live: where pushed frames go in a stream's region of the device frame pool, the wrap copy, which
stacks become ready after each push, and the session's arguments.  LiveSession itself runs with its device work replaced by a model
of the pool, which checks that every pass reads the frames its stacks name, inside their stream's region, and that each rally is
covered by exactly predict's stacks; the k rule, the per-stream flush, the errors and the model check run as they do on the GPU.
No GPU needed."""
import numpy as np
import pytest
import torch

from upliftingtabletennis_b200.live import BALL, TABLE, LiveSession, check_live_args, push_plan, ready_stacks


def test_push_plan_writes_in_order_and_wraps_at_the_region_end():
    assert push_plan(0, 0, 5, 8) == ([('write', 0, 0, 5)], 5, 5)
    # the last two frames of the open rally go to the start of the region
    assert push_plan(6, 30, 5, 8) == ([('write', 6, 0, 2), ('wrap', 6, 0, 2), ('write', 2, 2, 5)], 5, 35)
    # a rally that has one frame, or none yet, when the region is full
    assert push_plan(8, 1, 1, 8) == ([('wrap', 7, 0, 1), ('write', 1, 0, 1)], 2, 2)
    assert push_plan(8, 0, 3, 8) == ([('wrap', 8, 0, 0), ('write', 0, 0, 3)], 3, 3)
    # one push longer than the region wraps several times
    steps, w, n = push_plan(3, 0, 20, 8)
    assert steps == [('write', 3, 0, 5), ('wrap', 6, 0, 2), ('write', 2, 5, 11), ('wrap', 6, 0, 2), ('write', 2, 11, 17),
                     ('wrap', 6, 0, 2), ('write', 2, 17, 20)]
    assert (w, n) == (5, 20)
    assert push_plan(4, 2, 0, 8) == ([], 4, 2)


def test_ready_stacks_after_each_push():
    # ball stacks need their third frame, table stacks their frame
    assert ready_stacks(0, 1, 1, BALL) == [] and ready_stacks(1, 2, 2, BALL) == []
    assert ready_stacks(2, 3, 3, BALL) == [(0, 0)]
    assert ready_stacks(0, 5, 5, BALL) == [(0, 0), (1, 1), (2, 2)]
    assert ready_stacks(0, 5, 7, TABLE) == [(j, j + 2) for j in range(5)]
    assert ready_stacks(35, 38, 5, BALL) == [(33, 0), (34, 1), (35, 2)]      # after a wrap: frames 33, 34 were copied to slots 0, 1
    assert ready_stacks(4, 4, 4, BALL) == [] and ready_stacks(4, 4, 4, TABLE) == []


class FakeSession(LiveSession):
    """LiveSession with its device work replaced by a model of the pool (each slot holds a frame's (stream, rally, index) label):
    the bookkeeping under test is the session's own."""

    def __init__(self, streams, slots, k):
        super().__init__(FakePipe(), 50.0, streams, k, slots)
        self.rally = [0] * streams
        self.labels = {}                # id(frame) -> (stream, rally, index)
        self.keep = []
        self.launched = {}              # (stream, rally, frames per stack) -> stack indices, in launch order
        self.passes = []                # (frames per stack, [(stream, stack indices)])

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

    def _alloc_pool(self, shape):
        return [None] * (self.streams * self.slots)

    def _device_write(self, frames, p0):
        self._pool[p0:p0 + len(frames)] = [self.labels[id(f)] for f in frames]

    def _device_wrap(self, src, dst, m):
        assert dst + m <= src or m == 0
        self._pool[dst:dst + m] = self._pool[src:src + m]

    def _device_pass(self, fps, first, runs):
        self.passes.append((fps, runs))
        stacks = [(st, j) for st, idx in runs for j in idx]
        assert len(stacks) == len(first)
        for (st, j), p in zip(stacks, first):
            assert st * self.slots <= p and p + fps <= (st + 1) * self.slots          # inside the stream's region
            assert self._pool[p:p + fps] == [(st, self.rally[st], j + i) for i in range(fps)]       # its frames, none overwritten
            self.launched.setdefault((st, self.rally[st], fps), []).append(j)

    def _finish(self, s, n):
        return s, self.rally[s], n


class FakePipe:
    def __init__(self):
        self.models = []
        for _ in range(5):
            m = torch.nn.Linear(2, 2)
            m.compute_dtype = 'tf32'
            self.models.append(m)

    def _parts(self):
        return [type('Part', (), {'model': m})() for m in self.models]


def _push(session, s, count):
    session.push(s, session.frames(s, count))
    # the k rule: after a push, fewer than k stacks of each kind wait
    assert len(session._pending[BALL]) < session.k and len(session._pending[TABLE]) < session.k


def _check_coverage(session, lengths):
    for (s, r), n in lengths.items():
        # exactly predict's sliding windows: n - 2 ball stacks and n table stacks, each launched once, in order
        assert session.launched.get((s, r, BALL), []) == list(range(max(n - 2, 0))), (s, r)
        assert session.launched.get((s, r, TABLE), []) == list(range(n)), (s, r)


@pytest.mark.parametrize('slots,k', [(8, 16), (8, 1), (4, 3), (64, 16), (5, 100)])
def test_one_stream_ragged_pushes_and_back_to_back_rallies(slots, k):
    live = FakeSession(1, slots, k)
    lengths = {}
    for chunks in ([1, 5, 2, 17, 1, 1, 9], [3], [20], [7, 7, 7, 1, 20], [60]):
        for c in chunks:
            _push(live, 0, c)
        r = live.rally[0]
        assert live.end_rally(0) == (0, r, sum(chunks))
        lengths[(0, r)] = sum(chunks)
        assert not live._pending[BALL] and not live._pending[TABLE]
    _check_coverage(live, lengths)
    if k <= slots - 2:
        # a push launches a pass once k stacks are ready (a smaller region flushes at every wrap before k gather)
        assert any(len([j for _, idx in runs for j in idx]) >= k for _, runs in live.passes)


@pytest.mark.parametrize('slots,k', [(8, 16), (8, 4), (64, 16), (6, 2)])
def test_three_streams_interleaved(slots, k):
    import random
    rng = random.Random(slots * 31 + k)
    live = FakeSession(3, slots, k)
    targets = [[23, 9, 41], [12, 30, 3, 17], [49, 5]]          # rally lengths per stream, ending at different times
    done, left, lengths = [0, 0, 0], [t[0] for t in targets], {}
    while any(d < len(t) for d, t in zip(done, targets)):
        s = rng.choice([i for i in range(3) if done[i] < len(targets[i])])
        c = min(rng.choice([1, 1, 2, 5, 9]), left[s])
        if c:
            _push(live, s, c)
            left[s] -= c
        if left[s] == 0:
            others = [x for x in live._pending[TABLE] if x[0] != s]
            r = live.rally[s]
            assert live.end_rally(s) == (s, r, targets[s][done[s]])
            lengths[(s, r)] = targets[s][done[s]]
            assert live._pending[TABLE] == others           # end_rally flushes its own stream's stacks only
            done[s] += 1
            left[s] = targets[s][done[s]] if done[s] < len(targets[s]) else 0
    _check_coverage(live, lengths)
    assert sorted(lengths.values()) == sorted(n for t in targets for n in t)


def test_short_rallies_and_bad_frames():
    live = FakeSession(1, 8, 16)
    for n in (0, 1, 2):
        _push(live, 0, n) if n else None
        with pytest.raises(ValueError):
            live.end_rally(0)
        assert live._n[0] == 0
    _push(live, 0, 5)
    for bad in (np.zeros((4, 2, 3), np.uint8), np.zeros((2, 2, 3), np.float32), np.zeros((2, 2, 4), np.uint8)):
        with pytest.raises(ValueError):
            live.push(0, bad)
    assert live._n[0] == 5                                  # a refused push changes nothing
    _push(live, 0, 4)
    r = live.rally[0]
    assert live.end_rally(0) == (0, r, 9)
    _check_coverage(live, {(0, r): 9})
    with pytest.raises(ValueError):
        live.push(1, live.frames(0, 1))                     # no such stream
    live.close()
    with pytest.raises(RuntimeError):
        live.push(0, live.frames(0, 1))


@pytest.mark.parametrize('change', ['compute_dtype', 'in_place', 'load_state_dict', 'replaced'])
def test_a_model_change_drops_the_open_rally(change):
    live = FakeSession(2, 8, 16)
    _push(live, 0, 5)
    _push(live, 1, 5)
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
    if change == 'replaced':                                # a push compares version counters only; end_rally the whole fingerprint
        _push(live, 0, 1)
        with pytest.raises(RuntimeError):
            live.end_rally(0)
    else:
        with pytest.raises(RuntimeError):
            live.push(0, live.frames(0, 1))
    assert live._n[0] == 0 and not [x for x in live._pending[TABLE] if x[0] == 0]
    with pytest.raises(RuntimeError):
        live.end_rally(1)                                   # the other stream's rally was open too
    for s in (0, 1):                                        # new rallies start with the new models
        _push(live, s, 6)
        r = live.rally[s]
        assert live.end_rally(s) == (s, r, 6)


def test_arguments_are_validated():
    check_live_args(1, 1, 4)
    check_live_args(4, 16, 64)
    for streams, k, slots in ((0, 16, 64), (-1, 16, 64), (1.5, 16, 64), (True, 16, 64), ('2', 16, 64), (1, 0, 64), (1, None, 64),
                              (1, 2.0, 64), (1, 16, 3), (1, 16, 0)):
        with pytest.raises(ValueError):
            check_live_args(streams, k, slots)
    # the session checks them before it touches the pipeline or the GPU
    for kw in ({'streams': 0}, {'k': 0}, {'slots': 2}):
        with pytest.raises(ValueError):
            LiveSession(None, 50.0, **kw)
