"""Live sessions of TableTennisPipeline (TableTennisPipeline.live): frames are detected as the cameras deliver them, and each rally's
spin and trajectory come back as soon as the caller ends it, exactly as predict would return them for the rally's frames.

Entries: a session serves its streams from one entry (devices=None: the current device, driven on the caller's thread) or from one
entry per item of `devices` (a contiguous block of streams each, sharding.shard_range), each with its own device state, its own copy
of the five models and one launcher thread that runs the entry's device work in push order.

Device frame pool: stream s owns the `slots` frames s * slots .. (s + 1) * slots - 1 of the session, held in its entry's uint8 CUDA
tensor from (s - first stream of the entry) * slots on, and writes them in order.  When its write position reaches the region's end,
the last two frames of the open rally are copied to the start of the region (on the copy stream, after the compute stream) and writing
goes on from there, so every stack of every stream is "first frame + 0, 1, 2" inside the pool and a pass that mixes the streams of an
entry is one ttk_preprocess_stacks_indexed call, as in predict_clips.

The bookkeeping is kept in pure functions (push_plan, ready_stacks, check_live_args) so that it can be checked without a GPU."""
import functools
import itertools
import numbers
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _lib, ops, sharding
from .interface import _Detector, _fingerprint, _upload_tables, check_table_keypoints, check_timestamps, parse_devices

DEFAULT_K = 16          # ready stacks that launch a pass: _Detector.chunk, predict's pass size; 137-143 frames/s for k = 4..32 on
                        # WASB + HRNet (profiles/r06_live_timing.json), so no reason to give ViTPose's GEMMs fewer M tiles
DEFAULT_SLOTS = 64      # frames per stream (398 MB at 1080p): a wrap, and with it a pass of fewer than k stacks, at most every 62 frames
BALL, TABLE = 3, 1      # frames per stack

_SESSIONS = itertools.count()       # distinguishes the replicas of sessions in the pipeline's replica cache


def check_live_args(streams, k, slots):
    """TableTennisPipeline.live's integer arguments: streams >= 1, k >= 1, slots >= 4 (a wrap copies two frames, which must not overlap
    the two slots they go to).  Raises ValueError."""
    for name, v, lo in (('streams', streams, 1), ('k', k, 1), ('slots', slots, 4)):
        if isinstance(v, bool) or not isinstance(v, numbers.Integral) or v < lo:
            raise ValueError('%s must be an integer >= %d, got %r' % (name, lo, v))


def push_plan(w, n, count, slots):
    """Where `count` frames pushed to one stream go.  The stream's region has `slots` slots, its next frame goes to slot w, and its
    open rally holds n frames, the last min(n, w) of them in slots w - min(n, w) .. w - 1.  Returns (steps, w, n), the state after
    the push, with steps in order:
      ('wrap', src, dst, m): the region is full; copy slots src .. src + m - 1 (the last m = min(n, 2) frames of the rally) to
                             dst .. dst + m - 1 (the start of the region) and write on from dst + m;
      ('write', slot, a, b): frames a .. b - 1 of the push go to slots slot .. slot + b - a - 1."""
    steps, a = [], 0
    while a < count:
        if w == slots:
            m = min(n, 2)
            steps.append(('wrap', slots - m, 0, m))
            w = m
        b = a + min(count - a, slots - w)
        steps.append(('write', w, a, b))
        w, n, a = w + b - a, n + b - a, b
    return steps, w, n


def ready_stacks(n_before, n_after, w_after, frames_per_stack):
    """The stacks of a rally that become ready when it grows from n_before to n_after frames, its frame n_after - 1 now in slot
    w_after - 1: [(stack index in the rally, slot of its first frame)].  Stack j is frames j .. j + frames_per_stack - 1, predict's
    sliding window; it is ready once its last frame has been pushed."""
    lo, hi = max(n_before - frames_per_stack + 1, 0), max(n_after - frames_per_stack + 1, 0)
    return [(j, w_after - (n_after - j)) for j in range(lo, hi)]


class _Entry:
    """One entry of a session: the contiguous block `streams` of its streams and the device state that serves them.  The entry's pool
    holds the session's frames base .. base + len(streams) * slots - 1.
    launcher: a single-thread executor that runs the entry's device work in the order it is submitted (devices=[...]), or None: the
    work runs on the caller's thread, on the current device (devices=None)."""

    def __init__(self, device, streams, slots, launcher=None, slot=None):
        self.device, self.streams, self.base, self.launcher = device, streams, streams.start * slots, launcher
        self.pool = None
        self.copy = None                                    # copy stream (devices=None: the pipeline ball detector's)
        self.uploaded = None                                # event after the last write on the copy stream
        self.pending = {BALL: [], TABLE: []}                # ready stacks not yet launched: (stream, stack index, session frame)
        self.pos = {s: [None] * 4 for s in streams}         # per stream: ball, ball aux, table, table aux positions
        self.slot, self.parts, self.key = slot, None, None  # devices=[...]: replica cache key, the five models, fingerprint at build
        self.rings = {}                                     # devices=[...]: staging rings of host (False) and CUDA (True) frames
        self.error = None                                   # the first exception of a launcher task

    def submit(self, fn, *args, waited=False):
        """A Future of fn(*args) on the launcher, after everything submitted before it.  Once a task has failed, the later ones raise
        its error instead of running: the entry's device state is then unknown.  waited: the caller waits for this task's result, and
        a ValueError of it (a rally predict would refuse) goes to the caller only and leaves the entry usable."""
        def run():
            if self.error is not None:
                raise self.error
            try:
                return fn(*args)
            except BaseException as e:      # noqa: BLE001 - kept for the caller's next call on this entry
                if not (waited and isinstance(e, ValueError)):
                    self.error = e
                raise
        return self.launcher.submit(run)


class _Ring:
    """A staging ring of an entry: frame buffers `slots`, per slot the Future of the launcher's write out of it, the next slot."""

    def __init__(self, slots):
        self.slots, self.busy, self.next = slots, [None] * len(slots), 0


class LiveSession:
    """TableTennisPipeline.live(fps, streams=1, k=DEFAULT_K, slots=DEFAULT_SLOTS, devices=None).  A stream is one camera.

    push(stream, frames) appends one HWC uint8 BGR frame, or a list of them (numpy arrays or torch CPU / CUDA tensors, one frame
    shape per session; one push takes host frames or CUDA frames, not both), to the stream's open rally.  It returns once host frames
    have been copied into pinned staging memory (the caller may then reuse their memory).  CUDA frames may be on any GPU; they are
    copied on the caller's current stream (of their device), so work the caller queues on it afterwards (overwriting a frame, or the
    allocator reusing a freed one) comes after the copy; work on other streams is the caller's to order, as for any CUDA tensor.  Device memory is bounded: when the GPU falls behind, push waits for it.  Whenever k stacks are ready over the streams of
    one entry (a ball stack once its third frame is in, a table stack once its frame is in), one pass of each of the four detectors
    runs over them.

    end_rally(stream) runs the stream's ready stacks, then predict's tail (TableTennisPipeline._tail), and returns (spin, pos3d):
    exactly what pipe.predict(the frames pushed since the last end_rally, fps) returns, the spin on the pipeline's device.
    end_rally(stream, cameras=True) returns (spin, pos3d, camera) instead, camera the rally's interface.RallyCamera, exactly what
    pipe.predict_clips([the rally's frames], fps, cameras=True)[0] holds; it is computed by the same task as the tail (on the entry's
    launcher with devices=[...]) and comes back as numpy.  (With
    devices=[...] the spin is computed, and copied to the pipeline's device, on the launcher thread's default streams, as in
    predict_clips; a caller that reads it on another stream of that device orders that stream after the default stream.)  The stream
    then starts a new rally; it does so also when end_rally raises: ValueError for a rally of fewer than 3 frames, predict's ValueError
    for 0 or 50 or more agreeing ball detections.

    fps=None opens a timestamped session, for cameras whose frames are not 1 / fps apart (variable frame rate, dropped frames, or a
    caller that skips frames to keep up): push(stream, frames, timestamps=...) then takes the capture time of each frame in seconds
    (a number for a single frame), and end_rally returns exactly pipe.predict(the rally's frames, None, timestamps=their stamps).  Each
    stamp must be finite and later than the stream's previous stamp in the open rally; the stamps are kept per stream on the host and
    reset with the rally.  A wrong number of stamps, a bad stamp, stamps pushed to a session with fps or none to a timestamped session
    raise ValueError before the push does anything.

    set_table(stream, keypoints) gives a stream whose camera does not move its table, a (13, 3) array as predict's table_keypoints
    takes it (typically the RallyCamera.keypoints of an earlier rally's end_rally(stream, cameras=True)), or clears it with None.  It
    applies from the stream's next rally until it is changed, and raises ValueError while the stream has an open rally.  While it is
    set, the stream's pushes queue no table stacks (the table passes run over the other streams only) and end_rally returns exactly
    pipe.predict(the rally's frames, fps, table_keypoints=keypoints), with the stamps in a timestamped session.

    devices: None = one entry on the current device; push launches the passes on the caller's thread.  Otherwise a list of CUDA device
    indices, torch.device or 'cuda:N' strings, as predict_clips takes (a device may repeat): one entry per item, entry r serving
    streams sharding.shard_range(streams, r, len(devices)) -- contiguous blocks, the first streams % len(devices) entries one stream
    more -- on devices[r]; more entries than streams raises ValueError.  CUDA frames are best pushed on their stream's device (a frame on
    another GPU is copied across).  Each entry has its own frame pool, copy stream and copy of the five models (built from the
    pipeline's, rebuilt when they change), and one launcher thread that runs its writes, wraps, passes and tails in push order.  push
    stages the frames in a ring of the entry (pinned host memory, or device memory for CUDA frames) and queues their writes, so the
    caller's thread does not wait for the passes; it waits only when every slot of the ring still holds a frame the launcher has not
    written yet.  k and slots apply per entry.  An exception on a launcher is raised by the next push or end_rally on one of the
    entry's streams, and by close(); the entry's streams then keep raising it.

    A rally keeps the pipeline's models and compute_dtype of its first push.  If a compute_dtype or a weight tensor's contents
    (load_state_dict, in-place writes) change while the rally is open, the stream's next push or end_rally drops the rally and raises
    RuntimeError; a model whose tensors were replaced by other tensor objects is caught by end_rally at the latest.  (Each push
    compares the compute_dtypes and the tensors' version counters; the full _fingerprint, which builds five state dicts, runs when a
    rally opens and at end_rally.)  With devices=[...], a rally that opens under changed models rebuilds its entry's replicas, and the
    entry's other open rallies, detected with the old ones, are dropped the same way.  close() (or leaving a `with` block) waits for
    the launchers, frees the pools and raises the first launcher exception (leaving a `with` block because of another exception
    raises that one).

    The device work is in _alloc_pool, _alloc_ring, _stage, _device_write, _device_wrap, _device_pass, _build_parts and _finish;
    everything else is bookkeeping."""

    def __init__(self, pipe, fps, streams=1, k=None, slots=None, devices=None):
        k = DEFAULT_K if k is None else k
        slots = DEFAULT_SLOTS if slots is None else slots
        check_live_args(streams, k, slots)
        self.pipe, self.fps, self.streams, self.k, self.slots = pipe, fps, int(streams), int(k), int(slots)
        if devices is None:
            self._entries = [_Entry(None, range(self.streams), self.slots)]
        else:
            idx = parse_devices(devices, torch.cuda.device_count())
            if len(idx) > self.streams:
                raise ValueError('devices: %d entries for %d streams; each entry needs at least one stream' % (len(idx), self.streams))
            sid = next(_SESSIONS)
            self._entries = []
            for r, d in enumerate(idx):
                a, b = sharding.shard_range(self.streams, r, len(idx))
                launcher = ThreadPoolExecutor(1, 'ttk-live%d' % d, initializer=torch.cuda.set_device, initargs=(d,))
                self._entries.append(_Entry(torch.device('cuda', d), range(a, b), self.slots, launcher, ('live', sid, r)))
        self._entry = [e for e in self._entries for _ in e.streams]     # per stream
        self.shape = None                                   # frame shape, set by the first push
        self._pool = None
        self._w = [0] * self.streams                        # next slot each stream writes
        self._n = [0] * self.streams                        # frames of each stream's open rally
        self._models = [None] * self.streams                # per open rally: (full fingerprint, weight tensors, quick key)
        # fps=None: each stream's open rally's frame stamps, on the host (a wrap copies frames, not stamps)
        self._stamps = [[] for _ in range(self.streams)] if fps is None else None
        self._tables = [None] * self.streams                # set_table: each stream's known (13, 3) float64 table, or None
        self._stale = set()                                 # streams whose open rally was detected with replicas since rebuilt
        self._closed = False

    @property
    def _pending(self):
        """The ready stacks not yet launched, of all entries: {frames per stack: [(stream, stack index, session frame)]}."""
        return {fps: [x for e in self._entries for x in e.pending[fps]] for fps in (BALL, TABLE)}

    # ---- public --------------------------------------------------------------------------------------
    def push(self, stream, frames, timestamps=None):
        s = self._stream(stream)
        e = self._entry[s]
        if isinstance(frames, (np.ndarray, torch.Tensor)) and frames.ndim == 3:
            frames = [frames]
        frames = list(frames)
        stamps = self._check_stamps(s, len(frames), timestamps)
        if not frames:
            return
        self._check_frames(frames)
        self._check_models(s, full=False)
        steps, _, _ = push_plan(self._w[s], self._n[s], len(frames), self.slots)
        for step in steps:
            if step[0] == 'wrap':
                self._wrap(s, *step[1:])
            else:
                self._write(s, frames, *step[1:])
                if stamps is not None:
                    self._stamps[s] += stamps[step[2]:step[3]].tolist()
                if len(e.pending[BALL]) >= self.k or len(e.pending[TABLE]) >= self.k:
                    self._launch(e)

    def end_rally(self, stream, cameras=False):
        s = self._stream(stream)
        e, n = self._entry[s], self._n[s]
        try:
            self._check_models(s, full=True)
            if n < 3:
                raise ValueError('stream %d: a rally of %d frames; a rally needs at least 3 (one (prev, cur, next) ball stack)' % (s, n))
            self._launch(e, {s})
            finish = self._finish
            if self._stamps is not None:
                finish = functools.partial(finish, stamps=np.array(self._stamps[s], dtype=np.float64))
            if self._tables[s] is not None:
                finish = functools.partial(finish, table=self._tables[s])
            return self._run(e, finish, *((s, n, True) if cameras else (s, n)), wait=True)
        finally:
            self._reset(s)

    def set_table(self, stream, keypoints):
        """The known table of `stream` from its next rally on, a (13, 3) (x, y, v) array as predict's table_keypoints takes it, or None
        to detect the table again.  While it is set, the stream's frames go to the ball detectors only and end_rally returns
        predict(the rally's frames, fps, table_keypoints=keypoints).  Raises ValueError while the stream has an open rally, and for
        keypoints predict would refuse."""
        s = self._stream(stream)
        kp = None if keypoints is None else check_table_keypoints(keypoints, 'stream %d' % s)
        if self._n[s]:
            raise ValueError('stream %d: set_table with a rally of %d frames open; a table applies from the next rally, call it after '
                             'end_rally' % (s, self._n[s]))
        self._tables[s] = kp

    def close(self):
        if self._closed:
            return
        first = None
        for e in self._entries:
            if e.launcher is None:
                if e.uploaded is not None:
                    # nothing else records the pool's use on the copy stream: later allocations of this stream must come after its copies
                    torch.cuda.current_stream().wait_stream(self._copy_stream(e))
            else:
                done = e.launcher.submit(self._release, e)      # not e.submit: it runs after a failed task too
                e.launcher.shutdown(wait=True)
                first = first or e.error or done.exception()
                getattr(self.pipe, '_replicas', {}).pop(e.slot, None)
            e.pool, e.pos, e.parts, e.rings, e.uploaded = None, None, None, {}, None
            e.pending = {BALL: [], TABLE: []}
        self._pool = None
        self._closed = True
        if first is not None:
            raise first

    def __enter__(self):
        return self

    def __exit__(self, exc_type, *exc):
        try:
            self.close()
        except BaseException:
            if exc_type is None:            # otherwise the exception that left the block is the one to see
                raise
        return False

    # ---- checks --------------------------------------------------------------------------------------
    def _stream(self, stream):
        if self._closed:
            raise RuntimeError('this LiveSession is closed')
        if isinstance(stream, bool) or not isinstance(stream, numbers.Integral) or not 0 <= stream < self.streams:
            raise ValueError('stream must be an integer in [0, %d), got %r' % (self.streams, stream))
        error = self._entry[int(stream)].error
        if error is not None:
            raise error
        return int(stream)

    def _check_frames(self, frames):
        shape = self.shape or tuple(frames[0].shape)
        for f in frames:
            u8 = f.dtype == (torch.uint8 if isinstance(f, torch.Tensor) else np.uint8)
            if tuple(f.shape) != shape or len(shape) != 3 or shape[2] != 3 or not u8:
                raise ValueError('frames must be HWC uint8 BGR arrays of the session frame shape %s; got %s %s' % (shape, tuple(f.shape), f.dtype))
        on_device = [isinstance(f, torch.Tensor) and f.is_cuda for f in frames]
        if any(on_device) and not all(on_device):
            raise ValueError('one push takes host frames (numpy, torch CPU) or CUDA frames, not both')
        if self._pool is None:
            self.shape = shape
            self._pool = self._alloc_pool(shape)

    def _check_stamps(self, s, count, timestamps):
        """The float64 stamps of `count` frames pushed to stream s (None for a session with fps).  Raises ValueError, before any device
        work, when a timestamped session gets no stamps or the wrong number, a non-finite one, one that does not increase, or one not
        after the rally's previous frame, and when a session with fps gets stamps."""
        if self._stamps is None:
            if timestamps is not None:
                raise ValueError('stream %d: this session runs at fps=%r and takes no timestamps; open it with fps=None to push them'
                                 % (s, self.fps))
            return None
        if timestamps is None:
            raise ValueError('stream %d: this session (fps=None) needs timestamps=, one capture time per frame' % s)
        ts = check_timestamps([timestamps] if np.ndim(timestamps) == 0 else timestamps, count, 'stream %d' % s)     # (one frame, one stamp)
        if count and self._n[s] and not ts[0] > self._stamps[s][-1]:
            raise ValueError("stream %d: timestamp %r does not follow the rally's previous frame at %r; timestamps must increase strictly"
                             % (s, float(ts[0]), self._stamps[s][-1]))
        return ts

    def _check_models(self, s, full):
        parts = self.pipe._parts()
        e = self._entry[s]
        if s in self._stale:
            self._reset(s)
            raise RuntimeError('stream %d: the models changed while a rally was open; the rally (detected with the old models) is '
                               'dropped' % s)
        if self._n[s] == 0:
            key = tuple(_fingerprint(p.model) for p in parts)
            tensors = [v for p in parts for v in p.model.state_dict().values()]
            self._models[s] = (key, tensors, self._quick_key(parts, tensors))
            if e.launcher is not None and key != e.key:
                self._rebuild(e, key)
            return
        key, tensors, quick = self._models[s]
        if self._quick_key(parts, tensors) != quick or (full and tuple(_fingerprint(p.model) for p in parts) != key):
            self._reset(s)
            raise RuntimeError('stream %d: a model or its compute_dtype changed while a rally was open; the rally (detected with the old '
                               'models) is dropped' % s)

    @staticmethod
    def _quick_key(parts, tensors):
        return tuple(p.model.compute_dtype for p in parts), tuple(t._version for t in tensors)

    # ---- bookkeeping ---------------------------------------------------------------------------------
    def _run(self, e, fn, *args, wait=False):
        """fn(*args) as device work of entry e: now, or (devices=[...]) queued to its launcher; wait: return its result."""
        if e.launcher is None:
            return fn(*args)
        done = e.submit(fn, *args, waited=wait)
        return done.result() if wait else done

    def _rebuild(self, e, key):
        """A rally opens on entry e under models other than its replicas': every other open rally of the entry was detected with the
        old replicas and is dropped (its pending stacks now, the rally at its stream's next call), and the replicas are rebuilt after
        the work already queued, so that no pass mixes the two."""
        for s in e.streams:
            if self._n[s]:
                self._stale.add(s)
        for fps in (BALL, TABLE):
            e.pending[fps] = [x for x in e.pending[fps] if x[0] not in self._stale]
        e.key = key
        self._run(e, self._build_parts, e)

    def _write(self, s, frames, slot, a, b):
        e = self._entry[s]
        base = s * self.slots
        if e.launcher is None:
            self._device_write(frames[a:b], base + slot)
        else:
            self._hand_off(e, frames[a:b], base + slot)
        n0 = self._n[s]
        self._n[s], self._w[s] = n0 + b - a, slot + b - a
        for fps in (BALL, TABLE) if self._tables[s] is None else (BALL,):         # a known table needs no table stacks
            e.pending[fps] += [(s, j, base + f) for j, f in ready_stacks(n0, self._n[s], self._w[s], fps)]

    def _wrap(self, s, src, dst, m):
        e = self._entry[s]
        self._launch(e, {s})                    # the stream's ready stacks still read the slots about to be overwritten
        base = s * self.slots
        self._run(e, self._device_wrap, base + src, base + dst, m)
        self._w[s] = dst + m

    def _launch(self, e, streams=None):
        """One pass of each detector over entry e's pending stacks (of `streams` only, when given)."""
        for fps in (BALL, TABLE):
            take = [x for x in e.pending[fps] if streams is None or x[0] in streams]
            if not take:
                continue
            e.pending[fps] = [x for x in e.pending[fps] if not (streams is None or x[0] in streams)]
            take.sort(key=lambda x: x[0])       # stable: each stream's stacks stay in order, one contiguous run per stream
            runs = [(st, [x[1] for x in grp]) for st, grp in itertools.groupby(take, key=lambda x: x[0])]
            self._run(e, self._device_pass, fps, [x[2] for x in take], runs)

    def _reset(self, s):
        self._n[s], self._models[s] = 0, None
        if self._stamps is not None:
            self._stamps[s] = []
        self._stale.discard(s)
        e = self._entry[s]
        for fps in (BALL, TABLE):
            e.pending[fps] = [x for x in e.pending[fps] if x[0] != s]

    # ---- device work ---------------------------------------------------------------------------------
    def _alloc_pool(self, shape):
        for e in self._entries:
            size = (len(e.streams) * self.slots,) + shape
            if e.launcher is None:
                e.pool = torch.empty(size, dtype=torch.uint8, device=self.pipe.device)
            else:
                # on the stream the launcher computes on, which _release makes wait for the copy stream before the pool is freed
                with torch.cuda.device(e.device), torch.cuda.stream(torch.cuda.default_stream(e.device)):
                    e.pool = torch.empty(size, dtype=torch.uint8, device=e.device)
                e.copy = torch.cuda.Stream(device=e.device)
        return [e.pool for e in self._entries]

    def _copy_stream(self, e):
        if e.launcher is not None:
            return e.copy
        det = self.pipe.ball_detector
        if getattr(det, '_copy_stream', None) is None:
            det._copy_stream = torch.cuda.Stream(device=self.pipe.device)
        return det._copy_stream

    def _hand_off(self, e, frames, p0):
        """devices=[...], on the caller's thread: stages `frames` in entry e's ring for their kind, one slot per frame, and queues the
        write of each slot into session frame p0 + i to the launcher.  A slot is filled again once the launcher's write out of it has
        been queued and has finished, which bounds how far a launcher falls behind; push waits only then, never for queued passes."""
        cuda = isinstance(frames[0], torch.Tensor) and frames[0].is_cuda
        ring = e.rings.get(cuda)
        if ring is None:
            ring = e.rings[cuda] = _Ring(self._alloc_ring(e, cuda))
        for i, f in enumerate(frames):
            k = ring.next
            ring.next = (k + 1) % len(ring.slots)
            done = None if ring.busy[k] is None else ring.busy[k].result()     # (raises the launcher's error, if any)
            staged = self._stage(e, ring.slots[k], f, done)
            ring.busy[k] = e.submit(self._device_write, [ring.slots[k]], p0 + i, staged)

    def _alloc_ring(self, e, cuda):
        """_Detector.stage_slots frame buffers of entry e: pinned host memory, or (CUDA frames) device memory on the entry's device."""
        size = (_Detector.stage_slots,) + self.shape
        if not cuda:
            return torch.empty(size, dtype=torch.uint8).pin_memory()
        with torch.cuda.device(e.device), torch.cuda.stream(torch.cuda.default_stream(e.device)):
            return torch.empty(size, dtype=torch.uint8, device=e.device)

    def _stage(self, e, slot, f, done):
        """Frame f into ring slot `slot`, once `done` (the event after the launcher's last write out of the slot, or None) has
        passed.  A CUDA frame is copied on the caller's current stream, which so orders the caller's later work on f after the copy;
        returns the event the launcher's write waits for.  A host frame is copied here; returns None."""
        if isinstance(f, torch.Tensor) and f.is_cuda:
            with torch.cuda.device(e.device):
                caller = torch.cuda.current_stream()
                if done is not None:
                    caller.wait_event(done)
                slot.copy_(f, non_blocking=True)        # (from another GPU: one cudaMemcpyAsync, after the caller's stream there)
                return caller.record_event()
        if done is not None:
            done.synchronize()
        u = f.numpy() if isinstance(f, torch.Tensor) else f
        if u.flags['C_CONTIGUOUS']:
            _lib.check(_lib.lib.ttk_host_copy_stream(slot.data_ptr(), u.ctypes.data, u.nbytes))
        else:
            slot.numpy()[...] = u
        return None

    def _device_write(self, frames, p0, staged=None):
        """frames into session frames p0 .. on the copy stream.  devices=None: through the pinned staging ring of _Detector._upload
        unless they are CUDA tensors.  devices=[...] (on the launcher): `frames` are ring slots, written after the event `staged`
        (CUDA slots) when given; returns the event after the copy."""
        e = self._entry[p0 // self.slots]
        if e.launcher is not None:
            with torch.cuda.stream(e.copy):
                if staged is not None:
                    e.copy.wait_event(staged)
                for i, f in enumerate(frames):
                    e.pool[p0 - e.base + i].copy_(f, non_blocking=True)
                e.uploaded = torch.cuda.current_stream().record_event()
            return e.uploaded
        _, _, ready = self.pipe.ball_detector._upload(frames, self.pipe.device, out=e.pool[p0:p0 + len(frames)])
        e.uploaded = ready[-1][1]               # (host frames: waits until the last one is staged and its copy enqueued)
        if isinstance(frames[0], torch.Tensor) and frames[0].is_cuda:
            torch.cuda.current_stream().wait_event(e.uploaded)      # the caller's later work on its frames comes after the copy

    def _device_wrap(self, src, dst, m):
        e = self._entry[dst // self.slots]
        copy = self._copy_stream(e)
        copy.wait_stream(torch.cuda.current_stream())
        if m:
            src, dst = src - e.base, dst - e.base
            with torch.cuda.stream(copy):
                e.pool[dst:dst + m].copy_(e.pool[src:src + m], non_blocking=True)

    def _device_pass(self, fps, first, runs):
        """The two detectors of this stack kind over the session frames `first`; runs = [(stream, its stack indices)] in that order,
        all of one entry."""
        e = self._entry[runs[0][0]]
        if e.launcher is None:
            parts, dev = self.pipe._parts(), self.pipe.device
        else:
            parts, dev = e.parts, e.device
        first = [p - e.base for p in first]
        main = torch.cuda.current_stream()
        first_d = torch.tensor(first, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)
        main.wait_event(e.uploaded)
        with torch.no_grad():
            for d in ((0, 1) if fps == BALL else (2, 3)):
                pos = parts[d]._run(e.pool, 1, len(first), False, None, first=(first, first_d))[0]
                a = 0
                for st, idx in runs:
                    self._store(e, st, d, idx[0], pos[a:a + len(idx)])
                    a += len(idx)

    @staticmethod
    def _store(e, s, d, j0, p):
        """Rows j0 .. of stream s's positions of detector d, in a device buffer of entry e that grows by doubling."""
        buf = e.pos[s][d]
        need = j0 + p.shape[0]
        if buf is None or buf.shape[0] < need:
            cap = 64 if buf is None else buf.shape[0]
            while cap < need:
                cap *= 2
            grown = torch.empty((cap,) + tuple(p.shape[1:]), dtype=p.dtype, device=p.device)
            if buf is not None:
                grown[:j0].copy_(buf[:j0])
            e.pos[s][d] = buf = grown
        buf[j0:need].copy_(p)

    def _build_parts(self, e):
        """On entry e's launcher: its replicas of the pipeline's five models (TableTennisPipeline._replica_parts)."""
        e.parts = self.pipe._replica_parts(e.slot, e.device.index)

    def _release(self, e):
        """On entry e's launcher, at close(): everything queued on the entry's device (the caller's copies into the CUDA ring among
        it) has finished before the pool, the rings and the position buffers are freed."""
        if e.copy is not None:
            torch.cuda.synchronize()

    def _finish(self, s, n, cameras=False, stamps=None, table=None):
        """stamps: the rally's n frame stamps (fps=None).  table: the stream's known (13, 3) float64 table, copied to the entry's
        device, or None: the table filter over the rally's table positions."""
        e = self._entry[s]
        b, b_aux, t, t_aux = e.pos[s]
        centre = None if stamps is None else stamps[1:n - 1]
        keypoints = ops.filter_table(t[:n], t_aux[:n]) if table is None else _upload_tables(table, b.device)
        if e.launcher is None:
            return self.pipe._tail(b[:n - 2, 0], b_aux[:n - 2, 0], keypoints, self.fps, cameras=cameras, stamps=centre)
        out = self.pipe._tail(b[:n - 2, 0], b_aux[:n - 2, 0], keypoints, self.fps, e.parts[4], cameras=cameras, stamps=centre)
        return (out[0].to(self.pipe._home_device()),) + out[1:]
