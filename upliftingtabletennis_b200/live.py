"""Live sessions of TableTennisPipeline (TableTennisPipeline.live): frames are detected as the cameras deliver them, and each rally's
spin and trajectory come back as soon as the caller ends it, exactly as predict would return them for the rally's frames.

Device frame pool: one uint8 CUDA tensor of streams x slots frames; stream s owns the contiguous region [s * slots, (s + 1) * slots)
and writes it in order.  When its write position reaches the region's end, the last two frames of the open rally are copied to the
start of the region (on the copy stream, after the compute stream) and writing goes on from there, so every stack of every stream is
"first frame + 0, 1, 2" inside the pool and a pass that mixes streams is one ttk_preprocess_stacks_indexed call, as in predict_clips.

The bookkeeping is kept in pure functions (push_plan, ready_stacks, check_live_args) so that it can be checked without a GPU."""
import itertools
import numbers

import numpy as np
import torch

from .interface import _fingerprint

DEFAULT_K = 16          # ready stacks that launch a pass: _Detector.chunk, predict's pass size; 137-143 frames/s for k = 4..32 on
                        # WASB + HRNet (profiles/r06_live_timing.json), so no reason to give ViTPose's GEMMs fewer M tiles
DEFAULT_SLOTS = 64      # frames per stream (398 MB at 1080p): a wrap, and with it a pass of fewer than k stacks, at most every 62 frames
BALL, TABLE = 3, 1      # frames per stack


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


class LiveSession:
    """TableTennisPipeline.live(fps, streams=1, k=DEFAULT_K, slots=DEFAULT_SLOTS).  A stream is one camera.

    push(stream, frames) appends one HWC uint8 BGR frame, or a list of them (numpy arrays or torch CPU / CUDA tensors, one frame
    shape per session; one push takes host frames or CUDA frames, not both), to the stream's open rally.  It returns once host frames
    have been copied into the pinned staging ring (the caller may then reuse their memory) and the detector passes they complete have
    been launched.  CUDA frames are copied on the copy stream and the caller's current stream waits for that copy, so work the caller
    queues on it afterwards (overwriting a frame, or the allocator reusing a freed one) comes after the copy; work on other streams is
    the caller's to order, as for any CUDA tensor.  push does not wait for the GPU, except that a stream's device memory is bounded:
    when the GPU falls behind, push waits for it.  Whenever k stacks are ready over all streams (a ball stack once its third frame is
    in, a table stack once its frame is in), one pass of each of the four detectors runs over them.

    end_rally(stream) runs the stream's ready stacks, then predict's tail (TableTennisPipeline._tail), and returns (spin, pos3d):
    exactly what pipe.predict(the frames pushed since the last end_rally, fps) returns.  The stream then starts a new rally; it does
    so also when end_rally raises: ValueError for a rally of fewer than 3 frames, predict's ValueError for 0 or 50 or more agreeing
    ball detections.

    A rally keeps the pipeline's models and compute_dtype of its first push.  If a compute_dtype or a weight tensor's contents
    (load_state_dict, in-place writes) change while the rally is open, the stream's next push or end_rally drops the rally and raises
    RuntimeError; a model whose tensors were replaced by other tensor objects is caught by end_rally at the latest.  (Each push
    compares the compute_dtypes and the tensors' version counters; the full _fingerprint, which builds five state dicts, runs when a
    rally opens and at end_rally.)  close() (or leaving a `with` block) frees the pool.

    The device work is in _alloc_pool, _device_write, _device_wrap, _device_pass and _finish; everything else is bookkeeping."""

    def __init__(self, pipe, fps, streams=1, k=None, slots=None):
        k = DEFAULT_K if k is None else k
        slots = DEFAULT_SLOTS if slots is None else slots
        check_live_args(streams, k, slots)
        self.pipe, self.fps, self.streams, self.k, self.slots = pipe, fps, int(streams), int(k), int(slots)
        self.shape = None                                   # frame shape, set by the first push
        self._pool = None
        self._w = [0] * self.streams                        # next slot each stream writes
        self._n = [0] * self.streams                        # frames of each stream's open rally
        self._models = [None] * self.streams                # per open rally: (full fingerprint, weight tensors, quick key)
        self._pending = {BALL: [], TABLE: []}               # ready stacks not yet launched: (stream, stack index, pool frame)
        self._pos = [[None] * 4 for _ in range(self.streams)]      # per stream: ball, ball aux, table, table aux positions
        self._uploaded = None                               # event after the last upload on the copy stream
        self._closed = False

    # ---- public --------------------------------------------------------------------------------------
    def push(self, stream, frames):
        s = self._stream(stream)
        if isinstance(frames, (np.ndarray, torch.Tensor)) and frames.ndim == 3:
            frames = [frames]
        frames = list(frames)
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
                if len(self._pending[BALL]) >= self.k or len(self._pending[TABLE]) >= self.k:
                    self._launch()

    def end_rally(self, stream):
        s = self._stream(stream)
        n = self._n[s]
        try:
            self._check_models(s, full=True)
            if n < 3:
                raise ValueError('stream %d: a rally of %d frames; a rally needs at least 3 (one (prev, cur, next) ball stack)' % (s, n))
            self._launch({s})
            return self._finish(s, n)
        finally:
            self._reset(s)

    def close(self):
        if self._uploaded is not None:
            # nothing else records the pool's use on the copy stream: later allocations of this stream must come after its copies
            torch.cuda.current_stream().wait_stream(self._copy_stream())
        self._pool, self._pos, self._pending, self._uploaded = None, None, None, None
        self._closed = True

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    # ---- checks --------------------------------------------------------------------------------------
    def _stream(self, stream):
        if self._closed:
            raise RuntimeError('this LiveSession is closed')
        if isinstance(stream, bool) or not isinstance(stream, numbers.Integral) or not 0 <= stream < self.streams:
            raise ValueError('stream must be an integer in [0, %d), got %r' % (self.streams, stream))
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

    def _check_models(self, s, full):
        parts = self.pipe._parts()
        if self._n[s] == 0:
            key = tuple(_fingerprint(p.model) for p in parts)
            tensors = [v for p in parts for v in p.model.state_dict().values()]
            self._models[s] = (key, tensors, self._quick_key(parts, tensors))
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
    def _write(self, s, frames, slot, a, b):
        base = s * self.slots
        self._device_write(frames[a:b], base + slot)
        n0 = self._n[s]
        self._n[s], self._w[s] = n0 + b - a, slot + b - a
        for fps in (BALL, TABLE):
            self._pending[fps] += [(s, j, base + f) for j, f in ready_stacks(n0, self._n[s], self._w[s], fps)]

    def _wrap(self, s, src, dst, m):
        self._launch({s})                       # the stream's ready stacks still read the slots about to be overwritten
        base = s * self.slots
        self._device_wrap(base + src, base + dst, m)
        self._w[s] = dst + m

    def _launch(self, streams=None):
        """One pass of each detector over the pending stacks (of `streams` only, when given)."""
        for fps in (BALL, TABLE):
            take = [x for x in self._pending[fps] if streams is None or x[0] in streams]
            if not take:
                continue
            self._pending[fps] = [x for x in self._pending[fps] if not (streams is None or x[0] in streams)]
            take.sort(key=lambda x: x[0])       # stable: each stream's stacks stay in order, one contiguous run per stream
            runs = [(st, [x[1] for x in grp]) for st, grp in itertools.groupby(take, key=lambda x: x[0])]
            self._device_pass(fps, [x[2] for x in take], runs)

    def _reset(self, s):
        self._n[s], self._models[s] = 0, None
        for fps in (BALL, TABLE):
            self._pending[fps] = [x for x in self._pending[fps] if x[0] != s]

    # ---- device work ---------------------------------------------------------------------------------
    def _alloc_pool(self, shape):
        return torch.empty((self.streams * self.slots,) + shape, dtype=torch.uint8, device=self.pipe.device)

    def _copy_stream(self):
        det = self.pipe.ball_detector
        if getattr(det, '_copy_stream', None) is None:
            det._copy_stream = torch.cuda.Stream(device=self.pipe.device)
        return det._copy_stream

    def _device_write(self, frames, p0):
        """frames into pool frames p0 .. on the copy stream, through the pinned staging ring unless they are CUDA tensors."""
        _, _, ready = self.pipe.ball_detector._upload(frames, self.pipe.device, out=self._pool[p0:p0 + len(frames)])
        self._uploaded = ready[-1][1]           # (host frames: waits until the last one is staged and its copy enqueued)
        if isinstance(frames[0], torch.Tensor) and frames[0].is_cuda:
            torch.cuda.current_stream().wait_event(self._uploaded)      # the caller's later work on its frames comes after the copy

    def _device_wrap(self, src, dst, m):
        copy = self._copy_stream()
        copy.wait_stream(torch.cuda.current_stream())
        if m:
            with torch.cuda.stream(copy):
                self._pool[dst:dst + m].copy_(self._pool[src:src + m], non_blocking=True)

    def _device_pass(self, fps, first, runs):
        """The two detectors of this stack kind over the pool frames `first`; runs = [(stream, its stack indices)] in that order."""
        parts = self.pipe._parts()
        main = torch.cuda.current_stream()
        first_d = torch.tensor(first, dtype=torch.int32).pin_memory().to(self.pipe.device, non_blocking=True)
        main.wait_event(self._uploaded)
        with torch.no_grad():
            for d in ((0, 1) if fps == BALL else (2, 3)):
                pos = parts[d]._run(self._pool, 1, len(first), False, None, first=(first, first_d))[0]
                a = 0
                for st, idx in runs:
                    self._store(st, d, idx[0], pos[a:a + len(idx)])
                    a += len(idx)

    def _store(self, s, d, j0, p):
        """Rows j0 .. of stream s's positions of detector d, in a device buffer that grows by doubling."""
        buf = self._pos[s][d]
        need = j0 + p.shape[0]
        if buf is None or buf.shape[0] < need:
            cap = 64 if buf is None else buf.shape[0]
            while cap < need:
                cap *= 2
            grown = torch.empty((cap,) + tuple(p.shape[1:]), dtype=p.dtype, device=p.device)
            if buf is not None:
                grown[:j0].copy_(buf[:j0])
            self._pos[s][d] = buf = grown
        buf[j0:need].copy_(p)

    def _finish(self, s, n):
        b, b_aux, t, t_aux = self._pos[s]
        return self.pipe._tail(b[:n - 2, 0], b_aux[:n - 2, 0], t[:n], t_aux[:n], self.fps)
