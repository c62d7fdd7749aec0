"""Drop-in for the reference's ``interface.py`` (BallDetector, TableDetector, UpliftingModel,
TableTennisPipeline; reference ``interface.py:83-312``) with the hot path on libttk.

Same names, arguments, return types and error behaviour as the reference.  Differences are internal:
frames are uploaded once and processed as a batch on the GPU (the reference loops B=1 with a host
round-trip per frame), and the segformer++ detectors, whose architecture is not part of the reference
repository (fetched from another hub repo at construction time, ``balldetection/models/segformer_pp.py:12-19``),
are substituted by the in-repo WASB / HRNet architectures unless their weights are unavailable.
"""
import os
import zipfile

import numpy as np
import torch

from . import _lib, ops, sharding
from .detector import MyHRNet, WASBNet
from .precision import BF16, FP16, TF32, TF32X3, canonical
from .vitpose import TableVitPose, VitPose
from .uplift import MASK_FORMAT_ERROR, MultiStageModel, get_model as get_uplifting_model

HEIGHT, WIDTH = 1080, 1920          # inference/utils.py:22
BALL_VISIBLE = 1
KEYPOINT_VISIBLE, KEYPOINT_INVISIBLE = 1, 0
SEQ_LEN = 50                        # inference/utils.py:293

WEIGHTS_ZIP_URL = "https://mediastore.rz.uni-augsburg.de/get/TL7oQRStHG/"     # interface.py:29
ZIP_FILENAME = "tt_uplifting_weights.zip"
EXTRACTED_FOLDER_NAME = "weights"


def _get_weights_path(relative_path):
    """interface.py:34-73: locate (download + extract if needed) a file of the released weights tree."""
    hub_dir = torch.hub.get_dir()
    download_dir = os.path.join(hub_dir, "checkpoints")
    os.makedirs(download_dir, exist_ok=True)
    zip_path = os.path.join(download_dir, ZIP_FILENAME)
    extract_path = os.path.join(download_dir, "tt_uplifting_extracted")
    target_file = os.path.join(extract_path, EXTRACTED_FOLDER_NAME, relative_path)
    if os.path.exists(target_file):
        return target_file
    print(f"Weights not found at {target_file}.")
    if not os.path.exists(zip_path):
        print(f"Downloading weights from {WEIGHTS_ZIP_URL}...")
        try:
            torch.hub.download_url_to_file(WEIGHTS_ZIP_URL, zip_path, progress=True)
        except Exception as e:
            raise RuntimeError(f"Failed to download weights: {e}")
    if not os.path.exists(extract_path) or not os.path.exists(target_file):
        print("Extracting weights... this may take a moment.")
        try:
            with zipfile.ZipFile(zip_path, 'r') as zip_ref:
                zip_ref.extractall(extract_path)
            print("Extraction complete.")
        except Exception as e:
            raise RuntimeError(f"Failed to extract weights: {e}")
    return target_file


def _device():
    if not torch.cuda.is_available():
        raise RuntimeError('upliftingtabletennis_b200 needs a B200 (sm_100) GPU; there is no CPU fallback')
    return torch.device('cuda')


# ---- loaders (inference/inference_balldetection.py:40-61, inference_tabledetection.py:40-57, inference_uplifting.py:33-58) ----
class _DetectorTransform:
    """Stand-in for the reference's Compose([Resize, NormalizeImage]) (balldetection/transforms.py:504-508).
    Callable on the same dicts; the work happens in the fused CUDA pre-processing kernel."""

    def __init__(self, resolution):
        self.resolution = tuple(resolution)

    def __call__(self, data):
        dev = _device()
        out = dict(data)
        for k in ('image', 'prev_image', 'next_image'):
            if k in data and data[k] is not None:
                f = torch.from_numpy(np.ascontiguousarray(data[k])).to(dev)[None]
                x = ops.preprocess_stacks(f, 1, 1, 1, self.resolution[0], self.resolution[1], layout='nchw')
                out[k] = x[0].permute(1, 2, 0).double().cpu().numpy()       # HWC float64 like the reference
        return out


def _unsupported(model_name):
    return NotImplementedError(
        f"model '{model_name}': its architecture is not part of the reference repository (segformer++ is fetched from "
        "KieDani/SegformerPlusPlus at construction time); available: 'wasb' / 'hrnet' / 'vitpose'")


BALL_MODELS, TABLE_MODELS = ('wasb', 'vitpose'), ('hrnet', 'vitpose')      # architectures that are part of the reference repository


def _check_model_name(model_name, available):
    """Unsupported names fail before anything is downloaded or unpickled."""
    if model_name not in available:
        raise _unsupported(model_name)


def load_ball_model(model_path, dtype=None):
    """inference/inference_balldetection.py:40-61.  dtype: arithmetic class ('tf32' / 'tf32x3' / 'fp32' / 'bf16', and 'fp16' for
    WASB; see precision.py); None = the architecture's default."""
    load_dict = torch.load(model_path, map_location=torch.device('cpu'), weights_only=False)
    info = load_dict['additional_info']
    model_name, resolution, in_frames = info['model_name'], info['image_resolution'], info['in_frames']
    if model_name == 'wasb':                 # get_model, balldetection/train.py:249-271
        model = WASBNet(in_frames=in_frames, resolution=resolution, pretraining=False, dtype=dtype)
    elif model_name == 'vitpose':
        model = VitPose(in_frames=in_frames, model_size='small', resolution=resolution, pretraining=False, dtype=dtype)
    else:
        raise _unsupported(model_name)
    model.load_state_dict(load_dict['model_state_dict'])
    model.eval()
    print(f'Loaded BallDetection model: {model_name} with resolution {resolution}')
    print(f" - in_frames: {in_frames}, lr: {info.get('lr')}")
    return model, _DetectorTransform(resolution)


def load_table_model(model_path, dtype=None):
    """inference/inference_tabledetection.py:40-57."""
    load_dict = torch.load(model_path, map_location=torch.device('cpu'), weights_only=False)
    info = load_dict['additional_info']
    model_name, resolution = info['model_name'], info['image_resolution']
    if model_name == 'hrnet':                # get_model, tabledetection/train.py:205-225
        model = MyHRNet(resolution=resolution, pretraining=False, dtype=dtype)
    elif model_name == 'vitpose':
        model = TableVitPose(model_size='small', resolution=resolution, pretraining=False, dtype=dtype)
    else:
        raise _unsupported(model_name)
    model.load_state_dict(load_dict['model_state_dict'])
    model.eval()
    print(f'Loaded tabledetection model: {model_name} with resolution {resolution}')
    return model, _DetectorTransform(resolution)


class NormalizeImgCoords:
    """uplifting/transformations.py:252-266 (divides by 2560 x 1440, uplifting/helper.py:26)."""

    def __call__(self, data):
        r_img, table_img = data['r_img'], data['table_img']
        r_img = r_img / np.array([2560, 1440])
        table_img[..., :2] = table_img[..., :2] / np.array([2560, 1440])
        data['r_img'], data['table_img'] = r_img, table_img
        return data


def load_uplifting_model(model_path, dtype=None):
    """inference/inference_uplifting.py:33-58."""
    d = torch.load(model_path, weights_only=False, map_location=torch.device('cpu'))
    info = d['additional_info']
    model = get_uplifting_model(info['name'], size=info['size'], mode=info['tabletoken_mode'], time_rotation=info['time_rotation'], dtype=dtype)
    model.load_state_dict(d['model_state_dict'])
    model.eval()
    print(f"Loaded Uplifting model: {info['name']} with size {info['size']}, tabletoken_mode: {info['tabletoken_mode']}, "
          f"time_rotation: {info['time_rotation']}, transform_mode: {info['transform_mode']}")
    return model, NormalizeImgCoords(), info['transform_mode']


# ---- glue (inference/utils.py) ------------------------------------------------------------------
def _f64_cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(_device())


def filter_trajectory_ball(pred_positions1, pred_positions2, fps):
    """inference/utils.py:70-102: keep frames where both detectors see the ball and agree within 20 px
    (ttk_filter_ball; numpy in, numpy out like the reference)."""
    xy, idx, times, offs = ops.filter_ball(_f64_cuda(pred_positions1), _f64_cuda(pred_positions2), float(fps))
    n = int(offs[1].item())
    if n == 0:       # the reference slices np.array([])[:, :2] here (:98)
        raise IndexError('too many indices for array: array is 1-dimensional, but 2 were indexed')
    return xy[:n].cpu().numpy(), idx[:n].cpu().numpy(), times[:n].cpu().numpy()


def filter_trajectory_table(pred_positions1, pred_positions2):
    """inference/utils.py:137-232: two-model agreement (< 10 px), then the centroid of the largest
    DBSCAN(eps=10, min_samples=3) cluster per keypoint (ttk_filter_table; numpy in, numpy out)."""
    return ops.filter_table(_f64_cuda(pred_positions1), _f64_cuda(pred_positions2)).cpu().numpy()


def _uplifting_transform(ball_coords, table_coords, times):
    """inference/utils.py:268-309 on the GPU (ttk_trajectory_pack): returns CUDA float32 tensors
    ball (1,50,2), table (1,13,3), times (1,50), mask (1,50)."""
    dev = _device()
    ball = torch.from_numpy(np.ascontiguousarray(ball_coords, dtype=np.float64)).to(dev)
    tms = torch.from_numpy(np.ascontiguousarray(times, dtype=np.float64)).to(dev)
    tab = torch.from_numpy(np.ascontiguousarray(table_coords, dtype=np.float64)).to(dev)[None]
    offs = torch.tensor([0, ball.shape[0]], dtype=torch.int32, device=dev)
    b, t, ti, m = ops.trajectory_pack(ball, tms, offs, tab, SEQ_LEN, WIDTH, HEIGHT)
    return b, t, ti, m


class _nvtx:
    """NVTX range around a stage of the path (visible in Nsight Systems / ncu --nvtx): `with _nvtx('ttk:decode'): ...`."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        torch.cuda.nvtx.range_pop()
        return False


class _ReadyMarks:
    """[(frame index, CUDA event)] marking how far an upload has got, filled in by the uploader thread while the caller already
    launches network passes: indexing (and len-1 style access) blocks the HOST only until that mark's event has been recorded on
    the copy stream; the device-side wait is the caller's `wait_event`."""

    def __init__(self, frames):
        import threading
        self.frames = frames
        self.events = [torch.cuda.Event() for _ in frames]
        self._recorded = [threading.Event() for _ in frames]
        self.error = None

    def __len__(self):
        return len(self.frames)

    def __getitem__(self, k):
        k = range(len(self.frames))[k]
        self._recorded[k].wait()
        if self.error is not None:
            raise self.error
        return self.frames[k], self.events[k]

    def record(self, k, stream):
        self.events[k].record(stream)
        self._recorded[k].set()

    def fail(self, exc):
        self.error = exc
        for r in self._recorded:
            r.set()


_POOL = None
_UPLOADERS = {}


def _uploader(device_index):
    """One background thread per device that walks the staging ring of an upload, so that predict() can launch the first network pass
    while later frames are still being staged (the staging loop on the calling thread held back every kernel launch for the whole upload:
    15 ms of a 66 ms call for 96 copied 1080p frames).  Per device, so that predict_clips' uploads to several GPUs run side by side."""
    if device_index not in _UPLOADERS:
        from concurrent.futures import ThreadPoolExecutor
        _UPLOADERS.setdefault(device_index, ThreadPoolExecutor(max_workers=1, thread_name_prefix='ttk-upload%d' % device_index))
    return _UPLOADERS[device_index]


def _staging_pool():
    global _POOL
    if _POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        # host threads that copy numpy frames into the pinned staging ring: up to 8, sharing the cores with the other ranks of the node
        ranks = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1') or 1))
        n = int(os.environ.get('TTK_STAGE_THREADS', '0') or 0) or max(2, min(8, (os.cpu_count() or 8) // ranks))
        _POOL = ThreadPoolExecutor(max_workers=n, thread_name_prefix='ttk-stage')
    return _POOL


# ---- several clips in one call (TableTennisPipeline.predict_clips) -----------------------------------
def clip_stack_plan(lengths, frames_per_stack):
    """Stacks of clips of the given lengths, concatenated in clip order: a sliding window of frames_per_stack frames over each clip
    (stride 1, like predict), never crossing a clip.  Returns the first frame of every stack and the (n + 1,) prefix sums of the stack
    counts per clip."""
    first, offsets, f0 = [], [0], 0
    for n in lengths:
        k = max(n - frames_per_stack + 1, 0)
        first.extend(range(f0, f0 + k))
        offsets.append(offsets[-1] + k)
        f0 += n
    return first, offsets


def clip_blocks(lengths, max_frames):
    """Contiguous [(first clip, end)] blocks of at most max_frames frames each (a longer clip is a block of its own): bounds the device
    memory of predict_clips like _Detector.segment bounds predict()'s."""
    blocks, a, frames = [], 0, 0
    for i, n in enumerate(lengths):
        if i > a and frames + n > max_frames:
            blocks.append((a, i))
            a, frames = i, 0
        frames += n
    if a < len(lengths):
        blocks.append((a, len(lengths)))
    return blocks


def parse_devices(devices, device_count):
    """predict_clips' `devices`: a list of CUDA device indices, torch.device('cuda', i) or 'cuda:i' strings (a device may repeat: one
    replica of the models per entry).  Returns the indices; anything else raises ValueError."""
    if isinstance(devices, (str, int, torch.device)) or not hasattr(devices, '__iter__'):
        raise ValueError('devices must be a list of CUDA devices (indices, torch.device or "cuda:N"), got %r' % (devices,))
    out = []
    for d in devices:
        if isinstance(d, bool) or not isinstance(d, (int, str, torch.device)):
            raise ValueError('devices: %r is not a CUDA device index, torch.device or "cuda:N" string' % (d,))
        if not isinstance(d, int):
            try:
                dv = torch.device(d)
            except (RuntimeError, ValueError) as e:
                raise ValueError('devices: %r is not a CUDA device (%s)' % (d, e)) from None
            if dv.type != 'cuda' or dv.index is None:
                raise ValueError('devices: %r is not an indexed CUDA device ("cuda:N")' % (d,))
            d = dv.index
        if not 0 <= d < device_count:
            raise ValueError('devices: CUDA device %d does not exist (%d visible)' % (d, device_count))
        out.append(d)
    if not out:
        raise ValueError('devices must name at least one CUDA device')
    return out


def _replicate(model, device):
    """A copy of a detector / uplifting model shell on `device`: same architecture, state dict and compute_dtype.  Its weights reach the
    library on its first forward, which must run with `device` current."""
    if isinstance(model, WASBNet):
        m = WASBNet(in_frames=model.in_ch // 3, resolution=model.resolution)
    elif isinstance(model, MyHRNet):
        m = MyHRNet(resolution=model.resolution)
    elif isinstance(model, VitPose):
        m = VitPose(in_frames=model.in_ch // 3, resolution=model.resolution)
    elif isinstance(model, TableVitPose):
        m = TableVitPose(resolution=model.resolution)
    elif isinstance(model, MultiStageModel):
        m = MultiStageModel(model.dim, model.depth, model.num_heads, model.mode, model.time_rotation, model.use_skipconnection)
    else:
        raise TypeError('no replica for %s' % type(model).__name__)
    m.compute_dtype = model.compute_dtype
    m.load_state_dict(model.state_dict())
    return m.to(device).eval()


def _fingerprint(model):
    """Changes when the model's compute_dtype, one of its tensors (replaced) or their contents (in-place writes, load_state_dict) do."""
    return model.compute_dtype, tuple((k, v.data_ptr(), v._version) for k, v in model.state_dict().items())


# ---- public classes ---------------------------------------------------------------------------------
class _Detector:
    frames_per_stack = 1
    chunk = 16                     # stacks per network pass: bounds the workspace and lets uploads overlap compute
    ramp = (4, 12)                 # stacks of the first passes while a clip's frames are still being uploaded

    def _run(self, frames_u8, stack_stride, n_stacks, return_heatmaps, ready=None, heatmaps_to_host=False, first=None):
        """frames_u8: (n, H, W, 3) uint8 CUDA.  Returns positions (n_stacks, C, 3) float64 CUDA and heatmaps or None.
        heatmaps_to_host: the heatmaps come back as ONE pinned host tensor (n_stacks, C, h, w) instead of a CUDA tensor: each pass's
        maps are copied out on a third stream while the next pass computes (predict() returns 3.6 MB per map to the host, like the
        reference does; through pageable memory that copy alone cost more than the network).
        `ready`: [(last frame index, event)] from _upload -- a chunk starts as soon as its frames have arrived, so the
        host->device copy of later frames overlaps the network on earlier ones.
        `first`: (host list, (n_stacks,) int32 CUDA tensor) of each stack's first frame, replacing s * stack_stride -- stacks of several
        clips (clip_stack_plan); the passes are then all full but the last."""
        w, h = self.model.resolution
        prec, dt = self.model.compute_dtype, self.model.storage_dtype
        pos, hms = [], []
        main = torch.cuda.current_stream()
        waited = 0
        # while frames are still arriving the first passes are short (4, then 12 stacks), so that the network starts after 6 frames
        # instead of 18; afterwards full chunks
        for s0, ns in self._pass_plan(n_stacks, self.chunk, ready is not None and first is None, self.ramp):
            if first is not None:
                f_hi = max(first[0][s0:s0 + ns]) + self.frames_per_stack - 1
            else:
                f0 = s0 * stack_stride
                f_hi = f0 + (ns - 1) * stack_stride + self.frames_per_stack - 1
            while ready is not None and waited < len(ready) and (waited == 0 or ready[waited - 1][0] < f_hi):
                main.wait_event(ready[waited][1])
                waited += 1
            if getattr(self.model, 'input_layout', 'nhwc16') == 'nchw':       # ViTPose: the reference's NCHW float32 tensor
                with _nvtx('ttk:preprocess'):
                    if first is not None:
                        x = ops.preprocess_stacks_indexed(frames_u8, self.frames_per_stack, first[1][s0:s0 + ns], w, h, layout='nchw')
                    else:
                        x = ops.preprocess_stacks(frames_u8[f0:f_hi + 1], self.frames_per_stack, stack_stride, ns, w, h, layout='nchw')
                with _nvtx('ttk:heatmap_network'):
                    hm = self.model.heatmaps(x)
            else:
                with _nvtx('ttk:preprocess'):
                    if first is not None:
                        x = ops.preprocess_stacks_indexed(frames_u8, self.frames_per_stack, first[1][s0:s0 + ns], w, h, layout='nhwc16', dtype=dt)
                    else:
                        x = ops.preprocess_stacks(frames_u8[f0:f_hi + 1], self.frames_per_stack, stack_stride, ns, w, h, layout='nhwc16', dtype=dt)
                with _nvtx('ttk:heatmap_network'):
                    hm = self.model.heatmaps_from_nhwc16(x, prec)
            # interface.py:116,169 decode with the TABLE variant of extract_position_torch_gaussian.  It runs on a second stream:
            # the per-map fit is a latency-bound kernel of one warp per map (~0.3 ms whatever the number of maps) that fits beside the
            # persistent convolution CTAs, so the decode of pass i hides under the network of pass i + 1.
            side = getattr(self, '_decode_stream', None)
            if side is None:
                side = self._decode_stream = torch.cuda.Stream(device=hm.device)
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(side), _nvtx('ttk:decode'):
                side.wait_event(done)
                p = ops.decode_heatmaps(hm, self.resolution[0], self.resolution[1], 'table')
            hm.record_stream(side)
            pos.append(p)
            if return_heatmaps and heatmaps_to_host:
                if not hms:                     # pinned blocks come from torch's caching host allocator: no cudaHostAlloc per call
                    hms.append(torch.empty((n_stacks,) + tuple(hm.shape[1:]), dtype=hm.dtype, pin_memory=True))
                    if getattr(self, '_d2h_stream', None) is None:
                        self._d2h_stream = torch.cuda.Stream(device=hm.device)
                d2h = self._d2h_stream
                with torch.cuda.stream(d2h):
                    d2h.wait_event(done)
                    hms[0][s0:s0 + ns].copy_(hm, non_blocking=True)
                hm.record_stream(d2h)
            elif return_heatmaps:
                hms.append(hm)
        main.wait_stream(side)
        for p in pos:
            p.record_stream(main)
        if return_heatmaps and heatmaps_to_host:
            self._d2h_stream.synchronize()
            return torch.cat(pos), hms[0]
        return torch.cat(pos), (torch.cat(hms) if return_heatmaps else None)

    @staticmethod
    def _frame_key(im):
        """Identity of a host frame: its memory (address, shape, strides, element type), for numpy arrays and torch CPU tensors alike."""
        if isinstance(im, torch.Tensor):
            return (im.data_ptr(), tuple(im.shape), tuple(im.stride()), str(im.dtype))
        return (im.__array_interface__['data'][0], tuple(im.shape), tuple(im.strides), im.dtype.str)

    @staticmethod
    def _pass_plan(n_stacks, chunk, streaming, ramp=(4, 12)):
        """[(first stack, stacks)] of the network passes over a clip: full chunks, except that a clip whose frames are still being
        uploaded starts with two short passes (4, then 12 stacks)."""
        bounds, s0 = [], 0
        ramp = list(ramp) if streaming and n_stacks >= chunk else []
        while s0 < n_stacks:
            ns = min(ramp.pop(0) if ramp else chunk, n_stacks - s0)
            bounds.append((s0, ns))
            s0 += ns
        return bounds

    stage_slots = 16               # pinned staging ring for numpy frames: 16 x 6.2 MB at 1080p, whatever the clip length
    segment = 512                  # stacks per upload of predict(): bounds device and pinned memory for arbitrarily long inputs
                                   # (514 1080p frames = 3.2 GB on the device; the reference streams frame by frame)

    def _predict_segments(self, images, return_heatmaps):
        """predict() over at most `segment` stacks at a time; the numpy results are concatenated."""
        pos, hms = [], []
        for s0 in range(0, max(len(images), 1), self.segment):
            p, hm = self.predict_device(images[s0:s0 + self.segment], return_heatmaps, heatmaps_to_host=True)
            pos.append(p.cpu().numpy())
            if return_heatmaps:
                hms.append(hm.numpy())          # (a view of the pinned block; the array keeps it alive)
        return (pos[0] if len(pos) == 1 else np.concatenate(pos)), ((hms[0] if len(hms) == 1 else np.concatenate(hms)) if return_heatmaps else None)

    def _upload(self, images, dev, out=None):
        """Upload each distinct frame once, asynchronously on a copy stream.  numpy frames (pageable memory, what cv2 delivers) go
        through a small ring of pinned staging slots: host threads copy frame i into slot i % stage_slots (numpy releases the GIL for
        it) as soon as the transfer that last used the slot has finished (one event per slot -- no stream-wide synchronisation), and
        the slot is sent as soon as it is staged, so the host memcpy pipelines with the PCIe transfer.  torch CPU tensors (e.g.
        already pinned) are copied directly.  Returns the (n, H, W, 3) uint8 CUDA tensor, per input image its row in it, and
        [(frame index, event)] marking how far the copy has got.
        out: a (len(images), H, W, 3) uint8 CUDA tensor to write into instead (a slice of a LiveSession's frame pool): every image gets
        its own row, in order, host tensors too go through the staging ring, and the caller keeps `out` alive until the copy stream
        has passed the last mark."""
        torch.cuda.nvtx.range_push('ttk:upload')
        try:
            return self._upload_frames(images, dev, out)
        finally:
            torch.cuda.nvtx.range_pop()

    def _upload_frames(self, images, dev, out=None):
        slots, order, uniq = {}, [], []
        if out is not None:
            uniq, order = list(images), list(range(len(images)))
        else:
            for im in images:
                # frames are recognised by their memory, not by the Python object: clip[i] creates a new view object on every indexing,
                # and a sliding window over a clip names every frame three times
                k = self._frame_key(im)
                if k not in slots:
                    slots[k] = len(uniq)
                    uniq.append(im)
                order.append(slots[k])
        fshape = tuple(uniq[0].shape)
        for u in uniq:
            if tuple(u.shape) != fshape or len(fshape) != 3 or fshape[2] != 3 or (u.dtype != torch.uint8 if isinstance(u, torch.Tensor) else u.dtype != np.uint8):
                raise ValueError('frames must be uint8 arrays of one common shape (H, W, 3); got %s %s (first frame %s)' % (tuple(u.shape), u.dtype, fshape))
        n = len(uniq)
        own = out is None
        if own:
            out = torch.empty((n,) + fshape, dtype=torch.uint8, device=dev)
        elif tuple(out.shape) != (n,) + fshape:
            raise ValueError('upload target of shape %s for %d frames of shape %s' % (tuple(out.shape), n, fshape))
        # into a given `out` (LiveSession.push), host tensors are staged like numpy frames: the caller may reuse them once the marks
        # are recorded, whereas a direct non_blocking copy from pinned memory would still be reading them
        all_torch = all(isinstance(u, torch.Tensor) and (own or u.is_cuda) for u in uniq)
        copy_stream = getattr(self, '_copy_stream', None)
        if copy_stream is None:
            copy_stream = self._copy_stream = torch.cuda.Stream(device=dev)
        copy_stream.wait_stream(torch.cuda.current_stream())
        ready = []

        def mark(i):
            if i % 2 == 1 or i == n - 1:      # an event every other frame: the first pass (4 stacks) starts after 6 frames
                ev = torch.cuda.Event()
                ev.record(copy_stream)
                ready.append((i, ev))

        if all_torch:
            with torch.cuda.stream(copy_stream):
                for i, u in enumerate(uniq):
                    out[i].copy_(u, non_blocking=True)
                    mark(i)
            return out, order, ready
        ns = self.stage_slots
        stage = getattr(self, '_stage', None)
        if stage is None or tuple(stage.shape[1:]) != fshape:
            stage = self._stage = torch.empty((ns,) + fshape, dtype=torch.uint8).pin_memory()
            self._stage_ev = [None] * ns
        view, slot_ev = stage.numpy(), self._stage_ev
        slot_ptr = [stage[k].data_ptr() for k in range(ns)]
        marks = _ReadyMarks([i for i in range(n) if i % 2 == 1 or i == n - 1])      # an event every other frame: the first pass (4 stacks) starts after 6 frames
        if own:
            out.record_stream(copy_stream)
        dev_index = torch.cuda.current_device()

        def stage_one(i, ev):
            if ev is not None:
                ev.synchronize()            # the transfer that last read this slot (possibly of an earlier call) has finished
            u = uniq[i]
            u = u.numpy() if isinstance(u, torch.Tensor) else u
            if u.flags['C_CONTIGUOUS']:     # non-temporal stores: 11.5 instead of 8.7 GB/s per thread (tools/host_staging_probe.py)
                _lib.check(_lib.lib.ttk_host_copy_stream(slot_ptr[i % ns], u.ctypes.data, u.nbytes))
            else:
                view[i % ns] = u

        def run():
            try:
                torch.cuda.set_device(dev_index)
                pool = _staging_pool()
                staged = {i: pool.submit(stage_one, i, slot_ev[i % ns]) for i in range(min(ns, n))}
                k = 0
                with torch.cuda.stream(copy_stream):
                    for i in range(n):
                        staged.pop(i).result()
                        out[i].copy_(stage[i % ns], non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(copy_stream)
                        slot_ev[i % ns] = ev
                        if i + ns < n:
                            staged[i + ns] = pool.submit(stage_one, i + ns, ev)
                        if i % 2 == 1 or i == n - 1:
                            marks.record(k, copy_stream)
                            k += 1
            except BaseException as e:      # noqa: BLE001 - handed to the thread that reads the marks
                marks.fail(e)

        _uploader(dev_index).submit(run)
        return out, order, marks


class BallDetector(_Detector):
    """interface.py:83-134."""
    frames_per_stack = 3

    def __init__(self, model_name='segformerpp_b2', dtype=None):
        """dtype: 'tf32' / 'tf32x3' / 'fp32' / 'bf16' (precision.py); None = the architecture's default tensor-core path."""
        _check_model_name(model_name, BALL_MODELS)
        self.device = _device()
        self.resolution = (WIDTH, HEIGHT)
        self.model, self.transform = load_ball_model(model_path=_get_weights_path(f"inference_balldetection/{model_name}/model.pt"), dtype=dtype)
        self.model.to(self.device)
        self.model.eval()

    def predict(self, images, return_heatmaps=True):
        """images: list (length B) of (prev, curr, next) HWC uint8 BGR frames.
        Returns pred_pos (B, 3) float64 [x, y, 1.0] and the heatmaps (B, 1, h, w) float32 (None if return_heatmaps=False)."""
        return self._predict_segments(images, return_heatmaps)

    def predict_device(self, images, return_heatmaps=False, heatmaps_to_host=False):
        """predict() without the device->host copy: positions (B, 3) float64 and heatmaps stay CUDA tensors."""
        flat = [im for triple in images for im in (triple[0], triple[1], triple[2])]
        frames, order, ready = self._upload(flat, self.device)
        consecutive = all(order[3 * i + j] == i + j for i in range(len(images)) for j in range(3))
        if consecutive:                 # a sliding window over one clip (TableTennisPipeline.predict): every frame uploaded once
            stride = 1
        else:
            stride = 3
            if order != list(range(len(flat))):
                torch.cuda.current_stream().wait_event(ready[-1][1])
                frames, ready = frames[torch.tensor(order, device=self.device)], None
        with torch.no_grad():
            pos, hm = self._run(frames, stride, len(images), return_heatmaps, ready, heatmaps_to_host)
        return pos[:, 0], hm

    def filter_trajectory(self, ball_positions, ball_positions_aux, fps):
        return filter_trajectory_ball(ball_positions, ball_positions_aux, fps)


class TableDetector(_Detector):
    """interface.py:137-186."""
    frames_per_stack = 1

    def __init__(self, model_name='segformerpp_b2', dtype=None):
        _check_model_name(model_name, TABLE_MODELS)
        self.device = _device()
        self.resolution = (WIDTH, HEIGHT)
        self.KEYPOINT_VISIBLE = KEYPOINT_VISIBLE
        self.model, self.transform = load_table_model(model_path=_get_weights_path(f"inference_tabledetection/{model_name}/model.pt"), dtype=dtype)
        self.model.to(self.device)
        self.model.eval()

    def predict(self, images, return_heatmaps=True):
        """images: list of HWC uint8 BGR frames -> pred_pos (B, 13, 3) float64, heatmaps (B, 1, 13, h, w)."""
        pos, hm = self._predict_segments(images, return_heatmaps)
        return pos, (hm[:, None] if return_heatmaps else None)

    def predict_device(self, images, return_heatmaps=False, heatmaps_to_host=False):
        frames, order, ready = self._upload(list(images), self.device)
        if order != list(range(len(images))):
            torch.cuda.current_stream().wait_event(ready[-1][1])
            frames, ready = frames[torch.tensor(order, device=self.device)], None
        with torch.no_grad():
            pos, hm = self._run(frames, 1, len(images), return_heatmaps, ready, heatmaps_to_host)
        return pos, hm

    def calibrate_camera(self, keypoints):
        return calibrate_camera(keypoints)

    def filter_trajectory(self, table_keypoints, table_keypoints_aux):
        return filter_trajectory_table(table_keypoints, table_keypoints_aux)


def calibrate_camera(table_coords):
    """inference/utils.py:312-329: DLT start + 100-hypothesis RANSAC of BFGS fits + refit on the inliers
    (dataprocessing/regress_cameramatrices.py), all hypotheses concurrently on the GPU (ttk_calibrate_camera).
    table_coords (13, 3) -> Mint (3, 4), Mext (4, 4) float64 numpy, like the reference returns."""
    kp = np.ascontiguousarray(table_coords, dtype=np.float64).reshape(1, 13, 3)
    samples = ops.ransac_sample_table(kp)
    dev = _device()
    mint, mext, info = ops.calibrate_camera(torch.from_numpy(kp).to(dev), torch.from_numpy(samples).to(dev), WIDTH, HEIGHT)
    info = info.cpu().numpy()[0]
    if not info[3]:
        raise ValueError("Intrinsic matrix K has K[2,2] close to zero, indicating a degenerate camera.")     # my_dlt.py:128
    if info[0] == 0:
        raise ValueError("RANSAC failed to find a valid model.")
    return mint[0].cpu().numpy(), mext[0].cpu().numpy()


class UpliftingModel:
    """interface.py:189-247."""

    def __init__(self, dtype=None):
        self.device = _device()
        self.model, self.transform, self.transform_mode = load_uplifting_model(model_path=_get_weights_path("inference_uplifting/ours/model.pt"), dtype=dtype)
        self.model.to(self.device)
        self.model.eval()

    def predict(self, ball_coords, table_coords, times):
        data = self.transform({'r_img': ball_coords, 'table_img': table_coords})
        ball_coords, table_coords = data['r_img'], data['table_img']
        mask = np.zeros((ball_coords.shape[0] + 1,), dtype=np.float32)
        mask[:-1] = 1.0
        return self.predict_without_normalization(ball_coords, table_coords, torch.tensor(mask).to(self.device), times)

    def predict_without_normalization(self, ball_coords, table_coords, mask, times):
        ball_coords, table_coords, mask, times = (a.to(self.device) for a in (ball_coords, table_coords, mask, times))
        with torch.no_grad():
            pred_rotation, pred_position = self.model(ball_coords, table_coords, mask, times)
            if self.transform_mode == 'global':
                pred_rotation_local = ops.rotation_local(pred_rotation, pred_position)
            else:
                pred_rotation_local = pred_rotation
        T_prime = int(mask.sum().item())
        pred_position = pred_position[:, :T_prime, :].cpu().numpy()
        return pred_rotation_local.squeeze(0), pred_position.squeeze(0)


class TableTennisPipeline:
    """interface.py:251-312.  The reference pairs segformerpp_b2 (main) with wasb / hrnet (auxiliary) and rejects frames where
    the two disagree.  The segformer++ architecture is not in the reference repository, so the main detectors default to the
    other in-repo architecture, ViTPose; the auxiliary detectors are the reference's own.  Like the reference, four separate
    detector objects are built (main and auxiliary never share one, even when they name the same model)."""

    def __init__(self, ball_model='vitpose', ball_model_aux='wasb', table_model='vitpose', table_model_aux='hrnet', dtype=None):
        """dtype: None / 'tf32' / 'tf32x3' = every component on its reference-class tensor-core path (TF32 convolutions, 3xTF32
        Linear layers and attention); 'bf16' or 'fp32' = every component on that path.  'fp16' is refused: only the WASB / HRNet
        detectors have an fp16 path (switch one with ``pipe.<detector>.model.compute_dtype = 'fp16'``)."""
        if dtype is not None and canonical(dtype) == FP16:
            raise NotImplementedError("TableTennisPipeline has no fp16 path: fp16 exists for the WASB / HRNet detectors only (ViTPose and "
                                      "the uplifting transformer have none); build the pipeline with another dtype and set "
                                      "pipe.ball_detector_aux.model.compute_dtype = 'fp16' / pipe.table_detector_aux.model.compute_dtype = "
                                      "'fp16' on a WASB / HRNet detector")
        self.device = _device()
        if dtype is not None and canonical(dtype) in (TF32, TF32X3):
            dtype = None
        self.ball_detector = BallDetector(model_name=ball_model, dtype=dtype)
        self.ball_detector_aux = BallDetector(model_name=ball_model_aux, dtype=dtype)
        self.table_detector = TableDetector(model_name=table_model, dtype=dtype)
        self.table_detector_aux = TableDetector(model_name=table_model_aux, dtype=dtype)
        self.uplifting_model = UpliftingModel(dtype=dtype)
        self.KEYPOINT_VISIBLE = self.table_detector.KEYPOINT_VISIBLE

    def predict(self, images, fps):
        """interface.py:263-289.  Detections, both filters, the normalise/pad step and the transformer stay on the
        device: the only host visit is the final result (and T' for slicing it, as in the reference)."""
        n = len(images)
        # every frame crosses PCIe once: the four detector passes (ball / table, main / auxiliary) share the uploaded clip, and the
        # first pass starts while later frames are still arriving
        frames, order, ready = self.ball_detector._upload(list(images), self.device)
        if order != list(range(n)):
            torch.cuda.current_stream().wait_event(ready[-1][1])
            frames, ready = frames[torch.tensor(order, device=self.device)], None
        with torch.no_grad():
            ball_positions = self.ball_detector._run(frames, 1, n - 2, False, ready)[0][:, 0]       # sliding (prev, cur, next) window
            ball_positions_aux = self.ball_detector_aux._run(frames, 1, n - 2, False, None)[0][:, 0]
            table_keypoints = self.table_detector._run(frames, 1, n, False, None)[0]
            table_keypoints_aux = self.table_detector_aux._run(frames, 1, n, False, None)[0]
        return self._tail(ball_positions, ball_positions_aux, table_keypoints, table_keypoints_aux, fps)

    def _tail(self, ball_positions, ball_positions_aux, table_keypoints, table_keypoints_aux, fps):
        """predict's steps after the four detectors, shared with LiveSession.end_rally: the ball filter, the table filters, the
        trajectory packing, the uplifting transformer and the spin rotation.  Takes the (n - 2, 3) ball and (n, K, 3) table positions
        of one clip on the device; returns predict's (spin, pos3d)."""
        ball_xy, _, times_ball, offsets = ops.filter_ball(ball_positions, ball_positions_aux, float(fps))
        with _nvtx('ttk:filters_pack'):
            filtered_table_keypoints = ops.filter_table(table_keypoints, table_keypoints_aux)
            ball_coords, table_coords, times, mask = ops.trajectory_pack(ball_xy, times_ball, offsets, filtered_table_keypoints[None],
                                                                        SEQ_LEN, WIDTH, HEIGHT)
        with _nvtx('ttk:uplift'):
            return self.uplifting_model.predict_without_normalization(ball_coords, table_coords, mask, times)

    def live(self, fps, streams=1, k=None, slots=None):
        """A LiveSession (upliftingtabletennis_b200/live.py) over `streams` cameras at `fps`: frames are pushed as they arrive, the
        detectors run on them while the rally goes on, and end_rally(stream) returns exactly what predict(the rally's frames, fps)
        returns.  k: ready stacks that launch a detector pass (default live.DEFAULT_K); slots: device frame slots per stream (default
        live.DEFAULT_SLOTS)."""
        from .live import LiveSession
        return LiveSession(self, fps, streams, k, slots)

    def predict_clips(self, clips, fps, devices=None):
        """Many rallies in one call: returns [(spin, pos3d), ...], exactly [self.predict(c, fps) for c in clips] (same types, spin on
        the same device, same values bit for bit).  clips: list of clips, each a list of HWC uint8 BGR frames like predict takes, all
        of one frame size.
        On one device each distinct frame is uploaded once; each detector runs full passes whose stacks come from several clips (no
        window crosses a clip); the ball and table filters, the trajectory packing, the uplifting transformer and the spin rotation run
        once for all clips.  Work goes a block of clips (at most _Detector.segment frames) at a time, which bounds device memory.
        devices: None = the current device.  Otherwise a list of CUDA device indices, torch.device or 'cuda:N' strings: the clips
        are split into contiguous blocks (sharding.shard_range), one per entry, and each entry runs the one-device path on its block
        from a launcher thread of its own, with its own copy of the five models (built from this pipeline's models, rebuilt when their
        state dict or compute_dtype change; the first entry on the pipeline's device uses the pipeline's models).  A device may
        appear twice.  Only the per-clip results come back to the calling thread, whose current device stays as it was.
        Raises ValueError, naming the clip, when predict would raise ValueError for one (0, or 50 or more agreeing ball detections:
        the first such clip), before any uplift runs; and for a clip of fewer than 3 frames, which has no ball stack."""
        clips = [list(c) for c in clips]
        for i, c in enumerate(clips):
            if len(c) < 3:
                raise ValueError('clip %d: %d frames; a clip needs at least 3 (one (prev, cur, next) ball stack)' % (i, len(c)))
        if devices is None:
            if not clips:
                return []
            parts = self._parts()
            packed, counts = self._detect_clips(parts, clips, fps)
            counts = counts.cpu().tolist()
            self._check_counts(counts, 0)
            spin, pos = self._uplift_clips(parts, packed, counts)
            return [(spin[i], pos[i, :c]) for i, c in enumerate(counts)]
        idx = parse_devices(devices, torch.cuda.device_count())
        if not clips:
            return []
        blocks = [sharding.shard_range(len(clips), r, len(idx)) for r in range(len(idx))]
        home = self._home_device()          # where predict computes, and where the spins are returned
        own = idx.index(home.index) if home.index in idx else -1
        pool = getattr(self, '_launchers', None)
        if pool is None or pool._max_workers < len(idx):
            from concurrent.futures import ThreadPoolExecutor
            pool = self._launchers = ThreadPoolExecutor(max_workers=len(idx), thread_name_prefix='ttk-launch')

        def detect(r):
            torch.cuda.set_device(idx[r])
            parts = self._parts() if r == own else self._replica_parts(r, idx[r])
            a, b = blocks[r]
            if a == b:
                return parts, None, []
            packed, counts = self._detect_clips(parts, clips[a:b], fps)
            return parts, packed, counts.cpu().tolist()

        def uplift(r, parts, packed, counts):
            torch.cuda.set_device(idx[r])
            if not counts:
                return []
            spin, pos = self._uplift_clips(parts, packed, counts)
            spin = spin.to(home)
            return [(spin[i], pos[i, :c]) for i, c in enumerate(counts)]

        stage1 = self._join([pool.submit(detect, r) for r in range(len(idx))])
        for r, (_, _, counts) in enumerate(stage1):
            self._check_counts(counts, blocks[r][0])
        stage2 = self._join([pool.submit(uplift, r, *stage1[r]) for r in range(len(idx))])
        return [res for part in stage2 for res in part]

    @staticmethod
    def _join(futures):
        """Results in order, after every launcher has finished (a failing one does not leave the others running)."""
        from concurrent.futures import wait
        wait(futures)
        return [f.result() for f in futures]

    def _parts(self):
        return self.ball_detector, self.ball_detector_aux, self.table_detector, self.table_detector_aux, self.uplifting_model

    def _home_device(self):
        return next(iter(self.uplifting_model.model.state_dict().values())).device

    def _replica_parts(self, slot, device_index):
        """The five models of launcher `slot` on device_index, rebuilt when the pipeline's models changed.  Runs on the launcher's
        thread with device_index current."""
        own = self._parts()
        key = (device_index,) + tuple(_fingerprint(p.model) for p in own)
        cache = self.__dict__.setdefault('_replicas', {})
        hit = cache.get(slot)
        if hit is not None and hit[0] == key:
            return hit[1]
        dev = torch.device('cuda', device_index)
        parts = []
        for p in own:
            q = type(p).__new__(type(p))
            q.__dict__.update({k: v for k, v in p.__dict__.items() if k not in ('model', '_copy_stream', '_decode_stream', '_d2h_stream',
                                                                                  '_stage', '_stage_ev')})
            q.device, q.model = dev, _replicate(p.model, dev)
            parts.append(q)
        cache[slot] = (key, tuple(parts))
        return cache[slot][1]

    def _detect_clips(self, parts, clips, fps):
        """Detectors, both filters and the trajectory packing of `clips` on the current device, a block of clips at a time.
        Returns the packed uplift inputs (ball, table, times, mask) of all clips and the (n,) int32 CUDA agreeing-detection counts."""
        ball, ball_aux, table, table_aux, _ = parts
        dev = torch.device('cuda', torch.cuda.current_device())
        packed, counts = [], []
        for a, b in clip_blocks([len(c) for c in clips], ball.segment):
            lengths = [len(c) for c in clips[a:b]]
            n = sum(lengths)
            frames, order, ready = ball._upload([f for c in clips[a:b] for f in c], dev)
            if order != list(range(n)):
                torch.cuda.current_stream().wait_event(ready[-1][1])
                frames, ready = frames[torch.tensor(order, device=dev)], None
            bfirst, boffs = clip_stack_plan(lengths, ball.frames_per_stack)
            tfirst, toffs = clip_stack_plan(lengths, table.frames_per_stack)
            plan = torch.tensor(bfirst + boffs + tfirst + toffs, dtype=torch.int32).pin_memory().to(dev, non_blocking=True)
            bfirst_d, boffs_d, tfirst_d, toffs_d = plan.split([len(bfirst), len(boffs), len(tfirst), len(toffs)])
            with torch.no_grad():
                bpos = ball._run(frames, 1, len(bfirst), False, ready, first=(bfirst, bfirst_d))[0][:, 0]
                bpos_aux = ball_aux._run(frames, 1, len(bfirst), False, None, first=(bfirst, bfirst_d))[0][:, 0]
                ball_xy, _, times_ball, offsets = ops.filter_ball_clips(bpos, bpos_aux, boffs_d, float(fps))
                tpos = table._run(frames, 1, len(tfirst), False, None, first=(tfirst, tfirst_d))[0]
                tpos_aux = table_aux._run(frames, 1, len(tfirst), False, None, first=(tfirst, tfirst_d))[0]
            with _nvtx('ttk:filters_pack'):
                tab = ops.filter_table_clips(tpos, tpos_aux, toffs_d)
                packed.append(ops.trajectory_pack(ball_xy, times_ball, offsets, tab, SEQ_LEN, WIDTH, HEIGHT))
                counts.append(offsets[1:] - offsets[:-1])
        return [torch.cat(x) for x in zip(*packed)], torch.cat(counts)

    @staticmethod
    def _check_counts(counts, first_clip):
        """predict() raises ValueError (the uplifting model's mask check) for 0 or >= SEQ_LEN agreeing detections."""
        for i, c in enumerate(counts):
            if c == 0 or c >= SEQ_LEN:
                raise ValueError('clip %d (%d agreeing ball detections): %s' % (first_clip + i, c, MASK_FORMAT_ERROR))

    @staticmethod
    def _uplift_clips(parts, packed, counts):
        """The uplifting transformer on the packed clips (one forward for all of them): spins (n, 3) on the device and positions
        (n, SEQ_LEN, 3) as one host array."""
        up = parts[4]
        ball, table, times, mask = packed
        with _nvtx('ttk:uplift'), torch.no_grad():
            if up.model.compute_dtype == BF16:
                # the bf16 stacks are not batch invariant: a row's tensor-core sums depend on where its keys sit in the 128-row tile,
                # and the 1-ulp differences can flip a bf16 rounding (tests/test_gpu_full_size.py); one trajectory per forward then
                # gives what predict computes
                outs = [up.model(ball[i:i + 1], table[i:i + 1], mask[i:i + 1], times[i:i + 1]) for i in range(len(counts))]
                rot, pos = torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs])
            else:
                rot, pos = up.model(ball, table, mask, times)
            spin = ops.rotation_local(rot, pos) if up.transform_mode == 'global' else rot
        return spin, pos.cpu().numpy()

    def calibrate_camera(self, keypoints):
        return calibrate_camera(keypoints)

    def reproject(self, positions_3d, Mint, Mext):
        """interface.py:301-312: numpy in, numpy out (float64 like the reference's numpy path)."""
        p = torch.from_numpy(np.asarray(positions_3d, dtype=np.float64)).to(self.device)
        out = ops.project(p, torch.from_numpy(np.asarray(Mext, dtype=np.float64)).to(self.device),
                          torch.from_numpy(np.asarray(Mint, dtype=np.float64)).to(self.device))
        return out.cpu().numpy()
