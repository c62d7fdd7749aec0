"""HRNet-W18-small heatmap networks on libttk: WASB ball detector and HRNet table detector.

Mirrors the reference seams ``model(x) -> (heatmap, None)`` (balldetection/models/wasb.py:596-608)
and ``model(x) -> heatmaps`` (tabledetection/models/hrnet.py:588-590) with ``nn.Module`` shells whose
``state_dict()`` has exactly the reference's keys, so reference checkpoints load strictly
(inference/inference_balldetection.py:40-61).  The arithmetic runs in the CUDA library."""
import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from ._lib import lib, check, ptr, stream_ptr
from .precision import PrecisionMixin, TF32, TF32X3, FP32, BF16, FP16, lib_enum, storage_dtype

BN_EPS = 1e-5


class HRNetEngine:
    """Owns a ttk_hrnet handle: conv list, folded weights, workspace."""

    def __init__(self, in_ch, out_ch, out_first, out_count):
        h = C.c_void_p()
        check(lib.ttk_hrnet_create(in_ch, out_ch, out_first, out_count, C.byref(h)))
        self.h = h
        self.in_ch, self.out_ch, self.out_first, self.out_count = in_ch, out_ch, out_first, out_count
        self.specs = []
        name, bn = C.create_string_buffer(128), C.create_string_buffer(128)
        ints = [C.c_int() for _ in range(4)]
        for i in range(lib.ttk_hrnet_num_convs(h)):
            check(lib.ttk_hrnet_conv_info(h, i, name, bn, *[C.byref(v) for v in ints]))
            self.specs.append((name.value.decode(), bn.value.decode(), ints[0].value, ints[1].value, ints[2].value, ints[3].value))
        self._ws = None
        self.loaded = False

    def __del__(self):
        if getattr(self, 'h', None) is not None and lib is not None:
            lib.ttk_hrnet_destroy(self.h)
            self.h = None

    def state_dict_layout(self):
        out = []
        for name, bn, cin, cout, k, _ in self.specs:
            out.append((name + '.weight', (cout, cin, k, k)))
            if bn:
                for t in ('weight', 'bias', 'running_mean', 'running_var'):
                    out.append(('%s.%s' % (bn, t), (cout,)))
                out.append((bn + '.num_batches_tracked', ()))
            else:
                out.append((name + '.bias', (cout,)))
        return out

    def load(self, sd):
        """Fold eval-mode batch norm into each conv (float64 on the host) and hand the result to the library."""
        _lib.require_device()
        for i, (name, bn, cin, cout, k, _) in enumerate(self.specs):
            w = sd[name + '.weight'].detach().double().cpu().numpy()
            if bn:
                g = sd[bn + '.weight'].detach().double().cpu().numpy()
                beta = sd[bn + '.bias'].detach().double().cpu().numpy()
                mu = sd[bn + '.running_mean'].detach().double().cpu().numpy()
                var = sd[bn + '.running_var'].detach().double().cpu().numpy()
                s = g / np.sqrt(var + BN_EPS)
                w = w * s[:, None, None, None]
                b = beta - mu * s
            else:
                b = sd[name + '.bias'].detach().double().cpu().numpy()
            w32 = np.ascontiguousarray(w.astype(np.float32))
            b32 = np.ascontiguousarray(b.astype(np.float32))
            assert w32.shape == (cout, cin, k, k)
            check(lib.ttk_hrnet_set_conv(self.h, i, ptr(w32), ptr(b32)))
        self.loaded = True

    def forward_nhwc16(self, x, out=None, precision=None):
        """x: (B, H, W, 16) float32, bfloat16 or float16 CUDA tensor -> (B, out_count, H, W) float32.
        precision: 'tf32' / 'tf32x3' / 'fp32' for float32 tensors (default 'fp32': the strict SIMT path), 'bf16' for bfloat16 tensors,
        'fp16' for float16 tensors."""
        assert self.loaded, 'weights not loaded'
        assert x.is_cuda and x.dim() == 4 and x.shape[3] == 16 and x.is_contiguous()
        B, H, W, _ = x.shape
        assert x.dtype in (torch.float32, torch.bfloat16, torch.float16)
        if precision is None:
            precision = {torch.float32: FP32, torch.bfloat16: BF16, torch.float16: FP16}[x.dtype]
        assert storage_dtype(precision) == x.dtype, 'precision %r needs %s tensors' % (precision, storage_dtype(precision))
        dt = lib_enum(precision)
        need = lib.ttk_hrnet_workspace_bytes(self.h, B, H, W, dt)
        if self._ws is None or self._ws.numel() < need or self._ws.device != x.device:
            self._ws = torch.empty((need,), dtype=torch.uint8, device=x.device)
        if out is None:
            out = torch.empty((B, self.out_count, H, W), dtype=torch.float32, device=x.device)
        check(lib.ttk_hrnet_forward(self.h, ptr(x), B, H, W, dt, ptr(out), ptr(self._ws), self._ws.numel(), stream_ptr()))
        return out

    def last_launches(self):
        return lib.ttk_hrnet_last_launches(self.h)


def _attach(root, key, tensor, is_param):
    parts = key.split('.')
    m = root
    for p in parts[:-1]:
        if not hasattr(m, p):
            m.add_module(p, nn.Module())
        m = getattr(m, p)
    if is_param:
        m.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))
    else:
        m.register_buffer(parts[-1], tensor)


class _HRNetModule(PrecisionMixin, nn.Module):
    """nn.Module shell: holds the reference-named tensors, folds them into the engine lazily.
    ``compute_dtype`` (constructor argument ``dtype``): 'tf32' (default: tcgen05 tensor cores at the precision class of the
    reference's cuDNN convolutions), 'tf32x3' (tcgen05 tensor cores, three TF32 products of split operands per product: fp32-level
    results, the class of the reference on a CPU or with cuDNN's TF32 off), 'fp32' (SIMT, strict parity), 'bf16' (tcgen05, bf16
    storage), 'fp16' (tcgen05, fp16 storage: the bf16 kernels with 10 mantissa bits, range +-65504)."""
    default_precision = TF32
    supported_precisions = (TF32, TF32X3, FP32, BF16, FP16)

    def __init__(self, in_ch, out_ch, out_first, out_count, dtype=None):
        super().__init__()
        if dtype is not None:
            self.compute_dtype = dtype
        self.engine = HRNetEngine(in_ch, out_ch, out_first, out_count)
        self.in_ch = in_ch
        for key, shape in self.engine.state_dict_layout():
            if key.endswith('num_batches_tracked'):
                _attach(self, key, torch.zeros((), dtype=torch.long), False)
            elif 'running_' in key:
                _attach(self, key, torch.ones(shape) if key.endswith('var') else torch.zeros(shape), False)
            else:
                _attach(self, key, torch.zeros(shape), True)
        self._dirty = True
        self.register_load_state_dict_post_hook(lambda module, incompatible: setattr(module, '_dirty', True))

    def _sync(self):
        if self._dirty:
            self.engine.load(self.state_dict())
            self._dirty = False

    def heatmaps_from_nhwc16(self, x, precision=None):
        """x in the storage type of the path; precision defaults to this module's compute_dtype when the tensor type fits it."""
        self._sync()
        if precision is None:
            precision = self.compute_dtype if storage_dtype(self.compute_dtype) == x.dtype else None
        return self.engine.forward_nhwc16(x, precision=precision)

    def _forward_nchw(self, x):
        if not x.is_cuda:
            raise RuntimeError('upliftingtabletennis_b200 runs on a B200 GPU only; move the input to CUDA (there is no CPU fallback)')
        B, Cc, H, W = x.shape
        assert Cc == self.in_ch, 'expected %d input channels, got %d' % (self.in_ch, Cc)
        y = torch.zeros((B, H, W, 16), dtype=self.storage_dtype, device=x.device)
        y[..., :Cc] = x.permute(0, 2, 3, 1)
        return self.heatmaps_from_nhwc16(y, self.compute_dtype)


class WASBNet(_HRNetModule):
    """Drop-in for balldetection/models/wasb.py:WASBNet (in_frames=3): forward -> (heatmap (B,1,H,W), None)."""

    def __init__(self, in_frames=3, resolution=(1280, 704), pretraining=False, classify_invisible=False, dtype=None):
        if classify_invisible or pretraining:
            raise NotImplementedError('classify_invisible / pretraining are training-time options outside the inference hot path')
        super().__init__(3 * in_frames, 3, 1, 1, dtype=dtype)
        self.resolution = tuple(resolution)

    def forward(self, x):
        return self._forward_nchw(x), None


class MyHRNet(_HRNetModule):
    """Drop-in for tabledetection/models/hrnet.py:MyHRNet: forward -> heatmaps (B,13,H,W)."""

    def __init__(self, resolution=(1280, 704), pretraining=False, dtype=None):
        assert not pretraining
        super().__init__(3, 13, 0, 13, dtype=dtype)
        self.resolution = tuple(resolution)

    def forward(self, x):
        return self._forward_nchw(x)
