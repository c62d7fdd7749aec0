"""2D->3D uplifting transformer on libttk.

Mirrors ``uplifting/model.py:get_model`` / ``MultiStageModel`` (forward(ball, table, mask, times) -> (rot, pos))
with an ``nn.Module`` shell whose ``state_dict()`` keys equal the reference's, so the reference checkpoint
(inference/inference_uplifting.py:33-58) loads strictly.  Arithmetic runs in the CUDA library."""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from ._lib import lib, check, ptr, stream_ptr
from .detector import _attach
from .precision import BF16, FP32, TF32X3, PrecisionMixin, lib_enum

MASK_FORMAT_ERROR = 'wrong format for masks. Should be 0, 1 or -1e9, 0.'
SIZES = {'small': (32, 8, 4), 'base': (64, 12, 4), 'large': (128, 16, 4), 'huge': (192, 16, 8)}   # uplifting/model.py:574-603
PARAM_SHAPES = {'cls_token': lambda d: (1, 1, d)}


class UpliftEngine:
    def __init__(self, dim, heads, depth, use_skipconnection):
        h = C.c_void_p()
        check(lib.ttk_uplift_create(dim, heads, depth, 1 if use_skipconnection else 0, C.byref(h)))
        self.h = h
        self.dim = dim
        self.params = []
        name, numel = C.create_string_buffer(128), C.c_int()
        for i in range(lib.ttk_uplift_num_params(h)):
            check(lib.ttk_uplift_param_info(h, i, name, C.byref(numel)))
            self.params.append((name.value.decode(), numel.value))
        self._ws = None
        self.loaded = False

    def __del__(self):
        if getattr(self, 'h', None) is not None and lib is not None:
            lib.ttk_uplift_destroy(self.h)
            self.h = None

    def load(self, sd):
        _lib.require_device()
        for i, (name, numel) in enumerate(self.params):
            t = sd[name].detach().float().cpu().contiguous()
            assert t.numel() == numel, (name, t.shape, numel)
            check(lib.ttk_uplift_set_param(self.h, i, ptr(t), numel))
        self.loaded = True

    TF32X3_CHUNK = 4096          # trajectories per library call on the tf32x3 path: its activations live in HBM (7.3 GB per 4096)

    def forward(self, ball, table, mask, times, dtype=torch.float32, mask_additive=False):
        """mask_additive False: mask in {0, 1}; True: mask holds the reference's additive {-1e9, 0} values, which it keeps as they are
        (uplifting/model.py:541-546), so padded rows attend to the valid frames instead of to nothing."""
        assert self.loaded
        B, T, _ = ball.shape
        dev = ball.device
        dt = lib_enum(dtype)
        if dt == _lib.TF32X3 and B > self.TF32X3_CHUNK:
            parts = [self.forward(ball[i:i + self.TF32X3_CHUNK], table[i:i + self.TF32X3_CHUNK], mask[i:i + self.TF32X3_CHUNK],
                                  times[i:i + self.TF32X3_CHUNK], dtype, mask_additive) for i in range(0, B, self.TF32X3_CHUNK)]
            return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])
        args = [a.to(torch.float32).contiguous() for a in (ball, table, mask, times)]
        need = lib.ttk_uplift_workspace_bytes(self.h, B, T, dt)
        if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
            self._ws = torch.empty((need,), dtype=torch.uint8, device=dev)
        rot = torch.empty((B, 3), dtype=torch.float32, device=dev)
        pos = torch.empty((B, T, 3), dtype=torch.float32, device=dev)
        check(lib.ttk_uplift_forward(self.h, ptr(args[0]), ptr(args[1]), ptr(args[2]), ptr(args[3]), B, T, int(bool(mask_additive)), dt,
                                     ptr(rot), ptr(pos), ptr(self._ws), self._ws.numel(), stream_ptr()))
        return rot, pos

    def last_launches(self):
        return lib.ttk_uplift_last_launches(self.h)


def _shape_of(name, numel, dim):
    if name == 'cls_token':
        return (1, 1, dim)
    if name.endswith('inv_freq') or name.endswith('.bias') or 'norm' in name:
        return (numel,)
    if name.endswith('.weight'):
        if 'qkv' in name:
            return (3 * dim, dim)
        for key, (o, i) in (('embed.fc1', (dim, 3)), ('ball_embed.fc1', (dim, 2)), ('table_embed.fc1', (dim, 2)),
                            ('head.fc1', (dim // 2, dim)), ('head.fc2', (dim // 4, dim // 2)), ('head.fc3', (3, dim // 4))):
            if key in name and not (key == 'embed.fc1' and ('ball' in name or 'table' in name)):
                return (o, i)
        return (dim, dim)
    raise KeyError(name)


class MultiStageModel(PrecisionMixin, nn.Module):
    """Drop-in for uplifting/model.py:MultiStageModel (tabletoken_mode 'dynamic', time_rotation 'new').
    ``compute_dtype`` (constructor argument ``dtype``): 'tf32x3' (default: tcgen05 tensor cores with split operands, fp32-level
    results like the reference's fp32 Linear layers on a GPU), 'fp32' (fused SIMT stacks, the strict parity path) or 'bf16'
    (fused tcgen05 stacks, bf16 operands)."""
    default_precision = TF32X3
    supported_precisions = (TF32X3, FP32, BF16)

    def __init__(self, dim, depth, num_heads, mode='dynamic', time_rotation='new', use_skipconnection=False, dtype=None):
        super().__init__()
        if dtype is not None:
            self.compute_dtype = dtype
        if mode != 'dynamic' or time_rotation != 'new':
            raise NotImplementedError("only tabletoken_mode='dynamic' with time_rotation='new' (the released 'ours' model) has kernels")
        self.engine = UpliftEngine(dim, num_heads, depth, use_skipconnection)
        self.dim, self.mode, self.time_rotation, self.use_skipconnection = dim, mode, time_rotation, use_skipconnection
        self.depth, self.num_heads = depth, num_heads
        for name, numel in self.engine.params:
            shape = _shape_of(name, numel, dim)
            assert int(torch.tensor(shape).prod()) == numel, (name, shape, numel)
            _attach(self, name, torch.zeros(shape), True)
        self._dirty = True
        self.register_load_state_dict_post_hook(lambda module, incompatible: setattr(module, '_dirty', True))

    def _sync(self):
        if self._dirty:
            self.engine.load(self.state_dict())
            self._dirty = False

    def forward(self, ball_pos, table_pos, mask, times):
        if not ball_pos.is_cuda:
            raise RuntimeError('upliftingtabletennis_b200 runs on a B200 GPU only; move the inputs to CUDA (there is no CPU fallback)')
        # uplifting/model.py:541-546 -- same host-side check (and the same ValueError on an all-ones mask); like the reference, an
        # additive {-1e9, 0} mask is used as it is
        mn, mx = float(mask.min()), float(mask.max())
        if mn == 0 and mx == 1:
            additive = False
        elif mx == 0 and mn < -1e8:
            additive = True
        else:
            raise ValueError(MASK_FORMAT_ERROR)
        self._sync()
        return self.engine.forward(ball_pos, table_pos, mask, times, self.compute_dtype, mask_additive=additive)


def get_model(name='singlestage', size='small', mode='stacked', time_rotation='new', dtype=None):
    """uplifting/model.py:574-603.  Only the multi-stage family is on the hot path."""
    assert time_rotation in ['old', 'new'], 'time_rotation should be either "old" or "new"'
    if name not in ('multistage', 'connectstage'):
        raise NotImplementedError("only 'multistage' / 'connectstage' have B200 kernels (got %r)" % name)
    if size not in SIZES:
        raise ValueError(f'Unknown model size {size}')
    dim, depth, heads = SIZES[size]
    model = MultiStageModel(dim, depth, heads, mode=mode, time_rotation=time_rotation, use_skipconnection=(name == 'connectstage'), dtype=dtype)
    model.time_rotation = time_rotation
    return model
