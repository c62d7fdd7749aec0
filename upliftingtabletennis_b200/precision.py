"""Arithmetic classes of the network paths and how callers name them.

  'tf32' : fp32 tensors in HBM, products on the tcgen05 tensor cores with TF32 operands (nearest-even rounding by TMA, fp32
           accumulate) -- what cuDNN does for the reference's convolutions on a GPU (torch enables TF32 for cuDNN by default).
  'tf32x3' : fp32 tensors, every product as three TF32 tensor-core products of split operands (a_hi b_hi + a_lo b_hi + a_hi b_lo,
           fp32 accumulate): fp32-level results on the tensor cores -- the class of the reference's fp32 Linear layers (torch keeps
           TF32 off for matmul on a GPU).  The uplifting transformer's default.
  'fp32' : fp32 SIMT kernels (no tensor cores): the strict parity path against the CPU reference at 1e-4.
  'bf16' : bf16 tensors and operands on the tensor cores, fp32 accumulate; reported separately with its own bound.
  'fp16' : IEEE fp16 tensors and operands on the tensor cores, fp32 accumulate (WASB / HRNet detectors only): the bf16 path's kernels and
           2-byte traffic with TF32's 10 mantissa bits -- the class of torch.autocast('cuda') and model.half().  Its range is +-65504; an
           activation past it becomes inf, as under autocast (nothing is rescaled).

Constructors and hub entry points take ``dtype=`` as one of these strings or the matching torch dtype
(``torch.float32`` means the strict fp32 path, ``torch.bfloat16`` the bf16 path, ``torch.float16`` the fp16 path)."""
import torch

from . import _lib

TF32, FP32, BF16, TF32X3, FP16 = 'tf32', 'fp32', 'bf16', 'tf32x3', 'fp16'
_ALIASES = {'tf32': TF32, 'tensorfloat32': TF32, 'tf32x3': TF32X3, '3xtf32': TF32X3, 'fp32': FP32, 'f32': FP32, 'float32': FP32, 'bf16': BF16, 'bfloat16': BF16,
            'fp16': FP16, 'f16': FP16, 'float16': FP16, 'half': FP16, torch.float32: FP32, torch.bfloat16: BF16, torch.float16: FP16}
_ENUM = {TF32: _lib.TF32, FP32: _lib.F32, BF16: _lib.BF16, TF32X3: _lib.TF32X3, FP16: _lib.F16}
_STORAGE = {BF16: torch.bfloat16, FP16: torch.float16}


def canonical(dtype):
    try:
        return _ALIASES[dtype.lower() if isinstance(dtype, str) else dtype]
    except KeyError:
        raise ValueError("dtype must be one of 'tf32', 'tf32x3', 'fp32', 'bf16', 'fp16' (or torch.float32 / torch.bfloat16 / torch.float16), "
                         "got %r" % (dtype,)) from None


def storage_dtype(precision):
    """torch dtype of the activation tensors of a path."""
    return _STORAGE.get(canonical(precision), torch.float32)


def lib_enum(precision):
    return _ENUM[canonical(precision)]


class PrecisionMixin:
    """``compute_dtype`` attribute of the model shells: settable with any alias, reads back canonical."""
    default_precision = FP32
    supported_precisions = (FP32, BF16)

    @property
    def compute_dtype(self):
        return getattr(self, '_precision', self.default_precision)

    @compute_dtype.setter
    def compute_dtype(self, value):
        p = canonical(value)
        if p not in self.supported_precisions:
            raise NotImplementedError('%s has no %s path (available: %s)' % (type(self).__name__, p, ', '.join(self.supported_precisions)))
        object.__setattr__(self, '_precision', p)

    @property
    def storage_dtype(self):
        return storage_dtype(self.compute_dtype)
