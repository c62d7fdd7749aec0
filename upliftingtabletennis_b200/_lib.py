"""ctypes binding of libttk.so (include/ttk.h).  There is no CPU fallback: if the CUDA library
is missing, or a call fails, this module raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libttk.so')

F32, BF16, TF32, TF32X3, F16 = 0, 1, 2, 3, 4
DECODE_TABLE, DECODE_BALL = 0, 1
LAYOUT_NCHW_F32, LAYOUT_NHWC16 = 0, 1


class TtkError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'libttk.so (the hand-written sm_100a CUDA kernels) is not built: run '
            '`python -m upliftingtabletennis_b200.build` or `python -c "import __graft_entry__ as g; g.build()"`. '
            'This package has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
    sig = {
        'ttk_version': (i32, []),
        'ttk_last_error': (C.c_char_p, []),
        'ttk_host_copy_stream': (i32, [vp, vp, sz]),
        'ttk_host_blocking_sync': (i32, [i32, C.POINTER(C.c_uint)]),
        'ttk_device_ok': (i32, []),
        'ttk_preprocess_stacks': (i32, [vp, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, i32, i32, vp]),
        'ttk_preprocess_stacks_indexed': (i32, [vp, i32, i32, i32, i32, vp, i32, i32, i32, vp, vp, i32, i32, vp]),
        'ttk_hrnet_create': (i32, [i32, i32, i32, i32, C.POINTER(vp)]),
        'ttk_hrnet_destroy': (None, [vp]),
        'ttk_hrnet_num_convs': (i32, [vp]),
        'ttk_hrnet_conv_info': (i32, [vp, i32, C.c_char_p, C.c_char_p] + [C.POINTER(i32)] * 4),
        'ttk_hrnet_set_conv': (i32, [vp, i32, vp, vp]),
        'ttk_hrnet_workspace_bytes': (sz, [vp, i32, i32, i32, i32]),
        'ttk_hrnet_forward': (i32, [vp, vp, i32, i32, i32, i32, vp, vp, sz, vp]),
        'ttk_hrnet_last_launches': (i32, [vp]),
        'ttk_hrnet_set_subbatch': (i32, [vp, i32]),
        'ttk_hrnet_set_profile': (i32, [vp, i32]),
        'ttk_hrnet_set_force_simt': (i32, [vp, i32]),
        'ttk_hrnet_debug_conv': (i32, [vp, i32, vp, i32, i32, i32, vp, i32, i32, vp, vp]),
        'ttk_hrnet_debug_conv_f16': (i32, [vp, i32, vp, i32, i32, i32, vp, i32, i32, vp, vp]),
        'ttk_hrnet_debug_block': (i32, [vp, i32, vp, i32, i32, i32, vp, vp]),
        'ttk_hrnet_set_block_fusion': (i32, [vp, i32]),
        'ttk_hrnet_profile_count': (i32, [vp]),
        'ttk_hrnet_profile_read': (i32, [vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        'ttk_vit_create': (i32, [i32, i32, i32, i32, C.POINTER(vp)]),
        'ttk_vit_destroy': (None, [vp]),
        'ttk_vit_num_params': (i32, [vp]),
        'ttk_vit_param_info': (i32, [vp, i32, C.c_char_p, C.POINTER(i32)]),
        'ttk_vit_set_param': (i32, [vp, i32, vp, i32]),
        'ttk_vit_tokens': (i32, [vp, C.POINTER(i32), C.POINTER(i32)]),
        'ttk_vit_set_subbatch': (i32, [vp, i32]),
        'ttk_vit_workspace_bytes': (sz, [vp, i32, i32]),
        'ttk_vit_forward': (i32, [vp, vp, i32, i32, vp, vp, sz, vp]),
        'ttk_vit_last_launches': (i32, [vp]),
        'ttk_vit_debug_gemm': (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
        'ttk_vit_debug_attention': (i32, [vp, vp, vp, sz, i32, i32, i32, vp]),
        'ttk_decode_workspace_bytes': (sz, [i32, i32, i32]),
        'ttk_heatmap_decode': (i32, [vp, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, sz, vp]),
        'ttk_decode_set_profile': (i32, [i32]),
        'ttk_decode_profile_read': (i32, [C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        'ttk_filter_ball': (i32, [vp, vp, i32, C.c_double, C.c_double, vp, vp, vp, vp, vp]),
        'ttk_filter_ball_clips': (i32, [vp, vp, i32, vp, i32, C.c_double, C.c_double, vp, vp, vp, vp, vp]),
        'ttk_filter_table_workspace_bytes': (sz, [i32, i32, i32]),
        'ttk_filter_table': (i32, [vp, vp, i32, i32, i32, C.c_double, C.c_double, i32, vp, vp, sz, vp]),
        'ttk_filter_table_clips': (i32, [vp, vp, i32, vp, i32, i32, C.c_double, C.c_double, i32, vp, vp, sz, vp]),
        'ttk_calibrate_workspace_bytes': (sz, [i32, i32]),
        'ttk_calibrate_camera': (i32, [vp, vp, vp, i32, i32, i32, i32, i32, C.c_double, vp, vp, vp, vp, sz, vp]),
        'ttk_trajectory_pack': (i32, [vp, vp, vp, vp, i32, i32, C.c_double, C.c_double, vp, vp, vp, vp, vp]),
        'ttk_uplift_create': (i32, [i32, i32, i32, i32, C.POINTER(vp)]),
        'ttk_uplift_destroy': (None, [vp]),
        'ttk_uplift_num_params': (i32, [vp]),
        'ttk_uplift_param_info': (i32, [vp, i32, C.c_char_p, C.POINTER(i32)]),
        'ttk_uplift_set_param': (i32, [vp, i32, vp, i32]),
        'ttk_uplift_workspace_bytes': (sz, [vp, i32, i32, i32]),
        'ttk_uplift_forward': (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, sz, vp]),
        'ttk_uplift_last_launches': (i32, [vp]),
        'ttk_uplift_debug_gemm3': (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
        'ttk_uplift_debug_attention3': (i32, [i32, i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
        'ttk_rotation_local': (i32, [vp, vp, i32, i32, vp, vp]),
        'ttk_project': (i32, [vp, vp, vp, i32, i32, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)       # AttributeError if include/ttk.h and the library disagree
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTS = _load()


def check(rc):
    if rc != 0:
        raise TtkError('libttk error %d: %s' % (rc, lib.ttk_last_error().decode()))


def require_device():
    if not lib.ttk_device_ok():
        raise TtkError('libttk needs an sm_100 (B200) CUDA device; none is visible and there is no CPU fallback')


def host_blocking_sync(device=None):
    """Host threads waiting for `device` (default: the current one) sleep instead of spin.  For hosts that run one rank per GPU with few
    cores per GPU, where spinning waiters take the cores from the frame-staging threads; process-global for the device.  Returns the
    previous device flags."""
    import torch
    old = C.c_uint(0)
    check(lib.ttk_host_blocking_sync(torch.cuda.current_device() if device is None else int(device), C.byref(old)))
    return old.value


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


def ptr(t):
    """Device (or host) pointer of a contiguous torch tensor / numpy array."""
    if t is None:
        return C.c_void_p(0)
    if hasattr(t, 'data_ptr'):
        assert t.is_contiguous(), 'libttk needs contiguous tensors'
        return C.c_void_p(t.data_ptr())
    assert t.flags['C_CONTIGUOUS']
    return C.c_void_p(t.ctypes.data)
