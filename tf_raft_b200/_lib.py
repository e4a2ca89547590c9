"""ctypes binding of libraft_b200.so -- the C ABI declared in include/raft_b200.h.

PyTorch is used for device memory and streams only: every compute call below hands raw device
pointers and the current CUDA stream to the shared library.  There is no Python/torch fallback:
if the library has not been built, importing an op raises with the build command.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# RAFT_B200_LIB: load another build of the same sources (kernel experiments, tools/epi_exp.sh); the default is the in-tree build.
LIB_PATH = os.environ.get('RAFT_B200_LIB') or os.path.join(_HERE, 'libraft_b200.so')

PREC_FP32 = 0
PREC_F16X2 = 1
VARIANT_BASIC = 0
VARIANT_SMALL = 1
MAX_LEVELS = 8

_PRECISIONS = {'fp32': PREC_FP32, 'f16x2': PREC_F16X2, PREC_FP32: PREC_FP32, PREC_F16X2: PREC_F16X2}


def resolve_precision(precision=None):
    """None -> $RAFT_B200_PRECISION or 'f16x2' (the tcgen05 path)."""
    if precision is None:
        precision = os.environ.get('RAFT_B200_PRECISION', 'f16x2')
    try:
        return _PRECISIONS[precision]
    except KeyError:
        raise ValueError(f'unknown precision {precision!r}; expected one of fp32, f16x2') from None


class RaftConv(ctypes.Structure):
    """struct raft_conv: HWIO kernel + bias device pointers and dims."""
    _fields_ = [('kernel', ctypes.c_void_p), ('bias', ctypes.c_void_p),
                ('kh', ctypes.c_int), ('kw', ctypes.c_int), ('cin', ctypes.c_int), ('cout', ctypes.c_int)]


class RaftNorm(ctypes.Structure):
    """struct raft_norm"""
    _fields_ = [('gamma', ctypes.c_void_p), ('beta', ctypes.c_void_p), ('moving_mean', ctypes.c_void_p),
                ('moving_variance', ctypes.c_void_p)]


class RaftResBlock(ctypes.Structure):
    """struct raft_resblock"""
    _fields_ = [('conv1', RaftConv), ('conv2', RaftConv), ('norm1', RaftNorm), ('norm2', RaftNorm),
                ('downsample', RaftConv), ('downsample_norm', RaftNorm)]


class RaftEncoderWeights(ctypes.Structure):
    """struct raft_encoder_weights"""
    _fields_ = [('conv1', RaftConv), ('norm1', RaftNorm), ('block', RaftResBlock * 6), ('conv2', RaftConv)]


NORM_TYPES = {None: 0, 'instance': 1, 'batch': 2}

_vp, _i, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
_SIGNATURES = {
    'raft_b200_strerror': (ctypes.c_char_p, [_i]),
    'raft_b200_abi_version': (_i, []),
    'raft_b200_device_ok': (_i, [_i]),
    'raft_b200_launch_count': (ctypes.c_longlong, []),
    'raft_b200_launch_count_reset': (None, []),
    'raft_b200_debug_timeline': (None, [_i, _vp]),
    'raft_b200_profile_loop': (None, [_i]),
    'raft_b200_profile_read': (_i, [ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float), ctypes.POINTER(_i)]),
    'raft_b200_corr_pyramid_sizes': (_i, [_i, _i, _i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_corr_workspace_bytes': (_i, [_i, _i, _i, _i, _i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_corr_pyramid_build': (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.POINTER(_vp), _vp, _sz, _i, _vp]),
    'raft_b200_corr_lookup': (_i, [ctypes.POINTER(_vp), _vp, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    'raft_b200_corr_lookup_backward': (_i, [ctypes.POINTER(_vp), _vp, _vp, _i, _i, _i, _i, _i, _vp, ctypes.POINTER(_vp), _vp]),
    'raft_b200_sumsq': (_i, [_vp, _sz, _vp, _sz, _vp, _vp]),
    'raft_b200_adamw_step': (_i, [_vp, _vp, _vp, _vp, _sz, _vp, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                  ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp]),
    'raft_b200_bilinear_sampler': (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    'raft_b200_coords_grid': (_i, [_i, _i, _i, _vp, _vp]),
    'raft_b200_update_prepared_bytes': (_i, [_i, _i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_update_prepare': (_i, [_i, _vp, _vp, _sz, _i, _vp]),
    'raft_b200_update_workspace_bytes': (_i, [_i, _i, _i, _i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_update_basic': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _i, _vp]),
    'raft_b200_update_small': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _i, _vp]),
    'raft_b200_upsample_convex': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    'raft_b200_upflow8': (_i, [_vp, _i, _i, _i, _vp, _vp]),
    'raft_b200_encoder_prepared_bytes': (_i, [_i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_encoder_prepare': (_i, [_i, _i, _i, _vp, _vp, _sz, _vp]),
    'raft_b200_encoder_workspace_bytes': (_i, [_i, _i, _i, _i, ctypes.POINTER(_sz)]),
    'raft_b200_encoder_forward': (_i, [_i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    'raft_b200_context_split': (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    'raft_b200_conv2d': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    'raft_b200_forward_loop': (_i, [_i, _vp, ctypes.POINTER(_vp), _i, _i, _vp, _vp, _vp, ctypes.POINTER(_vp), _i,
                                    _i, _i, _i, _vp, _sz, _i, _vp]),
    'raft_b200_forward_interpolate': (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """The loaded shared library (loads on first use; raises if it was never built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f'{LIB_PATH} is missing: the sm_100a CUDA library has not been built. '
                'Run `python -c "import __graft_entry__ as g; g.build()"` (or `python -m tf_raft_b200.build`) '
                'from the repository root. There is no CPU / PyTorch fallback for the RAFT hot path.')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.raft_b200_abi_version() != 1:
            raise ImportError('libraft_b200.so ABI version mismatch; rebuild it')
        _lib = handle
    return _lib


def strerror(status):
    return lib().raft_b200_strerror(status).decode()


def check(status, what=''):
    if status != 0:
        raise RuntimeError(f'raft_b200 {what} failed: [{status}] {strerror(status)}')


def ptr(t):
    """Device pointer of a tensor (or NULL for None)."""
    return ctypes.c_void_p(None if t is None else t.data_ptr())


def ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError('tf_raft_b200 runs on CUDA tensors only (sm_100a); got a CPU tensor. '
                               'There is no CPU fallback for this path.')
        if t.dtype != torch.float32 or not t.is_contiguous():
            raise RuntimeError('expected contiguous float32 tensors')


def f32c(t):
    """contiguous float32 view/copy of a CUDA tensor."""
    if not t.is_cuda:
        raise RuntimeError('tf_raft_b200 runs on CUDA tensors only (sm_100a); got a CPU tensor. '
                           'There is no CPU fallback for this path.')
    return t.to(torch.float32).contiguous()


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def launch_count():
    return int(lib().raft_b200_launch_count())


def launch_count_reset():
    lib().raft_b200_launch_count_reset()
