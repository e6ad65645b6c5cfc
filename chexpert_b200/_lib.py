"""ctypes binding of libaaconv_b200.so (C ABI declared in include/aaconv_b200.h).

There is no fallback: if the shared object is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libaaconv_b200.so')

FP32, BF16 = 0, 1
PRECISIONS = {'fp32': FP32, 'bf16': BF16}


class Dims(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in
                ('B', 'Cin', 'Hin', 'Win', 'Cout', 'H', 'W', 'ksize', 'stride', 'pad', 'dil', 'dk', 'dv', 'nh',
                 'relative')]


class Io(ctypes.Structure):
    """aaconv_io: element types of x / y, batch stride of y (feature-buffer destination), fused InstanceNorm + ReLU prologue."""
    _fields_ = [('x_dtype', ctypes.c_int32), ('y_dtype', ctypes.c_int32), ('y_batch_stride', ctypes.c_int64),
                ('fuse_in_relu', ctypes.c_int32), ('in_eps', ctypes.c_float)]


class Params(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ('conv_w', 'qkv_w', 'out_w', 'key_rel_h', 'key_rel_w')]


class ParamGrads(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ('conv_w', 'qkv_w', 'out_w', 'key_rel_h', 'key_rel_w')]


# every symbol the header declares: name -> (restype, argtypes)
_P = ctypes.c_void_p
_DP = ctypes.POINTER(Dims)
_IOP = ctypes.POINTER(Io)
SYMBOLS = {
    'aaconv_abi_version': (ctypes.c_int, []),
    'aaconv_last_error': (ctypes.c_char_p, []),
    'aaconv_validate': (ctypes.c_int, [_DP, ctypes.c_int]),
    'aaconv_saved_bytes': (ctypes.c_size_t, [_DP, ctypes.c_int]),
    'aaconv_scratch_bytes': (ctypes.c_size_t, [_DP, ctypes.c_int, ctypes.c_int]),
    'aaconv_saved_bytes_io': (ctypes.c_size_t, [_DP, ctypes.c_int, _IOP]),
    'aaconv_scratch_bytes_io': (ctypes.c_size_t, [_DP, ctypes.c_int, _IOP]),
    'aaconv_forward_io': (ctypes.c_int, [_DP, ctypes.c_int, _IOP, _P, ctypes.POINTER(Params), _P, _P, _P, _P, _P]),
    'aaconv_backward_io': (ctypes.c_int, [_DP, ctypes.c_int, _IOP, _P, ctypes.POINTER(Params), _P, _P, _P, _P,
                                          ctypes.POINTER(ParamGrads), _P]),
    'aaconv_saved_offset': (ctypes.c_int64, [_DP, ctypes.c_int, ctypes.c_char_p]),
    'aaconv_forward': (ctypes.c_int, [_DP, ctypes.c_int, _P, ctypes.POINTER(Params), _P, _P, _P, _P, _P]),
    'aaconv_backward': (ctypes.c_int, [_DP, ctypes.c_int, _P, ctypes.POINTER(Params), _P, _P, _P, _P,
                                       ctypes.POINTER(ParamGrads), _P]),
    'aaconv_bce_forward_backward': (ctypes.c_int, [_P, _P, ctypes.c_int, _P, ctypes.c_int, ctypes.c_int,
                                                   _P, _P, _P, _P, _P]),
    'aaconv_ensemble_mean': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, _P, _P]),
    'aaconv_auroc_workspace_bytes': (ctypes.c_size_t, [ctypes.c_int]),
    'aaconv_auroc': (ctypes.c_int, [_P, _P, ctypes.c_int, ctypes.c_int, _P, _P, _P]),
    'aaconv_bn_relu_workspace_bytes': (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    'aaconv_bn_relu_forward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, _P, _P, _P, _P,
                                              ctypes.c_float, ctypes.c_float, _P, _P, _P, ctypes.c_int, _P]),
    'aaconv_bn_relu_backward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, _P, _P, _P, _P,
                                               _P, _P, _P, _P, _P]),
    'aaconv_bn_relu_backward_acc': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, _P, _P, _P, _P,
                                                   _P, ctypes.c_int64, _P, _P, _P, _P]),
    'aaconv_bn_relu_cl_workspace_bytes': (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    'aaconv_bn_stats_nchw': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, _P, ctypes.c_int,
                                            ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), _P]),
    'aaconv_bn_relu_cl_forward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                                 _P, _P, _P, _P, ctypes.c_float, ctypes.c_float, _P, _P, _P, _P, ctypes.c_int, ctypes.c_int, _P]),
    'aaconv_bn_relu_cl_backward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                                  _P, _P, _P, _P, _P, ctypes.c_int64, ctypes.c_int, _P, _P, _P, _P]),
    'aaconv_slice_layout': (ctypes.c_int, [_P, _P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int, _P]),
    'aaconv_bn_relu_eval': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                           _P, _P, _P, _P, ctypes.c_float, _P, ctypes.c_int, _P]),
    'aaconv_bn_relu_pool_workspace_bytes': (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    'aaconv_bn_relu_pool_forward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                                   ctypes.c_int, _P, _P, _P, _P, ctypes.c_float, ctypes.c_float, _P, _P, _P, ctypes.c_int,
                                                   ctypes.c_int, _P]),
    'aaconv_bn_relu_pool_backward': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                                    _P, _P, _P, _P, _P, ctypes.c_int64, ctypes.c_int, _P, _P, _P, _P]),
    'aaconv_radiograph_prep': (ctypes.c_int, [_P, ctypes.c_int64, _P, ctypes.c_int, ctypes.c_int, ctypes.c_int, _P, _P]),
    'aaconv_grad_cam': (ctypes.c_int, [_P, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, _P, _P,
                                       _P, _P, ctypes.c_float, _P, ctypes.c_int, _P, _P, ctypes.c_int, _P, _P]),
    'aaconv_launch_count': (ctypes.c_longlong, []),
    'aaconv_debug_set_timeline': (None, [_P]),
    'aaconv_debug_set_mode': (None, [ctypes.c_int]),
    'aaconv_debug_read_mbar_log': (ctypes.c_int, [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]),
    'aaconv_profile_begin': (ctypes.c_int, [_P]),
    'aaconv_profile_end': (ctypes.c_int, [ctypes.c_char_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_float), ctypes.c_int]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Load (once) and return the CDLL; raises RuntimeError if the extension was not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f'{LIB_PATH} is missing: build it with `python chexpert_b200/csrc/build.py` '
                    '(or __graft_entry__.build()). chexpert_b200 has no CPU / eager fallback.')
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SYMBOLS.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            if lib.aaconv_abi_version() != 2:
                raise RuntimeError('libaaconv_b200.so ABI version mismatch')
            _lib = lib
    return _lib


def check(code, what):
    if code != 0:
        msg = load().aaconv_last_error().decode(errors='replace')
        raise RuntimeError(f'{what} failed (code {code}): {msg}')


def launch_count():
    return int(load().aaconv_launch_count())


def profile_begin(stream_ptr):
    check(load().aaconv_profile_begin(ctypes.c_void_p(stream_ptr)), 'aaconv_profile_begin')


def profile_end(max_entries=4096):
    """-> list of (kernel name, milliseconds) in launch order since profile_begin()."""
    names = ctypes.create_string_buffer(max_entries * 40)
    ms = (ctypes.c_float * max_entries)()
    n = load().aaconv_profile_end(names, len(names), ms, max_entries)
    if n < 0:
        check(n, 'aaconv_profile_end')
    ns = names.value.decode().split('\n')
    return [(ns[i] if i < len(ns) else '?', float(ms[i])) for i in range(n)]
