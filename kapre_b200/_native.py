"""ctypes binding of libkapre_b200.so (the C ABI in include/kapre_b200.h).

The CUDA library is the product: there is NO fallback.  If the shared object is missing
the import fails loudly with the build command.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, '_lib', 'libkapre_b200.so')

OUT_COMPLEX, OUT_MAG, OUT_MAG_DB, OUT_FB, OUT_FB_DB, OUT_MAG_PHASE = range(6)


class KapreNativeError(RuntimeError):
    pass


class WaveDesc(Structure):
    _fields_ = [('batch', c_int32), ('channels', c_int32), ('length', c_int32),
                ('stride_b', c_int64), ('stride_c', c_int64), ('stride_l', c_int64)]


class SpecDesc(Structure):
    _fields_ = [('stride_b', c_int64), ('stride_c', c_int64), ('stride_t', c_int64),
                ('stride_f', c_int64)]


class DbCfg(Structure):
    _fields_ = [('ref_value', c_float), ('amin', c_float), ('dynamic_range', c_float)]


# every symbol declared in include/kapre_b200.h: (name, restype, argtypes)
SYMBOLS = [
    ('kapre_stft_plan_create', c_int, [c_int, c_int, c_int, c_void_p, POINTER(c_void_p)]),
    ('kapre_stft_plan_destroy', None, [c_void_p]),
    ('kapre_stft_num_frames', c_int, [c_void_p, c_int, c_int, c_int]),
    ('kapre_stft_supports_mode', c_int, [c_void_p, c_int]),
    ('kapre_stft_forward', c_int, [c_void_p, c_void_p, POINTER(WaveDesc), c_int, c_int, c_int, c_void_p,
                                   POINTER(SpecDesc), c_void_p, POINTER(DbCfg), c_void_p, c_void_p]),
    ('kapre_istft_plan_create', c_int, [c_int, c_int, c_int, c_void_p, POINTER(c_void_p)]),
    ('kapre_istft_plan_destroy', None, [c_void_p]),
    ('kapre_istft_inverse', c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(SpecDesc), c_void_p,
                                    POINTER(WaveDesc), c_void_p]),
    ('kapre_filterbank_create', c_int, [c_void_p, c_int, c_int, POINTER(c_void_p)]),
    ('kapre_filterbank_destroy', None, [c_void_p]),
    ('kapre_apply_filterbank', c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(SpecDesc), c_void_p,
                                       POINTER(SpecDesc), c_void_p]),
    ('kapre_magnitude', c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    ('kapre_phase', c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    ('kapre_magnitude_to_decibel', c_int, [c_void_p, c_void_p, c_int64, c_int64, POINTER(DbCfg), c_void_p, c_void_p]),
    ('kapre_delta', c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    ('kapre_frame', c_int, [c_void_p, POINTER(WaveDesc), c_int, c_int, c_int, c_float, c_void_p, POINTER(SpecDesc), c_void_p]),
    ('kapre_energy', c_int, [c_void_p, POINTER(WaveDesc), c_int, c_int, c_int, c_float, c_float, c_void_p, POINTER(WaveDesc), c_void_p]),
    ('kapre_concat_frequency_map', c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p]),
    ('kapre_spec_augment', c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p, c_int, c_float, c_void_p]),
    ('kapre_stft_backward', c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(SpecDesc), c_int, c_int, c_void_p,
                                    POINTER(WaveDesc), c_void_p]),
    ('kapre_istft_backward', c_int, [c_void_p, c_void_p, POINTER(WaveDesc), c_void_p, c_int, POINTER(SpecDesc), c_void_p]),
    ('kapre_spectral_backward', c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, POINTER(SpecDesc), c_void_p,
                                        POINTER(SpecDesc), c_void_p, POINTER(SpecDesc), POINTER(DbCfg), c_void_p, c_void_p,
                                        POINTER(SpecDesc), c_void_p]),
    ('kapre_magnitude_to_decibel_backward', c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64,
                                                    c_int64, POINTER(DbCfg), c_void_p, c_void_p]),
    ('kapre_last_error', c_char_p, []),
    ('kapre_version', c_int, []),
    ('kapre_launch_count', c_uint64, []),
    ('kapre_last_launch_info', c_char_p, []),
    ('kapre_profile_enable', c_int, [c_int]),
    ('kapre_profile_read', c_int, [POINTER(ctypes.c_double), POINTER(c_uint64)]),
    ('kapre_tc_set_debug', c_int, [c_void_p]),
    ('kapre_tc_dft_stage1', c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_int, POINTER(c_int), c_void_p, c_void_p]),
]

_lib = None


def lib():
    """Load (once) and return the shared library; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KapreNativeError(
                'kapre_b200: CUDA library %s not found.  Build it with '
                '`python -c "import __graft_entry__ as g; g.build()"` (nvcc, sm_100a).  '
                'There is no CPU or PyTorch fallback.' % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(handle, name)  # AttributeError if the ABI and the header drifted apart
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(rc: int):
    if rc != 0:
        msg = lib().kapre_last_error()
        raise KapreNativeError('kapre_b200 error %d: %s' % (rc, msg.decode() if msg else '?'))


def launch_count() -> int:
    return int(lib().kapre_launch_count())


def last_launch_info() -> str:
    s = lib().kapre_last_launch_info()
    return s.decode() if s else ''


def profile_enable(on, every: int = 1):
    """Bracket every `every`-th launch of the dominant kernels with CUDA events (0 / False: off)."""
    lib().kapre_profile_enable(int(every) if on else 0)


def profile_read():
    """(total kernel milliseconds, launches) recorded since the last read."""
    ms, n = ctypes.c_double(0.0), c_uint64(0)
    lib().kapre_profile_read(ctypes.byref(ms), ctypes.byref(n))
    return float(ms.value), int(n.value)
