"""Builds and drives the CPU emulation of the backward kernel bodies (tests/emu/kb_emu_grad.cpp).

Test infrastructure, like emu_harness.py: runs the exact source the GPU compiles for the STFT adjoint, the decibel
statistics and the spectral VJP on the CPU.
"""
import ctypes
import os
import subprocess

import numpy as np

from emu_harness import _CSRC, _fp, _strides4

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, 'emu', 'kb_emu_grad.cpp')
_OUT = os.path.join(_HERE, 'emu', '_build', 'libkb_emu_grad.so')


def _needs_build():
    if not os.path.exists(_OUT):
        return True
    t = os.path.getmtime(_OUT)
    deps = [_SRC] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC) if f.endswith(('.h', '.cuh'))]
    return any(os.path.getmtime(d) > t for d in deps)


def load():
    if _needs_build():
        os.makedirs(os.path.dirname(_OUT), exist_ok=True)
        subprocess.check_call(['g++', '-O2', '-std=c++17', '-shared', '-fPIC', '-DKB_HOST_EMU',
                               '-Wno-unknown-pragmas', '-o', _OUT, _SRC])
    return ctypes.CDLL(_OUT)


def emu_stft_adjoint(G, x_len, n_fft, win_length, hop, window, pad_begin, spec_fmt, wave_fmt, seg=0, n_warps=4, n_cta=3):
    """STFT adjoint (kapre_stft_backward) on the inverse kernel bodies: seg=k the streaming body with tiles of k hops,
    seg=0 the direct body.  G: complex64 (B, T, F, C) / (B, C, T, F); returns the (B, L, C) / (B, C, L) gradient."""
    lib = load()
    G = np.ascontiguousarray(G, dtype=np.complex64)
    if spec_fmt == 'channels_last':
        B, T, F, C = G.shape
    else:
        B, C, T, F = G.shape
    _, (sb, sc, st, sk) = _strides4((B, C, T, F), spec_fmt)
    L = int(x_len)
    if wave_fmt == 'channels_last':
        y = np.full((B, L, C), np.nan, dtype=np.float32)
        ysb, ysl, ysc = L * C, C, 1
    else:
        y = np.full((B, C, L), np.nan, dtype=np.float32)
        ysb, ysc, ysl = C * L, L, 1
    window = np.ascontiguousarray(window, dtype=np.float32)
    pad_left = (n_fft - hop) if pad_begin else 0
    LL = ctypes.c_longlong
    rc = lib.kb_emu_stft_adjoint(_fp(G), LL(sb), LL(sc), LL(st), LL(sk), B, C, T, n_fft, win_length, hop, _fp(window),
                                 pad_left, L, _fp(y), LL(ysb), LL(ysc), LL(ysl), int(seg), n_warps, n_cta)
    assert rc == 0, rc
    return y


def _strides_of(a):
    return [s // a.itemsize for s in a.strides]


def emu_dbstat(y, g, dynamic_range, chunks, order=None):
    """Decibel VJP statistics (kb_dbstat_cta) of 4-D (items, d1, d2, d3) arrays -> (n_items, 4) float32:
    max(y), #ties, clamped value (-inf if the clamp does not bind), clamped gradient sum.  ``order``: CTA order."""
    lib = load()
    y = np.asarray(y, dtype=np.float32)
    g = np.asarray(g, dtype=np.float32)
    n, d1, d2, d3 = y.shape
    stats = np.zeros((n, 4), np.float32)
    order = np.arange(n * chunks, dtype=np.int32) if order is None else np.ascontiguousarray(order, dtype=np.int32)
    LL = ctypes.c_longlong
    ys, gs = _strides_of(y), _strides_of(g)
    rc = lib.kb_emu_dbstat(_fp(y), *[LL(s) for s in ys], _fp(g), *[LL(s) for s in gs], n, d1, d2, d3, int(chunks),
                           ctypes.c_float(dynamic_range), _fp(order), _fp(stats))
    assert rc == 0, rc
    return stats


def emu_specvjp(X, g, y, fmt, fb=None, db=False, amin=1e-5, stats=None, n_warps=4, n_cta=5):
    """Spectral VJP (kb_specvjp_cta): complex X (B, T, F, C) / (B, C, T, F), upstream g and forward output y in the
    same layout with K = F or the band count -> complex64 gradient of X."""
    lib = load()
    X = np.ascontiguousarray(X, dtype=np.complex64)
    g = np.asarray(g, dtype=np.float32)
    y = np.ascontiguousarray(g if y is None else y, dtype=np.float32)
    if fmt == 'channels_last':
        B, T, F, C = X.shape
        perm = (0, 3, 1, 2)
    else:
        B, C, T, F = X.shape
        perm = (0, 1, 2, 3)
    xs = [s // 8 for s in X.strides]
    xs = [xs[i] for i in perm]
    gs = [_strides_of(g)[i] for i in perm]
    ys = [_strides_of(y)[i] for i in perm]
    G = np.full_like(X, np.nan)
    fb_p, nb = None, 0
    if fb is not None:
        fb = np.ascontiguousarray(fb, dtype=np.float32)
        fb_p, nb = _fp(fb), fb.shape[1]
    st = np.ascontiguousarray(stats if stats is not None else np.zeros((B, 4)), dtype=np.float32)
    LL = ctypes.c_longlong
    rc = lib.kb_emu_specvjp(_fp(X), *[LL(s) for s in xs], g.ctypes.data_as(ctypes.c_void_p), *[LL(s) for s in gs],
                            _fp(y), *[LL(s) for s in ys], B, C, T, F, fb_p, nb, int(bool(db)), ctypes.c_float(amin),
                            _fp(st), _fp(G), n_warps, n_cta)
    assert rc == 0, rc
    return G
