"""Tightening the parity pin (VERDICT round 1, item 8).

* the mel matrix is held to an independent, scalar float64 evaluation of the librosa >= 0.11 formula
  (``librosa.filters.mel`` as called at kapre/backend.py:222-230) at <= 1 float32 ulp -- not to torchaudio at 1e-5;
* ``tests/golden/regen_with_real_libs.py`` regenerates the reference cases with the REAL tensorflow / librosa whenever
  they are importable and must agree with the committed stand-in fixtures (skipped where they are not installed).
"""
import importlib.util
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))


def _hz_to_mel(f, htk):
    if htk:
        return 2595.0 * math.log10(1.0 + f / 700.0)
    f_sp = 200.0 / 3
    if f >= 1000.0:
        return 15.0 + math.log(f / 1000.0) / (math.log(6.4) / 27.0)
    return f / f_sp


def _mel_to_hz(m, htk):
    if htk:
        return 700.0 * (10.0 ** (m / 2595.0) - 1.0)
    f_sp = 200.0 / 3
    if m >= 15.0:
        return 1000.0 * math.exp((math.log(6.4) / 27.0) * (m - 15.0))
    return f_sp * m


def librosa_mel_scalar(sr, n_fft, n_mels, fmin, fmax, htk, slaney):
    """librosa.filters.mel written out element by element in Python floats (float64); float32 storage of the triangle
    before the Slaney scaling, as librosa does (weights is a float32 array, `weights *= enorm` rounds once more)."""
    if fmax is None:
        fmax = sr / 2.0
    n_freq = 1 + n_fft // 2
    fftfreqs = [k * (sr / 2.0) / (n_freq - 1) for k in range(n_freq)]
    lo, hi = _hz_to_mel(fmin, htk), _hz_to_mel(fmax, htk)
    mel_f = [_mel_to_hz(lo + (hi - lo) * i / (n_mels + 1), htk) for i in range(n_mels + 2)]
    W = np.zeros((n_mels, n_freq), dtype=np.float32)
    for i in range(n_mels):
        for k in range(n_freq):
            lower = -(mel_f[i] - fftfreqs[k]) / (mel_f[i + 1] - mel_f[i])
            upper = (mel_f[i + 2] - fftfreqs[k]) / (mel_f[i + 2] - mel_f[i + 1])
            W[i, k] = np.float32(max(0.0, min(lower, upper)))
        if slaney:
            enorm = 2.0 / (mel_f[i + 2] - mel_f[i])
            for k in range(n_freq):
                W[i, k] = np.float32(float(W[i, k]) * enorm)
    return W.T


def _ulps(a, b):
    a = np.asarray(a, dtype=np.float32) + np.float32(0.0)      # -0.0 -> +0.0 (librosa's max(0, min(..)) may return either)
    b = np.asarray(b, dtype=np.float32) + np.float32(0.0)
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


@pytest.mark.parametrize('sr,n_freq,n_mels,fmin,fmax,htk,norm', [
    (22050, 513, 128, 0.0, None, False, 'slaney'),        # cfg2 / README configuration
    (16000, 513, 128, 0.0, None, False, 'slaney'),        # cfg5
    (16000, 257, 64, 0.0, None, False, 'slaney'),         # cfg1
    (44100, 1025, 96, 30.0, 18000.0, True, 'slaney'),
    (22050, 201, 40, 0.0, 8000.0, False, None),
])
def test_mel_matrix_within_one_ulp_of_the_scalar_librosa_formula(sr, n_freq, n_mels, fmin, fmax, htk, norm):
    import kapre_b200.backend as KB       # pure NumPy: importable without a GPU
    ref = librosa_mel_scalar(sr, (n_freq - 1) * 2, n_mels, fmin, fmax, htk, norm == 'slaney')
    for name, fb in (('oracle', O.filterbank_mel(sr, n_freq, n_mels, fmin, fmax, htk, norm)),
                     ('product', KB.filterbank_mel(sr, n_freq, n_mels, fmin, fmax, htk, norm))):
        fb = np.asarray(fb)
        assert fb.shape == ref.shape and fb.dtype == np.float32
        assert ((fb != 0) == (ref != 0)).all(), name          # identical support
        assert _ulps(fb, ref).max() <= 1, (name, int(_ulps(fb, ref).max()))


def test_reference_cases_regenerate_with_real_tensorflow_and_librosa():
    """Runs only where the real dependencies exist (not in the build container, not on the GPU box)."""
    if importlib.util.find_spec('tensorflow') is None or importlib.util.find_spec('librosa') is None:
        pytest.skip('tensorflow / librosa not installed: the committed fixtures come from the stand-in '
                    '(tests/golden/tf_standin.py); run tests/golden/regen_with_real_libs.py where they exist')
    ref_root = os.environ.get('KAPRE_REFERENCE_ROOT')
    if not ref_root or not os.path.isdir(os.path.join(ref_root, 'kapre')):
        pytest.skip('KAPRE_REFERENCE_ROOT does not name a directory holding the kapre 0.4.0 package')
    out = subprocess.run([sys.executable, os.path.join(HERE, 'golden', 'regen_with_real_libs.py'), '--check'],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
