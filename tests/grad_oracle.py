"""Float64 vector-Jacobian products of the hot-path layers: the checker of the backward kernels.

TEST INFRASTRUCTURE ONLY (like ``oracle/``, which stays the forward checker and is not changed by these).  Each
function restates the TensorFlow gradient registered for the ops the reference calls, composed the way the layer
composes them.  A complex gradient is dL/dRe + i dL/dIm, PyTorch's convention for a real loss.

  STFT            tf.pad -> slice (ops/array_grad.py _PadGrad); tf.signal.frame -> scatter-add (overlap-add);
                  window multiply (Mul); RFFT -> _rfft_grad_helper (ops/signal/fft_ops.py)
  InverseSTFT     IRFFT -> _irfft_grad_helper (ops/signal/fft_ops.py); dual-window Mul; overlap_and_add -> frame
  Magnitude       ComplexAbs -> _ComplexAbsGrad (ops/math_grad.py): div_no_nan(g X, |X|)
  ApplyFilterbank tensordot = MatMul -> _MatMulGrad (ops/math_grad.py): g fb^T
  dB              Log -> _LogGrad, Maximum -> _MaximumGrad (the gradient goes to x where x >= y), Max (reduce) ->
                  _MinOrMaxGrad (split equally among the tied maxima), all in ops/math_grad.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle  # noqa: E402
from oracle.reference import CH_LAST, resolve_data_format  # noqa: E402


def _eff(n_fft, win_length, hop_length):
    win_length = n_fft if win_length is None else win_length
    hop_length = win_length // 4 if hop_length is None else hop_length
    return win_length, hop_length


def stft_layer_vjp(x_shape, G, n_fft=2048, win_length=None, hop_length=None, window_name=None, pad_begin=False,
                   pad_end=False, input_data_format='default', output_data_format='default'):
    """Gradient of kapre.STFT.call w.r.t. its waveform (shape ``x_shape``) for the complex spectrum gradient ``G``.

    RFFT's gradient (_rfft_grad_helper) maps G_t to g_t[n] = sum_{k <= N/2} Re(G_t[k] e^{+2 pi i k n / N}) for the
    n < min(win_length, N) samples the FFT reads (the rest of the frame is cropped or zero padding); the window
    multiplies it; frame's scatter-add overlap-adds the frames at t*hop; pad's slice drops the pad_begin prefix and
    the pad_end tail."""
    win_length, hop = _eff(n_fft, win_length, hop_length)
    idf, odf = resolve_data_format(input_data_format), resolve_data_format(output_data_format)
    G = np.asarray(G, dtype=np.complex128)
    if odf == CH_LAST:
        G = np.transpose(G, (0, 3, 1, 2))                       # (b, c, t, f)
    B, C, T, F = G.shape
    L = x_shape[1] if idf == CH_LAST else x_shape[2]
    w = oracle.get_window(window_name, win_length)
    we = min(win_length, n_fft)
    k = np.arange(F)
    n = np.arange(we)
    E = np.exp(2j * np.pi * np.outer(k, n) / n_fft)             # (f, n)
    frames = np.real(G @ E) * w[:we]                            # (b, c, t, n)
    pad_left = (n_fft - hop) if pad_begin else 0
    total = max(pad_left + L, (T - 1) * hop + we if T > 0 else 0)
    acc = np.zeros((B, C, total))
    for t in range(T):
        acc[..., t * hop:t * hop + we] += frames[..., t, :]
    gx = acc[..., pad_left:pad_left + L]
    if idf == CH_LAST:
        gx = np.transpose(gx, (0, 2, 1))
    return gx


def istft_layer_vjp(gy, n_fft=2048, win_length=None, hop_length=None, forward_window_name=None, frames=None,
                    input_data_format='default', output_data_format='default'):
    """Gradient of kapre.InverseSTFT.call w.r.t. its complex spectrum (``frames`` frames) for the waveform gradient
    ``gy``.  overlap_and_add's gradient frames gy; the dual window multiplies; IRFFT's gradient (_irfft_grad_helper)
    is (c_k / N) sum_n d[n] gy_t[n] e^{-2 pi i k n / N}, c_0 = c_{N/2} = 1, c_k = 2 otherwise."""
    win_length, hop = _eff(n_fft, win_length, hop_length)
    idf, odf = resolve_data_format(input_data_format), resolve_data_format(output_data_format)
    gy = np.asarray(gy, dtype=np.float64)
    if odf == CH_LAST:
        gy = np.transpose(gy, (0, 2, 1))                        # (b, c, l)
    fwd = oracle.get_window(forward_window_name, win_length)
    dual = oracle.inverse_stft_window(win_length, hop, fwd)
    we = min(win_length, n_fft)
    T = frames
    F = n_fft // 2 + 1
    fr = np.stack([gy[..., t * hop:t * hop + we] for t in range(T)], axis=-2) * dual[:we]   # (b, c, t, n)
    k = np.arange(F)
    E = np.exp(-2j * np.pi * np.outer(np.arange(we), k) / n_fft)   # (n, f)
    ck = np.full(F, 2.0)
    ck[0] = 1.0
    if n_fft % 2 == 0:
        ck[-1] = 1.0
    G = (fr @ E) * ck / n_fft
    G[..., 0] = G[..., 0].real                                   # irfft ignores Im of DC and Nyquist
    if n_fft % 2 == 0:
        G[..., -1] = G[..., -1].real
    if idf == CH_LAST:
        G = np.transpose(G, (0, 2, 3, 1))
    return G


def magnitude_vjp(X, g):
    """_ComplexAbsGrad: g X / |X|, 0 where |X| = 0 (div_no_nan)."""
    X = np.asarray(X, dtype=np.complex128)
    m = np.abs(X)
    with np.errstate(divide='ignore', invalid='ignore'):
        return np.where(m > 0, np.asarray(g, np.float64) * X / np.where(m > 0, m, 1.0), 0.0)


def apply_filterbank_vjp(g, filterbank, data_format='default'):
    """_MatMulGrad of the tensordot over the frequency axis: g fb^T."""
    df = resolve_data_format(data_format)
    fbT = np.asarray(filterbank, dtype=np.float64).T
    g = np.asarray(g, dtype=np.float64)
    if df == CH_LAST:
        return np.transpose(np.tensordot(np.transpose(g, (0, 1, 3, 2)), fbT, axes=(3, 0)), (0, 1, 3, 2))
    return np.tensordot(g, fbT, axes=(3, 0))


def magnitude_to_decibel_vjp(x, g, ref_value=1.0, amin=1e-5, dynamic_range=80.0):
    """kapre/backend.py:186-192 backward.  l = 10 log10(max(x, amin)) - c, m = max_item(l), thr = m - dynamic_range,
    y = max(l, thr):  _MaximumGrad gives g to l where l >= thr and the rest to thr = m - dr; _MinOrMaxGrad splits
    that equally among the items' tied maxima; _LogGrad and the max(x, amin) give 10 / (ln 10 x) where x >= amin."""
    x = np.asarray(x, dtype=np.float64)
    g = np.asarray(g, dtype=np.float64)
    l = 10.0 * np.log10(np.maximum(x, amin)) - 10.0 * np.log10(max(amin, ref_value))
    axis = tuple(range(x.ndim))[1:] if x.ndim > 1 else None
    m = np.max(l, axis=axis, keepdims=True)
    thr = m - dynamic_range
    keep = l >= thr
    clamped_sum = np.sum(np.where(keep, 0.0, g), axis=axis, keepdims=True)
    ismax = l == m
    dl = np.where(keep, g, 0.0) + ismax * clamped_sum / np.sum(ismax, axis=axis, keepdims=True)
    return dl * np.where(x >= amin, 10.0 / (np.log(10.0) * np.maximum(x, amin)), 0.0)


def melspectrogram_vjp(x, g, n_fft=2048, win_length=None, hop_length=None, window_name=None, pad_begin=False,
                       pad_end=False, sample_rate=22050, n_mels=128, mel_f_min=0.0, mel_f_max=None, mel_htk=False,
                       mel_norm='slaney', return_decibel=False, db_amin=1e-5, db_ref_value=1.0, db_dynamic_range=80.0,
                       input_data_format='default', output_data_format='default', filterbank=None):
    """Gradient of get_melspectrogram_layer (STFT -> Magnitude -> ApplyFilterbank [-> MagnitudeToDecibel]) w.r.t.
    the waveform: the chain rule through the VJPs above.  ``filterbank`` replaces the mel matrix (log filterbanks)."""
    X = oracle.stft_layer(x, n_fft, win_length, hop_length, window_name, pad_begin, pad_end, input_data_format,
                          output_data_format)
    mag = np.abs(X)
    fb = filterbank if filterbank is not None else oracle.filterbank_mel(
        sample_rate, n_fft // 2 + 1, n_mels, mel_f_min, mel_f_max, mel_htk, mel_norm, dtype=np.float32)
    fb = np.asarray(fb, np.float64)
    if return_decibel:
        mel = oracle.apply_filterbank(mag, fb, output_data_format)
        g = magnitude_to_decibel_vjp(mel, g, db_ref_value, db_amin, db_dynamic_range)
    gm = apply_filterbank_vjp(g, fb, output_data_format)
    return stft_layer_vjp(np.shape(x), magnitude_vjp(X, gm), n_fft, win_length, hop_length, window_name, pad_begin,
                          pad_end, input_data_format, output_data_format)


def stft_magnitude_vjp(x, g, n_fft=2048, win_length=None, hop_length=None, window_name=None, pad_begin=False,
                       pad_end=False, return_decibel=False, db_amin=1e-5, db_ref_value=1.0, db_dynamic_range=80.0,
                       input_data_format='default', output_data_format='default'):
    """Gradient of get_stft_magnitude_layer (STFT -> Magnitude [-> MagnitudeToDecibel]) w.r.t. the waveform."""
    X = oracle.stft_layer(x, n_fft, win_length, hop_length, window_name, pad_begin, pad_end, input_data_format,
                          output_data_format)
    if return_decibel:
        g = magnitude_to_decibel_vjp(np.abs(X), g, db_ref_value, db_amin, db_dynamic_range)
    return stft_layer_vjp(np.shape(x), magnitude_vjp(X, g), n_fft, win_length, hop_length, window_name, pad_begin,
                          pad_end, input_data_format, output_data_format)
