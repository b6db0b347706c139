"""Functional layer over the C ABI: torch tensors in, torch tensors out.

PyTorch is only the device-memory carrier and the stream provider here; every computation
is a launch of the kernels in ``csrc/`` through ``libkapre_b200.so``.  There is no fallback:
a missing library, a CPU-only process or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes
import threading

import numpy as np
import torch

from . import _native as N
from .backend import _CH_FIRST_STR, _CH_LAST_STR

_lock = threading.Lock()


def _require_cuda():
    if not torch.cuda.is_available():
        raise N.KapreNativeError('kapre_b200 needs a CUDA device (B200, sm_100a); there is no CPU path')


def _stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def to_device(x, dtype=None):
    """NumPy array / CPU tensor / CUDA tensor -> CUDA tensor on the current device.
    Returns (tensor, was_host)."""
    _require_cuda()
    was_host = True
    if isinstance(x, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(x))
    elif isinstance(x, torch.Tensor):
        t = x
        was_host = not x.is_cuda
    else:
        t = torch.as_tensor(np.asarray(x))
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    if not t.is_cuda:
        t = t.to(torch.device('cuda', torch.cuda.current_device()), non_blocking=True)
    return t, was_host


def to_host(t: torch.Tensor) -> np.ndarray:
    """CUDA tensor -> NumPy through pinned memory (torch's caching host allocator)."""
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


_ws_cache = {}
_ws_retired = []   # outgrown workspaces stay alive: a captured CUDA graph may have their address baked in


def new_workspace(n_items: int, device) -> torch.Tensor:
    """Zeroed scratch of the decibel modes: 2 words per item (maximum + clamp-pass arrival counter)."""
    return torch.zeros(2 * max(int(n_items), 1), dtype=torch.int32, device=device)


def _workspace(n_items: int, device) -> torch.Tensor:
    """Per-(device, stream) zero-initialised scratch for the per-item dB maxima.  The kernels leave
    it zeroed (self-cleaning contract of the C ABI), so it is allocated and cleared only once.
    Objects that record launches into a CUDA graph own a private workspace instead (``workspace=``
    of ``stft_forward``), so nothing this cache does can invalidate a captured address."""
    n = max(int(n_items), 1)
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < 2 * n:
        if ws is not None:
            _ws_retired.append(ws)
        ws = new_workspace(max(n, 1024), device)
        _ws_cache[key] = ws
    return ws


def _device_of_first_arg(fn):
    """Run an op with the device of its first (tensor) argument current; host inputs keep the current device."""
    import functools

    @functools.wraps(fn)
    def wrapped(x, *a, **k):
        if isinstance(x, torch.Tensor) and x.is_cuda:
            with torch.cuda.device(x.device):
                return fn(x, *a, **k)
        return fn(x, *a, **k)
    return wrapped


def _on_device_of(t: torch.Tensor):
    """Context that makes the tensor's device current: plans, filterbanks, workspaces and the launch
    stream are all taken from the CURRENT device, which must be the one that owns the data."""
    if not t.is_cuda:
        raise N.KapreNativeError('kapre_b200 needs CUDA tensors (there is no CPU path)')
    return torch.cuda.device(t.device)


class _Handle:
    """Owns one C-ABI object and frees it with the matching destroy function."""

    def __init__(self, ptr, destroy):
        self.ptr = ptr
        self._destroy = destroy

    def __del__(self):
        try:
            if self.ptr:
                self._destroy(self.ptr)
                self.ptr = None
        except Exception:
            pass


class StftPlan:
    """kapre_stft_plan per CUDA device for one (n_fft, win_length, hop, window)."""

    def __init__(self, n_fft, win_length, hop_length, window: np.ndarray):
        self.n_fft, self.win_length, self.hop_length = int(n_fft), int(win_length), int(hop_length)
        self.window = np.ascontiguousarray(window, dtype=np.float32)
        if self.window.shape != (self.win_length,):
            raise ValueError('window must have win_length=%d samples, got %s' % (self.win_length, self.window.shape))
        self._per_device = {}

    def handle(self):
        _require_cuda()
        dev = torch.cuda.current_device()
        with _lock:
            h = self._per_device.get(dev)
            if h is None:
                lib = N.lib()
                out = ctypes.c_void_p()
                N.check(lib.kapre_stft_plan_create(self.n_fft, self.win_length, self.hop_length,
                                                   self.window.ctypes.data_as(ctypes.c_void_p), ctypes.byref(out)))
                h = _Handle(out, lib.kapre_stft_plan_destroy)
                self._per_device[dev] = h
        return h.ptr

    def num_frames(self, length, pad_begin, pad_end):
        lp = int(length) + ((self.n_fft - self.hop_length) if pad_begin else 0)
        if pad_end:
            return -(-lp // self.hop_length)
        return max(0, 1 + (lp - self.win_length) // self.hop_length)

    def supports_mode(self, mode):
        return bool(N.lib().kapre_stft_supports_mode(self.handle(), int(mode)))


class IstftPlan:
    def __init__(self, n_fft, win_length, hop_length, dual_window: np.ndarray):
        self.n_fft, self.win_length, self.hop_length = int(n_fft), int(win_length), int(hop_length)
        self.dual = np.ascontiguousarray(dual_window, dtype=np.float32)
        self._per_device = {}

    def handle(self):
        _require_cuda()
        dev = torch.cuda.current_device()
        with _lock:
            h = self._per_device.get(dev)
            if h is None:
                lib = N.lib()
                out = ctypes.c_void_p()
                N.check(lib.kapre_istft_plan_create(self.n_fft, self.win_length, self.hop_length,
                                                    self.dual.ctypes.data_as(ctypes.c_void_p), ctypes.byref(out)))
                h = _Handle(out, lib.kapre_istft_plan_destroy)
                self._per_device[dev] = h
        return h.ptr


class Filterbank:
    """kapre_filterbank per CUDA device for one (n_freq, n_bands) matrix."""

    def __init__(self, matrix: np.ndarray):
        self.matrix = np.ascontiguousarray(matrix, dtype=np.float32)
        if self.matrix.ndim != 2:
            raise ValueError('filterbank must be (n_freq, n_bands)')
        self.n_freq, self.n_bands = self.matrix.shape
        self._per_device = {}

    def handle(self):
        _require_cuda()
        dev = torch.cuda.current_device()
        with _lock:
            h = self._per_device.get(dev)
            if h is None:
                lib = N.lib()
                out = ctypes.c_void_p()
                N.check(lib.kapre_filterbank_create(self.matrix.ctypes.data_as(ctypes.c_void_p), self.n_freq,
                                                    self.n_bands, ctypes.byref(out)))
                h = _Handle(out, lib.kapre_filterbank_destroy)
                self._per_device[dev] = h
        return h.ptr


def _wave_desc(t: torch.Tensor, data_format: str):
    """(B, L, C) channels_last or (B, C, L) channels_first -> kapre_wave_desc."""
    if t.dim() != 3:
        raise ValueError('waveform batch must be 3-D, got shape %s' % (tuple(t.shape),))
    if data_format == _CH_LAST_STR:
        B, L, C = t.shape
        sb, sl, sc = t.stride()
    else:
        B, C, L = t.shape
        sb, sc, sl = t.stride()
    return N.WaveDesc(B, C, L, sb, sc, sl), (B, C, L)


def _spec_alloc(B, C, T, K, data_format, dtype, device):
    if data_format == _CH_LAST_STR:
        out = torch.empty((B, T, K, C), dtype=dtype, device=device)
        sb, st, sk, sc = out.stride()
    else:
        out = torch.empty((B, C, T, K), dtype=dtype, device=device)
        sb, sc, st, sk = out.stride()
    return out, N.SpecDesc(sb, sc, st, sk)


def _spec_desc(t: torch.Tensor, data_format: str):
    if t.dim() != 4:
        raise ValueError('spectrogram batch must be 4-D, got shape %s' % (tuple(t.shape),))
    if data_format == _CH_LAST_STR:
        B, T, K, C = t.shape
        sb, st, sk, sc = t.stride()
    else:
        B, C, T, K = t.shape
        sb, sc, st, sk = t.stride()
    return N.SpecDesc(sb, sc, st, sk), (B, C, T, K)


def stft_forward(x: torch.Tensor, plan: StftPlan, input_data_format, output_data_format, pad_begin, pad_end,
                 mode=N.OUT_COMPLEX, fb: Filterbank = None, db=None, workspace: torch.Tensor = None):
    """One fused launch: waveform -> (complex STFT | magnitude | filterbank) [-> dB].
    ``db`` = (ref_value, amin, dynamic_range); ``workspace``: caller-owned decibel scratch (``new_workspace``)."""
    if not x.is_cuda:
        raise N.KapreNativeError('stft_forward needs a CUDA tensor')
    with _on_device_of(x):
        return _stft_forward(x, plan, input_data_format, output_data_format, pad_begin, pad_end, mode, fb, db, workspace)


def _stft_forward(x, plan, input_data_format, output_data_format, pad_begin, pad_end, mode, fb, db, workspace):
    if x.dtype != torch.float32:
        x = x.float()
    if pad_begin and plan.hop_length > plan.n_fft:
        # kapre/time_frequency.py:169-172 pads by n_fft - hop_length; tf.pad rejects a negative amount
        raise ValueError('pad_begin needs hop_length <= n_fft: the padding is n_fft - hop_length = %d'
                         % (plan.n_fft - plan.hop_length))
    xd, (B, C, L) = _wave_desc(x, input_data_format)
    T = plan.num_frames(L, pad_begin, pad_end)
    fbmode = mode in (N.OUT_FB, N.OUT_FB_DB)
    K = fb.n_bands if fbmode else plan.n_fft // 2 + 1
    dtype = torch.complex64 if mode == N.OUT_COMPLEX else torch.float32
    c_out = 2 * C if mode == N.OUT_MAG_PHASE else C   # mag+phase: phases in channels [C, 2C)
    out, od = _spec_alloc(B, c_out, T, K, output_data_format, dtype, x.device)
    dbc, ws = None, None
    if mode in (N.OUT_MAG_DB, N.OUT_FB_DB) or (mode == N.OUT_MAG_PHASE and db is not None):
        dbc = N.DbCfg(float(db[0]), float(db[1]), float(db[2]))
        ws = workspace if workspace is not None else _workspace(B, x.device)
        if ws.device != x.device or ws.numel() < 2 * B:
            raise ValueError('decibel workspace must live on %s and hold 2 x %d words' % (x.device, B))
    if out.numel() == 0:
        return out
    try:
        N.check(N.lib().kapre_stft_forward(
            plan.handle(), _ptr(x), ctypes.byref(xd), int(bool(pad_begin)), int(bool(pad_end)), int(mode), _ptr(out),
            ctypes.byref(od), fb.handle() if fbmode else None, ctypes.byref(dbc) if dbc is not None else None,
            _ptr(ws) if ws is not None else None, _stream_ptr()))
    except N.KapreNativeError:
        if ws is not None and not torch.cuda.is_current_stream_capturing():
            ws.zero_()          # a failed call may have left maxima behind: restore the all-zero contract
        raise
    return out


@_device_of_first_arg
def istft(X: torch.Tensor, plan: IstftPlan, input_data_format, output_data_format):
    if not X.is_cuda:
        raise N.KapreNativeError('istft needs a CUDA tensor')
    if X.dtype != torch.complex64:
        X = X.to(torch.complex64)
    sd, (B, C, T, F) = _spec_desc(X, input_data_format)
    if F != plan.n_fft // 2 + 1:
        raise ValueError('expected %d frequency bins for n_fft=%d, got %d' % (plan.n_fft // 2 + 1, plan.n_fft, F))
    out_len = (T - 1) * plan.hop_length + plan.win_length if T > 0 else 0
    if output_data_format == _CH_LAST_STR:
        y = torch.empty((B, out_len, C), dtype=torch.float32, device=X.device)
        sb, sl, sc = y.stride()
    else:
        y = torch.empty((B, C, out_len), dtype=torch.float32, device=X.device)
        sb, sc, sl = y.stride()
    if y.numel() == 0:
        return y
    yd = N.WaveDesc(B, C, out_len, sb, sc, sl)
    N.check(N.lib().kapre_istft_inverse(plan.handle(), _ptr(X), B, C, T, ctypes.byref(sd), _ptr(y),
                                        ctypes.byref(yd), _stream_ptr()))
    return y


@_device_of_first_arg
def apply_filterbank(x: torch.Tensor, fb: Filterbank, data_format):
    if not x.is_cuda:
        raise N.KapreNativeError('apply_filterbank needs a CUDA tensor')
    if x.dtype != torch.float32:
        x = x.float()
    xd, (B, C, T, F) = _spec_desc(x, data_format)
    if F != fb.n_freq:
        raise ValueError('filterbank expects %d frequency bins, input has %d' % (fb.n_freq, F))
    out, od = _spec_alloc(B, C, T, fb.n_bands, data_format, torch.float32, x.device)
    if out.numel() == 0:
        return out
    N.check(N.lib().kapre_apply_filterbank(fb.handle(), _ptr(x), B, C, T, ctypes.byref(xd), _ptr(out),
                                           ctypes.byref(od), _stream_ptr()))
    return out


@_device_of_first_arg
def magnitude(x: torch.Tensor):
    if not x.is_cuda:
        raise N.KapreNativeError('magnitude needs a CUDA tensor')
    if not x.is_complex():
        return x.abs()  # tf.abs of a real tensor: plain |x| (not on the hot path)
    x = x.to(torch.complex64).contiguous()
    out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    if out.numel():
        N.check(N.lib().kapre_magnitude(_ptr(x), _ptr(out), x.numel(), _stream_ptr()))
    return out


@_device_of_first_arg
def phase(x: torch.Tensor):
    if not x.is_cuda:
        raise N.KapreNativeError('phase needs a CUDA tensor')
    x = x.to(torch.complex64).contiguous()
    out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    if out.numel():
        N.check(N.lib().kapre_phase(_ptr(x), _ptr(out), x.numel(), _stream_ptr()))
    return out


@_device_of_first_arg
def magnitude_to_decibel(x, ref_value=1.0, amin=1e-5, dynamic_range=80.0):
    t, was_host = to_device(x, torch.float32)
    t = t.contiguous()
    out = torch.empty_like(t)
    if t.numel():
        if t.dim() > 1:
            n_items, item = t.shape[0], t.numel() // t.shape[0]
        else:
            n_items, item = 1, t.numel()
        ws = _workspace(n_items, t.device)
        dbc = N.DbCfg(float(ref_value), float(amin), float(dynamic_range))
        N.check(N.lib().kapre_magnitude_to_decibel(_ptr(t), _ptr(out), n_items, item, ctypes.byref(dbc), _ptr(ws),
                                                   _stream_ptr()))
    return to_host(out) if was_host and isinstance(x, np.ndarray) else out


# ------------------------------------------------------------------------------- adjacent layers
_PAD_MODES = {'symmetric': 0, 'reflect': 1, 'constant': 2}


@_device_of_first_arg
def delta(x: torch.Tensor, win_length: int, mode: str, data_format: str):
    """kapre.Delta along the time axis of (b, t, f, ch) / (b, ch, t, f)."""
    if not x.is_cuda:
        raise N.KapreNativeError('delta needs a CUDA tensor')
    x = x.float().contiguous()
    if x.dim() != 4:
        raise ValueError('Delta expects a 4-D batch, got shape %s' % (tuple(x.shape),))
    if data_format == _CH_LAST_STR:
        outer, frames, inner = x.shape[0], x.shape[1], x.shape[2] * x.shape[3]
    else:
        outer, frames, inner = x.shape[0] * x.shape[1], x.shape[2], x.shape[3]
    out = torch.empty_like(x)
    if x.numel():
        N.check(N.lib().kapre_delta(_ptr(x), _ptr(out), outer, frames, inner, int(win_length),
                                    _PAD_MODES[mode.lower()], _stream_ptr()))
    return out


@_device_of_first_arg
def concat_frequency_map(x: torch.Tensor, data_format: str):
    """kapre.ConcatenateFrequencyMap: (b, t, f, ch) -> (b, t, f, ch + 1) or (b, ch, t, f) -> (b, ch + 1, t, f)."""
    if not x.is_cuda:
        raise N.KapreNativeError('concat_frequency_map needs a CUDA tensor')
    x = x.float().contiguous()
    if x.dim() != 4:
        raise ValueError('ConcatenateFrequencyMap expects a 4-D batch, got shape %s' % (tuple(x.shape),))
    cl = data_format == _CH_LAST_STR
    if cl:
        B, T, F, C = x.shape
        out = torch.empty((B, T, F, C + 1), dtype=torch.float32, device=x.device)
    else:
        B, C, T, F = x.shape
        out = torch.empty((B, C + 1, T, F), dtype=torch.float32, device=x.device)
    if out.numel():
        N.check(N.lib().kapre_concat_frequency_map(_ptr(x), _ptr(out), B, C, T, F, int(cl), _stream_ptr()))
    return out


@_device_of_first_arg
def spec_augment(x: torch.Tensor, time_masks: np.ndarray, freq_masks: np.ndarray, mask_value: float, data_format: str):
    """kapre.SpecAugment with given masks: x (b, t, f, 1) or (b, 1, t, f); masks (b, n, 2) int32 (start, width)."""
    if not x.is_cuda:
        raise N.KapreNativeError('spec_augment needs a CUDA tensor')
    x = x.float().contiguous()
    if data_format == _CH_LAST_STR:
        B, T, F, C = x.shape
    else:
        B, C, T, F = x.shape
    if C != 1:
        raise RuntimeError('SpecAugment does not support spectrograms with depth greater than 1')
    out = torch.empty_like(x)
    if x.numel() == 0:
        return out
    tm = torch.as_tensor(np.ascontiguousarray(time_masks, dtype=np.int32).reshape(B, -1, 2)).to(x.device)
    fm = torch.as_tensor(np.ascontiguousarray(freq_masks, dtype=np.int32).reshape(B, -1, 2)).to(x.device)
    N.check(N.lib().kapre_spec_augment(_ptr(x), _ptr(out), B, T, F, _ptr(tm) if tm.numel() else None, tm.shape[1],
                                       _ptr(fm) if fm.numel() else None, fm.shape[1], ctypes.c_float(mask_value), _stream_ptr()))
    return out


def _frames_for(length, frame_length, hop, pad_end):
    return -(-length // hop) if pad_end else max(0, 1 + (length - frame_length) // hop)


@_device_of_first_arg
def frame(x: torch.Tensor, frame_length, hop_length, pad_end, pad_value, data_format):
    """kapre.Frame: (b, t, ch) -> (b, frames, frame_length, ch) or (b, ch, t) -> (b, ch, frames, frame_length)."""
    if not x.is_cuda:
        raise N.KapreNativeError('frame needs a CUDA tensor')
    x = x.float()
    xd, (B, C, L) = _wave_desc(x, data_format)
    T = _frames_for(L, frame_length, hop_length, pad_end)
    out, od = _spec_alloc(B, C, T, frame_length, data_format, torch.float32, x.device)
    if out.numel():
        N.check(N.lib().kapre_frame(_ptr(x), ctypes.byref(xd), int(frame_length), int(hop_length), int(bool(pad_end)),
                                    ctypes.c_float(pad_value), _ptr(out), ctypes.byref(od), _stream_ptr()))
    return out


@_device_of_first_arg
def energy(x: torch.Tensor, frame_length, hop_length, pad_end, pad_value, scale, data_format):
    """kapre.Energy: scale * sum of squares per frame; (b, t, ch) -> (b, frames, ch), (b, ch, t) -> (b, ch, frames)."""
    if not x.is_cuda:
        raise N.KapreNativeError('energy needs a CUDA tensor')
    x = x.float()
    xd, (B, C, L) = _wave_desc(x, data_format)
    T = _frames_for(L, frame_length, hop_length, pad_end)
    if data_format == _CH_LAST_STR:
        out = torch.empty((B, T, C), dtype=torch.float32, device=x.device)
        sb, st, sc = out.stride()
    else:
        out = torch.empty((B, C, T), dtype=torch.float32, device=x.device)
        sb, sc, st = out.stride()
    if out.numel():
        od = N.WaveDesc(B, C, T, sb, sc, st)
        N.check(N.lib().kapre_energy(_ptr(x), ctypes.byref(xd), int(frame_length), int(hop_length), int(bool(pad_end)),
                                     ctypes.c_float(pad_value), ctypes.c_float(scale), _ptr(out), ctypes.byref(od),
                                     _stream_ptr()))
    return out


# ------------------------------------------------------------------------------- backward (VJPs)
def grad_workspace(n_items: int, device) -> torch.Tensor:
    """Zeroed scratch of the decibel VJP statistics (C ABI: >= 1056 * n_items + 16 bytes, zero on entry, left zero)."""
    n = max(int(n_items), 1)
    return torch.zeros(((n * 4 + 15) // 16 * 16 + 1040 * n) // 4, dtype=torch.int32, device=device)


def _resolved(t: torch.Tensor) -> torch.Tensor:
    """Materialise torch's lazy conjugate / negative views (their bits are not what the strides describe)."""
    return t.resolve_conj().resolve_neg() if t.is_complex() else t.resolve_neg()


def transposed(fb: Filterbank) -> Filterbank:
    """The (n_bands, n_freq) transpose of a filterbank: ApplyFilterbank's VJP is ApplyFilterbank with it."""
    t = getattr(fb, '_transposed', None)
    if t is None:
        t = fb._transposed = Filterbank(fb.matrix.T)
    return t


@_device_of_first_arg
def stft_backward(G: torch.Tensor, plan: StftPlan, spec_format, wave_format, pad_begin, pad_end, length):
    """VJP of the STFT: complex gradient of the spectrum (layout ``spec_format``) -> float32 gradient of the waveform
    (layout ``wave_format``, ``length`` samples).  One launch of the windowed overlap-add of inverse real FFTs."""
    if not G.is_cuda:
        raise N.KapreNativeError('stft_backward needs a CUDA tensor')
    G = _resolved(G.to(torch.complex64))
    sd, (B, C, T, F) = _spec_desc(G, spec_format)
    L = int(length)
    if F != plan.n_fft // 2 + 1:
        raise ValueError('expected %d frequency bins for n_fft=%d, got %d' % (plan.n_fft // 2 + 1, plan.n_fft, F))
    if wave_format == _CH_LAST_STR:
        gx = torch.empty((B, L, C), dtype=torch.float32, device=G.device)
        sb, sl, sc = gx.stride()
    else:
        gx = torch.empty((B, C, L), dtype=torch.float32, device=G.device)
        sb, sc, sl = gx.stride()
    if gx.numel():
        xd = N.WaveDesc(B, C, L, sb, sc, sl)
        N.check(N.lib().kapre_stft_backward(plan.handle(), _ptr(G), B, C, T, ctypes.byref(sd), int(bool(pad_begin)),
                                            int(bool(pad_end)), _ptr(gx), ctypes.byref(xd), _stream_ptr()))
    return gx


@_device_of_first_arg
def istft_backward(gy: torch.Tensor, plan: IstftPlan, spec_format, wave_format, frames):
    """VJP of the inverse STFT: float gradient of the waveform -> complex64 gradient of the ``frames``-frame spectrum."""
    if not gy.is_cuda:
        raise N.KapreNativeError('istft_backward needs a CUDA tensor')
    gy = _resolved(gy.to(torch.float32))
    yd, (B, C, L) = _wave_desc(gy, wave_format)
    G, gd = _spec_alloc(B, C, int(frames), plan.n_fft // 2 + 1, spec_format, torch.complex64, gy.device)
    if G.numel():
        N.check(N.lib().kapre_istft_backward(plan.handle(), _ptr(gy), ctypes.byref(yd), _ptr(G), int(frames),
                                             ctypes.byref(gd), _stream_ptr()))
    return G


@_device_of_first_arg
def spectral_backward(X: torch.Tensor, g: torch.Tensor, y, mode, fb: Filterbank, db, data_format, out=None):
    """VJP of |.| [-> filterbank] [-> dB] at the complex STFT ``X`` (4-D, ``data_format``): upstream gradient ``g`` and,
    for the decibel modes, forward output ``y`` (both (B, C, T, K) in ``data_format``) -> complex gradient of ``X``.
    ``out`` may be ``X`` itself (in place)."""
    if not X.is_cuda:
        raise N.KapreNativeError('spectral_backward needs a CUDA tensor')
    if X.dtype != torch.complex64:
        raise ValueError('spectral_backward needs a complex64 spectrum')
    xd, (B, C, T, F) = _spec_desc(X, data_format)
    g = _resolved(g.to(torch.float32))
    gd, _ = _spec_desc(g, data_format)
    fbmode = mode in (N.OUT_FB, N.OUT_FB_DB)
    dbmode = mode in (N.OUT_MAG_DB, N.OUT_FB_DB)
    if out is None:
        out, od = _spec_alloc(B, C, T, F, data_format, torch.complex64, X.device)
    else:
        od, _ = _spec_desc(out, data_format)
    yd, dbc, ws = None, None, None
    if dbmode:
        yd, _ = _spec_desc(y, data_format)
        dbc = N.DbCfg(float(db[0]), float(db[1]), float(db[2]))
        ws = grad_workspace(B, X.device)
    if out.numel():
        N.check(N.lib().kapre_spectral_backward(
            fb.handle() if fbmode else None, int(mode), _ptr(X), B, C, T, F, ctypes.byref(xd), _ptr(g), ctypes.byref(gd),
            _ptr(y) if dbmode else None, ctypes.byref(yd) if dbmode else None, ctypes.byref(dbc) if dbmode else None,
            _ptr(ws) if dbmode else None, _ptr(out), ctypes.byref(od), _stream_ptr()))
    return out


def _items(t: torch.Tensor):
    """(n_items, item_size) of the decibel layer: per batch item, or one item for a 1-D tensor (kapre/backend.py:178-179)."""
    if t.dim() > 1:
        return t.shape[0], t.numel() // t.shape[0]
    return 1, t.numel()


@_device_of_first_arg
def magnitude_to_decibel_backward(x: torch.Tensor, y: torch.Tensor, g: torch.Tensor, ref_value, amin, dynamic_range):
    """VJP of MagnitudeToDecibel: contiguous float32 input ``x`` and output ``y`` of the forward, upstream gradient ``g``
    (any strides) -> float32 gradient of ``x``."""
    if not x.is_cuda:
        raise N.KapreNativeError('magnitude_to_decibel_backward needs a CUDA tensor')
    gx = torch.empty_like(x)
    if x.numel() == 0:
        return gx
    n_items, item = _items(x)
    g2 = _resolved(g.to(torch.float32)).reshape(n_items, item)
    ws = grad_workspace(n_items, x.device)
    dbc = N.DbCfg(float(ref_value), float(amin), float(dynamic_range))
    N.check(N.lib().kapre_magnitude_to_decibel_backward(_ptr(x), _ptr(y), _ptr(g2), g2.stride(0), g2.stride(1), _ptr(gx),
                                                        n_items, item, ctypes.byref(dbc), _ptr(ws), _stream_ptr()))
    return gx


@_device_of_first_arg
def magnitude_backward(X: torch.Tensor, g: torch.Tensor):
    """VJP of Magnitude (tf.abs of a complex tensor): G = g X / |X|, 0 where |X| = 0."""
    if not X.is_cuda:
        raise N.KapreNativeError('magnitude_backward needs a CUDA tensor')
    Xc = X.to(torch.complex64).contiguous()
    F = Xc.shape[-1] if Xc.dim() else 1
    X2 = Xc.reshape(1, 1, -1, F)
    g2 = _resolved(g.to(torch.float32)).reshape(1, 1, -1, F)
    # a (rows, F) tensor is a (1, 1, rows, F) channels_first spectrogram
    return spectral_backward(X2, g2, None, N.OUT_MAG, None, None, _CH_FIRST_STR).reshape(Xc.shape)
