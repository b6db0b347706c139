"""Mirrors of the hot-path factories of ``kapre/composed.py`` plus the ``Sequential`` container.

``get_melspectrogram_layer`` (reference kapre/composed.py:138-261), ``get_stft_magnitude_layer``
(:32-135) and ``get_perfectly_reconstructing_stft_istft`` (:388-417) keep their signatures and
return the same layer stacks.  ``Sequential`` recognises the stack
``[STFT, Magnitude, (ApplyFilterbank), (MagnitudeToDecibel)]`` and runs it as ONE fused CUDA
launch (magnitudes never reach HBM); ``.layers`` remains usable one by one
(kapre/composed.py:5-12) and gives the same results through the stand-alone kernels.
"""
from __future__ import annotations

import os
import weakref

import numpy as np
import torch

from . import _native as N
from . import autograd, backend, ops
from .backend import _CH_DEFAULT_STR, _CH_FIRST_STR, _CH_LAST_STR
from .time_frequency import (STFT, ApplyFilterbank, InverseSTFT, Layer, Magnitude, MagnitudeToDecibel, Phase,
                             get_registered_object)

__all__ = ['CapturedSequential', 'Sequential', 'StftMagPhase', 'get_stft_magnitude_layer', 'get_melspectrogram_layer',
           'get_log_frequency_spectrogram_layer', 'get_perfectly_reconstructing_stft_istft', 'get_stft_mag_phase']


_streams = {}


_copy_pool = None


def _get_copy_pool():
    global _copy_pool
    if _copy_pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _copy_pool = ThreadPoolExecutor(8)
    return _copy_pool


def _host_copy(dst, src, min_bytes=1 << 20):
    """Host-to-host copy of a contiguous tensor with a few memcpy threads (NumPy releases the GIL in ``copyto``).
    ``Tensor.copy_`` between CPU tensors runs an OpenMP loop that was measured 50x slower than one memcpy on
    CPU-restricted hosts (thread oversubscription); one thread moves ~12 GB/s, PCIe needs ~55 GB/s."""
    d = dst.numpy().reshape(-1)
    a = src.numpy().reshape(-1)
    n = d.size
    try:
        ncpu = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        ncpu = os.cpu_count() or 1
    k = max(1, min(8, ncpu, d.nbytes // min_bytes))
    if k == 1:
        np.copyto(d, a)
        return
    step = -(-n // k)
    list(_get_copy_pool().map(lambda j: np.copyto(d[j * step:(j + 1) * step], a[j * step:(j + 1) * step]), range(k)))


def _side_streams(dev):
    """(copy-in, copy-out) streams per device for the pipelined host path."""
    key = dev.index
    if key not in _streams:
        _streams[key] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    return _streams[key]


class Sequential(Layer):
    """Minimal ``keras.Sequential``: ``add``, ``layers``, ``__call__``, ``predict``, config."""

    def __init__(self, layers=None, name=None, fuse=True):
        super().__init__(name=name)
        self.layers = []
        self.fuse = fuse
        for layer in (layers or []):
            self.add(layer)

    def add(self, layer):
        if not isinstance(layer, Layer):
            raise TypeError('Sequential only takes kapre_b200 layers, got %r' % (layer,))
        self.layers.append(layer)

    # -- fusion -----------------------------------------------------------------------------
    def _fused_prefix(self):
        """(n_layers_consumed, mode, stft, filterbank_layer, db_layer) for the longest leading
        run that one fused launch covers, or None."""
        ls = self.layers
        if not self.fuse or len(ls) < 2 or type(ls[0]) is not STFT or type(ls[1]) is not Magnitude:
            return None
        stft = ls[0]
        n, mode, fbl, dbl = 2, N.OUT_MAG, None, None
        if len(ls) > n and type(ls[n]) is ApplyFilterbank and hasattr(ls[n], 'filterbank') \
                and ls[n].data_format == stft.output_data_format \
                and ls[n].filterbank.shape[0] == stft.n_fft // 2 + 1:
            fbl, mode, n = ls[n], N.OUT_FB, n + 1
        if len(ls) > n and type(ls[n]) is MagnitudeToDecibel:
            dbl, n = ls[n], n + 1
            mode = N.OUT_FB_DB if fbl is not None else N.OUT_MAG_DB
        if not stft.plan.supports_mode(mode):
            return None
        return n, mode, stft, fbl, dbl

    def call(self, x):
        start = 0
        fused = self._fused_prefix() if (isinstance(x, torch.Tensor) and x.is_cuda and x.dim() == 3) else None
        if fused is not None:
            n, mode, stft, fbl, dbl = fused
            db = None
            if dbl is not None:
                # same call-time validation as backend.magnitude_to_decibel (kapre/backend.py:168-173)
                if dbl.ref_value <= 0:
                    raise ValueError('ref_value must be positive, got: %s' % (dbl.ref_value,))
                if dbl.amin <= 0:
                    raise ValueError('amin must be positive, got: %s' % (dbl.amin,))
                if dbl.dynamic_range <= 0:
                    raise ValueError('dynamic_range must be positive, got: %s' % (dbl.dynamic_range,))
                db = (dbl.ref_value, dbl.amin, dbl.dynamic_range)
            if autograd.wants_grad(x):
                x = autograd.FusedSpectrogramFn.apply(x, stft, mode, fbl.fb if fbl is not None else None, db)
            else:
                x = ops.stft_forward(x, stft.plan, stft.input_data_format, stft.output_data_format, stft.pad_begin,
                                     stft.pad_end, mode, fbl.fb if fbl is not None else None, db)
            start = n
        for layer in self.layers[start:]:
            x = layer.call(x)
        return x

    def _pinned_result(self, shape, dtype):
        """Page-locked result buffer and the NumPy array over it that ``predict`` returns.

        ``cudaHostAlloc`` of a result-sized block costs 10-70 ms (measured: it was the whole gap between
        predict() and the PCIe bound), so finished buffers are recycled.  A buffer is handed out again
        only when the array returned for it -- and every view derived from it -- is gone: NumPy keeps the
        array's ``base`` (a tensor aliasing the buffer) alive exactly that long, and a weak reference to
        that base tells."""
        pool = self.__dict__.setdefault('_result_pool', [])
        entry = None
        for e in pool:
            if e['t'].shape == shape and e['t'].dtype == dtype and (e['ref'] is None or e['ref']() is None):
                entry = e
                break
        if entry is None:
            entry = {'t': torch.empty(shape, dtype=dtype, pin_memory=True), 'ref': None}
            pool.append(entry)
            if len(pool) > 4:       # drop one idle buffer of another shape / an older one
                for i, e in enumerate(pool):
                    if e is not entry and (e['ref'] is None or e['ref']() is None):
                        del pool[i]
                        break
        arr = entry['t'].numpy()
        entry['ref'] = weakref.ref(arr.base)
        return entry['t'], arr

    def predict(self, x, batch_size=None, verbose=0, **kwargs):
        """Like ``keras.Model.predict``: host array in, host array out.

        Host inputs are streamed: the batch is cut into chunks of ``batch_size`` items (default:
        an eighth of the batch) and chunk i+1's host->device copy, chunk i's kernels and chunk
        i-1's device->host copy run on three CUDA streams, so PCIe runs in both directions while
        the SMs compute.  Results do not depend on the chunking: every op on the path, including
        the decibel clamp, is per batch item (kapre/backend.py:178-179)."""
        if isinstance(x, torch.Tensor) and x.is_cuda:
            return ops.to_host(self.call(x))
        xh = torch.from_numpy(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else torch.as_tensor(x)
        B = xh.shape[0]
        if B == 0:
            return ops.to_host(self.call(xh.cuda()))
        chunk = int(batch_size) if batch_size and batch_size > 0 else max(1, -(-B // 8))
        ops._require_cuda()
        dev = torch.device('cuda', torch.cuda.current_device())
        s_comp = torch.cuda.current_stream()
        s_in, s_out = _side_streams(dev)
        s_in.wait_stream(s_comp)
        out_host = None
        keep = []
        # Pageable input (what a kapre user's NumPy array is): a cudaMemcpy from pageable memory goes through the driver's own
        # small staging buffer and blocks the host (~10 GB/s, nothing overlaps).  Instead every chunk is copied into its own
        # page-locked staging buffer by a memcpy thread (all chunks at once: one thread moves ~12 GB/s, PCIe needs ~55), and
        # the loop below only waits for chunk i's copy before it queues chunk i's DMA.  More than 16 chunks: a ring of three
        # buffers, each reused only after the event recorded behind its DMA has completed.
        n_chunks = -(-B // chunk)
        stage = futs = None
        if not xh.is_pinned():
            stage = self._staging_ring((min(chunk, B),) + tuple(xh.shape[1:]), xh.dtype, n_chunks if n_chunks <= 16 else 3)
            if n_chunks <= 16:
                pool = _get_copy_pool()
                futs = [pool.submit(_host_copy, stage[ci]['t'][:min(chunk, B - ci * chunk)], xh[ci * chunk:(ci + 1) * chunk], 1 << 62)
                        for ci in range(n_chunks)]
        for ci, i in enumerate(range(0, B, chunk)):
            src = xh[i:i + chunk]
            if stage is not None:
                slot = stage[ci % len(stage)]
                buf = slot['t'][:src.shape[0]]
                if futs is not None:
                    futs[ci].result()
                else:
                    if slot['ev'] is not None:
                        slot['ev'].synchronize()
                    _host_copy(buf, src)
                src = buf
            with torch.cuda.stream(s_in):
                xd = src.to(dev, non_blocking=True)
                ev_in = torch.cuda.Event()
                ev_in.record(s_in)
            if stage is not None:
                slot['ev'] = ev_in
            s_comp.wait_event(ev_in)
            xd.record_stream(s_comp)
            yd = self.call(xd)
            ev_c = torch.cuda.Event()
            ev_c.record(s_comp)
            if out_host is None:
                out_host, out_arr = self._pinned_result((B,) + tuple(yd.shape[1:]), yd.dtype)
            s_out.wait_event(ev_c)
            yd.record_stream(s_out)
            with torch.cuda.stream(s_out):
                out_host[i:i + chunk].copy_(yd, non_blocking=True)
            keep.append((xd, yd))
        s_out.synchronize()
        return out_arr

    def _staging_ring(self, shape, dtype, n=3):
        """``n`` page-locked staging buffers for pageable host inputs.  ``cudaHostAlloc`` is slow (10-70 ms for a
        cfg2-sized chunk), so the buffers are kept and only ever grow: a smaller chunk shape is a view of the same bytes."""
        need = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        ring = self.__dict__.setdefault('_stage_ring', [])
        for slot in ring:
            if slot['raw'].numel() < need:
                slot['raw'] = torch.empty((max(need, 1),), dtype=torch.uint8, pin_memory=True)
        while len(ring) < n:
            ring.append({'raw': torch.empty((max(need, 1),), dtype=torch.uint8, pin_memory=True), 'ev': None})
        for slot in ring:
            slot['t'] = slot['raw'][:need].view(dtype).view(shape)
        return ring[:n]

    def capture(self, example):
        """Freeze this model for one input shape into a CUDA graph (``CapturedSequential``): replaying it
        costs one graph launch instead of one kernel launch + Python / ctypes dispatch per layer, which is
        what bounds small batches (cfg1: 13 us of kernel under ~40 us of submission)."""
        return CapturedSequential(self, example)

    # -- serialisation ------------------------------------------------------------------------
    def get_config(self):
        return {'name': self.name,
                'layers': [{'class_name': type(l).__name__,
                            'registered_name': getattr(type(l), '_registered_name', None),
                            'config': l.get_config()} for l in self.layers]}

    @classmethod
    def from_config(cls, config):
        layers = []
        for item in config['layers']:
            klass = get_registered_object(item.get('registered_name')) or globals().get(item['class_name'])
            if klass is None:
                raise ValueError('Unknown layer class %r' % (item['class_name'],))
            layers.append(klass.from_config(dict(item['config'])))
        return cls(layers, name=config.get('name'))


class CapturedSequential:
    """A ``Sequential`` captured into a CUDA graph for a fixed input shape / dtype / device.

    ``captured(x)`` copies ``x`` (host or device) into the graph's static input, replays the graph and
    returns the static output tensor (valid until the next call; ``.clone()`` it to keep it).  The
    kernels are the same C-ABI launches as in eager mode, recorded once on a private stream."""

    def __init__(self, model, example):
        ops._require_cuda()
        x, _ = ops.to_device(example)
        self.model = model
        self.static_in = x.clone()
        cur = torch.cuda.current_stream()
        self._stream = torch.cuda.Stream(device=x.device)
        self._stream.wait_stream(cur)
        with torch.cuda.stream(self._stream):      # warm-up on the capture stream: plans, workspace, smem attrs
            for _ in range(2):
                model.call(self.static_in)
        self._stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self._stream):
            self.static_out = model.call(self.static_in)
        cur.wait_stream(self._stream)

    def __call__(self, x):
        if not isinstance(x, torch.Tensor):
            x = torch.from_numpy(np.ascontiguousarray(x))
        if tuple(x.shape) != tuple(self.static_in.shape):
            raise ValueError('captured for input shape %s, got %s' % (tuple(self.static_in.shape), tuple(x.shape)))
        self.static_in.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.static_out

    def predict(self, x, **kwargs):
        return ops.to_host(self(x))


def get_stft_magnitude_layer(input_shape=None, n_fft=2048, win_length=None, hop_length=None, window_name=None,
                             pad_begin=False, pad_end=False, return_decibel=False, db_amin=1e-5,
                             db_ref_value=1.0, db_dynamic_range=80.0, input_data_format='default',
                             output_data_format='default', name='stft_magnitude'):
    """``Sequential([STFT, Magnitude, (MagnitudeToDecibel)])`` -- kapre/composed.py:32-135."""
    backend.validate_data_format_str(input_data_format)
    backend.validate_data_format_str(output_data_format)
    stft_kwargs = {}
    if input_shape is not None:
        stft_kwargs['input_shape'] = input_shape
    waveform_to_stft = STFT(**stft_kwargs, n_fft=n_fft, win_length=win_length, hop_length=hop_length,
                            window_name=window_name, pad_begin=pad_begin, pad_end=pad_end,
                            input_data_format=input_data_format, output_data_format=output_data_format)
    layers = [waveform_to_stft, Magnitude()]
    if return_decibel:
        layers.append(MagnitudeToDecibel(ref_value=db_ref_value, amin=db_amin, dynamic_range=db_dynamic_range))
    return Sequential(layers, name=name)


def get_melspectrogram_layer(input_shape=None, n_fft=2048, win_length=None, hop_length=None, window_name=None,
                             pad_begin=False, pad_end=False, sample_rate=22050, n_mels=128, mel_f_min=0.0,
                             mel_f_max=None, mel_htk=False, mel_norm='slaney', return_decibel=False,
                             db_amin=1e-5, db_ref_value=1.0, db_dynamic_range=80.0, input_data_format='default',
                             output_data_format='default', name='melspectrogram'):
    """``Sequential([STFT, Magnitude, ApplyFilterbank('mel'), (MagnitudeToDecibel)])`` --
    kapre/composed.py:138-261.  Called on a CUDA tensor the whole stack is one fused kernel."""
    backend.validate_data_format_str(input_data_format)
    backend.validate_data_format_str(output_data_format)
    stft_kwargs = {}
    if input_shape is not None:
        stft_kwargs['input_shape'] = input_shape
    waveform_to_stft = STFT(**stft_kwargs, n_fft=n_fft, win_length=win_length, hop_length=hop_length,
                            window_name=window_name, pad_begin=pad_begin, pad_end=pad_end,
                            input_data_format=input_data_format, output_data_format=output_data_format)
    kwargs = {'sample_rate': sample_rate, 'n_freq': n_fft // 2 + 1, 'n_mels': n_mels, 'f_min': mel_f_min,
              'f_max': mel_f_max, 'htk': mel_htk, 'norm': mel_norm}
    stftm_to_melgram = ApplyFilterbank(type='mel', filterbank_kwargs=kwargs, data_format=output_data_format)
    layers = [waveform_to_stft, Magnitude(), stftm_to_melgram]
    if return_decibel:
        layers.append(MagnitudeToDecibel(ref_value=db_ref_value, amin=db_amin, dynamic_range=db_dynamic_range))
    return Sequential(layers, name=name)


def get_log_frequency_spectrogram_layer(input_shape=None, n_fft=2048, win_length=None, hop_length=None,
                                        window_name=None, pad_begin=False, pad_end=False, sample_rate=22050,
                                        log_n_bins=84, log_f_min=None, log_bins_per_octave=12, log_spread=0.125,
                                        return_decibel=False, db_amin=1e-5, db_ref_value=1.0,
                                        db_dynamic_range=80.0, input_data_format='default',
                                        output_data_format='default', name='log_frequency_spectrogram'):
    """Same stack with the log-frequency filterbank -- kapre/composed.py:264-385."""
    backend.validate_data_format_str(input_data_format)
    backend.validate_data_format_str(output_data_format)
    stft_kwargs = {}
    if input_shape is not None:
        stft_kwargs['input_shape'] = input_shape
    waveform_to_stft = STFT(**stft_kwargs, n_fft=n_fft, win_length=win_length, hop_length=hop_length,
                            window_name=window_name, pad_begin=pad_begin, pad_end=pad_end,
                            input_data_format=input_data_format, output_data_format=output_data_format)
    kwargs = {'sample_rate': sample_rate, 'n_freq': n_fft // 2 + 1, 'n_bins': log_n_bins,
              'bins_per_octave': log_bins_per_octave, 'f_min': log_f_min, 'spread': log_spread}
    stftm_to_loggram = ApplyFilterbank(type='log', filterbank_kwargs=kwargs, data_format=output_data_format)
    layers = [waveform_to_stft, Magnitude(), stftm_to_loggram]
    if return_decibel:
        layers.append(MagnitudeToDecibel(ref_value=db_ref_value, amin=db_amin, dynamic_range=db_dynamic_range))
    return Sequential(layers, name=name)


def get_perfectly_reconstructing_stft_istft(n_fft, hop_length, waveform_data_format, stft_data_format,
                                            stft_name=None, istft_name=None):
    """The (STFT, InverseSTFT) pair of kapre/composed.py:388-417: Hann window of ``n_fft`` samples,
    ``pad_begin`` and ``pad_end`` on, so that STFT -> InverseSTFT reproduces the waveform after
    trimming the first ``n_fft - hop_length`` samples."""
    stft = STFT(n_fft=n_fft, win_length=n_fft, hop_length=hop_length, window_name='hann_window', pad_begin=True,
                pad_end=True, input_data_format=waveform_data_format, output_data_format=stft_data_format,
                name=stft_name)
    istft = InverseSTFT(n_fft=n_fft, win_length=n_fft, hop_length=hop_length, forward_window_name='hann_window',
                        input_data_format=stft_data_format, output_data_format=waveform_data_format,
                        name=istft_name)
    return stft, istft


class StftMagPhase(Layer):
    """The functional model built by ``get_stft_mag_phase`` (kapre/composed.py:478-511): STFT, then
    Magnitude (optionally MagnitudeToDecibel) and Phase, concatenated on the channel axis.  On the
    fused path all of it is one kernel launch writing both halves of the output tensor."""

    def __init__(self, stft, magnitude, phase, mag_to_decibel, ch_axis, name=None):
        super().__init__(name=name)
        self.stft, self.magnitude, self.phase, self.mag_to_decibel = stft, magnitude, phase, mag_to_decibel
        self.ch_axis = ch_axis
        self.layers = [stft, magnitude, phase] + ([mag_to_decibel] if mag_to_decibel is not None else [])

    def call(self, x):
        stft, db = self.stft, self.mag_to_decibel
        natural_axis = 1 if stft.output_data_format == _CH_FIRST_STR else 3
        if x.dim() == 3 and self.ch_axis == natural_axis and stft.plan.supports_mode(N.OUT_MAG_PHASE):
            dbt = None
            if db is not None:
                for nm in ('ref_value', 'amin', 'dynamic_range'):   # kapre/backend.py:168-173
                    if getattr(db, nm) <= 0:
                        raise ValueError('%s must be positive, got: %s' % (nm, getattr(db, nm)))
                dbt = (db.ref_value, db.amin, db.dynamic_range)
            return ops.stft_forward(x, stft.plan, stft.input_data_format, stft.output_data_format, stft.pad_begin,
                                    stft.pad_end, N.OUT_MAG_PHASE, None, dbt)
        s = stft.call(x)
        mag = self.magnitude.call(s)
        ph = self.phase.call(s)
        if db is not None:
            mag = db.call(mag)
        return torch.cat([mag, ph], dim=self.ch_axis)

    def predict(self, x, batch_size=None, verbose=0, **kwargs):
        y = self(x)
        return ops.to_host(y) if isinstance(y, torch.Tensor) else y


def get_stft_mag_phase(input_shape, n_fft=2048, win_length=None, hop_length=None, window_name=None, pad_begin=False,
                       pad_end=False, return_decibel=False, db_amin=1e-5, db_ref_value=1.0, db_dynamic_range=80.0,
                       input_data_format='default', output_data_format='default', name='stft_mag_phase'):
    """Magnitude and phase of the STFT side by side on the channel axis -- kapre/composed.py:420-511.
    Output ``(batch, time, freq, 2*ch)`` / ``(batch, 2*ch, time, freq)``: ``[ch magnitude; ch phase]``.
    ``input_shape`` is accepted for signature compatibility (the reference needs it for ``keras.Input``)."""
    backend.validate_data_format_str(input_data_format)
    backend.validate_data_format_str(output_data_format)
    waveform_to_stft = STFT(n_fft=n_fft, win_length=win_length, hop_length=hop_length, window_name=window_name,
                            pad_begin=pad_begin, pad_end=pad_end, input_data_format=input_data_format,
                            output_data_format=output_data_format)
    mag_to_decibel = MagnitudeToDecibel(ref_value=db_ref_value, amin=db_amin, dynamic_range=db_dynamic_range) \
        if return_decibel else None
    ch_axis = 1 if output_data_format == _CH_FIRST_STR else 3     # sic: the unresolved string, composed.py:504
    return StftMagPhase(waveform_to_stft, Magnitude(), Phase(), mag_to_decibel, ch_axis, name=name)
