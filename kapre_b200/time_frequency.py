"""Drop-in mirrors of the hot-path layers of ``kapre/time_frequency.py``.

``STFT``, ``InverseSTFT``, ``Magnitude``, ``Phase``, ``MagnitudeToDecibel`` and
``ApplyFilterbank`` keep the reference's constructor signatures, defaults, validation order
and ``get_config()`` keys (/root/reference/kapre/time_frequency.py:61-559), but ``call`` runs
hand-written sm_100a CUDA through the C ABI instead of ``tf.signal``.

Keras is not a dependency: ``Layer`` below is the minimal part of the Keras layer protocol the
reference relies on (``__call__`` -> ``call``, ``name``, ``get_config`` / ``from_config``).
Inputs may be NumPy arrays or CPU tensors (copied to the current CUDA device, result returned
as NumPy, like ``model.predict``) or CUDA tensors (result stays on the device).
"""
from __future__ import annotations

import itertools

import numpy as np
import torch

from . import _native as N
from . import autograd, backend, ops
from .backend import _CH_DEFAULT_STR, _CH_FIRST_STR, _CH_LAST_STR

__all__ = ['Layer', 'STFT', 'InverseSTFT', 'Magnitude', 'Phase', 'MagnitudeToDecibel', 'ApplyFilterbank', 'Delta']

_name_counters = {}
_REGISTRY = {}


def register_keras_serializable(package='Kapre'):
    """Same registration key as the reference ('Kapre>ClassName', time_frequency.py:60)."""

    def deco(cls):
        _REGISTRY['%s>%s' % (package, cls.__name__)] = cls
        cls._registered_name = '%s>%s' % (package, cls.__name__)
        return cls

    return deco


def get_registered_object(name):
    return _REGISTRY.get(name)


def _auto_name(cls_name):
    # keras-style snake_case auto names: stft, stft_1, ...
    snake = ''.join(('_' + c.lower()) if c.isupper() and i and not cls_name[i - 1].isupper() else c.lower()
                    for i, c in enumerate(cls_name))
    c = _name_counters.setdefault(snake, itertools.count())
    i = next(c)
    return snake if i == 0 else '%s_%d' % (snake, i)


class Layer:
    """The slice of ``keras.layers.Layer`` the kapre layers use."""

    def __init__(self, name=None, trainable=True, dtype=None, input_shape=None, **kwargs):
        kwargs.pop('batch_input_shape', None)
        kwargs.pop('batch_size', None)
        if kwargs:
            raise TypeError('Unrecognized keyword arguments passed to %s: %s' % (type(self).__name__, kwargs))
        self.name = name if name is not None else _auto_name(type(self).__name__)
        self.trainable = trainable
        self.dtype = dtype or backend._get_floatx()
        self.input_shape_arg = input_shape
        self.built = True

    # -- tensor plumbing ----------------------------------------------------------------
    def __call__(self, x, *args, **kwargs):
        kwargs.pop('training', None)
        t, was_host = ops.to_device(x)
        y = self.call(t, *args, **kwargs)
        if was_host and isinstance(y, torch.Tensor):
            return ops.to_host(y)
        return y

    def call(self, x):  # pragma: no cover - abstract
        raise NotImplementedError

    @property
    def weights(self):
        return []

    def count_params(self):
        return 0

    # -- serialisation ------------------------------------------------------------------
    # constructor keywords a subclass reports in get_config(): (config key, attribute holding the value)
    _config_fields = ()

    def get_config(self):
        config = {'name': self.name, 'trainable': self.trainable, 'dtype': self.dtype}
        for key, attr in self._config_fields:
            config[key] = getattr(self, attr)
        return config

    @classmethod
    def from_config(cls, config):
        return cls(**config)


def _unwrap_format(fmt):
    # kapre/time_frequency.py:118-124: workaround for dict-wrapped strings from Keras deserialisation
    return fmt['config'] if isinstance(fmt, dict) else fmt


def _resolve(fmt):
    return backend.image_data_format() if fmt == _CH_DEFAULT_STR else fmt


@register_keras_serializable(package='Kapre')
class STFT(Layer):
    """Short-time Fourier transform layer (reference: kapre/time_frequency.py:61-203).

    ``(batch, time, ch)`` / ``(batch, ch, time)`` float32 waveforms ->
    complex64 ``(batch, time, freq, ch)`` / ``(batch, ch, time, freq)``.
    Semantics of ``tf.signal.stft`` as kapre calls it: frames of ``win_length`` every
    ``hop_length`` samples, window from ``window_name``, right zero-pad to ``n_fft``, one-sided
    FFT; ``pad_begin`` prepends ``n_fft - hop_length`` zeros (sic, :169-172), ``pad_end`` pads
    the tail so that ``ceil(len / hop)`` frames come out.
    """

    def __init__(self, n_fft=2048, win_length=None, hop_length=None, window_name=None, pad_begin=False,
                 pad_end=False, input_data_format='default', output_data_format='default', **kwargs):
        super().__init__(**kwargs)
        for data_format in (input_data_format, output_data_format):
            backend.validate_data_format_str(data_format)  # raises before the dict unwrap, like :115-116
        input_data_format = _unwrap_format(input_data_format)
        output_data_format = _unwrap_format(output_data_format)
        if win_length is None:
            win_length = n_fft
        if hop_length is None:
            hop_length = win_length // 4  # :128-129
        self.n_fft = n_fft
        self.win_length = win_length
        self.hop_length = hop_length
        self.window_name = window_name
        self.window_fn = backend.get_window_fn(window_name)
        self.pad_begin = pad_begin
        self.pad_end = pad_end
        self.input_data_format_original = input_data_format
        self.output_data_format_original = output_data_format
        self.output_data_format = _resolve(output_data_format)
        self.input_data_format = _resolve(input_data_format)
        self._plan = None

    @property
    def plan(self) -> ops.StftPlan:
        if self._plan is None:
            self._plan = ops.StftPlan(self.n_fft, self.win_length, self.hop_length,
                                      self.window_fn(self.win_length))
        return self._plan

    def call(self, x):
        if autograd.wants_grad(x):
            return autograd.StftFn.apply(x, self)
        return ops.stft_forward(x, self.plan, self.input_data_format, self.output_data_format,
                                self.pad_begin, self.pad_end, N.OUT_COMPLEX)

    _config_fields = (
        ('n_fft', 'n_fft'),
        ('win_length', 'win_length'),
        ('hop_length', 'hop_length'),
        ('window_name', 'window_name'),
        ('pad_begin', 'pad_begin'),
        ('pad_end', 'pad_end'),
        ('input_data_format', 'input_data_format_original'),
        ('output_data_format', 'output_data_format_original'),
    )


@register_keras_serializable(package='Kapre')
class InverseSTFT(Layer):
    """Inverse STFT layer (reference: kapre/time_frequency.py:207-333).

    complex64 ``(batch, time, freq, ch)`` / ``(batch, ch, time, freq)`` -> float32 waveform of
    length ``(frames - 1) * hop_length + win_length`` (not trimmed, :213-214): irfft(n_fft),
    first ``win_length`` samples, times the dual of ``forward_window_name``
    (``tf.signal.inverse_stft_window_fn``, :278-280), overlap-add.
    """

    def __init__(self, n_fft=2048, win_length=None, hop_length=None, forward_window_name=None,
                 input_data_format='default', output_data_format='default', **kwargs):
        super().__init__(**kwargs)
        for data_format in (input_data_format, output_data_format):
            backend.validate_data_format_str(data_format)
        input_data_format = _unwrap_format(input_data_format)
        output_data_format = _unwrap_format(output_data_format)
        if win_length is None:
            win_length = n_fft
        if hop_length is None:
            hop_length = win_length // 4
        self.n_fft = n_fft
        self.win_length = win_length
        self.hop_length = hop_length
        self.forward_window_name = forward_window_name
        self.window_fn = backend.inverse_stft_window_fn(
            frame_step=hop_length, forward_window_fn=backend.get_window_fn(forward_window_name))
        self.input_data_format_original = input_data_format
        self.output_data_format_original = output_data_format
        self.output_data_format = _resolve(output_data_format)
        self.input_data_format = _resolve(input_data_format)
        self._plan = None

    @property
    def plan(self) -> ops.IstftPlan:
        if self._plan is None:
            self._plan = ops.IstftPlan(self.n_fft, self.win_length, self.hop_length,
                                       self.window_fn(self.win_length))
        return self._plan

    def call(self, x):
        if autograd.wants_grad(x):
            return autograd.IstftFn.apply(x, self)
        return ops.istft(x, self.plan, self.input_data_format, self.output_data_format)

    _config_fields = (
        ('n_fft', 'n_fft'),
        ('win_length', 'win_length'),
        ('hop_length', 'hop_length'),
        ('forward_window_name', 'forward_window_name'),
        ('input_data_format', 'input_data_format_original'),
        ('output_data_format', 'output_data_format_original'),
    )


@register_keras_serializable(package='Kapre')
class Magnitude(Layer):
    """``tf.abs`` of the complex input (reference: kapre/time_frequency.py:337-359)."""

    def call(self, x):
        if autograd.wants_grad(x) and x.is_complex():
            return autograd.MagnitudeFn.apply(x)
        return ops.magnitude(x)


@register_keras_serializable(package='Kapre')
class Phase(Layer):
    """``tf.math.angle`` of the complex input (reference: kapre/time_frequency.py:363-411).
    ``approx_atan_accuracy`` (the TFLite-compatible approximation) is accepted and stored for
    config round trips; the exact angle is returned either way."""

    def __init__(self, approx_atan_accuracy=None, **kwargs):
        super().__init__(**kwargs)
        self.approx_atan_accuracy = approx_atan_accuracy

    def call(self, x):
        return ops.phase(x)

    _config_fields = (('approx_atan_accuracy', 'approx_atan_accuracy'),)


@register_keras_serializable(package='Kapre')
class MagnitudeToDecibel(Layer):
    """Decibel scaling (reference: kapre/time_frequency.py:415-465 -> backend.py:126-194).
    Parameters are validated when the layer is called, like the reference."""

    def __init__(self, ref_value=1.0, amin=1e-5, dynamic_range=80.0, **kwargs):
        super().__init__(**kwargs)
        self.ref_value = ref_value
        self.amin = amin
        self.dynamic_range = dynamic_range

    def call(self, x):
        if autograd.wants_grad(x):
            return autograd.MagnitudeToDecibelFn.apply(x, self.ref_value, self.amin, self.dynamic_range)
        return backend.magnitude_to_decibel(x, ref_value=self.ref_value, amin=self.amin,
                                            dynamic_range=self.dynamic_range)

    _config_fields = (('amin', 'amin'), ('dynamic_range', 'dynamic_range'), ('ref_value', 'ref_value'))


@register_keras_serializable(package='Kapre')
class ApplyFilterbank(Layer):
    """Apply a (n_freq, n_filterbanks) filterbank along the frequency axis
    (reference: kapre/time_frequency.py:469-559).  ``type`` is ``'mel'`` or ``'log'``; any other
    value leaves ``self.filterbank`` undefined, as in the reference (:519-522)."""

    def __init__(self, type, filterbank_kwargs, data_format='default', **kwargs):
        super().__init__(**kwargs)
        backend.validate_data_format_str(data_format)
        data_format = _unwrap_format(data_format)
        self.type = type
        self.filterbank_kwargs = filterbank_kwargs
        if type == 'log':
            self.filterbank = backend.filterbank_log(**filterbank_kwargs)
        elif type == 'mel':
            self.filterbank = backend.filterbank_mel(**filterbank_kwargs)
        self.data_format_original = data_format
        self.data_format = _resolve(data_format)
        self.freq_axis = 3 if self.data_format == _CH_FIRST_STR else 2
        self._fb = None

    @property
    def fb(self) -> ops.Filterbank:
        if self._fb is None:
            self._fb = ops.Filterbank(np.asarray(self.filterbank))
        return self._fb

    def call(self, x):
        if autograd.wants_grad(x):
            return autograd.ApplyFilterbankFn.apply(x, self)
        return ops.apply_filterbank(x, self.fb, self.data_format)

    _config_fields = (
        ('type', 'type'),
        ('filterbank_kwargs', 'filterbank_kwargs'),
        ('data_format', 'data_format_original'),
    )


@register_keras_serializable(package='Kapre')
class Delta(Layer):
    """Local estimate of the time derivative (reference: kapre/time_frequency.py:563-644):
    ``sum_{m=-n..n} m * x[t+m] / (2 * sum_{m=1..n} m^2)`` with ``n = (win_length - 1) // 2`` on the time
    axis, the input extended by ``mode`` ('symmetric', 'reflect' or 'constant', as ``tf.pad``)."""

    def __init__(self, win_length=5, mode='symmetric', data_format='default', **kwargs):
        super().__init__(**kwargs)
        backend.validate_data_format_str(data_format)
        data_format = _unwrap_format(data_format)
        if not win_length >= 3:
            raise ValueError('win_length should be equal or bigger than 3, but it is %d' % win_length)
        if win_length % 2 != 1:
            raise ValueError('win_length should be an odd number, but it is %d' % win_length)
        if mode.lower() not in ('symmetric', 'reflect', 'constant'):
            raise ValueError('mode.lower() should be one of %sbut it is %s'
                             % (str(('symmetric', 'reflect', 'constant')), mode))
        self.data_format_original = data_format
        self.data_format = _resolve(data_format)
        self.win_length = win_length
        self.mode = mode
        self.n = (self.win_length - 1) // 2
        self.denom = 2 * sum([_n ** 2 for _n in range(1, self.n + 1, 1)])

    def call(self, x):
        return ops.delta(x, self.win_length, self.mode, self.data_format)

    _config_fields = (('win_length', 'win_length'), ('mode', 'mode'), ('data_format', 'data_format_original'))


@register_keras_serializable(package='Kapre')
class ConcatenateFrequencyMap(Layer):
    """Adds a frequency-information channel: ``linspace(0, 1, n_freq)`` along the frequency axis, broadcast over batch
    and time, concatenated on the channel axis (reference: kapre/time_frequency.py:648-744)."""

    def __init__(self, data_format='default', **kwargs):
        super().__init__(**kwargs)
        backend.validate_data_format_str(data_format)
        data_format = _unwrap_format(data_format)
        self.data_format_original = data_format
        self.data_format = _resolve(data_format)

    def call(self, x):
        return ops.concat_frequency_map(x, self.data_format)

    _config_fields = (('data_format', 'data_format_original'),)

