"""Autograd for the hot-path layers: ``torch.autograd.Function``s over the backward kernels of the C ABI.

The layers (``STFT``, ``InverseSTFT``, ``Magnitude``, ``ApplyFilterbank``, ``MagnitudeToDecibel`` and the fused
``Sequential`` prefix) route through these only when ``torch.is_grad_enabled()`` and the input requires grad;
otherwise they run their forward kernels exactly as before.  The gradients restate TensorFlow's registered
gradients of the ops the reference calls (see include/kapre_b200.h).  Every Function is once-differentiable: the
backward kernels have no gradient of their own.

The fused backward does not keep the complex spectrum from the forward (the forward never writes it): it recomputes
it with the forward kernel, turns it into the spectrum's gradient in place (decibel statistics + spectral VJP) and
runs the STFT adjoint -- four launches.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import _native as N
from . import backend, ops


def _like(grad: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    return grad if grad.dtype == x.dtype else grad.to(x.dtype)


def wants_grad(x) -> bool:
    return isinstance(x, torch.Tensor) and torch.is_grad_enabled() and x.requires_grad


class StftFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, layer):
        ctx.layer = layer
        ctx.length = x.shape[1] if layer.input_data_format == backend._CH_LAST_STR else x.shape[2]
        ctx.x_dtype = x.dtype
        return ops.stft_forward(x, layer.plan, layer.input_data_format, layer.output_data_format, layer.pad_begin,
                                layer.pad_end, N.OUT_COMPLEX)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        s = ctx.layer
        gx = ops.stft_backward(g, s.plan, s.output_data_format, s.input_data_format, s.pad_begin, s.pad_end, ctx.length)
        return gx.to(ctx.x_dtype), None


class IstftFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, layer):
        ctx.layer = layer
        ctx.frames = X.shape[1] if layer.input_data_format == backend._CH_LAST_STR else X.shape[2]
        ctx.x_dtype = X.dtype
        return ops.istft(X, layer.plan, layer.input_data_format, layer.output_data_format)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        s = ctx.layer
        G = ops.istft_backward(g, s.plan, s.input_data_format, s.output_data_format, ctx.frames)
        return G.to(ctx.x_dtype), None


class MagnitudeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X):
        ctx.save_for_backward(X)
        return ops.magnitude(X)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        X, = ctx.saved_tensors
        return _like(ops.magnitude_backward(X, g), X)


class ApplyFilterbankFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, layer):
        ctx.layer = layer
        ctx.x_dtype = x.dtype
        return ops.apply_filterbank(x, layer.fb, layer.data_format)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        s = ctx.layer
        # g_mag = g_fb fb^T: the stand-alone filterbank kernel with the transposed matrix
        return ops.apply_filterbank(g, ops.transposed(s.fb), s.data_format).to(ctx.x_dtype), None


class MagnitudeToDecibelFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ref_value, amin, dynamic_range):
        xc = x.to(torch.float32).contiguous()
        y = backend.magnitude_to_decibel(xc, ref_value=ref_value, amin=amin, dynamic_range=dynamic_range)
        ctx.save_for_backward(xc, y)
        ctx.db = (ref_value, amin, dynamic_range)
        ctx.x_dtype = x.dtype
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        xc, y = ctx.saved_tensors
        return ops.magnitude_to_decibel_backward(xc, y, g, *ctx.db).to(ctx.x_dtype), None, None, None


class FusedSpectrogramFn(torch.autograd.Function):
    """STFT -> Magnitude [-> ApplyFilterbank] [-> MagnitudeToDecibel] in one forward launch (Sequential's fused prefix)."""

    @staticmethod
    def forward(ctx, x, stft, mode, fb, db):
        y = ops.stft_forward(x, stft.plan, stft.input_data_format, stft.output_data_format, stft.pad_begin, stft.pad_end,
                             mode, fb, db)
        ctx.stft, ctx.mode, ctx.fb, ctx.db = stft, mode, fb, db
        ctx.x_dtype = x.dtype
        ctx.save_for_backward(x, y if db is not None else None)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        x, y = ctx.saved_tensors
        s = ctx.stft
        length = x.shape[1] if s.input_data_format == backend._CH_LAST_STR else x.shape[2]
        X = ops.stft_forward(x, s.plan, s.input_data_format, s.output_data_format, s.pad_begin, s.pad_end, N.OUT_COMPLEX)
        ops.spectral_backward(X, g, y, ctx.mode, ctx.fb, ctx.db, s.output_data_format, out=X)
        gx = ops.stft_backward(X, s.plan, s.output_data_format, s.input_data_format, s.pad_begin, s.pad_end, length)
        return gx.to(ctx.x_dtype), None, None, None, None
