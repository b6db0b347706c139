"""GPU tier of the backward path: the layers' gradients (CUDA backward kernels through torch.autograd) against the
float64 VJPs of tests/grad_oracle.py, plus the properties the kernels promise (adjoint identities, determinism,
stride-0 upstream gradients, unchanged no-grad path).

Tolerances: 1e-5 of the largest reference gradient for the linear ops (float32 FFTs of a few thousand terms), 1e-4 for
chains through the decibel layer (its 1/x factor amplifies float32 rounding of small magnitudes)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import grad_oracle as GO  # noqa: E402
import oracle  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FMTS = ['channels_last', 'channels_first']


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('needs a GPU')
    return torch


def _wave(rng, B, C, L, fmt):
    x = rng.standard_normal((B, C, L)).astype(np.float32)
    return np.ascontiguousarray(np.transpose(x, (0, 2, 1))) if fmt == 'channels_last' else x


def _close(got, ref, rel):
    ref = np.asarray(ref)
    err = np.abs(np.asarray(got, dtype=ref.dtype) - ref).max()
    assert err <= rel * np.abs(ref).max(), (err, np.abs(ref).max())


STFT_GRID = [
    # n_fft, win, hop, pad_begin, pad_end
    (256, 256, 64, False, False), (512, 400, 128, True, True), (1024, 1024, 256, True, False),
    (2048, 2048, 512, False, True), (400, 400, 160, True, True), (1000, 1000, 250, False, True),
    (75, 60, 25, True, False), (256, 200, 300, False, True), (512, 600, 128, False, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize('C', [1, 3])
@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('cfg', STFT_GRID)
def test_stft_gradient(cfg, fmt, C):
    torch = _torch()
    import kapre_b200 as K
    n_fft, win, hop, pb, pe = cfg
    rng = np.random.default_rng(0)
    x = _wave(rng, 2, C, 4000, fmt)
    layer = K.STFT(n_fft=n_fft, win_length=win, hop_length=hop, window_name='hann_window', pad_begin=pb, pad_end=pe,
                   input_data_format=fmt, output_data_format=fmt)
    xt = torch.from_numpy(x).cuda().requires_grad_()
    y = layer(xt)
    G = (rng.standard_normal(tuple(y.shape)) + 1j * rng.standard_normal(tuple(y.shape))).astype(np.complex64)
    (y.real * torch.from_numpy(G.real).cuda() + y.imag * torch.from_numpy(G.imag).cuda()).sum().backward()
    ref = GO.stft_layer_vjp(x.shape, G, n_fft, win, hop, 'hann_window', pb, pe, fmt, fmt)
    assert xt.grad.shape == xt.shape and xt.grad.dtype == xt.dtype
    _close(xt.grad.cpu().numpy(), ref, 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('n_fft,win,hop', [(256, 256, 64), (1024, 1024, 256), (400, 400, 100), (1000, 1000, 250),
                                           (75, 75, 25), (512, 300, 128)])
def test_istft_gradient(n_fft, win, hop, fmt):
    torch = _torch()
    import kapre_b200 as K
    rng = np.random.default_rng(1)
    T, C, F = 20, 2, n_fft // 2 + 1
    shape = (2, T, F, C) if fmt == 'channels_last' else (2, C, T, F)
    X = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    layer = K.InverseSTFT(n_fft=n_fft, win_length=win, hop_length=hop, forward_window_name='hann_window',
                          input_data_format=fmt, output_data_format=fmt)
    Xt = torch.from_numpy(X).cuda().requires_grad_()
    y = layer(Xt)
    g = rng.standard_normal(tuple(y.shape)).astype(np.float32)
    (y * torch.from_numpy(g).cuda()).sum().backward()
    ref = GO.istft_layer_vjp(g, n_fft, win, hop, 'hann_window', T, fmt, fmt)
    _close(Xt.grad.cpu().numpy(), ref, 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('fb_type', ['mel', 'log'])
@pytest.mark.parametrize('fmt', FMTS)
def test_magnitude_filterbank_decibel_gradients(fmt, fb_type):
    torch = _torch()
    import kapre_b200 as K
    rng = np.random.default_rng(2)
    shape = (2, 30, 513, 2) if fmt == 'channels_last' else (2, 2, 30, 513)
    X = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    X.flat[5] = 0
    Xt = torch.from_numpy(X).cuda().requires_grad_()
    m = K.Magnitude()(Xt)
    g = rng.standard_normal(shape).astype(np.float32)
    (m * torch.from_numpy(g).cuda()).sum().backward()
    _close(Xt.grad.cpu().numpy(), GO.magnitude_vjp(X, g), 1e-5)
    kw = dict(sample_rate=16000, n_freq=513) if fb_type == 'mel' else dict(sample_rate=16000, n_freq=513, n_bins=84)
    fbl = K.ApplyFilterbank(fb_type, kw, data_format=fmt)
    a = rng.uniform(0, 1, shape).astype(np.float32)
    at = torch.from_numpy(a).cuda().requires_grad_()
    z = fbl(at)
    gz = rng.standard_normal(tuple(z.shape)).astype(np.float32)
    (z * torch.from_numpy(gz).cuda()).sum().backward()
    _close(at.grad.cpu().numpy(), GO.apply_filterbank_vjp(gz, np.asarray(fbl.filterbank), fmt), 1e-5)
    # decibel layer on data with silence: the clamp binds
    d = (rng.uniform(0, 1, (3, 40, 64)) ** 4).astype(np.float32)
    d[:, 10:30] = 0.0
    dt = torch.from_numpy(d).cuda().requires_grad_()
    yd = K.MagnitudeToDecibel(dynamic_range=40.0)(dt)
    gd = rng.standard_normal(d.shape).astype(np.float32)
    (yd * torch.from_numpy(gd).cuda()).sum().backward()
    _close(dt.grad.cpu().numpy(), GO.magnitude_to_decibel_vjp(d, gd, dynamic_range=40.0), 1e-4)


def _mel_layer(K, fmt, n_fft=1024, hop=256, fuse=True, db=True, n_mels=128):
    layer = K.get_melspectrogram_layer(n_fft=n_fft, hop_length=hop, sample_rate=16000, n_mels=n_mels,
                                       return_decibel=db, input_data_format=fmt, output_data_format=fmt)
    layer.fuse = fuse
    return layer


def _tone(B, C, L, fmt):
    t = np.arange(L) / 16000.0
    rng = np.random.default_rng(3)
    x = np.sin(2 * np.pi * 440 * t)[None, None] * (1 + rng.uniform(0, 1, (B, C, 1))) + 0.05 * rng.standard_normal((B, C, L))
    x[..., L // 3:L // 2] = 0.0                                   # digital silence: the dB clamp binds
    x = x.astype(np.float32)
    return np.ascontiguousarray(np.transpose(x, (0, 2, 1))) if fmt == 'channels_last' else x


@pytest.mark.gpu
@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('n_fft,hop', [(1024, 256), (400, 160)])
def test_logmel_gradient_fused_and_unfused(fmt, n_fft, hop):
    torch = _torch()
    import kapre_b200 as K
    x = _tone(2, 2, 16000, fmt)
    kw = dict(n_fft=n_fft, hop_length=hop, sample_rate=16000, n_mels=64, return_decibel=True, input_data_format=fmt,
              output_data_format=fmt)
    y_ref = oracle.melspectrogram_layer(x, **kw)
    g = np.random.default_rng(4).standard_normal(y_ref.shape).astype(np.float32)
    ref = GO.melspectrogram_vjp(x, g, **kw)
    grads = []
    for fuse in (True, False):
        xt = torch.from_numpy(x).cuda().requires_grad_()
        y = _mel_layer(K, fmt, n_fft, hop, fuse, n_mels=64)(xt)
        (y * torch.from_numpy(g).cuda()).sum().backward()
        grads.append(xt.grad.cpu().numpy())
        _close(grads[-1], ref, 1e-4)
    _close(grads[0], grads[1], 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['mag', 'mag_db', 'fb', 'fb_db'])
def test_fused_and_unfused_gradients_agree(mode):
    torch = _torch()
    import kapre_b200 as K
    fmt = 'channels_first'
    x = _tone(2, 1, 12000, fmt)
    out = []
    for fuse in (True, False):
        if mode.startswith('fb'):
            layer = _mel_layer(K, fmt, 512, 128, fuse, db=mode.endswith('db'), n_mels=40)
        else:
            layer = K.get_stft_magnitude_layer(n_fft=512, hop_length=128, return_decibel=mode.endswith('db'),
                                               input_data_format=fmt, output_data_format=fmt)
            layer.fuse = fuse
        xt = torch.from_numpy(x).cuda().requires_grad_()
        y = layer(xt)
        g = torch.from_numpy(np.random.default_rng(5).standard_normal(tuple(y.shape)).astype(np.float32)).cuda()
        (y * g).sum().backward()
        out.append(xt.grad.cpu().numpy())
    _close(out[0], out[1], 1e-4)


@pytest.mark.gpu
def test_adjoint_identities_at_cfg2_size():
    """<STFT x, G> = <x, STFT^T G> and <ISTFT X, g> = <X, ISTFT^T g> at B256 x 5 s, n_fft 1024, hop 256."""
    torch = _torch()
    import kapre_b200 as K
    from kapre_b200 import _native as N, ops
    B, L = 256, 80000
    gen = torch.Generator(device='cuda').manual_seed(0)
    x = torch.randn((B, L, 1), device='cuda', generator=gen)
    stft = K.STFT(n_fft=1024, hop_length=256, window_name='hann_window', input_data_format='channels_last',
                  output_data_format='channels_last')
    Y = stft(x)
    G = torch.randn(Y.shape, dtype=torch.complex64, device='cuda', generator=gen)
    gx = ops.stft_backward(G, stft.plan, 'channels_last', 'channels_last', False, False, L)
    lhs = (Y.real.double() * G.real.double() + Y.imag.double() * G.imag.double()).sum()
    rhs = (x.double() * gx.double()).sum()
    assert abs(float(lhs - rhs)) <= 1e-5 * float(x.double().norm() * G.abs().double().norm())
    ist = K.InverseSTFT(n_fft=1024, hop_length=256, forward_window_name='hann_window', input_data_format='channels_last',
                        output_data_format='channels_last')
    yw = ist(G)
    g = torch.randn(yw.shape, device='cuda', generator=gen)
    GX = ops.istft_backward(g, ist.plan, 'channels_last', 'channels_last', G.shape[1])
    lhs = (yw.double() * g.double()).sum()
    # the istft reads only Re of bins 0 and N/2: its adjoint has 0 there, so compare on what it reads
    Gr = G.clone()
    Gr[:, :, 0] = Gr[:, :, 0].real.to(torch.complex64)
    Gr[:, :, -1] = Gr[:, :, -1].real.to(torch.complex64)
    rhs = (Gr.real.double() * GX.real.double() + Gr.imag.double() * GX.imag.double()).sum()
    assert abs(float(lhs - rhs)) <= 1e-5 * float(G.abs().double().norm() * g.double().norm())
    del N


@pytest.mark.gpu
def test_perfect_reconstruction_pair_gradient():
    torch = _torch()
    import kapre_b200 as K
    stft, istft = K.get_perfectly_reconstructing_stft_istft(512, 128, 'channels_last', 'channels_last')
    rng = np.random.default_rng(6)
    X = stft(torch.from_numpy(_wave(rng, 2, 1, 8000, 'channels_last')).cuda()).detach().requires_grad_()
    y = istft(X)
    g = rng.standard_normal(tuple(y.shape)).astype(np.float32)
    (y * torch.from_numpy(g).cuda()).sum().backward()
    ref = GO.istft_layer_vjp(g, 512, 512, 128, istft.forward_window_name, X.shape[1], 'channels_last', 'channels_last')
    _close(X.grad.cpu().numpy(), ref, 1e-5)


@pytest.mark.gpu
def test_sum_backward_stride0_and_determinism():
    torch = _torch()
    import kapre_b200 as K
    x = torch.from_numpy(_tone(4, 1, 16000, 'channels_last')).cuda()
    layer = _mel_layer(K, 'channels_last', 512, 128, n_mels=64)
    grads = []
    for _ in range(2):
        xt = x.clone().requires_grad_()
        layer(xt).sum().backward()                                   # upstream gradient: expanded, all strides 0
        grads.append(xt.grad.clone())
    assert torch.isfinite(grads[0]).all()
    assert torch.equal(grads[0], grads[1])
    ref = GO.melspectrogram_vjp(x.cpu().numpy(), np.ones(tuple(layer(x).shape)), n_fft=512, hop_length=128,
                                sample_rate=16000, n_mels=64, return_decibel=True, input_data_format='channels_last',
                                output_data_format='channels_last')
    _close(grads[0].cpu().numpy(), ref, 1e-4)
    st = K.STFT(n_fft=256, hop_length=64, input_data_format='channels_last', output_data_format='channels_last')
    xs = x[:, :3000].clone().requires_grad_()
    st(xs).abs().sum().backward()
    assert torch.isfinite(xs.grad).all()


@pytest.mark.gpu
def test_no_behaviour_change_without_grad():
    torch = _torch()
    import kapre_b200 as K
    from kapre_b200 import _native as N
    x = torch.from_numpy(_tone(4, 1, 16000, 'channels_last')).cuda()
    layer = _mel_layer(K, 'channels_last', 512, 128, n_mels=64)
    torch.cuda.synchronize()
    c0 = N.launch_count()
    y0 = layer(x)
    c1 = N.launch_count()
    with torch.no_grad():
        y1 = layer(x.clone().requires_grad_())
    c2 = N.launch_count()
    y2 = layer(x.clone().requires_grad_())
    c3 = N.launch_count()
    assert y0.grad_fn is None and y2.grad_fn is not None
    assert c1 - c0 == c2 - c1 == c3 - c2
    assert torch.equal(y0, y1) and torch.equal(y0, y2.detach())
    for l in (K.STFT(n_fft=512, hop_length=128, input_data_format='channels_last', output_data_format='channels_last'),):
        a = l(x)
        b = l(x.clone().requires_grad_())
        assert torch.equal(a, b.detach())


@pytest.mark.skipif(shutil.which('cuobjdump') is None or not os.path.exists(
    os.path.join(ROOT, 'kapre_b200', '_lib', 'libkapre_b200.so')), reason='needs cuobjdump and the built library')
def test_backward_kernel_resources():
    """The adjoint instantiations of the streaming inverse kernel fit its launch bounds (128 threads x 4 CTAs: 128
    registers) without meaningful spills; the new kernels do not spill."""
    import re
    out = subprocess.run(['cuobjdump', '-res-usage', os.path.join(ROOT, 'kapre_b200', '_lib', 'libkapre_b200.so')],
                         capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.search(r'Function (\S+):', line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r'REG:(\d+) STACK:(\d+)', line)
        if m and cur:
            res[cur] = (int(m.group(1)), int(m.group(2)))
            cur = None
    adj = {k: v for k, v in res.items() if re.search(r'kb_istft2_kernelILi\d+ELb1E', k)}
    assert len(adj) == 4
    for name, (regs, stack) in adj.items():
        assert regs <= 128 and stack <= 64, (name, regs, stack)
    for key in ('kb_specvjp_kernel', 'kb_dbstat_kernel', 'kb_db_backward_kernel', 'kb_istft_grad_edges_kernel'):
        found = [v for k, v in res.items() if key in k]
        assert found and all(stack == 0 for _, stack in found), (key, found)


@pytest.mark.gpu
@pytest.mark.parametrize('n_fft,hop', [(1024, 256), (256, 64)])
def test_stft_gradient_pad_begin_many_tiles(n_fft, hop):
    """pad_begin on long signals: many streaming tiles per signal, the first of which starts inside the dropped prefix."""
    torch = _torch()
    import kapre_b200 as K
    rng = np.random.default_rng(7)
    x = _wave(rng, 8, 1, 80000, 'channels_last')
    layer = K.STFT(n_fft=n_fft, hop_length=hop, window_name='hann_window', pad_begin=True, pad_end=True,
                   input_data_format='channels_last', output_data_format='channels_last')
    xt = torch.from_numpy(x).cuda().requires_grad_()
    y = layer(xt)
    G = (rng.standard_normal(tuple(y.shape)) + 1j * rng.standard_normal(tuple(y.shape))).astype(np.complex64)
    (y.real * torch.from_numpy(G.real).cuda() + y.imag * torch.from_numpy(G.imag).cuda()).sum().backward()
    ref = GO.stft_layer_vjp(x.shape, G, n_fft, n_fft, hop, 'hann_window', True, True, 'channels_last', 'channels_last')
    _close(xt.grad.cpu().numpy(), ref, 1e-5)
