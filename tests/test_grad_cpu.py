"""CPU tier of the backward path: the float64 VJPs of tests/grad_oracle.py against central finite differences of the
oracle forward, and the backward kernel bodies (run on the CPU through tests/emu) against those VJPs."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import emu_grad as E  # noqa: E402
import grad_oracle as GO  # noqa: E402
import oracle  # noqa: E402

FMTS = ['channels_last', 'channels_first']


def _wave(rng, B, C, L, fmt):
    x = rng.standard_normal((B, C, L))
    return np.transpose(x, (0, 2, 1)).copy() if fmt == 'channels_last' else x


def _fd_check(f, vjp_val, x, g, eps=1e-6, rtol=1e-6, complex_input=False, seed=0):
    """<vjp, v> against (f(x + eps v) - f(x - eps v)) . g / (2 eps) for a random direction v."""
    rng = np.random.default_rng(seed)
    v = rng.standard_normal(np.shape(x))
    if complex_input:
        v = v + 1j * rng.standard_normal(np.shape(x))
    fd = np.sum((f(x + eps * v) - f(x - eps * v)) * g) / (2 * eps)
    an = np.sum(np.real(vjp_val) * np.real(v)) + (np.sum(np.imag(vjp_val) * np.imag(v)) if complex_input else 0.0)
    scale = np.sqrt(np.sum(np.abs(vjp_val) ** 2) * np.sum(np.abs(v) ** 2))
    assert abs(fd - an) <= rtol * scale, (fd, an, scale)


STFT_CASES = [
    # n_fft, win, hop, pad_begin, pad_end, L
    (16, 16, 4, False, False, 61),
    (16, 12, 4, True, True, 53),       # win < n_fft
    (16, 24, 6, False, True, 70),      # win > n_fft
    (16, 6, 9, False, False, 64),      # hop > win: uncovered gaps
    (15, 15, 5, True, False, 47),      # odd n_fft
    (75, 75, 25, False, True, 260),
]


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('C', [1, 3])
@pytest.mark.parametrize('case', STFT_CASES)
def test_stft_vjp_finite_differences(case, C, fmt):
    n_fft, win, hop, pb, pe, L = case
    rng = np.random.default_rng(1)
    x = _wave(rng, 2, C, L, fmt)
    kw = dict(n_fft=n_fft, win_length=win, hop_length=hop, window_name='hann_window', pad_begin=pb, pad_end=pe,
              input_data_format=fmt, output_data_format=fmt)
    y = oracle.stft_layer(x, **kw)
    G = rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape)
    f = lambda z: oracle.stft_layer(z, **kw)  # noqa: E731
    gx = GO.stft_layer_vjp(x.shape, G, **kw)
    assert gx.shape == x.shape
    # <f(x), G>_R = sum Re f Re G + Im f Im G is linear: its exact directional derivative checks the VJP
    _fd_check(lambda z: np.concatenate([np.real(f(z)).ravel(), np.imag(f(z)).ravel()]), gx, x,
              np.concatenate([np.real(G).ravel(), np.imag(G).ravel()]))
    if hop > win:   # samples no frame reads get no gradient
        Lp = L + ((n_fft - hop) if pb else 0)
        cov = np.zeros(Lp, bool)
        for t in range(y.shape[1] if fmt == 'channels_last' else y.shape[2]):
            cov[t * hop:t * hop + min(win, n_fft)] = True
        cov = cov[(n_fft - hop) if pb else 0:]
        gl = gx[0, :, 0] if fmt == 'channels_last' else gx[0, 0]
        assert np.all(gl[~cov[:L]] == 0)


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('n_fft,win,hop', [(16, 16, 4), (15, 10, 5), (16, 20, 8), (75, 75, 25)])
def test_istft_vjp_finite_differences(n_fft, win, hop, fmt):
    rng = np.random.default_rng(2)
    T, C = 5, 3 if fmt == 'channels_first' else 1
    F = n_fft // 2 + 1
    shape = (2, T, F, C) if fmt == 'channels_last' else (2, C, T, F)
    X = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    kw = dict(n_fft=n_fft, win_length=win, hop_length=hop, forward_window_name='hann_window', input_data_format=fmt,
              output_data_format=fmt)
    f = lambda z: oracle.istft_layer(z, **kw)  # noqa: E731
    g = rng.standard_normal(f(X).shape)
    G = GO.istft_layer_vjp(g, frames=T, **kw)
    assert G.shape == X.shape
    _fd_check(f, G, X, g, complex_input=True)
    bins = G[:, :, [0, -1] if n_fft % 2 == 0 else [0], :] if fmt == 'channels_last' else G[..., [0, -1] if n_fft % 2 == 0 else [0]]
    assert np.all(np.imag(bins) == 0)


def test_magnitude_and_filterbank_vjps():
    rng = np.random.default_rng(3)
    X = rng.standard_normal((2, 3, 4, 9)) + 1j * rng.standard_normal((2, 3, 4, 9))
    X[0, 0, 0, 0] = 0
    g = rng.standard_normal(X.shape)
    G = GO.magnitude_vjp(X, g)
    assert G[0, 0, 0, 0] == 0
    Xn = X.copy()
    Xn[0, 0, 0, 0] = 1.0     # |.| is not differentiable at 0: check elsewhere
    _fd_check(np.abs, GO.magnitude_vjp(Xn, g), Xn, g, complex_input=True)
    for fmt in FMTS:
        x = rng.standard_normal((2, 5, 9, 3)) if fmt == 'channels_last' else rng.standard_normal((2, 3, 5, 9))
        fb = rng.uniform(0, 1, (9, 4))
        y = oracle.apply_filterbank(x, fb, fmt)
        g = rng.standard_normal(y.shape)
        _fd_check(lambda z: oracle.apply_filterbank(z, fb, fmt), GO.apply_filterbank_vjp(g, fb, fmt), x, g)


def _tone_with_silence(L, C, fmt, sr=8000):
    t = np.arange(L) / sr
    x = np.sin(2 * np.pi * 440 * t) + 0.05 * np.random.default_rng(11).standard_normal(L)   # noise: no near-tied maxima
    x[L // 3:2 * L // 3] = 0.0                                    # digital silence: the dB clamp binds
    x = np.stack([x * (1 + 0.1 * c) for c in range(C)], 0)[None]
    return np.transpose(x, (0, 2, 1)).copy() if fmt == 'channels_last' else x


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('C', [1, 3])
def test_logmel_vjp_finite_differences_with_binding_clamp(fmt, C):
    x = _tone_with_silence(1200, C, fmt)
    kw = dict(n_fft=64, hop_length=16, sample_rate=8000, n_mels=12, return_decibel=True, pad_begin=True,
              db_dynamic_range=25.0, input_data_format=fmt, output_data_format=fmt)
    y = oracle.melspectrogram_layer(x, **kw)
    thr = y.max() - 25.0
    assert np.sum(y <= thr + 1e-9) > 10                          # the clamp binds on many elements
    g = np.random.default_rng(4).standard_normal(y.shape)
    gx = GO.melspectrogram_vjp(x, g, **kw)
    _fd_check(lambda z: oracle.melspectrogram_layer(z, **kw), gx, x, g, eps=1e-7, rtol=1e-5)
    kw2 = dict(kw)
    for k in ('sample_rate', 'n_mels'):
        kw2.pop(k)
    gx2 = GO.stft_magnitude_vjp(x, g[..., :1].repeat(33, axis=-1) if fmt == 'channels_first' else
                                np.broadcast_to(g[:, :, :1, :], oracle.stft_magnitude_layer(x, **kw2).shape), **kw2)
    assert np.all(np.isfinite(gx2))


def test_db_vjp_tied_maxima_split_equally():
    """Two tied maxima share the gradient of the clamped elements equally; clamped elements get none."""
    x = np.array([[1.0, 1.0, 0.5, 1e-12, 0.0, 1e-9]])            # the last three are clamped (dynamic range 40 dB)
    g = np.array([[1.0, 2.0, 3.0, 4.0, 5.0, 6.0]])
    dx = GO.magnitude_to_decibel_vjp(x, g, dynamic_range=40.0)
    k = 10.0 / np.log(10.0)
    S = 4.0 + 5.0 + 6.0
    np.testing.assert_allclose(dx[0, :3], [(1.0 + S / 2) * k, (2.0 + S / 2) * k, 3.0 * k / 0.5], rtol=1e-12)
    assert np.all(dx[0, 3:] == 0)
    y = oracle.magnitude_to_decibel(x, dynamic_range=40.0)
    assert y[0, 0] == y[0, 1] and np.all(y[0, 3:] == y[0, 0] - 40.0)


@pytest.mark.parametrize('shape', [(3, 2, 4, 5), (7,)])
def test_db_vjp_finite_differences(shape):
    rng = np.random.default_rng(5)
    x = rng.uniform(0, 1, shape) ** 6
    x.flat[1] = 0.0
    g = rng.standard_normal(shape)
    f = lambda z: oracle.magnitude_to_decibel(np.abs(z), dynamic_range=30.0)  # noqa: E731
    _fd_check(f, GO.magnitude_to_decibel_vjp(x, g, dynamic_range=30.0), x, g, eps=1e-9, rtol=1e-5)


# ------------------------------------------------------------------------------------ emulated kernel bodies
# seg = m * FR - (R - 1) hops per tile, as the library launches the streaming body (FR = 4 warps * 32 / Q frames per
# round, R = ceil(min(win, n_fft) / hop)), and shorter tiles; tile counts that leave several tiles per emulated CTA.
# With pad_begin, a tile that overran its segment into the next one (after clamping its start to the dropped prefix)
# overwrote the next tile's first samples whenever it ran after it.
@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('n_fft,win,hop,pb,pe,L,seg', [
    (256, 256, 64, True, True, 3000, 29),
    (256, 200, 64, False, False, 4100, 61),
    (256, 300, 128, True, False, 6500, 31),      # win > n_fft
    (512, 512, 128, False, True, 9000, 13),
    (256, 100, 160, False, True, 9900, 32),      # hop > win
    # tiles shorter than one round: every tile of a signal in another emulated CTA, tile 1 before tile 0
    (256, 256, 64, True, True, 3000, 3),
    (256, 256, 64, True, True, 3000, 5),
    (512, 400, 128, True, False, 9000, 7),
])
def test_emu_stft_adjoint_streaming(n_fft, win, hop, pb, pe, L, seg, fmt):
    rng = np.random.default_rng(6)
    C = 2
    T = oracle.num_frames(L + ((n_fft - hop) if pb else 0), win, hop, pe)
    F = n_fft // 2 + 1
    shape = (2, T, F, C) if fmt == 'channels_last' else (2, C, T, F)
    G = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    w = oracle.get_window('hann_window', win)
    xshape = (2, L, C) if fmt == 'channels_last' else (2, C, L)
    ref = GO.stft_layer_vjp(xshape, G, n_fft, win, hop, 'hann_window', pb, pe, fmt, fmt)
    other = 'channels_first' if fmt == 'channels_last' else 'channels_last'
    for body_seg in (seg, 0):
        got = E.emu_stft_adjoint(G, L, n_fft, win, hop, w, pb, fmt, fmt, seg=body_seg, n_cta=4)
        np.testing.assert_allclose(got, ref, atol=1e-5 * np.abs(ref).max())
    got = E.emu_stft_adjoint(np.transpose(G, (0, 3, 1, 2) if fmt == 'channels_last' else (0, 2, 3, 1)), L, n_fft, win,
                             hop, w, pb, other, fmt, seg=seg)
    np.testing.assert_allclose(got, ref, atol=1e-5 * np.abs(ref).max())


@pytest.mark.parametrize('n_fft,win,hop,pb,pe,L', [(75, 75, 25, True, True, 400), (400, 400, 160, False, True, 1700),
                                                   (15, 10, 20, False, False, 100), (16, 16, 4, False, False, 10)])
def test_emu_stft_adjoint_direct(n_fft, win, hop, pb, pe, L):
    rng = np.random.default_rng(7)
    T = oracle.num_frames(L + ((n_fft - hop) if pb else 0), win, hop, pe)
    F = n_fft // 2 + 1
    G = (rng.standard_normal((1, 2, T, F)) + 1j * rng.standard_normal((1, 2, T, F))).astype(np.complex64)
    w = oracle.get_window('hann_window', win)
    ref = GO.stft_layer_vjp((1, 2, L), G, n_fft, win, hop, 'hann_window', pb, pe, 'channels_first', 'channels_first')
    got = E.emu_stft_adjoint(G, L, n_fft, win, hop, w, pb, 'channels_first', 'channels_first', seg=0)
    np.testing.assert_allclose(got, ref, atol=1e-5 * max(np.abs(ref).max(), 1.0))


def _stats_ref(y, g, dr):
    n = y.shape[0]
    yf, gf = y.reshape(n, -1).astype(np.float64), g.reshape(n, -1).astype(np.float64)
    out = np.zeros((n, 4))
    for i in range(n):
        mx, mn = yf[i].max(), yf[i].min()
        binds = mn <= (mx - dr) + 2 ** -20 * (abs(mx) + dr)
        out[i] = [mx, np.sum(yf[i] == mx), mn if binds else -np.inf, gf[i][yf[i] == mn].sum() if binds else 0.0]
    return out


@pytest.mark.parametrize('shape,chunks', [((3, 2, 7, 33), 1), ((2, 1, 40, 1000), 3), ((4, 1, 1, 5000), 64),
                                          ((1, 3, 9, 17), 5)])
def test_emu_db_statistics(shape, chunks):
    rng = np.random.default_rng(8)
    l = (10 * np.log10(np.maximum(rng.uniform(0, 1, shape) ** 8, 1e-5))).astype(np.float32)
    y = np.maximum(l, l.reshape(shape[0], -1).max(1)[:, None, None, None] - np.float32(60.0))
    y[0].flat[3] = y[0].max()                                      # a tie
    g = rng.standard_normal(shape).astype(np.float32)
    got = E.emu_dbstat(y, g, 60.0, chunks)
    ref = _stats_ref(y, g, 60.0)
    np.testing.assert_allclose(got[:, :3], ref[:, :3], rtol=0)
    np.testing.assert_allclose(got[:, 3], ref[:, 3], rtol=1e-5, atol=1e-4)
    assert got[0, 1] >= 2
    perm = np.random.default_rng(9).permutation(shape[0] * chunks)
    np.testing.assert_array_equal(E.emu_dbstat(y, g, 60.0, chunks, order=perm), got)   # arrival order is irrelevant
    gb = np.broadcast_to(np.float32(0.5), shape)                    # stride-0 upstream gradient
    np.testing.assert_allclose(E.emu_dbstat(y, gb, 60.0, chunks)[:, 3], _stats_ref(y, np.full(shape, 0.5), 60.0)[:, 3],
                               rtol=1e-6)


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('mode', ['MAG', 'MAG_DB', 'FB', 'FB_DB'])
def test_emu_spectral_vjp(mode, fmt):
    rng = np.random.default_rng(10)
    x = _tone_with_silence(2000, 2, fmt) + 0.01 * _wave(rng, 1, 2, 2000, fmt)
    x = np.concatenate([x, 0.5 * x[:, ::-1]], 0)
    n_fft, hop = 256, 64
    X = oracle.stft_layer(x, n_fft, n_fft, hop, 'hann_window', True, True, fmt, fmt)
    mag = np.abs(X)
    fb = oracle.filterbank_mel(8000, n_fft // 2 + 1, 20, dtype=np.float32) if mode.startswith('FB') else None
    z = oracle.apply_filterbank(mag, fb.astype(np.float64), fmt) if fb is not None else mag
    db = mode.endswith('DB')
    y = oracle.magnitude_to_decibel(z, dynamic_range=30.0).astype(np.float32) if db else None
    g = rng.standard_normal(z.shape)
    gz = GO.magnitude_to_decibel_vjp(z, g, dynamic_range=30.0) if db else g
    gm = GO.apply_filterbank_vjp(gz, fb, fmt) if fb is not None else gz
    ref = GO.magnitude_vjp(X, gm)
    stats = None
    if db:
        y4 = np.transpose(y, (0, 3, 1, 2)) if fmt == 'channels_last' else y
        g4 = np.transpose(g, (0, 3, 1, 2)) if fmt == 'channels_last' else g
        stats = E.emu_dbstat(np.ascontiguousarray(y4), np.ascontiguousarray(g4, np.float32), 30.0, 2)
        assert np.all(np.isfinite(stats[:, 2]))                     # the clamp binds in every item
    got = E.emu_specvjp(X.astype(np.complex64), g.astype(np.float32), y, fmt, fb=fb, db=db, stats=stats)
    np.testing.assert_allclose(got, ref, atol=1e-4 * np.abs(ref).max())
