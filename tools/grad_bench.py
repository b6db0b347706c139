"""Times the backward path of the log-mel front end on the GPU and writes profiles/grad_cfg2.json.

cfg2: B256 x 5 s mono at 22.05 kHz, n_fft 1024, hop 256, 128 mel, dB, channels_last.  CUDA events around each item after
warm-up, median of `--reps` repetitions of `--iters` launches; the input (113 MB) and the recomputed spectrum (453 MB)
exceed the 126 MB L2.  Also times the n_fft 400 / hop 160 configuration, whose STFT adjoint is the direct O(n_fft)
body.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kapre_b200 as K  # noqa: E402
from kapre_b200 import _native as N, ops  # noqa: E402


def _time(fn, iters, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return float(np.median(out))


def _card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ''
    return q or torch.cuda.get_device_name()


def bench_cfg(B, L, sr, n_fft, hop, n_mels, iters, reps):
    fmt = 'channels_last'
    layer = K.get_melspectrogram_layer(n_fft=n_fft, hop_length=hop, sample_rate=sr, n_mels=n_mels,
                                       return_decibel=True, input_data_format=fmt, output_data_format=fmt)
    stft, fbl, dbl = layer.layers[0], layer.layers[2], layer.layers[3]
    gen = torch.Generator(device='cuda').manual_seed(0)
    x = torch.rand((B, L, 1), device='cuda', generator=gen) * 2 - 1
    xg = x.clone().requires_grad_()
    y = layer(x)
    g = torch.randn(y.shape, device='cuda', generator=gen)
    db = (dbl.ref_value, dbl.amin, dbl.dynamic_range)
    X = ops.stft_forward(x, stft.plan, fmt, fmt, stft.pad_begin, stft.pad_end, N.OUT_COMPLEX)
    T = X.shape[1]

    def fwd_bwd():
        xg.grad = None
        (layer(xg) * g).sum().backward()

    r = {'batch': B, 'samples': L, 'sample_rate': sr, 'n_fft': n_fft, 'hop': hop, 'n_mels': n_mels, 'frames': T}
    r['forward_ms'] = _time(lambda: layer(x), iters, reps)
    r['forward_backward_ms'] = _time(fwd_bwd, iters, reps)
    r['bwd_recompute_stft_ms'] = _time(
        lambda: ops.stft_forward(x, stft.plan, fmt, fmt, stft.pad_begin, stft.pad_end, N.OUT_COMPLEX), iters, reps)
    r['bwd_stats_and_spectral_vjp_ms'] = _time(
        lambda: ops.spectral_backward(X, g, y, N.OUT_FB_DB, fbl.fb, db, fmt, out=torch.empty_like(X)), iters, reps)
    r['bwd_stft_adjoint_ms'] = _time(
        lambda: ops.stft_backward(X, stft.plan, fmt, fmt, stft.pad_begin, stft.pad_end, L), iters, reps)
    ist = K.InverseSTFT(n_fft=n_fft, hop_length=hop, input_data_format=fmt, output_data_format=fmt)
    r['istft_inverse_same_shape_ms'] = _time(lambda: ist(X), iters, reps)
    r['spectrum_bytes'] = int(X.numel() * 8)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'grad_cfg2.json'))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('grad_bench needs a GPU')
    res = {'card': _card(), 'timing': 'CUDA events, median of %d x %d launches after warm-up' % (a.reps, a.iters),
           'cfg2': bench_cfg(256, 110250, 22050, 1024, 256, 128, a.iters, a.reps),
           'nfft400': bench_cfg(256, 80000, 16000, 400, 160, 128, max(2, a.iters // 4), a.reps)}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
