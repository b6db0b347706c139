"""Generates tests/golden/kapre_ref_cases.npz + kapre_ref_cases.json by RUNNING THE REFERENCE.

Run in the build container only (``python tests/golden/make_golden_ref.py``): it imports the
unmodified sources under /root/reference/kapre with tf_standin.py registered in place of TensorFlow /
Keras / librosa (neither is installed here), feeds float64 inputs through the reference's own layers
and composed models, and stores what they return (as float32 / complex64).  See tf_standin.py for
what this does and does not pin: kapre's own code is executed line by line; the inside of
``tf.signal`` / ``librosa`` is the stand-in's re-statement (cross-checked in make_golden.py), except
for the ``stft_tflite`` cases, where the reference's own DFT-matrix STFT (float32, elementary ops only,
kapre/tflite_compatible_stft.py:153-192) provides the spectrum.

The manifest lists, per case, the layer / factory name, its keyword arguments and the input key, so
tests/test_ref_golden.py can drive the oracle and the CUDA path through the same cases.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import tf_standin  # noqa: E402

tf_standin.install()
sys.path.insert(0, '/root/reference')
import kapre  # noqa: E402  (the reference package)
from kapre import backend as KB  # noqa: E402
from kapre import composed as KC  # noqa: E402
from kapre.time_frequency_tflite import STFTTflite  # noqa: E402

assert kapre.__file__.startswith('/root/reference/'), kapre.__file__

REF_FIXTURE = '/root/reference/tests/speech_test_file.npz'


def main():
    rng = np.random.default_rng(20240917)
    speech = np.load(REF_FIXTURE)['audio_data'].astype(np.float32)[:4000]
    inputs = {
        'noise_cl': rng.uniform(-1, 1, size=(2, 3000, 2)).astype(np.float32),      # (b, t, ch)
        'speech_cl': np.stack([speech, speech[::-1]], 0)[:, :, None].astype(np.float32),
        'tone_cl': (0.5 * np.sin(2 * np.pi * 440.0 / 16000 * np.arange(3000)))[None, :, None].astype(np.float32),
    }
    inputs['noise_cf'] = np.ascontiguousarray(np.transpose(inputs['noise_cl'], (0, 2, 1)))
    out = dict(('in_' + k, v) for k, v in inputs.items())
    manifest = []

    def record(key, kind, kwargs, in_key, value, **extra):
        value = np.asarray(value)
        value = value.astype(np.complex64 if np.iscomplexobj(value) else np.float32)
        out[key] = value
        manifest.append(dict(key=key, kind=kind, kwargs=kwargs, input=in_key, shape=list(value.shape), **extra))

    def x64(k):
        return inputs[k].astype(np.float64)

    # ---- STFT layer: kapre/time_frequency.py:61-203 ------------------------------------------------
    stft_cases = [
        dict(n_fft=512, hop_length=128),
        dict(n_fft=512, win_length=400, hop_length=160, window_name='hamming_window', pad_end=True),
        dict(n_fft=1024, hop_length=256, pad_begin=True),
        dict(n_fft=1000, win_length=512, hop_length=250, pad_end=True),
        dict(n_fft=256, hop_length=64, window_name='kaiser_window', pad_begin=True, pad_end=True),
        dict(n_fft=512, hop_length=256, window_name='vorbis_window'),
        dict(n_fft=2048, hop_length=1024, window_name='kaiser_bessel_derived_window'),
    ]
    for i, kw in enumerate(stft_cases):
        for in_key, fmts in (('noise_cl', ('channels_last', 'channels_last')),
                             ('noise_cf', ('channels_first', 'channels_first')),
                             ('noise_cl', ('channels_last', 'channels_first'))):
            if i > 1 and fmts[0] != fmts[1]:
                continue
            kwargs = dict(kw, input_data_format=fmts[0], output_data_format=fmts[1])
            y = kapre.STFT(**kwargs)(x64(in_key))
            record('stft_%d_%s' % (i, fmts[0][9] + fmts[1][9]), 'STFT', kwargs, in_key, y)

    # ---- the reference's own DFT-matrix STFT (float32): kapre/time_frequency_tflite.py, tflite_compatible_stft.py
    for i, kw in enumerate([dict(n_fft=512, hop_length=128), dict(n_fft=1000, win_length=512, hop_length=250,
                                                                   pad_end=True)]):
        kwargs = dict(kw, input_data_format='channels_last', output_data_format='channels_last')
        y = STFTTflite(**kwargs)(inputs['speech_cl'][:1])      # batch size 1 only (tflite restriction)
        record('stft_tflite_%d' % i, 'STFTTflite', kwargs, 'speech_cl', y[..., 0] + 1j * y[..., 1], batch=1)

    # ---- Magnitude / Phase / MagnitudeToDecibel: :336-465, backend.py:126-195 --------------------
    s = kapre.STFT(n_fft=512, hop_length=128)(x64('speech_cl'))
    record('magnitude_0', 'Magnitude', {}, 'stft:speech_cl:512:128', kapre.Magnitude()(s))
    record('phase_0', 'Phase', {}, 'stft:speech_cl:512:128', kapre.Phase()(s))
    for i, kw in enumerate([dict(), dict(ref_value=0.1, amin=1e-4, dynamic_range=40.0),
                            dict(ref_value=2.0, amin=1e-10, dynamic_range=120.0)]):
        record('mag2db_%d' % i, 'MagnitudeToDecibel', kw, 'magnitude_0', kapre.MagnitudeToDecibel(**kw)(np.abs(s)))
    # non-batch input: the maximum is taken over everything (backend.py:178-181)
    record('mag2db_1d', 'backend.magnitude_to_decibel', dict(ref_value=1.0, amin=1e-5, dynamic_range=30.0),
           'magnitude_0[0,:,5,0]', KB.magnitude_to_decibel(np.abs(s)[0, :, 5, 0], 1.0, 1e-5, 30.0))

    # ---- filterbanks: backend.py:198-299 ----------------------------------------------------------
    for i, kw in enumerate([dict(sample_rate=22050, n_freq=257, n_mels=40, f_min=0.0, f_max=8000.0, htk=False,
                                 norm='slaney'),
                            dict(sample_rate=16000, n_freq=513, n_mels=128, f_min=0.0, f_max=None, htk=True,
                                 norm='slaney'),
                            dict(sample_rate=44100, n_freq=1025, n_mels=96, f_min=30.0, f_max=16000.0, htk=False,
                                 norm=None)]):
        record('fb_mel_%d' % i, 'backend.filterbank_mel', kw, None, KB.filterbank_mel(**kw))
    for i, kw in enumerate([dict(sample_rate=22050, n_freq=257, n_bins=84, bins_per_octave=12, f_min=None, spread=0.125),
                            dict(sample_rate=16000, n_freq=513, n_bins=48, bins_per_octave=24, f_min=110.0,
                                 spread=0.25)]):
        record('fb_log_%d' % i, 'backend.filterbank_log', kw, None, KB.filterbank_log(**kw))

    # ---- composed models: composed.py:42-414 -----------------------------------------------------
    comp = [
        ('get_stft_magnitude_layer', dict(n_fft=512, hop_length=128, return_decibel=True), 'noise_cl'),
        ('get_stft_magnitude_layer', dict(n_fft=1024, win_length=800, hop_length=200, pad_end=True,
                                          return_decibel=False, input_data_format='channels_first',
                                          output_data_format='channels_first'), 'noise_cf'),
        ('get_melspectrogram_layer', dict(n_fft=512, hop_length=128, sample_rate=16000, n_mels=40,
                                          return_decibel=True), 'speech_cl'),
        ('get_melspectrogram_layer', dict(n_fft=1024, hop_length=256, sample_rate=22050, n_mels=128,
                                          return_decibel=True, pad_end=True), 'noise_cl'),
        ('get_melspectrogram_layer', dict(n_fft=512, hop_length=256, sample_rate=16000, n_mels=64, mel_f_min=50.0,
                                          mel_f_max=7000.0, mel_htk=True, mel_norm=None, return_decibel=False,
                                          input_data_format='channels_first', output_data_format='channels_first'),
         'noise_cf'),
        ('get_melspectrogram_layer', dict(n_fft=2048, hop_length=1024, sample_rate=44100, n_mels=96, pad_begin=True,
                                          return_decibel=True, db_amin=1e-7, db_ref_value=0.5,
                                          db_dynamic_range=60.0, output_data_format='channels_first'), 'noise_cl'),
        ('get_log_frequency_spectrogram_layer', dict(n_fft=512, hop_length=128, sample_rate=22050,
                                                     log_n_bins=84, return_decibel=True), 'tone_cl'),
    ]
    for i, (fn, kw, in_key) in enumerate(comp):
        kw = dict(kw)
        kw.setdefault('input_data_format', 'channels_last')
        kw.setdefault('output_data_format', 'channels_last')
        model = getattr(KC, fn)(**kw)
        record('composed_%d' % i, fn, kw, in_key, model(x64(in_key)))

    # ---- get_stft_mag_phase: composed.py:420-511 (keras functional API: Input -> STFT -> Magnitude || Phase -> Concatenate)
    for i, (kw, in_key) in enumerate([
            (dict(n_fft=512, hop_length=128, return_decibel=True), 'speech_cl'),
            (dict(n_fft=1024, hop_length=256, return_decibel=False, pad_end=True), 'noise_cl'),
            (dict(n_fft=512, hop_length=256, return_decibel=True, db_dynamic_range=40.0,
                  input_data_format='channels_first', output_data_format='channels_first'), 'noise_cf')]):
        kw = dict(kw)
        kw.setdefault('input_data_format', 'channels_last')
        kw.setdefault('output_data_format', 'channels_last')
        shape = inputs[in_key].shape[1:]
        model = KC.get_stft_mag_phase(input_shape=shape, **kw)
        record('mag_phase_%d' % i, 'get_stft_mag_phase', dict(kw, input_shape=list(shape)), in_key, model(x64(in_key)))

    # ---- InverseSTFT: time_frequency.py:207-333, composed.py:417-433 -----------------------------
    for i, (kw, in_key) in enumerate([(dict(n_fft=512, hop_length=128), 'noise_cl'),
                                      (dict(n_fft=1024, win_length=1024, hop_length=256,
                                            forward_window_name='hamming_window',
                                            input_data_format='channels_first',
                                            output_data_format='channels_first'), 'noise_cf'),
                                      (dict(n_fft=512, win_length=384, hop_length=96), 'speech_cl')]):
        kw = dict(kw)
        kw.setdefault('input_data_format', 'channels_last')
        kw.setdefault('output_data_format', 'channels_last')
        fkw = dict(n_fft=kw['n_fft'], win_length=kw.get('win_length'), hop_length=kw['hop_length'],
                   window_name=kw.get('forward_window_name'), input_data_format=kw['input_data_format'],
                   output_data_format=kw['input_data_format'])
        spec = kapre.STFT(**fkw)(x64(in_key))
        record('istft_in_%d' % i, 'STFT', fkw, in_key, spec)
        record('istft_%d' % i, 'InverseSTFT', kw, 'istft_in_%d' % i, kapre.InverseSTFT(**kw)(spec))
    rkw = dict(n_fft=512, hop_length=128, waveform_data_format='channels_last', stft_data_format='channels_first')
    stft, istft = KC.get_perfectly_reconstructing_stft_istft(**rkw)
    record('roundtrip_0', 'get_perfectly_reconstructing_stft_istft', rkw, 'noise_cl', istft(stft(x64('noise_cl'))))

    # ---- adjacent layers: Delta (:563-644), Frame / Energy / LogmelToMFCC (signal.py) ----------
    mel = KC.get_melspectrogram_layer(n_fft=512, hop_length=128, sample_rate=16000, n_mels=40, return_decibel=True,
                                      input_data_format='channels_last', output_data_format='channels_last')(
        x64('speech_cl'))
    record('logmel_0', 'get_melspectrogram_layer',
           dict(n_fft=512, hop_length=128, sample_rate=16000, n_mels=40, return_decibel=True,
                input_data_format='channels_last', output_data_format='channels_last'), 'speech_cl', mel)
    for i, kw in enumerate([dict(win_length=5, mode='symmetric'), dict(win_length=3, mode='reflect'),
                            dict(win_length=9, mode='constant')]):
        kw = dict(kw, data_format='channels_last')
        record('delta_%d' % i, 'Delta', kw, 'logmel_0', kapre.Delta(**kw)(mel))
    record('mfcc_0', 'LogmelToMFCC', dict(n_mfccs=13, data_format='channels_last'), 'logmel_0',
           kapre.LogmelToMFCC(n_mfccs=13, data_format='channels_last')(mel))
    for i, kw in enumerate([dict(frame_length=400, hop_length=160, pad_end=False),
                            dict(frame_length=512, hop_length=128, pad_end=True, pad_value=0.5)]):
        kw = dict(kw, data_format='channels_last')
        record('frame_%d' % i, 'Frame', kw, 'noise_cl', kapre.Frame(**kw)(x64('noise_cl')))
    for i, kw in enumerate([dict(sample_rate=16000, ref_duration=0.1, frame_length=400, hop_length=160),
                            dict(sample_rate=22050, ref_duration=0.05, frame_length=512, hop_length=256, pad_end=True)]):
        kw = dict(kw, data_format='channels_last')
        record('energy_%d' % i, 'Energy', kw, 'noise_cl', kapre.Energy(**kw)(x64('noise_cl')))

    np.savez_compressed(os.path.join(HERE, 'kapre_ref_cases.npz'), **out)
    with open(os.path.join(HERE, 'kapre_ref_cases.json'), 'w') as f:
        json.dump(dict(generator='tests/golden/make_golden_ref.py', reference_version=kapre.__version__,
                       cases=manifest), f, indent=1)
    size = os.path.getsize(os.path.join(HERE, 'kapre_ref_cases.npz'))
    print('wrote %d cases, %.1f KiB' % (len(manifest), size / 1024.0))


if __name__ == '__main__':
    main()
