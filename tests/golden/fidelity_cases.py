"""Keyword sets of the reference-fidelity checks (tests/test_reference_fidelity.py).

Shared by make_golden_fidelity.py, which recorded the reference's answers to them, and by the tests, which put
the same keyword sets to this repository's layers and oracle.  Pure NumPy: nothing here imports the reference.
"""
import numpy as np

LAYER_SETS = 150     # random keyword sets per layer class (valid and invalid)
FUZZ_CONFIGS = 120   # random STFT / mel configurations of the oracle check
SAMPLE = 16          # stored reference elements per fuzz output (with its shape, max |.| and sum |.|)


def api_cases(n=LAYER_SETS):
    """(layers, factories, filterbanks): lists of (name, kwargs).  ``layers`` names a layer class, ``factories`` a
    function of ``composed``, ``filterbanks`` a function of ``backend``."""
    rng = np.random.default_rng(1)

    def pick(options):
        return options[int(rng.integers(len(options)))]

    def flip():
        return bool(rng.random() < 0.5)

    layers = []
    for _ in range(n):
        fmt_i = pick(['channels_first', 'channels_last', 'default', 'weird', 3])
        fmt_o = pick(['channels_first', 'channels_last', 'default', 'weird', 3])
        n_fft = pick([256, 512, 1000])
        win, hop = pick([None, 200, 256]), pick([None, 64, 100])
        wn = pick([None, 'hann_window', 'hamming_window', 'nope'])
        layers.append(('STFT', dict(n_fft=n_fft, win_length=win, hop_length=hop, window_name=wn, pad_begin=flip(),
                                    pad_end=flip(), input_data_format=fmt_i, output_data_format=fmt_o)))
        layers.append(('InverseSTFT', dict(n_fft=n_fft, win_length=win, hop_length=hop, forward_window_name=wn,
                                           input_data_format=fmt_i, output_data_format=fmt_o)))
        layers.append(('MagnitudeToDecibel', dict(ref_value=pick([1.0, 0.1]), amin=pick([1e-5, 1e-10]),
                                                  dynamic_range=pick([80.0, 40.0]))))
        layers.append(('Delta', dict(win_length=pick([2, 3, 4, 5, 9]),
                                     mode=pick(['symmetric', 'reflect', 'constant', 'wrap', 'SYMMETRIC']),
                                     data_format=fmt_i)))
        layers.append(('Frame', dict(frame_length=pick([100, 512]), hop_length=pick([50, 200]), pad_end=flip(),
                                     pad_value=pick([0, 1.5]), data_format=fmt_i)))
        layers.append(('Energy', dict(sample_rate=pick([8000, 22050]), ref_duration=pick([0.1, 0.05]),
                                      frame_length=pick([100, 2205]), hop_length=pick([50, 1102]), pad_end=flip(),
                                      data_format=fmt_i)))
        layers.append(('LogmelToMFCC', dict(n_mfccs=pick([13, 20]), data_format=fmt_i)))
        layers.append(('Magnitude', {}))
        layers.append(('Phase', {}))
        layers.append(('ApplyFilterbank', dict(type=pick(['mel', 'log', 'tri']),
                                               filterbank_kwargs=dict(sample_rate=16000, n_freq=n_fft // 2 + 1,
                                                                      n_mels=8),
                                               data_format=fmt_i)))
    factories = []
    for _ in range(max(10, n // 5)):
        kw = dict(n_fft=pick([256, 512, 1024]), win_length=pick([None, 200]), hop_length=pick([None, 64]),
                  window_name=pick([None, 'hamming_window']), pad_begin=flip(), pad_end=flip(),
                  return_decibel=flip(), db_amin=pick([1e-5, 1e-7]), db_ref_value=pick([1.0, 0.5]),
                  db_dynamic_range=pick([80.0, 50.0]),
                  input_data_format=pick(['channels_first', 'channels_last', 'default']),
                  output_data_format=pick(['channels_first', 'channels_last', 'default']))
        factories.append(('get_stft_magnitude_layer', kw))
        factories.append(('get_melspectrogram_layer', dict(kw, sample_rate=pick([16000, 22050]), n_mels=pick([40, 128]),
                                                           mel_f_min=pick([0.0, 30.0]), mel_f_max=pick([None, 7000.0]),
                                                           mel_htk=flip(), mel_norm=pick(['slaney', None]))))
        factories.append(('get_log_frequency_spectrogram_layer',
                          dict(kw, sample_rate=22050, log_n_bins=pick([48, 84]), log_f_min=pick([None, 55.0]),
                               log_bins_per_octave=pick([12, 24]), log_spread=pick([0.125, 0.25]))))
    filterbanks = []
    for _ in range(20):
        sr, n_freq = pick([8000, 16000, 44100]), pick([129, 257, 513])
        filterbanks.append(('filterbank_mel', dict(sample_rate=sr, n_freq=n_freq, n_mels=pick([10, 40, 96]),
                                                   f_min=pick([0.0, 50.0]), f_max=pick([None, sr / 2.5]), htk=flip(),
                                                   norm=pick(['slaney', None]))))
        filterbanks.append(('filterbank_log', dict(sample_rate=sr, n_freq=n_freq, n_bins=pick([24, 60]),
                                                   bins_per_octave=pick([12, 24]), f_min=pick([None, 40.0]),
                                                   spread=pick([0.125, 0.3]))))
    return layers, factories, filterbanks


def encode(v):
    """JSON form of a get_config() value that keeps tuples apart from lists (``decode`` inverts it)."""
    if isinstance(v, tuple):
        return {'__tuple__': [encode(e) for e in v]}
    if isinstance(v, list):
        return [encode(e) for e in v]
    if isinstance(v, dict):
        return dict((k, encode(e)) for k, e in v.items())
    assert v is None or type(v) in (str, bool, int, float), (type(v), v)
    return v


def decode(v):
    if isinstance(v, dict):
        if list(v) == ['__tuple__']:
            return tuple(decode(e) for e in v['__tuple__'])
        return dict((k, decode(e)) for k, e in v.items())
    if isinstance(v, list):
        return [decode(e) for e in v]
    return v


def fuzz_cases(n=FUZZ_CONFIGS, seed=0):
    """[(STFT layer kwargs, float64 input, mel factory kwargs or None)].  Every value is drawn whatever the
    reference did with the previous configuration, so the list is the same wherever it is generated."""
    rng = np.random.default_rng(seed)
    cases = []
    for _ in range(n):
        n_fft = int(rng.choice([64, 100, 256, 500, 512]))
        win = int(rng.integers(2, n_fft + 1)) if rng.random() < 0.5 else None
        hop = int(rng.integers(1, n_fft + 1)) if rng.random() < 0.7 else None
        wname = rng.choice([None, 'hann_window', 'hamming_window', 'kaiser_window', 'vorbis_window'])
        wname = None if wname is None else str(wname)
        pb, pe = bool(rng.random() < 0.5), bool(rng.random() < 0.5)
        ifmt = str(rng.choice(['channels_first', 'channels_last', 'default']))
        ofmt = str(rng.choice(['channels_first', 'channels_last', 'default']))
        C, L = int(rng.integers(1, 4)), int(rng.integers(n_fft, 4 * n_fft + 50))
        x = rng.uniform(-1, 1, size=(2, L, C) if ifmt != 'channels_first' else (2, C, L))
        kw = dict(n_fft=n_fft, win_length=win, hop_length=hop, window_name=wname, pad_begin=pb, pad_end=pe,
                  input_data_format=ifmt, output_data_format=ofmt)
        mk = dict(kw, sample_rate=int(rng.choice([8000, 16000, 22050])), n_mels=int(rng.integers(2, 40)),
                  mel_htk=bool(rng.random() < 0.5), return_decibel=bool(rng.random() < 0.7),
                  db_dynamic_range=float(rng.choice([80.0, 30.0])))
        cases.append((kw, x, mk if rng.random() < 0.4 else None))
    return cases
