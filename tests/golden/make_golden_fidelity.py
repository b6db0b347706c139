"""Generates tests/golden/kapre_ref_fidelity.json + kapre_ref_fidelity.npz by RUNNING THE REFERENCE.

  KAPRE_REFERENCE_ROOT=<directory holding the kapre 0.4.0 package> python tests/golden/make_golden_fidelity.py

Imports the unmodified reference package over tf_standin.py (as make_golden_ref.py does) and records its answers
to the keyword sets of fidelity_cases.py, which tests/test_reference_fidelity.py puts to this repository:
* per layer keyword set: the exception type the constructor raises, or its ``get_config()``;
* per composed factory call: the layer classes in order, each with its config (arrays as their shapes);
* the ``backend.filterbank_mel`` / ``filterbank_log`` matrices, whole;
* per STFT / mel fuzz configuration: whether the reference raises, and otherwise the output's shape, max |.|,
  sum |.| and its values at SAMPLE seeded positions (float64).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import fidelity_cases as FC  # noqa: E402
import tf_standin  # noqa: E402

REF_ROOT = os.path.abspath(os.environ['KAPRE_REFERENCE_ROOT'])
tf_standin.install()
sys.path.insert(0, REF_ROOT)
import kapre as R  # noqa: E402  (the reference package)
from kapre import backend as RB  # noqa: E402
from kapre import composed as RC  # noqa: E402

assert R.__file__.startswith(REF_ROOT + os.sep), R.__file__


def _config(obj):
    cfg = obj.get_config()
    for k in ('name', 'trainable', 'dtype'):
        cfg.pop(k, None)
    return cfg


def _outcome(fn):
    try:
        return {'config': FC.encode(fn())}
    except Exception as e:  # noqa: BLE001
        return {'raises': type(e).__name__}


def _layer_list(model):
    return [(type(lay).__name__, dict((k, np.asarray(v).shape if hasattr(v, 'shape') else v)
                                      for k, v in _config(lay).items())) for lay in model.layers]


def main():
    layers, factories, filterbanks = FC.api_cases()
    out = {'generator': 'tests/golden/make_golden_fidelity.py', 'reference_version': R.__version__}
    table, index = [], {}

    def intern(v):                            # most answers recur: the records point into a table of distinct ones
        key = json.dumps(v, sort_keys=True)
        if key not in index:
            index[key] = len(table)
            table.append(v)
        return index[key]

    out['table'] = table
    out['layers'] = [intern(_outcome(lambda: _config(getattr(R, name)(**kw)))) for name, kw in layers]
    out['factories'] = [[intern(FC.encode(entry)) for entry in _layer_list(getattr(RC, fn)(**kw))]
                        for fn, kw in factories]
    fbs = [np.asarray(getattr(RB, fn)(**kw)) for fn, kw in filterbanks]
    assert all(a.dtype == np.float32 for a in fbs)
    out['filterbanks'] = [list(a.shape) for a in fbs]

    rng = np.random.default_rng(7)
    samples = {'stft': ([], []), 'mel': ([], [])}

    def digest(kind, a):
        d = dict(shape=list(a.shape), absmax=float(np.abs(a).max()) if a.size else 0.0, l1=float(np.abs(a).sum()),
                 row=None)
        if a.size:
            idx = rng.integers(0, a.size, FC.SAMPLE)
            d['row'] = len(samples[kind][0])
            samples[kind][0].append(idx)
            samples[kind][1].append(a.reshape(-1)[idx])
        return d

    out['fuzz'] = []
    for kw, x, mk in FC.fuzz_cases():
        try:
            a = R.STFT(**kw)(x)
        except Exception as e:  # noqa: BLE001
            out['fuzz'].append({'stft': {'raises': type(e).__name__}, 'mel': None})
            continue
        rec = {'stft': digest('stft', a), 'mel': None}
        if a.size and mk is not None:
            rec['mel'] = digest('mel', np.asarray(RC.get_melspectrogram_layer(**mk)(x)))
        out['fuzz'].append(rec)

    np.savez_compressed(os.path.join(HERE, 'kapre_ref_fidelity.npz'),
                        filterbanks=np.concatenate([a.reshape(-1) for a in fbs]),
                        stft_idx=np.stack(samples['stft'][0]).astype(np.int32),
                        stft_val=np.stack(samples['stft'][1]).astype(np.complex128),
                        mel_idx=np.stack(samples['mel'][0]).astype(np.int32),
                        mel_val=np.stack(samples['mel'][1]).astype(np.float64))
    with open(os.path.join(HERE, 'kapre_ref_fidelity.json'), 'w') as f:
        json.dump(out, f, separators=(',', ':'))
        f.write('\n')
    print('%d layer keyword sets, %d factory calls, %d filterbanks, %d fuzz configurations (%d raise)'
          % (len(layers), len(factories), len(fbs), len(out['fuzz']),
             sum('raises' in r['stft'] for r in out['fuzz'])))


if __name__ == '__main__':
    main()
