"""The layer mirrors and the oracle against answers recorded from the reference's own code
(tests/golden/make_golden_fidelity.py: the unmodified kapre 0.4.0 sources over tf_standin.py, stored in
tests/golden/kapre_ref_fidelity.json / .npz).  The keyword sets come from tests/golden/fidelity_cases.py;
nothing here imports the reference."""
import json
import os

import numpy as np

import kapre_b200 as M
import oracle as O
from golden import fidelity_cases as FC

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, 'golden', 'kapre_ref_fidelity.json')) as _f:
    REF = json.load(_f)
_npz = np.load(os.path.join(HERE, 'golden', 'kapre_ref_fidelity.npz'))


def _config(obj):
    cfg = obj.get_config()
    for k in ('name', 'trainable', 'dtype'):
        cfg.pop(k, None)
    return cfg


def _outcome(fn):
    try:
        return {'config': fn()}
    except Exception as e:  # noqa: BLE001
        return {'raises': type(e).__name__}


def _layer_list(model):
    return [(type(lay).__name__, dict((k, np.asarray(v).shape if hasattr(v, 'shape') else v)
                                      for k, v in _config(lay).items())) for lay in model.layers]


def test_layer_constructors_and_get_config_match_the_reference():
    """Every mirrored layer, for random keyword sets (valid and invalid), raises the exception type the reference
    raised or returns its get_config(); the composed factories build the same layer classes in the same order with
    the same configs; the filterbank matrices agree."""
    layers, factories, filterbanks = FC.api_cases()
    table = [FC.decode(v) for v in REF['table']]
    bad = []
    for (name, kw), i in zip(layers, REF['layers'], strict=True):
        got = _outcome(lambda: _config(getattr(M, name)(**kw)))
        if got != table[i]:
            bad.append(('layer differs', name, kw, table[i], got))
    for (fn, kw), rows in zip(factories, REF['factories'], strict=True):
        want = [table[i] for i in rows]
        got = _layer_list(getattr(M, fn)(**kw))
        if got != want:
            bad.append(('factory differs', fn, kw, want, got))
    flat, off = _npz['filterbanks'], 0
    for (fn, kw), shape in zip(filterbanks, REF['filterbanks'], strict=True):
        a = flat[off:off + int(np.prod(shape))].reshape(shape)
        off += a.size
        b = np.asarray(getattr(M.backend, fn)(**kw))
        if a.shape != b.shape or np.abs(a - b).max() > 2e-6 * max(1.0, np.abs(a).max()):
            bad.append((fn + ' differs', kw))
    assert off == flat.size
    assert not bad, '%d disagreements, first: %r' % (len(bad), bad[:3])


def _compare(kind, got, want, tol):
    """None if `got` matches the reference output summarised by `want` (shape, max |.|, sum |.|, sampled elements)
    within tol * max(1, max |.|) per element, else what differs."""
    got = np.asarray(got)
    if list(got.shape) != want['shape']:
        return 'shape %s, reference %s' % (got.shape, want['shape'])
    if not got.size:
        return None
    bound = tol * max(1.0, want['absmax'])
    sample = got.reshape(-1)[_npz[kind + '_idx'][want['row']]]
    err = max(abs(float(np.abs(got).max()) - want['absmax']),
              float(np.abs(sample - _npz[kind + '_val'][want['row']]).max()))
    if err > bound:
        return 'max |err| %.3g > %.3g' % (err, bound)
    if abs(float(np.abs(got).sum()) - want['l1']) > tol * want['l1']:
        return 'sum |.| %r, reference %r' % (float(np.abs(got).sum()), want['l1'])
    return None


def test_oracle_agrees_with_the_reference_code_on_random_configurations():
    """Random STFT layer configurations (and a mel factory on some): the oracle raises where the reference raised
    and otherwise returns its output."""
    bad = []
    for (kw, x, mk), rec in zip(FC.fuzz_cases(), REF['fuzz'], strict=True):
        if 'raises' in rec['stft']:
            try:
                O.stft_layer(x, **kw)
            except Exception:  # noqa: BLE001
                continue
            bad.append(('reference raised %s, oracle did not' % rec['stft']['raises'], kw))
            continue
        why = _compare('stft', O.stft_layer(x, **kw), rec['stft'], 1e-9)
        if why:
            bad.append(('STFT: ' + why, kw))
        if rec['mel'] is not None:
            why = _compare('mel', O.melspectrogram_layer(x, **mk), rec['mel'], 1e-7)
            if why:
                bad.append(('mel: ' + why, mk))
    assert not bad, '%d disagreements, first: %r' % (len(bad), bad[:3])
