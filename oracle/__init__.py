"""CPU oracle for the kapre STFT -> |.| -> filterbank -> dB hot path (and InverseSTFT).

TEST INFRASTRUCTURE ONLY.  Nothing under ``kapre_b200/`` may import this package; only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs use it, and only as the checker / the baseline, never as the product.

PARITY PINNING STATUS: pinned by outputs of the reference's own code run in the build container,
with one stated limit.  The reference (kapre 0.4.0) is pure Python over TensorFlow + librosa;
neither is installed (no network) and the repository stores no golden output vectors (its tests
compare against librosa evaluated at test time).  ``tests/golden/make_golden_ref.py`` therefore
imports the UNMODIFIED sources under /root/reference/kapre over ``tests/golden/tf_standin.py`` -- a
NumPy stand-in for the TensorFlow / Keras / librosa entry points they call -- and records what the
reference's layers and composed models return for 55 cases (``tests/golden/kapre_ref_cases.*``);
``tests/test_ref_golden.py`` holds the oracle (CPU tier) and the CUDA path (GPU tier) to them.

* Pinned by the reference's own code: everything kapre itself does -- data-format transposes,
  ``pad_begin`` / ``pad_end`` wiring, the arguments it passes to ``tf.signal.stft`` /
  ``inverse_stft`` / ``inverse_stft_window_fn``, magnitude / phase, the decibel formula and its
  per-item clamp, the filterbank contraction, ``filterbank_log``, Delta / Frame / Energy / MFCC, the
  composed models -- and, through ``STFTTflite``, the reference's own DFT-matrix STFT
  (``kapre/tflite_compatible_stft.py``, float32, elementary ops only).
* NOT the reference: the inside of ``tf.signal.*`` and ``librosa.filters.mel``.  Those are restated in
  the stand-in from their published algorithms and cross-checked against independent
  implementations present in the container: ``torch.stft(center=False)``,
  ``torchaudio.functional.melscale_fbanks``, ``scipy.signal.get_window``, ``numpy.fft``, the
  reference's literal dB test matrix (``tests/test_backend.py:20-22``) and analytic known-answer
  tests (impulse, DC, bin-centred cosine, Parseval, STFT->ISTFT identity).

``tests/test_reference_fidelity.py`` additionally holds the oracle to the reference's outputs on random
STFT / mel configurations (including which argument combinations raise), and every layer mirror to the
reference's constructor errors and ``get_config()``: answers of the reference's own classes recorded by
``tests/golden/make_golden_fidelity.py`` in ``tests/golden/kapre_ref_fidelity.*``.

See ``tests/golden/make_golden.py`` / ``make_golden_ref.py`` for the scripts that produced the committed fixtures.
"""
from .reference import *  # noqa: F401,F403
