"""The voice activity detector behind iContext::runCapture (whisper_b200/csrc/vad.h, host-only) against the reference's
(Whisper/Whisper/voiceActivityDetection.cpp): golden vectors generated from the reference's own code (tests/golden/vad.npz,
tests/golden/make_vad_golden.py).  Integer results (sample positions): must be identical.  The one stated difference of the pin: the
reference build the vectors come from evaluates its FFT twiddles with sinf / cosf in place of DirectXMath's XMScalarSinCos polynomial
(oracle/shim/stdafx.h)."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.golden.make_vad_golden import HELD_OUT_SEEDS, N_SIGNALS, drive, vad_signal

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "boundary", "_build", "libvad_test.so")


def _ours():
    if not os.path.exists(SHIM):
        pytest.fail("tests/boundary/_build/libvad_test.so is missing: run __graft_entry__.build()")
    return C.CDLL(SHIM)


@pytest.mark.parametrize("seed", range(N_SIGNALS))
def test_detector_matches_reference_golden(seed):
    g = np.load(os.path.join(HERE, "golden", "vad.npz"))
    got = drive(_ours(), "wvad", seed)
    assert got == g["s%d" % seed].tolist()


def test_golden_vectors_discriminate():
    g = np.load(os.path.join(HERE, "golden", "vad.npz"))
    distinct = [len(set(g[k].tolist())) for k in g.files]
    assert sum(d > 5 for d in distinct) >= N_SIGNALS // 2       # speech end positions move as the buffers grow
    assert any(g[k][-1] == 0 for k in g.files) or any(0 in g[k].tolist() for k in g.files)   # ... and "no speech" occurs


def test_detector_matches_live_reference():
    """Held-out signals: what the reference's detector returned for them when it was run (make_vad_golden.py)."""
    g = np.load(os.path.join(HERE, "golden", "vad.npz"))
    ours = _ours()
    for seed in HELD_OUT_SEEDS:
        assert drive(ours, "wvad", seed) == g["s%d" % seed].tolist(), seed


def test_features_of_known_frames():
    """Closed-form checks of the three features (voiceActivityDetection.cpp:66-125)."""
    L = _ours()
    L.wvad_create.restype = C.c_void_p
    L.wvad_features.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    h = L.wvad_create()
    out = (C.c_float * 3)()

    def feats(frame):
        frame = np.ascontiguousarray(frame, np.float32)
        L.wvad_features(h, frame.ctypes.data_as(C.POINTER(C.c_float)), out)
        return list(out)

    t = np.arange(256)
    # a pure tone in bin 16 (1 kHz): energy = rms in int16 units, dominant = 16 * 62.5 Hz, flatness large (one line over nothing)
    e, f, s = feats(0.25 * np.sin(2 * np.pi * 16 * t / 256))
    assert abs(e - 0.25 * 32768 / np.sqrt(2)) < 1.0 and f == 1000.0 and s > 30
    # an impulse has a flat spectrum: flatness 0 dB, energy = 32768 * a / 16
    x = np.zeros(256, np.float32); x[0] = 0.5
    e, f, s = feats(x)
    assert abs(e - 0.5 * 32768 / 16) < 1e-2 and abs(s) < 1e-3
    # digital silence: zero energy, bin 0, flatness NaN (0 / 0) exactly like the reference's arithmetic
    e, f, s = feats(np.zeros(256, np.float32))
    assert e == 0.0 and f == 0.0 and np.isnan(s)
    L.wvad_destroy.argtypes = [C.c_void_p]
    L.wvad_destroy(h)
