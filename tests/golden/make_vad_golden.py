"""TEST INFRASTRUCTURE — golden vectors for the voice activity detector behind iContext::runCapture.

Generates tests/golden/vad.npz from the REFERENCE's own detector (Whisper/Whisper/voiceActivityDetection.cpp, compiled unmodified into
oracle/_ref/liboracle_vad.so by oracle/Makefile): for each seeded synthetic signal the detector is driven the way the capture loop
drives it — detect() on a buffer that grows by ragged blocks, with an occasional clear() — and every returned value is recorded.

    python tests/golden/make_vad_golden.py
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
N_SIGNALS = 16
# a second, disjoint set of signals, recorded the same way (tests/test_vad.py::test_detector_matches_live_reference)
HELD_OUT_SEEDS = range(100, 130)


def vad_signal(seed: int, secs: int = 12) -> np.ndarray:
    """Noise floor plus a few bursts of amplitude-modulated harmonic tone ("voiced" sound) at 16 kHz."""
    rng = np.random.default_rng(seed)
    n = 16000 * secs
    t = np.arange(n) / 16000.0
    x = rng.standard_normal(n).astype(np.float32) * rng.choice([0.0005, 0.002, 0.01])
    for _ in range(rng.integers(1, 5)):
        a = rng.uniform(0, secs - 1.5); d = rng.uniform(0.3, 2.5); f0 = rng.uniform(90, 300); amp = rng.uniform(0.02, 0.4)
        m = (t >= a) & (t < a + d)
        v = sum(np.sin(2 * np.pi * f0 * k * t + rng.uniform(0, 6)) / k for k in range(1, 12))
        env = 0.5 * (1 + np.sin(2 * np.pi * rng.uniform(2, 6) * t))
        x = x + (amp * m * env * v).astype(np.float32)
    if seed % 5 == 4:
        x[16000 * 3:16000 * 4] = 0.0        # a second of digital silence: log10(0) in the energy threshold, NaN flatness
    return x.astype(np.float32)


def schedule(seed: int, n: int):
    """(buffer lengths handed to detect(), indices after which the buffer is cleared and restarted)"""
    rng = np.random.default_rng(1000 + seed)
    lengths, clears, pos = [], [], 0
    while pos < n:
        pos = min(n, pos + int(rng.integers(100, 6000)))
        lengths.append(pos)
        if rng.random() < 0.02:
            clears.append(len(lengths) - 1)
    return lengths, clears


def drive(lib, prefix: str, seed: int):
    """Run one signal through a detector exposing <prefix>_create/_detect/_clear/_destroy; returns the list of detect() results."""
    getattr(lib, prefix + "_create").restype = C.c_void_p
    det = getattr(lib, prefix + "_detect"); det.restype = C.c_uint64; det.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_uint64]
    getattr(lib, prefix + "_clear").argtypes = [C.c_void_p]
    getattr(lib, prefix + "_destroy").argtypes = [C.c_void_p]
    x = vad_signal(seed)
    lengths, clears = schedule(seed, x.size)
    h = getattr(lib, prefix + "_create")()
    out, base = [], 0
    for i, pos in enumerate(lengths):
        seg = np.ascontiguousarray(x[base:pos])
        out.append(int(det(h, seg.ctypes.data_as(C.POINTER(C.c_float)), seg.size)))
        if i in clears:                      # what Capture does after handing a buffer to the transcriber: pcm.clear(); vad.clear()
            getattr(lib, prefix + "_clear")(h)
            base = pos
    getattr(lib, prefix + "_destroy")(h)
    return out


if __name__ == "__main__":
    ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "liboracle_vad.so"))
    data = {}
    for seed in list(range(N_SIGNALS)) + list(HELD_OUT_SEEDS):
        res = drive(ref, "ora_vad", seed)
        data["s%d" % seed] = np.asarray(res, np.int64)
        print(seed, "calls", len(res), "distinct results", len(set(res)), "last", res[-1])
    np.savez_compressed(os.path.join(HERE, "vad.npz"), **data)
