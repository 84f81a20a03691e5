"""The numpy decoder deep into its context, against the reference (tests/golden/long_context.npz, made by tests/golden/make_long_context.py),
and the fast teacher-forced restatement (tests/teacher_forced.py) that the GPU depth tests compare with.  CPU only.

Every other decoder fixture stops at n_past <= 42; whisper_full carries up to 224 earlier tokens into a window's prompt and decodes on
to the end of the context, 447 rows.  The controls show that each comparison would notice a plausible fault of the step kernel's
deep paths: each injected fault moves the compared quantity by at least 10x the tolerance at the checkpoint concerned."""
import os

import numpy as np
import pytest

from oracle import whisper_np as wn
from tests import teacher_forced as tf
from tests.golden.make_golden import LOGIT_STEP
from tests.golden.make_long_context import LONG_MODEL, LONG_PREFILLS, LONG_THREADS
from whisper_b200 import synth

TOL_LOGIT = 3e-2      # the GPU parity tolerance (tests/test_gpu_parity.py); the numpy restatement stays within 1e-2 of the reference
TOL_KV = 4e-3


def golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "long_context.npz"))


def logit_tol(ref_row):
    """TOL_LOGIT, scaled with the logits' spread as in the other parity tests: rows after an arbitrary (unscripted) text id run at
    rms ~23 instead of ~1."""
    return TOL_LOGIT * max(1.0, float(np.std(ref_row)) / 3.0)


@pytest.fixture(scope="module")
def model_and_cross():
    g = golden()
    m = wn.NpModel(synth.model_path(LONG_MODEL))
    mel = wn.log_mel(synth.synth_pcm(int(g["chunk"])), m.filters)
    _, ck, cv = wn.encode(m, mel, 0)
    return m, ck, cv


@pytest.fixture(scope="module")
def restated(model_and_cross):
    """restate() of the fixture's single-step pass at every thread count of the fixture (logits at the checkpoints, whole self-KV)"""
    m, ck, cv = model_and_cross
    g = golden()
    return {th: tf.restate(m, ck, cv, g["tokens"], th, logit_rows=g["checkpoints"]) for th in LONG_THREADS}


def test_ring_geometry():
    """ring_rows / v_round_rows restate decode_flow.cu's Cfg<D>::CR and RR for the model widths the tests use"""
    assert [tf.ring_rows(d) for d in (128, 384, 1024, 1280)] == [128, 128, 128, 160]
    assert [tf.v_round_rows(128, t) for t in (1, 3, 4, 5, 8, 9, 12, 16)] == [128, 128, 128, 64, 64, 42, 42, 32]


@pytest.mark.parametrize("threads", LONG_THREADS)
def test_np_decoder_at_depth_vs_golden(threads, model_and_cross):
    """NpDecoder stepped one token at a time through the whole context (n_past 0 .. 446), then the carried-over and long prompts:
    logits at every checkpoint, last-row logits of every prompt and self-KV rows against the reference."""
    m, ck, cv = model_and_cross
    g = golden()
    toks, cps = g["tokens"], g["checkpoints"].tolist()
    idx = np.arange(0, m.n_vocab, LOGIT_STEP)
    dec = wn.NpDecoder(m, ck, cv, pv_threads=threads)
    worst = 0.0
    for p in range(len(toks)):
        lg, _ = dec.decode([int(toks[p])], p)
        if p in cps:
            ref = g["t%d_logits" % threads][cps.index(p)]
            err = float(np.abs(lg[0, idx] - ref).max())
            assert err < logit_tol(ref), (p, err)
            assert abs(float(lg[0].max()) - float(g["t%d_logits_max" % threads][cps.index(p)])) < logit_tol(ref)
            worst = max(worst, err / logit_tol(ref))
    last = m.n_text_layer - 1
    assert np.abs(dec.k[[0, last]][:, cps] - g["t%d_self_k" % threads].astype(np.float32)).max() < TOL_KV
    assert np.abs(dec.v[[0, last]][:, cps] - g["t%d_self_v" % threads].astype(np.float32)).max() < TOL_KV
    for i, (n_past, n) in enumerate(LONG_PREFILLS):
        k, v = dec.k.copy(), dec.v.copy()
        lg, _ = dec.decode(toks[n_past:n_past + n].tolist(), n_past)
        dec.k, dec.v = k, v                  # every prompt sees the single steps' rows before its n_past (make_long_context.LONG_PREFILLS)
        ref = g["t%d_prefill_logits" % threads][i]
        assert np.abs(lg[-1, idx] - ref).max() < logit_tol(ref), (n_past, n)
    print("threads %d: worst logit error %.2f of the tolerance" % (threads, worst))


@pytest.mark.parametrize("threads", [1, 3, 16])
def test_restatement_is_bitwise_np_decoder(threads, model_and_cross):
    """restate() computes exactly what NpDecoder computes one call at a time: logits and the self-KV cache, bit for bit, on 40 tokens
    (16 threads: most parts of the early rows are empty)."""
    m, ck, cv = model_and_cross
    toks = golden()["tokens"][:40]
    lg, k, v = tf.restate(m, ck, cv, toks, threads)
    dec = wn.NpDecoder(m, ck, cv, pv_threads=threads)
    ref = np.stack([dec.decode([int(toks[i])], i)[0][0] for i in range(len(toks))])
    assert np.array_equal(lg, ref)
    assert np.array_equal(k, dec.k[:, :len(toks)]) and np.array_equal(v, dec.v[:, :len(toks)])


@pytest.mark.parametrize("threads", LONG_THREADS)
def test_restatement_prefill_vs_golden(threads, model_and_cross, restated):
    """restate(prefill=True): one call of N rows shares the key partition ceil((n_past + N) / threads), as the reference's does"""
    m, ck, cv = model_and_cross
    g = golden()
    toks = g["tokens"]
    idx = np.arange(0, m.n_vocab, LOGIT_STEP)
    _, k, v = restated[threads]
    for i, (n_past, n) in enumerate(LONG_PREFILLS):
        lg, _, _ = tf.restate(m, ck, cv, toks[n_past:n_past + n], threads, n_past=n_past, prefix=(k, v), prefill=True, logit_rows=[n - 1])
        ref = g["t%d_prefill_logits" % threads][i]
        assert np.abs(lg[0, idx] - ref).max() < logit_tol(ref), (n_past, n)


# (fault, thread count, checkpoint n_past it must show at, compared quantity).  Moving the own V row into another part's chain only
# re-associates f16 roundings in the logits (about 1x the tolerance), and the positional rows of the scripted model are small (2x): those
# two faults are shown on the self-KV rows the GPU tests also compare, of the last layer and of layer 0.
CONTROLS = [
    ("lost_slot", 1, 129, "logits"),     # 129 cached rows: the first one past a single slot
    ("lost_slot", 4, 385, "logits"),
    ("last_round", 1, 255, "logits"),    # 1 thread: two V rounds once n > 128; at n = 256 the second holds 126 rows
    ("last_round", 2, 385, "logits"),    # 2 threads: two rounds once n > 256
    ("own_part", 1, 446, "k_last"),
    ("own_part", 2, 258, "k_last"),
    ("own_part", 4, 446, "k_last"),
    ("pos_shift", 1, 446, "k0"),
]


@pytest.mark.parametrize("bug,threads,at,what", CONTROLS)
def test_controls_move_the_compared_quantity(bug, threads, at, what, model_and_cross, restated):
    """A restatement with the fault injected misses the reference by >= 10x the tolerance at the checkpoint concerned (logits), or on
    the stored self-KV rows up to it, while the faithful restatement stays within the tolerance there."""
    m, ck, cv = model_and_cross
    g = golden()
    cps = g["checkpoints"].tolist()
    i = cps.index(at)
    lg, k, _ = tf.restate(m, ck, cv, g["tokens"][:at + 1], threads, logit_rows=[at], bug=bug)
    if what == "logits":
        idx = np.arange(0, m.n_vocab, LOGIT_STEP)
        ref = g["t%d_logits" % threads][i]
        good, bad, tol = restated[threads][0][i, idx], lg[0, idx], logit_tol(ref)
    else:
        layer, stored = (0, 0) if what == "k0" else (m.n_text_layer - 1, 1)
        ref = g["t%d_self_k" % threads][stored][:i + 1].astype(np.float32)
        good, bad, tol = restated[threads][1][layer][cps[:i + 1]], k[layer][cps[:i + 1]], TOL_KV
    assert np.abs(good - ref).max() < tol
    margin = float(np.abs(bad - ref).max()) / tol
    print("%s at %d threads, n_past %d, %s: %.0fx the tolerance" % (bug, threads, at, what, margin))
    assert margin >= 10, margin
