"""The GPU sampler (softmax + whisper_sample_best / whisper_sample_timestamp rules, kernels_decode.cu: sample_cluster_kernel) against the
reference's own sampler (Whisper/source/whisper.cpp:1875-1964) on hand-made and random distributions.

Protocol: logits -> GPU (wsp_test_sample) -> probs + sampled token, against what the reference's sampler returned when it was given
those very probability rows (oracle/_ref: ora_sample_from_probs writes a row where whisper_sample_best reads; tests/golden/sampler.npz,
make_golden.py --sampler).  ids and tids must be equal, p / pt / ptsum within 1e-6 (the reference sums in double; so does the kernel).
Exact ties are INCLUDED: the reference's top-4 comes from std::partial_sort, whose order among equal keys is an artefact of libstdc++'s
heap-select — the kernel detects a deciding tie and re-runs that very algorithm (kernels_decode.cu: emulatePartialSort), so even
all-zero probability ranges resolve identically."""
import os

import numpy as np
import pytest

from whisper_b200 import capi

pytestmark = pytest.mark.gpu

MODEL = "micro.en"          # the reference sampler's vocabulary layout (make_golden.py --sampler)
N_VOCAB, BEG, SOT, SOLM, NOT = 51864, 50363, 50257, 50361, 50362
SPECIAL4 = [BEG, SOT, SOLM, NOT]


def make_rows(seed=0):
    """(logits, force_timestamp, is_initial, label) groups.  Logit scales are chosen so that probabilities are well spread."""
    rng = np.random.default_rng(seed)
    groups = []

    def base(n, scale=3.0):
        return (rng.standard_normal((n, N_VOCAB)) * scale).astype(np.float32)

    # 1. plain random rows, three temperatures, all three sampling modes
    for scale in (1.0, 3.0, 8.0):
        groups.append((base(24, scale), False, False, "random x%.0f" % scale))
        # (at x8 a forced-timestamp row underflows EVERY timestamp probability to exactly 0 in the f16-table softmax: an all-way tie)
        groups.append((base(12, scale), True, False, "random forced-ts x%.0f" % scale))
        groups.append((base(12, scale), True, True, "random initial x%.0f" % scale))
    # 2. banned tokens (sot / solm / not) in the top 1, top 2, top 3 (whisper.cpp:1949-1956)
    lg = base(24)
    for r in range(24):
        order = [SOT, SOLM, NOT]
        rng.shuffle(order)
        k = 1 + r % 3
        for i, t in enumerate(order[:k]):
            lg[r, t] = 30.0 - i          # the k best tokens are banned ones
        lg[r, 100 + r] = 25.0 - 0.01 * r   # best admissible text token
    groups.append((lg, False, False, "banned in top-k"))
    # 3. sum of timestamp probabilities close to the best text probability, both sides (whisper.cpp:1921-1928)
    lg = np.full((32, N_VOCAB), -12.0, np.float32)
    lg += (rng.standard_normal(lg.shape) * 0.05).astype(np.float32)
    for r in range(32):
        lg[r, 77] = 4.0                                      # one text token with p ~ exp(4)
        n_ts = 20
        ts = BEG + rng.choice(1500, n_ts, replace=False)
        # 20 timestamps of equal weight whose total is exp(4) * (1 +- delta)
        delta = (r - 15.5) * 0.004
        lg[r, ts] = np.float32(4.0 + np.log((1.0 + delta) / n_ts)) + (rng.standard_normal(n_ts) * 0.02).astype(np.float32)
    groups.append((lg, False, False, "sum_ts ~ max_tx"))
    # 4. initial timestamp: the best timestamp lies beyond beg+100 and must be ignored (whisper.cpp:1902-1911)
    lg = base(16)
    for r in range(16):
        lg[r, BEG + 101 + 13 * r] = 30.0                     # (8 below the leader: far from the f16-table underflow at ~-16.6)
        lg[r, BEG + (7 * r) % 101] = 22.0
        lg[r, BEG + 100] += 5.0 if r % 2 else 0.0            # the boundary itself is admissible
    groups.append((lg, True, True, "initial cap at beg+100"))
    groups.append((lg.copy(), True, False, "same rows, not initial"))
    # 5. ties away from the top: equal logits for many tokens below the leaders, equal timestamp maxima (tid = first maximum)
    lg = np.full((16, N_VOCAB), -3.0, np.float32)
    for r in range(16):
        lg[r, 5 + r] = 6.0
        lg[r, BEG + 40 + r] = 2.0
        lg[r, BEG + 400 + r] = 2.0                            # two equal best timestamps: the lower id is reported as tid
    groups.append((lg, False, False, "ties below the top"))
    # 6. EXACT ties: logits drawn from four values (one of them deep in the underflow range), a few equal leaders, banned tokens among
    #    them.  The reference's answer is then whatever std::partial_sort( top 4 ) leaves first; the kernel re-runs that algorithm.
    for k in range(36):
        lg = rng.choice(np.array([-30.0, 0.0, 1.0, 5.0], np.float32), size=(1, N_VOCAB), p=[0.9, 0.05, 0.04, 0.01]).astype(np.float32)
        lg[0, rng.integers(0, N_VOCAB, 3)] = 6.0
        if k % 3 == 0:
            lg[0, [SOT, SOLM, NOT]] = 7.0
        if k % 4 == 0:
            lg[0, :BEG] = -30.0
            lg[0, rng.integers(0, BEG, 5)] = 2.0
        groups.append((lg, bool(k & 1), bool(k & 1) and bool(k & 2), "exact ties %d" % k))
    # 7. peaked rows (p ~ 1) and a row dominated by -inf-like logits
    lg = base(8, 1.0)
    for r in range(8):
        lg[r, [3, BEG + 5, 50256, SOT][r % 4]] = 60.0
    groups.append((lg, False, False, "peaked"))
    return groups


def test_gpu_sampler_matches_reference_rules():
    ref = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sampler.npz")))
    total = 0
    for lg, force_ts, initial, label in make_rows():
        probs, got = capi.test_sample(lg, SPECIAL4, force_ts, initial)
        assert np.allclose(probs.sum(-1), 1.0, atol=2e-5), label
        for r in range(lg.shape[0]):
            want = {k: v[total] for k, v in ref.items()}
            g = got[r]
            assert g["id"] == want["id"], (label, r, g, want)
            assert g["tid"] == want["tid"], (label, r, g, want)
            assert abs(g["p"] - want["p"]) <= 1e-6, (label, r, g, want)
            assert abs(g["ptsum"] - want["ptsum"]) <= 1e-6, (label, r, g, want)
            assert abs(g["pt"] - want["pt"]) <= 2e-6, (label, r, g, want)
            total += 1
    assert total == ref["id"].size and total >= 200


def test_sampler_close_call_switches_sides():
    """The 'sum_ts ~ max_tx' group really straddles the decision: both outcomes occur."""
    lg, force_ts, initial, _ = [g for g in make_rows() if g[3] == "sum_ts ~ max_tx"][0]
    _, got = capi.test_sample(lg, SPECIAL4, force_ts, initial)
    kinds = {t["id"] >= BEG for t in got}
    assert kinds == {True, False}
