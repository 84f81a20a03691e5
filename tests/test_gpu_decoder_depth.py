"""The decoder deep into its context and at full batch width, on a B200.

whisper_full carries up to 224 earlier tokens into each window's prompt and decodes on to the end of the context, so the step kernel
(decode_flow.cu) runs with up to 447 cached rows: self-attention keys in several ring slots of CR rows, V rows in several rounds, and
with B * H > 148 (chunks x heads), two or three attention units per CTA.  These tests pin that whole operating range against the
reference (tests/golden/long_context.npz) and against the teacher-forced numpy restatement (tests/teacher_forced.py, pinned by
tests/test_decoder_depth.py).  Every test that means to run a step kernel checks from the launch counter that it did: a host-token
call adds 2 launches (tokens, flags), then 1 for a step kernel without sampling, or 2 + 8 L on the kernel-per-op path.

Controls: next to each comparison, the restatement with a plausible kernel fault injected must miss the GPU by >= 10x the tolerance
(faults are only ever injected into numpy, never into a kernel)."""
import os
import tempfile

import numpy as np
import pytest

from oracle import whisper_np as wn
from tests import teacher_forced as tf
from tests.golden.make_golden import GAP_SAFE, LOGIT_STEP
from tests.golden.make_long_context import LONG_MODEL, LONG_PREFILLS, LONG_THREADS
from whisper_b200 import capi, synth

pytestmark = pytest.mark.gpu

TOL_LOGIT, TOL_KV = 3e-2, 4e-3
WSP_E_BOUNDS = -7


def golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "long_context.npz"))


def logit_tol(ref_row):
    return TOL_LOGIT * max(1.0, float(np.std(ref_row)) / 3.0)


def expected_launches(mode, N, L):
    """launches of one host-token decode call with DECODE_NO_SAMPLE"""
    return 2 + (1 if N == 1 and mode in (1, 2) else 2 + 8 * L)


class Run:
    """one model on the GPU, and the numpy model for the restatement"""

    def __init__(self, path, batch):
        self.m = capi.Model(path)
        self.e = capi.Engine(self.m, 0)
        self.c = capi.Context(self.e, batch)
        self.L = capi.lib()
        self.nm = wn.NpModel(path)

    def decode(self, rows, n_past, mode):
        rows = np.asarray(rows, np.int32)
        before = self.L.wsp_launch_count()
        self.c.decode(rows, n_past, rows.shape[0], capi.DECODE_NO_SAMPLE)
        n = self.L.wsp_launch_count() - before
        assert n == expected_launches(mode, rows.shape[1], self.m.n_text_layer), (mode, rows.shape, n_past, n)
        return self.c.logits(rows.shape[0])

    def kv(self, name, slot=0):
        m = self.m
        d, H, L = m.n_text_state, m.n_text_head, m.n_text_layer
        rows = m.n_text_ctx if name.startswith("self") else m.n_audio_ctx
        return self.c.get_tensor(name, slot).reshape(L, H, rows, 64).transpose(0, 2, 1, 3).reshape(L, rows, d)

    def close(self):
        self.c.close()
        self.e.close()
        self.m.close()


@pytest.fixture(scope="module")
def micro():
    g = golden()
    r = Run(synth.model_path(LONG_MODEL), 2)
    r.c.pcm_to_mel(0, synth.synth_pcm(int(g["chunk"])))
    r.c.encode(1)
    yield r
    r.c.set_step_mode(2)
    r.c.set_reference_threads(4)
    r.close()


@pytest.mark.parametrize("threads", LONG_THREADS)
@pytest.mark.parametrize("mode", [2, 1, 0])
def test_fixture_parity_at_depth(mode, threads, micro):
    """Single steps n_past 0 .. 446, then the row at n_past 447, then the long prompts, against the reference."""
    g = golden()
    c, m = micro.c, micro.m
    toks, cps = g["tokens"], g["checkpoints"].tolist()
    idx = np.arange(0, m.n_vocab, LOGIT_STEP)
    c.set_step_mode(mode)
    c.set_reference_threads(threads)
    errs = []
    for p in range(len(toks)):
        lg = micro.decode([[toks[p]]], p, mode)[0]
        if p in cps:
            ref = g["t%d_logits" % threads][cps.index(p)]
            err = float(np.abs(lg[idx] - ref).max())
            errs.append(err / logit_tol(ref))
            assert err < logit_tol(ref), (mode, threads, p, err)
            assert abs(float(lg.max()) - float(g["t%d_logits_max" % threads][cps.index(p)])) < logit_tol(ref), (mode, threads, p)
    last = m.n_text_layer - 1
    k, v = micro.kv("self_k"), micro.kv("self_v")
    kv_err = max(np.abs(k[[0, last]][:, cps] - g["t%d_self_k" % threads].astype(np.float32)).max(),
                 np.abs(v[[0, last]][:, cps] - g["t%d_self_v" % threads].astype(np.float32)).max())
    assert kv_err < TOL_KV, (mode, threads, kv_err)
    # the last row of the context: written by a call at n_past 447, which leaves row 446 as it was
    micro.decode([[toks[5]]], m.n_text_ctx - 1, mode)
    k2 = micro.kv("self_k")
    assert np.array_equal(k2[:, :m.n_text_ctx - 1], k[:, :m.n_text_ctx - 1])
    nm = micro.nm
    s = np.float32(np.power(64.0, -0.25))
    x = nm["decoder.token_embedding.weight"][[toks[5]]] + nm["decoder.positional_embedding"][m.n_text_ctx - 1:]
    want = wn.r16(wn.mul_mat(nm["decoder.blocks.0.attn.key.weight"], wn.norm(x, nm["decoder.blocks.0.attn_ln.weight"], nm["decoder.blocks.0.attn_ln.bias"])) * s)
    assert np.abs(k2[0, -1] - want[0]).max() < TOL_KV
    for i, (n_past, n) in enumerate(LONG_PREFILLS):
        lg = micro.decode([toks[n_past:n_past + n]], n_past, mode)[0]
        ref = g["t%d_prefill_logits" % threads][i]
        assert np.abs(lg[idx] - ref).max() < logit_tol(ref), (mode, threads, n_past, n)
    print("mode %d threads %d: worst logit error %.2f of the tolerance (n_past 0-3: %.2f, 443-446: %.2f), self-KV %.1e"
          % (mode, threads, max(errs), max(errs[:4]), max(errs[-4:]), kv_err))


def depth_checkpoints(d, n_ctx=448):
    """n_past on both sides of every multiple of the step kernel's ring slot, and the end of the context"""
    cr = tf.ring_rows(d)
    cps = [p for k in range(1, (n_ctx - 1) // cr + 1) for p in range(k * cr - 2, k * cr + 3) if p < n_ctx - 1]
    return sorted(set([0, 1] + cps + list(range(n_ctx - 5, n_ctx - 1))))


# (threads, a fault the restatement must show at some checkpoint; 16 threads never take two V rounds within 448 rows)
MORE_THREADS = [(3, "last_round"), (5, None), (8, None), (9, "last_round"), (12, None), (16, "lost_slot")]


@pytest.mark.parametrize("threads,bug", MORE_THREADS)
def test_thread_counts_beyond_the_fixture(threads, bug, micro):
    """Step mode 2 at reference thread counts the fixture lacks (PG = 2, 3, 4 parts per 64-thread group, RR = 64, 42, 32 V rows per
    slot; at 3 threads two V rounds once n > 384), against the restatement fed with the GPU's own cross-attention memories."""
    g = golden()
    c, m = micro.c, micro.m
    toks = g["tokens"]
    cps = depth_checkpoints(m.n_text_state)
    c.set_step_mode(2)
    c.set_reference_threads(threads)
    got = {}
    for p in range(len(toks)):
        lg = micro.decode([[toks[p]]], p, 2)[0]
        if p in cps:
            got[p] = lg
    ck, cv = micro.kv("cross_k"), micro.kv("cross_v")
    want, k, _ = tf.restate(micro.nm, ck, cv, toks, threads, logit_rows=cps)
    errs = [float(np.abs(got[p] - want[i]).max()) / logit_tol(want[i]) for i, p in enumerate(cps)]
    assert max(errs) < 1.0, dict(zip(cps, np.round(errs, 2)))
    gk = micro.kv("self_k")
    assert np.abs(gk[:, :len(toks)] - k).max() < TOL_KV
    print("threads %d: worst logit error %.2f of the tolerance" % (threads, max(errs)))
    if bug:
        bad = tf.restate(micro.nm, ck, cv, toks, threads, logit_rows=cps, bug=bug)[0]
        margin = max(float(np.abs(got[p] - bad[i]).max()) / logit_tol(want[i]) for i, p in enumerate(cps))
        print("  control %s: %.0fx" % (bug, margin))
        assert margin >= 10, (bug, margin)


def test_free_running_to_the_end_of_the_context(micro):
    """run_chunks with the CUDA graph: tokens fed back and n_past advanced on the device, across every ring slot boundary, until the
    context is full.  Teacher-forced along the GPU's own tokens, the restatement makes the same decision wherever its margin is clear."""
    g = golden()
    c, m = micro.c, micro.m
    c.set_step_mode(2)
    c.set_reference_threads(4)
    c.set_graph(True)
    prompt = m.prompt_init()
    n_decode = m.n_text_ctx - len(prompt)
    pcms = [synth.synth_pcm(int(g["chunk"])), synth.synth_pcm(int(g["chunk"]) + 2)]
    toks, _ = c.run_chunks(pcms, prompt, n_decode)
    assert toks.shape == (2, n_decode)
    checked = deep = 0
    for b in range(2):
        seq = np.concatenate([prompt, toks[b, :-1]])
        lg, _, _ = tf.restate(micro.nm, micro.kv("cross_k", b), micro.kv("cross_v", b), seq, 4)
        lg = lg[len(prompt) - 1:]
        for i in range(n_decode):
            srt = np.sort(lg[i])
            pr = wn.softmax_rows(lg[i][None])[0]
            s = wn.sample_best(micro.nm, pr, force_timestamp=i == 0, is_initial=i == 0)
            tx = float(pr[:m.special["beg"]].max())
            if srt[-1] - srt[-2] >= GAP_SAFE and abs(s["ptsum"] - tx) > 0.1 * tx:
                assert toks[b, i] == s["id"], (b, i)
                checked += 1
                deep += i >= 3 * tf.ring_rows(m.n_text_state)
    # most decisions are clear, and so are many in the last ring slot
    assert checked > n_decode and deep > 40, (checked, deep)
    print("free running: %d of %d decisions checked, %d of them past n_past 384" % (checked, 2 * n_decode, deep))


def test_bounds(micro):
    c, m = micro.c, micro.m
    c.set_step_mode(2)
    c.set_reference_threads(4)
    micro.decode([[1]], m.n_text_ctx - 1, 2)
    with pytest.raises(capi.WspError) as ex:
        c.decode([[1, 2]], m.n_text_ctx - 1, 1, capi.DECODE_NO_SAMPLE)
    assert ex.value.status == WSP_E_BOUNDS
    with pytest.raises(capi.WspError) as ex:
        c.run_chunks([synth.synth_pcm(0)], m.prompt_init(), m.n_text_ctx + 1 - len(m.prompt_init()))
    assert ex.value.status == WSP_E_BOUNDS


# ---- full batch width: a random model of large-v2's width ------------------------------------------------------------------------
WIDE = synth.HParams(n_vocab=51865, n_audio_state=1280, n_audio_head=20, n_audio_layer=2,
                     n_text_state=1280, n_text_head=20, n_text_layer=2)


@pytest.fixture(scope="module")
def wide_model():
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "ggml-wide.bin")
        synth.write_model(p, WIDE, seed=77)
        yield p


def wide_tokens(b, n):
    """a different sequence for every chunk: text ids and timestamps"""
    x = synth.lcg_u32(500 + b, n).astype(np.int64)
    t = np.where(x % 3 == 0, 50364 + (x >> 4) % 1500, (x >> 8) % 50257)
    t[0] = 50258
    return t.astype(np.int32)


@pytest.mark.parametrize("B", [9, 16])
def test_full_batch_width(B, wide_model):
    """B = 9 (the first two-tile batch) and 16 chunks x 20 heads = 180 and 320 attention units on 148 CTAs: a prompt across CR = 160
    rows, then single steps through n_past 159-161 and 319-321.  Chunks 0 and 8 (B = 9), 7 and 15 (B = 16) against the restatement,
    fed with the GPU's own cross-attention memories so that only the decoder is under test; every chunk against itself run alone in a
    batch of 1."""
    cr = tf.ring_rows(WIDE.n_text_state)
    assert cr == 160
    n0, n1 = cr - 1, 2 * cr + 2
    at = [cr - 1, cr, cr + 1, 2 * cr - 1, 2 * cr, 2 * cr + 1]
    seqs = [wide_tokens(b, n1) for b in range(B)]
    pcms = [synth.synth_pcm(20 + b) for b in range(B)]

    def run(r, chunks):
        for slot, b in enumerate(chunks):
            r.c.pcm_to_mel(slot, pcms[b])
        r.c.encode(len(chunks))
        r.c.set_step_mode(2)
        r.c.set_reference_threads(4)
        r.decode([seqs[b][:n0] for b in chunks], 0, 2)
        out = {}
        for p in range(n0, n1):
            lg = r.decode([[seqs[b][p]] for b in chunks], p, 2)
            if p in at:
                out[p] = lg
        return out

    r = Run(wide_model, B)
    try:
        got = run(r, list(range(B)))
        ck = {b: r.kv("cross_k", b) for b in ((0, 8) if B == 9 else (7, 15))}
        cv = {b: r.kv("cross_v", b) for b in ck}
    finally:
        r.close()
    # every chunk alone
    r1 = Run(wide_model, 1)
    try:
        for b in range(B):
            alone = run(r1, [b])
            for p in at:
                assert np.abs(alone[p][0] - got[p][b]).max() < 1e-4, (B, b, p)
    finally:
        r1.close()
    # chunks at the edges of the two tiles against the restatement (0 and 8 at B = 9, 7 and 15 at B = 16); the control swaps one head's
    # self-attention output between the two chunks
    nm = wn.NpModel(wide_model)
    keep = {}

    def capture(il, kind, A):
        keep[(il, kind)] = A.copy()
        return A

    def swap(il, kind, A):
        if kind == "self":
            A = A.copy()
            A[3] = keep[(il, kind)][3]
        return A

    rows = [p - n0 for p in at]
    worst, prefix = 0.0, {}
    for b in ck:
        prefix[b] = tf.restate(nm, ck[b], cv[b], seqs[b][:n0], 4, prefill=True, logit_rows=[])[1:]
        lg, _, _ = tf.restate(nm, ck[b], cv[b], seqs[b][n0:n1], 4, n_past=n0, prefix=prefix[b], logit_rows=rows,
                              attn_hook=capture if b == max(ck) else None)
        for i, p in enumerate(at):
            e = float(np.abs(got[p][b] - lg[i]).max()) / logit_tol(lg[i])
            worst = max(worst, e)
            assert e < 1.0, (B, b, p, e)
    b = min(ck)
    bad, _, _ = tf.restate(nm, ck[b], cv[b], seqs[b][n0:n1], 4, n_past=n0, prefix=prefix[b], logit_rows=rows, attn_hook=swap)
    margin = max(float(np.abs(got[p][b] - bad[i]).max()) / logit_tol(bad[i]) for i, p in enumerate(at))
    print("B %d: worst logit error %.2f of the tolerance; head-swap control (chunks %d, %d) %.0fx" % (B, worst, b, max(ck), margin))
    assert margin >= 10, margin
