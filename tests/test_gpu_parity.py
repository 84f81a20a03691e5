"""Parity of the CUDA hot path with the reference, on a B200, through the C ABI.

Oracle: the committed fixtures tests/golden/*.npz (outputs of oracle/_ref = the reference's unmodified CPU code).

Tolerances (floating point, activations O(1), logits rms ~3):
  mel 5e-4 · encoder tensors 8e-3 · f16 KV memories 4e-3 · logits 3e-2 (measured: 1e-4, 3e-3, 2e-3, 1e-2).
Greedy tokens must be IDENTICAL to the reference's for the whole free-running sequence.
"""
import os

import numpy as np
import pytest

from tests.golden.make_golden import CASES, LOGIT_STEP, MEL_STEP, N_STEPS, ROW_STEP, case_padded
from whisper_b200 import capi, synth

pytestmark = pytest.mark.gpu

TOL_MEL, TOL_ENC, TOL_KV, TOL_LOGIT = 5e-4, 8e-3, 4e-3, 3e-2

_cache = {}


def open_model(name, batch=1):
    key = (name, batch)
    if key not in _cache:
        m = capi.Model(synth.model_path(name))
        e = _cache.get(("engine", name)) or capi.Engine(m, 0)
        _cache[("engine", name)] = e
        _cache[key] = (m, e, capi.Context(e, batch))
    return _cache[key]


def golden(name):
    return np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))


@pytest.mark.parametrize("name", list(CASES))
def test_mel(name):
    model, _, n, off = CASES[name]
    m, e, c = open_model(model)
    g = golden(name)
    chunk = int(g["chunk"])
    c.pcm_to_mel(0, synth.synth_pcm(chunk, n))
    mel = c.get_mel(0)
    assert mel.shape == tuple(g["mel_shape"])
    assert np.abs(mel[:, ::MEL_STEP] - g["mel"]).max() < TOL_MEL


def test_mel_edge_cases():
    m, e, c = open_model("micro.en-sc")
    # shorter than one FFT window, and an empty buffer: n_len = n_samples / 160 frames, zero-padded frames (whisper.cpp:2080, 2105-2109)
    for n in (0, 100, 160, 399, 400, 16000):
        c.pcm_to_mel(0, synth.synth_pcm(3, n) if n else np.zeros(0, np.float32))
        mel = c.get_mel(0)
        assert mel.shape == (80, n // 160)
        assert np.isfinite(mel).all()
    # silence: log10 clamps at 1e-10 -> constant (-10 + 4)/4
    c.pcm_to_mel(0, np.zeros(32000, np.float32))
    assert np.allclose(c.get_mel(0), (-10.0 + 4.0) / 4.0)


def test_mel_streamed_window():
    """wsp_pcm_to_mel_window, the log-mel of iContext::runStreamed: one window normalised by its own maximum (floor 1e-20), or by a
    forced one (MelStreamer.cpp:128-183), against the numpy restatement oracle/whisper_np.py::log_mel_window."""
    from oracle import whisper_np as wn
    m, e, c = open_model("micro.en-sc")
    filters = wn.NpModel(synth.model_path("micro.en-sc")).filters
    pcm = np.concatenate([synth.synth_pcm(11), 0.05 * synth.synth_pcm(12)])          # 60 s, the second half 26 dB quieter
    for i0, n_frames, samples in ((0, 3000, 480240), (2500, 3000, 480240), (3100, 2900, 2900 * 160), (5990, 10, 1600), (0, 1, 100)):
        seg = pcm[i0 * 160:i0 * 160 + samples]
        want, found_want = wn.log_mel_window(seg, filters, n_frames)
        found = c.pcm_to_mel_window(0, seg, n_frames)
        got = c.get_mel(0)
        assert got.shape == (80, n_frames)
        assert abs(found - found_want) < 4 * TOL_MEL          # raw log10 units = 4 x the normalised ones
        assert np.abs(got - want).max() < TOL_MEL
    # a forced maximum (the streamer re-using the previous window's at the tail of a stream) moves the clamp level
    seg = pcm[3100 * 160:]
    want, _ = wn.log_mel_window(seg, filters, 2900, forced_max=3.5)
    found = c.pcm_to_mel_window(0, seg, 2900, forced_max=3.5)
    assert found < 3.0 and np.abs(c.get_mel(0) - want).max() < TOL_MEL and c.get_mel(0).min() >= (3.5 - 8 + 4) / 4 - 1e-6
    # silence: every band at log10(1e-10) = -10, maximum floored at 1e-20 -> clamp at -8 -> -1.0 everywhere
    found = c.pcm_to_mel_window(0, np.zeros(16000, np.float32), 100)
    assert found == float(np.float32(1e-20)) and np.all(c.get_mel(0) == -1.0)
    # no frames at all
    c.pcm_to_mel_window(0, np.zeros(0, np.float32), 0)
    assert c.get_mel(0).shape == (80, 0)
    # the whole-clip entry point is unaffected by what the window calls left behind
    g = golden("micro_en_30s")
    c.pcm_to_mel(0, synth.synth_pcm(int(g["chunk"])))
    assert np.abs(c.get_mel(0)[:, ::MEL_STEP] - g["mel"]).max() < TOL_MEL


@pytest.mark.parametrize("name", list(CASES))
def test_encoder_trace_points(name):
    """Same named intermediates the reference traces (whisper.cpp:1121-1432), layer by layer."""
    model, _, n, off = CASES[name]
    m, e, c = open_model(model)
    g = golden(name)
    chunk = int(g["chunk"])
    d, T, L = m.n_audio_state, m.n_audio_ctx, m.n_audio_layer
    c.pcm_to_mel(0, synth.synth_pcm(chunk, n))
    c.set_encoder_layers(0)
    c.encode(1, [off])
    conv1 = c.get_tensor("enc.conv1").reshape(3000, d)
    assert np.abs(conv1[::ROW_STEP * 2] - g["enc_temp1"]).max() < TOL_ENC
    assert np.abs(c.get_tensor("enc.x").reshape(T, d)[::ROW_STEP] - g["enc_layer0_in"]).max() < TOL_ENC
    c.set_encoder_layers(1)
    c.encode(1, [off])
    assert np.abs(c.get_tensor("enc.x").reshape(T, d)[::ROW_STEP] - g["enc_layer1_in"]).max() < TOL_ENC
    c.set_encoder_layers(-1)
    c.encode(1, [off])
    assert np.abs(c.get_tensor("enc.x").reshape(T, d)[::ROW_STEP] - g["enc_layers"]).max() < TOL_ENC
    # ln_post of the scripted models amplifies by SC_ENC_GAIN_CALIBRATED (synth.py): encode-out and the cross-KV carry that factor
    gain = synth.SC_ENC_GAIN_CALIBRATED
    assert np.abs(c.get_tensor("encode-out").reshape(T, d)[::ROW_STEP] - g["encode_out"]).max() < TOL_ENC * gain
    H, Ld = m.n_audio_head, m.n_text_layer
    for nm in ("cross_k", "cross_v"):
        got = c.get_tensor(nm).reshape(Ld, H, T, 64).transpose(0, 2, 1, 3).reshape(Ld, T, d)
        assert np.abs(got[:, ::ROW_STEP] - g[nm].astype(np.float32)).max() < TOL_KV * gain


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("threads", [1, 4, 6, 16])
def test_decoder_logits_teacher_forced(name, threads):
    model, _, n, off = CASES[name]
    m, e, c = open_model(model)
    g = golden(name)
    chunk = int(g["chunk"])
    c.set_reference_threads(threads)
    c.pcm_to_mel(0, synth.synth_pcm(chunk, n))
    c.encode(1, [off])
    prompt = g["prompt"].tolist()
    idx = np.arange(0, m.n_vocab, LOGIT_STEP)
    c.decode([prompt], 0, 1, capi.DECODE_ALL_LOGITS)
    lg = c.logits(len(prompt))
    # logits of rms ~3 in every regular case; the zero-padded case runs at rms ~25 (see make_golden.CASES): the tolerance scales with it
    tol = TOL_LOGIT * max(1.0, float(g["t%d_prompt_logits" % threads].std()) / 3.0)
    assert np.abs(lg[:, idx] - g["t%d_prompt_logits" % threads]).max() < tol
    assert np.abs(lg.max(-1) - g["t%d_prompt_logits_max" % threads]).max() < tol
    pr = c.probs(len(prompt))
    assert np.allclose(pr.sum(-1), 1.0, atol=1e-4)
    toks = g["t%d_tokens" % threads]
    s = c.decode([prompt], 0, 1, capi.DECODE_FORCE_TIMESTAMP | capi.DECODE_INITIAL)[0]
    pinned = not case_padded(name)     # the zero-padded case pins logits only: its decisions are not protected by GAP_SAFE
    if pinned:
        assert s["id"] == toks[0] and s["tid"] == g["t%d_tids" % threads][0]
        assert abs(s["p"] - g["t%d_token_p" % threads][0]) < 1e-3
    n_past = len(prompt)
    for i in range(1, N_STEPS):
        s = c.decode([[int(toks[i - 1])]], n_past, 1, 0)[0]
        n_past += 1
        lg = c.logits(1)
        assert np.abs(lg[0, idx] - g["t%d_step_logits" % threads][i - 1]).max() < tol, "step %d" % i
        if pinned:
            assert s["id"] == toks[i], "step %d" % i
            assert abs(s["p"] - g["t%d_token_p" % threads][i]) < 5e-3
    c.set_reference_threads(4)


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("threads", [1, 4, 6, 16])
@pytest.mark.parametrize("graph", [True, False])
def test_greedy_tokens_free_running(name, threads, graph):
    """The measured path (wsp_run_chunks: tokens fed back on the device, CUDA graph per step) reproduces the reference's
    greedy sequence exactly — when the window starts at frame 0, which is what run_chunks encodes."""
    model, _, n, off = CASES[name]
    if off != 0:
        pytest.skip("run_chunks always encodes the window at offset 0")
    if case_padded(name):
        pytest.skip("zero-padded window: decisions are not pinned (make_golden.CASES)")
    m, e, c = open_model(model)
    g = golden(name)
    chunk = int(g["chunk"])
    c.set_reference_threads(threads)
    c.set_graph(graph)
    toks, st = c.run_chunks([synth.synth_pcm(chunk, n)], g["prompt"].tolist(), N_STEPS)
    assert toks[0].tolist() == g["t%d_tokens" % threads].tolist()
    c.set_graph(True)
    c.set_reference_threads(4)


def test_batch_equals_single():
    """Independent chunks: a chunk's tokens do not depend on which batch slot it sits in or on its neighbours."""
    m, e, c1 = open_model("micro.en-sc", 1)
    _, _, c4 = open_model("micro.en-sc", 4)
    pcms = [synth.synth_pcm(i, 480000 - 16000 * i) for i in range(4)]
    prompt = m.prompt_init()
    t4, _ = c4.run_chunks(pcms, prompt, 12)
    for i in range(4):
        t1, _ = c1.run_chunks([pcms[i]], prompt, 12)
        assert t1[0].tolist() == t4[i].tolist()
    # permuting the batch permutes the results
    t4p, _ = c4.run_chunks(pcms[::-1], prompt, 12)
    assert t4p[::-1].tolist() == t4.tolist()
    # partial batch on a larger context
    t2, _ = c4.run_chunks(pcms[:2], prompt, 12)
    assert t2.tolist() == t4[:2].tolist()


@pytest.mark.parametrize("threads", [2, 3, 5, 8, 9, 12, 13, 16])
def test_step_kernels_agree_for_every_thread_count(threads):
    """The dataflow step kernel (mode 2), round 1's barrier kernel (mode 1) and the kernel-per-op path (mode 0) reproduce the same
    reference arithmetic: same greedy tokens, logits within the summation-order noise, at reference thread counts that put one,
    two, three and four key ranges on a 64-thread group of the step kernel (the fixtures pin 1, 4, 6, 16 against the reference)."""
    m, e, c = open_model("micro.en-sc", 2)
    g = golden("micro_en_30s")
    pcms = [synth.synth_pcm(int(g["chunk"])), synth.synth_pcm(int(g["chunk"]), 400000)]
    prompt = g["prompt"].tolist()
    c.set_reference_threads(threads)
    res = {}
    try:
        for mode in (2, 1, 0):
            c.set_step_mode(mode)
            toks, _ = c.run_chunks(pcms, prompt, N_STEPS)
            res[mode] = (toks.copy(), c.logits(2).copy())
    finally:
        c.set_step_mode(2)
        c.set_reference_threads(4)
    for mode in (1, 0):
        assert res[2][0].tolist() == res[mode][0].tolist(), (threads, mode)
        assert np.abs(res[2][1] - res[mode][1]).max() < TOL_LOGIT, (threads, mode)


def test_live_reference_when_prebuilt():
    """A model shape and clip that the parity cases above do not cover (tiny.en-sc, chunk 5): log-mel, cross-attention keys and 20 greedy
    tokens against the reference's (tests/golden/tiny_en_live.npz, make_golden.py --live)."""
    from tests.golden.make_golden import LIVE_CHUNK, LIVE_MODEL, LIVE_STEPS
    g = golden("tiny_en_live")
    m, e, c = open_model(LIVE_MODEL)
    pcm = synth.synth_pcm(LIVE_CHUNK)
    c.pcm_to_mel(0, pcm)
    mel = c.get_mel(0)
    assert mel.shape == tuple(g["mel_shape"])
    assert np.abs(mel[:, ::MEL_STEP] - g["mel"]).max() < TOL_MEL
    c.encode(1)
    d, T, H, L = m.n_audio_state, m.n_audio_ctx, m.n_audio_head, m.n_text_layer
    got = c.get_tensor("cross_k").reshape(L, H, T, 64).transpose(0, 2, 1, 3).reshape(L, T, d)
    assert np.abs(got[:, ::ROW_STEP] - g["cross_k"].astype(np.float32)).max() < TOL_KV * synth.SC_ENC_GAIN_CALIBRATED
    prompt = m.prompt_init()
    assert prompt == g["prompt"].tolist()
    toks, _ = c.run_chunks([pcm], prompt, LIVE_STEPS)
    assert toks[0].tolist() == g["tokens"].tolist()


@pytest.mark.parametrize("model", ["tiny.en-sc", "base.en-sc", "medium-sc", "large-sc"])
def test_real_model_shapes_match_reference_fixture(model):
    """BASELINE.json's model shapes on the scripted weights, all chunks as ONE batch: medium-sc = the bench configuration (8 chunks,
    32 tokens each), base.en-sc = 12 chunks (the two-tile path of the decoder step, B in 9..16), large-sc = configs[4]'s shape.  Greedy
    tokens identical to the reference's for every chunk (its margins are >= GAP_SAFE by construction of the fixture), last-step logits
    within tolerance (tests/golden/real_shapes.npz, made by `make_golden.py --real-shapes`)."""
    from tests.golden.make_golden import REAL_SHAPES
    g = golden("real_shapes")
    key = model.replace(".", "_").replace("-", "_")
    if key + "_tokens" not in g:
        pytest.skip("no fixture for " + model)
    n_chunks, steps = REAL_SHAPES[model]
    chunks = g[key + "_chunks"].tolist()
    assert len(chunks) == n_chunks
    m = capi.Model(synth.model_path(model))
    e = capi.Engine(m, 0)
    c = capi.Context(e, n_chunks)
    try:
        prompt = g[key + "_prompt"].tolist()
        assert prompt == m.prompt_init()
        # 4 threads is the reference's default; the bench configuration is also pinned at 16, the thread count its reference arm is timed with
        for th in (4, 16):
            pre = key + ("" if th == 4 else "_t%d" % th)
            if pre + "_tokens" not in g:
                continue
            c.set_reference_threads(th)
            toks, _ = c.run_chunks([synth.synth_pcm(ch) for ch in chunks], prompt, steps)
            logits = c.logits(n_chunks)
            for i, ch in enumerate(chunks):
                assert toks[i].tolist() == g[pre + "_tokens"][i].tolist(), (model, ch, th)
                assert np.abs(logits[i][::LOGIT_STEP] - g[pre + "_last_logits_sub"][i]).max() < TOL_LOGIT, (model, ch, th)
    finally:
        c.close()
        e.close()
        m.close()


def test_argument_errors():
    m, e, c = open_model("micro.en-sc")
    with pytest.raises(capi.WspError) as ex:
        c.encode(2)            # context was created for batch 1
    assert ex.value.status == -7
    with pytest.raises(capi.WspError):
        c.decode([[m.n_vocab + 5]], 0, 1, 0)
    with pytest.raises(capi.WspError):
        c.decode([[1]], m.n_text_ctx, 1, 0)
    with pytest.raises(capi.WspError):
        c.get_tensor("no-such-tensor")


def test_launch_counter_counts_kernels():
    L = capi.lib()
    m, e, c = open_model("micro.en-sc")
    before = L.wsp_launch_count()
    c.run_chunks([synth.synth_pcm(0)], m.prompt_init(), 4)
    assert L.wsp_launch_count() - before > 40   # encoder ~45 launches + 4 token steps (persistent decoder kernel + sampler)
