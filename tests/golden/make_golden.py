#!/usr/bin/env python
"""Generate tests/golden/*.npz from oracle/_ref — the reference's own CPU implementation (Whisper/source/{ggml.c,whisper.cpp},
compiled unmodified by oracle/Makefile).  The reference ships no golden vectors for this path (SURVEY.md §4), so these
fixtures ARE the pin: they are what the numpy restatement (oracle/whisper_np.py) and the CUDA engine are compared with on
machines where /root/reference (and hence a fresh oracle/_ref build) is not available.

Inputs are fully determined by whisper_b200/synth.py (model seed 1234, PCM chunk ids), so only outputs are stored, and large
tensors are stored as deterministic sub-samples to keep the fixtures small.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz
    python tests/golden/make_golden.py --sampler  # tests/golden/sampler.npz: needs a B200 besides oracle/_ref
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.ref import RefOracle  # noqa: E402
from whisper_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# deterministic sub-sampling shared with the tests
MEL_STEP = 10        # every 10th frame
ROW_STEP = 25        # every 25th time step of [T][d] tensors
LOGIT_STEP = 61      # every 61st vocabulary entry
N_STEPS = 40         # greedy steps stored per case
# The scripted models (whisper_b200/synth.py, "-sc") decide every text token between two equally scored candidates by the random
# part of the logits; the margin is Gaussian (std ~2.5).  A fixture only keeps inputs for which the REFERENCE's top-2 margin stays
# above GAP_SAFE at every stored step — 3x the logit tolerance of the parity tests — so "identical greedy tokens" is a fair demand.
GAP_SAFE = 0.1
MIN_DISTINCT = 10    # a fixture whose sequence has fewer distinct tokens is rejected (round 1's degenerate fixtures had 2)


def logits_sample(lg):
    idx = np.arange(0, lg.shape[-1], LOGIT_STEP)
    return lg[..., idx].astype(np.float32)


def top2_gap(lg):
    s = np.partition(lg, -2)[-2:]
    return float(s[1] - s[0])


def prompt_of(o):
    return [o.special["sot"]] + ([o.special["sot"] + 1, o.special["transcribe"]] if o.n_vocab == 51865 else [])


def greedy(o, prompt, n_steps, keep_logits=False):
    """The bench loop (BASELINE.md §2): prompt, first token by whisper_sample_timestamp(initial), then whisper_sample_best.  Returns
    tokens, tids, ps, gaps (top-2 logit margin of every step but the forced first one), per-step logits sub-samples, last logits."""
    lg, _ = o.decode(prompt, 0)
    prompt_logits = lg
    tok = o.sample(initial=True, force_timestamp=True)
    toks, ps, tids, gaps, step_logits = [tok["id"]], [tok["p"]], [tok["tid"]], [], []
    n_past = len(prompt)
    for _ in range(n_steps - 1):
        lg, _ = o.decode([toks[-1]], n_past)
        n_past += 1
        gaps.append(top2_gap(lg[0]))
        if keep_logits:
            step_logits.append(logits_sample(lg[0]))
        tok = o.sample()
        toks.append(tok["id"]); ps.append(tok["p"]); tids.append(tok["tid"])
    return dict(tokens=np.array(toks, np.int32), tids=np.array(tids, np.int32), p=np.array(ps, np.float32), gap=np.array(gaps, np.float32),
                step_logits=np.stack(step_logits) if keep_logits else None, last_logits=lg[0], prompt_logits=prompt_logits)


def make(model_name: str, chunk0: int, n_samples: int, offset: int, threads_list=(1, 4, 6, 16)):
    """Encoder trace points, cross-KV, teacher-forced logits and greedy tokens at 1, 4, 6 and 16 reference threads (the reference's
    V^T*P arithmetic depends on its thread count, ggml.c:4680-4722; 4 is its default, 6 and 16 exercise two and four key ranges per
    64-thread group of the decoder-step kernel); the PCM chunk id is the first one >= chunk0 whose greedy sequences are clear of
    near-ties at every thread count."""
    path = synth.model_path(model_name)
    for chunk in range(chunk0, chunk0 + 40):
        pcm = synth.synth_pcm(chunk, n_samples)
        o = RefOracle(path, threads=1)
        mel = o.pcm_to_mel(pcm)
        prompt = prompt_of(o)
        runs = {}
        for th in threads_list:
            oo = RefOracle(path, threads=th)
            oo.set_mel(mel)
            oo.encode(offset)
            runs[th] = greedy(oo, prompt, N_STEPS, keep_logits=True)
        worst = min(float(r["gap"].min()) for r in runs.values())
        distinct = min(len(set(r["tokens"].tolist())) for r in runs.values())
        print("  %s chunk %d: min gap %.3f, distinct %d" % (model_name, chunk, worst, distinct), flush=True)
        padded = n_samples < offset * 160 + 480000
        if (worst >= GAP_SAFE and distinct >= MIN_DISTINCT) or padded:
            break
    else:
        raise RuntimeError("no clean chunk for " + model_name)
    out = {"chunk": np.int32(chunk)}
    out["mel_shape"] = np.array(mel.shape, np.int32)
    out["mel"] = mel[:, ::MEL_STEP].astype(np.float32)
    o.trace(True)
    o.encode(offset)
    tr = o.trace_items()
    o.trace(False)
    d, T, L = o.n_audio_state, o.n_audio_ctx, o.n_audio_layer
    out["enc_temp1"] = tr["enc.temp1"].reshape(d, 3000).T[::ROW_STEP * 2].astype(np.float32)
    for il in (0, 1):
        out["enc_layer%d_in" % il] = tr["enc.layer[ %d ].in" % il].reshape(T, d)[::ROW_STEP].astype(np.float32)
    out["enc_layers"] = tr["enc.layers"].reshape(T, d)[::ROW_STEP].astype(np.float32)
    out["encode_out"] = tr["encode-out"].reshape(T, d)[::ROW_STEP].astype(np.float32)
    ck, cv = o.cross_kv()
    out["cross_k"] = ck[:, ::ROW_STEP].astype(np.float16)
    out["cross_v"] = cv[:, ::ROW_STEP].astype(np.float16)
    out["prompt"] = np.array(prompt, np.int32)
    for th, r in runs.items():
        lg = r["prompt_logits"]
        out["t%d_prompt_logits" % th] = logits_sample(lg)
        out["t%d_prompt_logits_max" % th] = lg.max(-1).astype(np.float32)
        out["t%d_prompt_argmax" % th] = lg.argmax(-1).astype(np.int32)
        out["t%d_tokens" % th] = r["tokens"]
        out["t%d_tids" % th] = r["tids"]
        out["t%d_token_p" % th] = r["p"]
        out["t%d_step_logits" % th] = r["step_logits"]
        out["t%d_gap" % th] = r["gap"]
    return out


CASES = {
    # name: (model, first PCM chunk id to try, n_samples, mel offset); the chunk id actually used is stored in the fixture ("chunk")
    "micro_en_30s": ("micro.en-sc", 0, 480000, 0),
    "micro_ml_30s": ("micro-sc", 3, 480000, 0),           # multilingual specials
    "micro_en_offset": ("micro.en-sc", 6, 640000, 1000),   # 40 s clip, window starting at frame 1000
    # short clip: the window is zero-padded (whisper.cpp:1104-1120).  A random encoder's response to silence throws the scripted decoder
    # off its script — logits of rms ~25, one token repeated — so this case pins mel / encoder / logits only, not token variety
    "micro_ml_11s": ("micro-sc", 1, 176000, 0),
}

def case_padded(name: str) -> bool:
    """the case's 30 s window reaches past the end of its clip (zero-padded mel): greedy decisions are not pinned there"""
    _model, _c, n, off = CASES[name]
    return n < off * 160 + 480000


# whisper_full() runs (the transcription driver, whisper.cpp:2765-3125) on the sparse-branch scripted models: every 30 s window yields
# 8 multi-token segments with increasing timestamps and an EOT; three text tokens per window are decided by the audio / the history
FULL_MODEL = "micro.en-sc1"
FULL_MODEL_ML = "micro-sc1"
FULL_SECONDS = 78
# every run stops before the clip's tail: a window that reaches past the end of the audio is zero-padded by the reference, and a random
# encoder's response to silence throws the scripted decoder off its script (thousands of garbage decodes per run)
FULL_DURATION_MS = 64000
FULL_RUNS = {
    # name: (model, eFullParamsFlags, max_tokens, offset_ms, duration_ms, language, calls)
    #   flags: 1 Translate, 2 NoContext, 4 SingleSegment, 8 PrintSpecial;  calls = 2: two consecutive runFull calls on one context
    #   WITHOUT NoContext, the second one is stored (prompt carry-over across calls, whisper.cpp:2850-2861)
    "plain": (FULL_MODEL, 0, 0, 0, FULL_DURATION_MS, "en", 1),
    "special": (FULL_MODEL, 8, 0, 0, FULL_DURATION_MS, "en", 1),
    "special_nocontext_max40": (FULL_MODEL, 8 | 2, 40, 0, FULL_DURATION_MS, "en", 1),
    "single_segment_max16": (FULL_MODEL, 4, 16, 0, FULL_DURATION_MS, "en", 1),
    "special_offset_duration": (FULL_MODEL, 8 | 2, 30, 10000, 32000, "en", 1),
    "context_second_call": (FULL_MODEL, 0, 0, 0, FULL_DURATION_MS, "en", 2),
    "ml_german": (FULL_MODEL_ML, 0, 0, 0, FULL_DURATION_MS, "de", 1),
    "ml_translate": (FULL_MODEL_ML, 1, 0, 0, FULL_DURATION_MS, "fr", 1),
    # token-level timestamps (flag 0x100 = TokenTimestamps, whisper.cpp:3374-3600) and max_len wrapping (:2713-2763)
    "token_ts": (FULL_MODEL, 0x100, 0, 0, FULL_DURATION_MS, "en", 1),
    "token_ts_maxlen12": (FULL_MODEL, 0x100 | 2, 0, 0, FULL_DURATION_MS, "en", 1),
}
FULL_MAX_LEN = {"token_ts_maxlen12": 12}


def full_pcm(base: int = 10):
    n = 16000 * FULL_SECONDS
    return np.concatenate([synth.synth_pcm(base + i) for i in range((n + 479999) // 480000)])[:n]


def run_full_reference(model, pcm, flags, max_tokens, off, dur, lang, calls, max_len=0):
    o = RefOracle(synth.model_path(model), threads=4, log_level=0)
    L = o.L
    o.gap_log(True)
    for _ in range(calls):
        rc = L.ora_full_ex2(o.ctx, pcm.ctypes.data_as(C.POINTER(C.c_float)), pcm.size, 4, flags, lang.encode(), max_tokens, off, dur, max_len)
        assert rc == 0
    gaps = o.gap_log()
    o.gap_log(False)
    segs = []
    for i in range(L.ora_full_n_segments(o.ctx)):
        toks = [L.ora_full_token_id(o.ctx, i, j) for j in range(L.ora_full_n_tokens(o.ctx, i))]
        tt = [(L.ora_full_token_t0(o.ctx, i, j), L.ora_full_token_t1(o.ctx, i, j)) for j in range(len(toks))]
        segs.append((L.ora_full_segment_t0(o.ctx, i), L.ora_full_segment_t1(o.ctx, i), toks, L.ora_full_segment_text(o.ctx, i), tt))
    return segs, gaps


def make_full():
    out = {}
    for name, (model, flags, max_tokens, off, dur, lang, calls) in FULL_RUNS.items():
        for base in range(10, 410, 10):
            pcm = full_pcm(base)
            segs, gaps = run_full_reference(model, pcm, flags, max_tokens, off, dur, lang, calls, FULL_MAX_LEN.get(name, 0))
            # (a run that leaves the script — hundreds of decoder calls per window while whisper_full retries — is not a useful pin)
            if gaps.size and gaps.min() >= GAP_SAFE and gaps.size <= 80 * calls * (FULL_SECONDS // 16 + 1):
                break
        else:
            raise RuntimeError("no clean PCM for full/" + name)
        out[name + "_pcm_base"] = np.int32(base)
        out[name + "_t"] = np.array([[s[0], s[1]] for s in segs], np.int64).reshape(-1, 2)
        out[name + "_ntok"] = np.array([len(s[2]) for s in segs], np.int32)
        out[name + "_tokens"] = np.array([t for s in segs for t in s[2]], np.int32)
        out[name + "_text"] = np.array([s[3].decode(errors="replace") for s in segs])
        out[name + "_token_t"] = np.array([t for s in segs for t in s[4]], np.int64).reshape(-1, 2)
        out[name + "_min_gap"] = np.float32(gaps.min())
        print("  full/%s: pcm base %d, %d segments, %d tokens (%d distinct), %d decoder calls, min gap %.3f" % (
            name, base, len(segs), out[name + "_tokens"].size, len(set(out[name + "_tokens"].tolist())), gaps.size, gaps.min()), flush=True)
    return out


def make_lang():
    """whisper_lang_auto_detect (whisper.cpp:2428-2495) on the multilingual scripted model, three clips."""
    out = {}
    o = RefOracle(synth.model_path("micro-sc"), threads=4)
    ids, probs = [], []
    for ch in (3, 5, 8):
        o.pcm_to_mel(synth.synth_pcm(ch, 480000))
        lid, pr = o.lang_auto_detect(0)
        ids.append(lid); probs.append(pr)
        print("  lang/chunk %d: id %d p %.4f (runner-up %.4f)" % (ch, lid, np.sort(pr)[-1], np.sort(pr)[-2]), flush=True)
    out["chunks"] = np.array([3, 5, 8], np.int32)
    out["lang_id"] = np.array(ids, np.int32)
    out["lang_probs"] = np.array(probs, np.float32)
    return out


# BASELINE.json's model shapes: greedy tokens of the bench loop at 4 reference threads, the last step's logits (sub-sampled) and the
# top-2 margins.  "medium-sc" is the BENCH CONFIGURATION itself (8 chunks, one batch); base.en runs 12 chunks (the two-tile path of the
# decoder step, B in 9..16); large is configs[4]'s shape (a few steps: its encoder alone takes the CPU a minute).
REAL_SHAPES = {"tiny.en-sc": (2, 24), "base.en-sc": (12, 16), "medium-sc": (8, 32), "large-sc": (1, 4)}
# the bench configuration is also pinned at 16 reference threads — the thread count the reference arm of bench.py is timed with
REAL_THREADS = {"medium-sc": (4, 16)}


def make_real_shapes(models=None):
    out = {}
    for model, (n_chunks, steps) in REAL_SHAPES.items():
        if models and model not in models:
            continue
        ths = REAL_THREADS.get(model, (4,))
        os_ = {th: RefOracle(synth.model_path(model), threads=th) for th in ths}
        o = os_[ths[0]]
        prompt = prompt_of(o)
        key = model.replace(".", "_").replace("-", "_")
        chosen = []
        toks, logits, gaps = ({th: [] for th in ths} for _ in range(3))
        ch = 0
        while len(chosen) < n_chunks:
            assert ch < 200, "no clean chunks for " + model
            mel = o.pcm_to_mel(synth.synth_pcm(ch))
            rs = {}
            for th in ths:
                os_[th].set_mel(mel)
                os_[th].encode(0)
                rs[th] = greedy(os_[th], prompt, steps)
            gap = min(float(r["gap"].min()) for r in rs.values())
            ok = gap >= GAP_SAFE and min(len(set(r["tokens"].tolist())) for r in rs.values()) >= min(MIN_DISTINCT, steps)
            print("  real/%s chunk %d: min gap %.3f %s tokens %s..." % (model, ch, gap, "keep" if ok else "skip", rs[ths[0]]["tokens"][:6].tolist()), flush=True)
            if ok:
                chosen.append(ch)
                for th in ths:
                    toks[th].append(rs[th]["tokens"]); logits[th].append(rs[th]["last_logits"][::LOGIT_STEP].astype(np.float32)); gaps[th].append(rs[th]["gap"])
            ch += 1
        out[key + "_chunks"] = np.array(chosen, np.int32)
        out[key + "_prompt"] = np.array(prompt, np.int32)
        for th in ths:
            pre = key + ("" if th == 4 else "_t%d" % th)     # the keys without a thread suffix are the reference's default, 4 threads
            out[pre + "_tokens"] = np.stack(toks[th])
            out[pre + "_last_logits_sub"] = np.stack(logits[th])
            out[pre + "_gap"] = np.stack(gaps[th])
        del os_, o
    return out


# A model shape and clip no other fixture covers (tests/test_gpu_parity.py::test_live_reference_when_prebuilt): log-mel, cross-attention
# keys and the greedy tokens of the bench loop at the reference's default 4 threads.
LIVE_MODEL, LIVE_CHUNK, LIVE_STEPS = "tiny.en-sc", 5, 20


def make_live():
    o = RefOracle(synth.model_path(LIVE_MODEL), threads=4)
    pcm = synth.synth_pcm(LIVE_CHUNK)
    mel = o.pcm_to_mel(pcm)
    o.encode(0)
    ck, _ = o.cross_kv()
    prompt = prompt_of(o)
    _, toks, _ = o.bench_chunk(pcm, prompt, LIVE_STEPS)
    return {"mel_shape": np.array(mel.shape, np.int32), "mel": mel[:, ::MEL_STEP].astype(np.float32),
            "cross_k": ck[:, ::ROW_STEP].astype(np.float16), "prompt": np.array(prompt, np.int32), "tokens": np.asarray(toks, np.int32)}


def make_sampler():
    """The reference's whisper_sample_best / whisper_sample_timestamp (ora_sample_from_probs) on the probability rows the GPU sampler's
    softmax makes of tests/test_gpu_sampler.make_rows(), in row order.  Needs a B200 and oracle/_ref on the same machine."""
    from tests.test_gpu_sampler import MODEL, SPECIAL4, make_rows
    from whisper_b200 import capi
    o = RefOracle(synth.model_path(MODEL), threads=1)
    res = {k: [] for k in ("id", "tid", "p", "pt", "ptsum")}
    for lg, force_ts, initial, _label in make_rows():
        probs, _ = capi.test_sample(lg, SPECIAL4, force_ts, initial)
        for row in probs:
            s = o.sample_from_probs(row, force_ts, initial)
            for k in res:
                res[k].append(s[k])
    return {k: np.array(v, np.int32 if k in ("id", "tid") else np.float32) for k, v in res.items()}


TOKENIZER_TEXTS = [b" hello hellox 12345!", b" hello world's , worlds 345 12", b" t12 t345", b""]


def make_tokenizer():
    """Prints the TOKENIZER_GOLDEN table of tests/test_gpu_com.py: whisper_tokenize of the reference on the "-words" vocabulary."""
    o = RefOracle(synth.model_path("micro.en-words"))
    for t in TOKENIZER_TEXTS:
        print("    %r: %r," % (t, o.tokenize(t)))


def save(name, data, merge=False):
    p = os.path.join(HERE, name + ".npz")
    if merge and os.path.exists(p):
        old = dict(np.load(p))
        old.update(data)
        data = old
    np.savez_compressed(p, **data)
    print(name, "%.0f KB" % (os.path.getsize(p) / 1024), flush=True)


if __name__ == "__main__":
    if "--tokenizer" in sys.argv:
        make_tokenizer()
        sys.exit(0)
    if "--real-shapes" in sys.argv:
        rest = [a for a in sys.argv[1:] if not a.startswith("--")]
        save("real_shapes", make_real_shapes(rest or None), merge=bool(rest))
        sys.exit(0)
    if "--full" in sys.argv:
        save("full_runs", make_full())
        sys.exit(0)
    if "--lang" in sys.argv:
        save("lang_detect", make_lang())
        sys.exit(0)
    if "--live" in sys.argv:
        save("tiny_en_live", make_live())
        sys.exit(0)
    if "--sampler" in sys.argv:
        save("sampler", make_sampler())
        sys.exit(0)
    if "--cases" in sys.argv:
        for name in [a for a in sys.argv[1:] if not a.startswith("--")] or list(CASES):
            save(name, make(*CASES[name]))
        sys.exit(0)
    save("full_runs", make_full())
    save("lang_detect", make_lang())
    save("tiny_en_live", make_live())
    for name, (model, chunk, n, off) in CASES.items():
        save(name, make(model, chunk, n, off))
