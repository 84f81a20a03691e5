"""Synthetic inputs for parity tests and bench.py: ggml model files and 16 kHz PCM.

There are no real `ggml-*.bin` files and no network in this environment (SURVEY.md §0.4), so every
correctness and performance run uses model files written here in the reference's exact on-disk format
(reader: /root/reference/Whisper/source/whisper.cpp:451-1072, Whisper/Whisper/WhisperModel.cpp:434-492;
layout summarised in SURVEY.md Appendix A).  Real model files load through the same path unchanged.

Both the CPU oracle and the CUDA engine read the *same file bytes*, and both get the *same PCM bytes*.
"""
from __future__ import annotations

import os
import struct
import tempfile
from dataclasses import dataclass

import numpy as np

GGML_MAGIC = 0x67676D6C  # whisper.cpp:466


@dataclass(frozen=True)
class HParams:
    """whisper_hparams in file order (whisper.cpp:248-260, :477-487)."""

    n_vocab: int = 51864
    n_audio_ctx: int = 1500
    n_audio_state: int = 384
    n_audio_head: int = 6
    n_audio_layer: int = 4
    n_text_ctx: int = 448
    n_text_state: int = 384
    n_text_head: int = 6
    n_text_layer: int = 4
    n_mels: int = 80
    f16: int = 1

    def as_list(self):
        return [self.n_vocab, self.n_audio_ctx, self.n_audio_state, self.n_audio_head, self.n_audio_layer,
                self.n_text_ctx, self.n_text_state, self.n_text_head, self.n_text_layer, self.n_mels, self.f16]


def _hp(d, h, l, vocab):
    return HParams(n_vocab=vocab, n_audio_state=d, n_audio_head=h, n_audio_layer=l,
                   n_text_state=d, n_text_head=h, n_text_layer=l)


# Model shapes (SURVEY.md §8 table).  "micro" is a test-only shape: the reference loader sizes its arenas by
# n_audio_layer ∈ {4,6,12,24,32} (whisper.cpp:490-508), so a 4-layer model with a small state loads in the oracle.
MODELS = {
    "micro.en": _hp(128, 2, 4, 51864),
    "micro": _hp(128, 2, 4, 51865),
    "tiny.en": _hp(384, 6, 4, 51864),
    "tiny": _hp(384, 6, 4, 51865),
    "base.en": _hp(512, 8, 6, 51864),
    "base": _hp(512, 8, 6, 51865),
    "small": _hp(768, 12, 12, 51865),
    "medium": _hp(1024, 16, 24, 51865),
    "large": _hp(1280, 20, 32, 51865),
}


def tensor_list(hp: HParams):
    """(name, ne[], is_f16, kind) for every tensor the loader requires (whisper.cpp:772-945).
    ne[0] is the fastest axis.  kind drives the synthetic distribution."""
    d, dt = hp.n_audio_state, hp.n_text_state
    out = []
    out.append(("encoder.positional_embedding", [d, hp.n_audio_ctx], False, "pos"))
    out.append(("encoder.conv1.weight", [3, hp.n_mels, d], True, "mat"))
    out.append(("encoder.conv1.bias", [1, d], False, "bias"))
    out.append(("encoder.conv2.weight", [3, d, d], True, "mat"))
    out.append(("encoder.conv2.bias", [1, d], False, "bias"))
    out.append(("encoder.ln_post.weight", [d], False, "gamma"))
    out.append(("encoder.ln_post.bias", [d], False, "bias"))
    for i in range(hp.n_audio_layer):
        p = f"encoder.blocks.{i}."
        out += [
            (p + "mlp_ln.weight", [d], False, "gamma"), (p + "mlp_ln.bias", [d], False, "bias"),
            (p + "mlp.0.weight", [d, 4 * d], True, "mat"), (p + "mlp.0.bias", [4 * d], False, "bias"),
            (p + "mlp.2.weight", [4 * d, d], True, "mat"), (p + "mlp.2.bias", [d], False, "bias"),
            (p + "attn_ln.weight", [d], False, "gamma"), (p + "attn_ln.bias", [d], False, "bias"),
            (p + "attn.query.weight", [d, d], True, "mat"), (p + "attn.query.bias", [d], False, "bias"),
            (p + "attn.key.weight", [d, d], True, "mat"),
            (p + "attn.value.weight", [d, d], True, "mat"), (p + "attn.value.bias", [d], False, "bias"),
            (p + "attn.out.weight", [d, d], True, "mat"), (p + "attn.out.bias", [d], False, "bias"),
        ]
    out.append(("decoder.positional_embedding", [dt, hp.n_text_ctx], False, "pos"))
    out.append(("decoder.token_embedding.weight", [dt, hp.n_vocab], True, "emb"))
    out.append(("decoder.ln.weight", [dt], False, "gamma"))
    out.append(("decoder.ln.bias", [dt], False, "bias"))
    for i in range(hp.n_text_layer):
        p = f"decoder.blocks.{i}."
        out += [
            (p + "mlp_ln.weight", [dt], False, "gamma"), (p + "mlp_ln.bias", [dt], False, "bias"),
            (p + "mlp.0.weight", [dt, 4 * dt], True, "mat"), (p + "mlp.0.bias", [4 * dt], False, "bias"),
            (p + "mlp.2.weight", [4 * dt, dt], True, "mat"), (p + "mlp.2.bias", [dt], False, "bias"),
            (p + "attn_ln.weight", [dt], False, "gamma"), (p + "attn_ln.bias", [dt], False, "bias"),
            (p + "attn.query.weight", [dt, dt], True, "mat"), (p + "attn.query.bias", [dt], False, "bias"),
            (p + "attn.key.weight", [dt, dt], True, "mat"),
            (p + "attn.value.weight", [dt, dt], True, "mat"), (p + "attn.value.bias", [dt], False, "bias"),
            (p + "attn.out.weight", [dt, dt], True, "mat"), (p + "attn.out.bias", [dt], False, "bias"),
            (p + "cross_attn_ln.weight", [dt], False, "gamma"), (p + "cross_attn_ln.bias", [dt], False, "bias"),
            (p + "cross_attn.query.weight", [dt, dt], True, "mat"), (p + "cross_attn.query.bias", [dt], False, "bias"),
            (p + "cross_attn.key.weight", [dt, dt], True, "mat"),
            (p + "cross_attn.value.weight", [dt, dt], True, "mat"), (p + "cross_attn.value.bias", [dt], False, "bias"),
            (p + "cross_attn.out.weight", [dt, dt], True, "mat"), (p + "cross_attn.out.bias", [dt], False, "bias"),
        ]
    return out


def _mel_filters(n_mel=80, n_fft=201, seed=7):
    """Triangular-ish non-negative filterbank.  The values are free parameters of the file (the reference reads
    them from the model, whisper.cpp:531-538); a banded bank keeps the log-mel dynamic range realistic."""
    f = np.zeros((n_mel, n_fft), np.float32)
    # mel-like warping: denser at low frequencies
    centres = np.expm1(np.linspace(0, np.log1p(n_fft - 2.0), n_mel))
    centres = np.maximum(centres, np.arange(n_mel) * 0.9 + 0.5)
    width = np.maximum(np.gradient(centres), 1.0) * 1.5
    k = np.arange(n_fft, dtype=np.float64)
    for j in range(n_mel):
        tri = np.maximum(0.0, 1.0 - np.abs(k - centres[j]) / width[j])
        s = tri.sum()
        f[j] = (tri / max(s, 1e-9) * 0.05).astype(np.float32)
    return f


def tokenizer_test_words(i: int) -> bytes:
    """Vocabulary of the "-words" model variants: letters, digits, space and a few multi-character entries, so that the GPT-2
    pre-split + greedy longest match of the reference tokenizer (whisper.cpp:2192-2245) has something to match."""
    special = {100: b" hello", 101: b"hel", 102: b"lo", 103: b" 12", 104: b"345", 105: b" wor", 106: b"ld", 107: b"'s", 108: b" ,", 109: b" world"}
    if i < 26:
        return bytes([97 + i])
    if i < 36:
        return bytes([48 + i - 26])
    if i == 36:
        return b" "
    if i in special:
        return special[i]
    return (" t%d" % i).encode() if i != 50256 else b""


# ---------------------------------------------------------------------------------------------------------------------
# "Scripted" synthetic models (name suffix "-sc").
#
# A decoder with purely random weights is useless as a parity fixture: whatever the audio and the history, it collapses onto one
# repeated token (a fixed point of token -> next token), so "identical greedy tokens" proves little.  A scripted model keeps
# random weights everywhere (every kernel still chews on generic data) but confines them to the last d-64 "noise" dimensions of
# the decoder's residual stream and uses the first 64 dimensions as a clean CODE channel:
#
#   * every ACTIVE token (64 text tokens, timestamps, EOT, sot / transcribe / translate) carries an orthogonal code in its
#     embedding row; all other rows have no code and can never win;
#   * the first hidden units of the LAST decoder layer's MLP are a lookup keyed on the input token's code: they erase it and
#     write the code of the SUCCESSOR — a Markov chain  init-timestamp -> 2-4 text tokens -> end timestamp -> start timestamp
#     -> text ... -> EOT  with increasing timestamps, i.e. what whisper_full's segment / seek logic expects (whisper.cpp:2926-3016);
#   * every text step writes the codes of TWO equally scored candidates; which one wins is decided by the ordinary random part of
#     the logits, which depends on the audio (cross-attention) and on the whole history (self-attention over the KV cache).
#
# Logits are therefore peaked (successor vs everything else: ~10), sequences vary from chunk to chunk, and a wrong KV cache or
# cross-attention flips branch decisions.  The branch margins are Gaussian (std ~3): fixtures record the reference's top-2 gap at
# every step, and the generator only keeps inputs whose gaps stay clear of the parity tolerance.
SC_NC = 64                      # code dimensions: [0,16) segment code, [16,32) step code, [32,64) special-token code
SC_SEG_LEN = (4, 3, 4, 2, 4, 3, 4, 4)
SC_GAMMA_NOISE = 3.0
# Calibration (tools/calibrate_script.py, stored in whisper_b200/script_calib.npz): a random network's outputs are ~95 % one constant
# vector.  The scripted models subtract the measured constant from the encoder's ln_post output and from the decoder's final
# LayerNorm output (noise dimensions) and amplify what is left — the part that depends on the audio, the position and the history.
SC_CENTER = None                # mean of the decoder's final LayerNorm output at unit gain, [d]
SC_GAIN = 1.0
SC_ENC_CENTER = None            # mean of the encoder's ln_post output at unit gain, [d]
SC_ENC_GAIN = 1.0
SC_NOISE_LOGIT_RMS = 0.9
SC_ENC_GAIN_CALIBRATED = 3.0


def _hadamard(n):
    h = np.array([[1.0]])
    while h.shape[0] < n:
        h = np.block([[h, h], [h, -h]])
    return h


SC_SPARSE = False               # "-sc1" models: only the first text token of segments 0, 3 and 6 is a branch (long whisper_full runs)


def script_tokens(n_vocab: int):
    """The active tokens of a scripted model and the successor table.  Returns (codes, succ):
    codes: {token_id: unit-norm float64[64] code},  succ: {token_id: [successor ids]} (two entries = a branch)."""
    sh = 1 if n_vocab == 51865 else 0
    eot, sot, beg = 50256 + sh, 50257 + sh, 50363 + sh      # multilingual files shift the specials by one (whisper.cpp:575-583)
    translate, transcribe = 50358, 50359
    h16 = _hadamard(16) / 4.0
    h32 = _hadamard(32) / np.sqrt(32.0)
    codes, succ = {}, {}

    def text_id(k, j, v):
        return 1000 + 400 * k + 50 * j + 7 * v + 3 * k * j

    def text_code(k, j, v):
        c = np.zeros(SC_NC)
        c[0:16] = h16[1 + k]
        c[16:32] = h16[1 + 2 * j + v]
        return c / np.sqrt(2.0)

    def special_code(i):
        c = np.zeros(SC_NC)
        c[32:64] = h32[1 + i]
        return c

    ts_end = [beg + 100 * (k + 1) for k in range(8)]
    ts_start = [t + 1 for t in ts_end[:7]]
    init, init2 = beg, beg + 4
    # multilingual models: two language tokens (en, de) are active so that the distribution after [sot] — what
    # whisper_lang_auto_detect reads (whisper.cpp:2428-2495) — is a real, audio-dependent decision between them
    langs = [sot + 1 + 0, sot + 1 + 2] if sh else []
    specials = [eot, sot, transcribe, translate, init, init2] + ts_end + ts_start + langs
    for i, t in enumerate(specials):
        codes[t] = special_code(i)
    for k in range(8):
        for j in range(4):
            for v in range(2):
                codes[text_id(k, j, v)] = text_code(k, j, v)
    assert len(set(codes)) == len(specials) + 64

    def seg_first(k):
        if SC_SPARSE and k not in (0, 3, 6):
            return [text_id(k, 0, k & 1)]
        return [text_id(k, 0, 0), text_id(k, 0, 1)]
    succ[sot] = langs if sh else [init]
    succ[transcribe] = [init]
    for t in langs:
        succ[t] = [transcribe]
    succ[translate] = [init2]
    succ[init] = seg_first(0)
    succ[init2] = seg_first(4)
    succ[eot] = seg_first(0)          # never used by whisper_full (it stops at EOT); keeps fixed-length benchmark loops varied
    for k in range(8):
        for j in range(4):
            for v in range(2):
                if j >= SC_SEG_LEN[k] - 1:
                    succ[text_id(k, j, v)] = [ts_end[k]]
                elif SC_SPARSE:
                    succ[text_id(k, j, v)] = [text_id(k, j + 1, v ^ (j & 1))]     # no branch: the variant follows from the segment's first token
                else:
                    succ[text_id(k, j, v)] = [text_id(k, j + 1, 0), text_id(k, j + 1, 1)]
        succ[ts_end[k]] = [ts_start[k]] if k < 7 else [eot]
        if k < 7:
            succ[ts_start[k]] = seg_first(k + 1)
    return codes, succ


def _script_patch(name: str, ne, kind: str, data: np.ndarray, hp: "HParams") -> np.ndarray:
    """Turn one freshly drawn random decoder tensor into its scripted form (see above).  `data` is flat, ne[0] fastest."""
    if not name.startswith("decoder."):
        # a random encoder collapses too: its output is ~95 % one constant vector.  Centre ln_post on the calibrated mean and
        # amplify what is left, so that the cross-attention memories really depend on the audio and on the position
        if name == "encoder.ln_post.weight":
            return data * np.float32(SC_ENC_GAIN)
        if name == "encoder.ln_post.bias" and SC_ENC_CENTER is not None:
            return (-SC_ENC_GAIN * SC_ENC_CENTER).astype(np.float32)
        return data
    d, L = hp.n_text_state, hp.n_text_layer
    # code amplitude in the embedding: it has to dominate the noise part of the residual stream, whose norm grows like a random walk
    # over the 3 L sub-layers (~2 sqrt(d) for the 4-layer models)
    ge = 3.0 * np.sqrt(d) * max(1.0, np.sqrt(L / 4.0))
    if name == "decoder.token_embedding.weight":
        rows = data.reshape(ne[1], ne[0])
        rows[:, :SC_NC] = 0.0
        codes, _ = script_tokens(hp.n_vocab)
        for t, c in codes.items():
            rows[t, :SC_NC] = (ge * np.sqrt(2.0) * c).astype(np.float32)
        return rows.reshape(-1)
    if name == "decoder.positional_embedding":
        rows = data.reshape(ne[1], ne[0])
        rows[:, :SC_NC] = 0.0
        return rows.reshape(-1)
    if name == "decoder.ln.weight":
        data = data * np.float32(SC_GAMMA_NOISE * SC_GAIN)           # noise logits: rms ~3
        data[:SC_NC] = np.float32(27.5 / (ge * np.sqrt(d)))   # code logits: successor ~25, same-segment runners-up ~10, everything else ~0
        return data
    if name == "decoder.ln.bias":
        if SC_CENTER is not None:
            data[SC_NC:] = (-SC_GAMMA_NOISE * SC_GAIN * SC_CENTER[SC_NC:]).astype(np.float32)
        data[:SC_NC] = 0.0
        return data
    if not name.startswith("decoder.blocks."):
        return data
    il = int(name.split(".")[2])
    leaf = name.split(".", 3)[3]
    last = il == L - 1
    if kind == "mat":
        w = data.reshape(ne[1], ne[0])           # [out][in]
        reads_stream = leaf in ("cross_attn.query.weight", "mlp.0.weight")     # self-attention reads the token codes too: history matters
        writes_stream = leaf in ("attn.out.weight", "cross_attn.out.weight", "mlp.2.weight")
        if reads_stream:
            w[:, :SC_NC] = 0.0
        if writes_stream:
            w[:SC_NC, :] = 0.0
        if last and leaf in ("mlp.0.weight", "mlp.2.weight"):
            codes, succ = script_tokens(hp.n_vocab)
            toks = sorted(codes)
            kappa = 26.7 / np.sqrt(d)          # full match: kappa * ge sqrt(2) / sigma ~ 24 with sigma ~ 1.1 ge sqrt(2 / d), whatever ge is
            for u, t in enumerate(toks):
                if leaf == "mlp.0.weight":
                    w[u, :] = 0.0
                    w[u, :SC_NC] = (kappa * codes[t]).astype(np.float32)
                else:
                    target = np.zeros(SC_NC)
                    for s_ in succ[t]:
                        target += codes[s_]
                    if len(succ[t]) == 2:      # both text candidates share the segment code: count it once (specials have none)
                        target[0:16] *= 0.5
                    col = (ge * np.sqrt(2.0) / 3.0) * (target - codes[t])
                    w[:, u] = 0.0
                    w[:SC_NC, u] = col.astype(np.float32)
        return w.reshape(-1)
    if leaf in ("attn.out.bias", "cross_attn.out.bias", "mlp.2.bias"):
        data[:SC_NC] = 0.0
        return data
    if last and leaf == "mlp.0.bias":
        codes, _ = script_tokens(hp.n_vocab)
        data[:len(codes)] = np.float32(-18.0)
        return data
    if leaf.endswith("_ln.weight"):
        data[:SC_NC] = 1.0
        return data
    if leaf.endswith("_ln.bias"):
        data[:SC_NC] = 0.0
        return data
    return data


def write_model(path: str, name_or_hp, seed: int = 1234, emb_scale: float = 3.0, ts_boost: float = 1.0, eot_boost: float = 1.0, words=None, script: bool = False) -> HParams:
    """Write a synthetic ggml model file.  Matrices ~ N(0, 1/fan_in) stored f16; LN gamma = 1 + N(0, 0.01);
    biases N(0, 0.01); positional embeddings N(0, 0.01) (SURVEY.md §8(d)); the token embedding is scaled by
    `emb_scale` so that greedy decisions are not near-ties on random weights (SURVEY.md §7 "Parity definition")."""
    hp = MODELS[name_or_hp] if isinstance(name_or_hp, str) else name_or_hp
    rng = np.random.default_rng(seed)
    tmp = path + ".tmp%d" % os.getpid()
    with open(tmp, "wb") as f:
        f.write(struct.pack("<I", GGML_MAGIC))
        f.write(struct.pack("<11i", *hp.as_list()))
        filt = _mel_filters(hp.n_mels, 201)
        f.write(struct.pack("<2i", hp.n_mels, 201))
        f.write(filt.astype("<f4").tobytes())
        n_words = 50257  # as in real files; the loader synthesises the remaining special tokens (whisper.cpp:585-607)
        f.write(struct.pack("<i", n_words))
        chunks = []
        for i in range(n_words):
            w = words(i) if words else ((" t%d" % i).encode() if i != 50256 else b"")
            chunks.append(struct.pack("<I", len(w)) + w)
        f.write(b"".join(chunks))
        for name, ne, is_f16, kind in tensor_list(hp):
            n = int(np.prod(ne))
            if kind == "mat":
                fan_in = ne[0] if len(ne) == 2 else ne[0] * ne[1]
                data = rng.standard_normal(n, dtype=np.float32) * np.float32(1.0 / np.sqrt(fan_in))
            elif kind == "emb":
                data = rng.standard_normal(n, dtype=np.float32) * np.float32(emb_scale / np.sqrt(ne[0]))
                if ts_boost != 1.0 or eot_boost != 1.0:
                    # "-ts" variants: larger timestamp / end-of-text rows, so that greedy decoding on random weights emits timestamps
                    # and EOT and the transcription driver's windowing / segment logic gets exercised
                    rows = data.reshape(ne[1], ne[0])
                    sh = 1 if hp.n_vocab == 51865 else 0
                    rows[50363 + sh:] *= np.float32(ts_boost)
                    rows[50256 + sh] *= np.float32(eot_boost)
            elif kind == "gamma":
                data = 1.0 + rng.standard_normal(n, dtype=np.float32) * np.float32(0.01)
            elif kind == "pos":
                data = rng.standard_normal(n, dtype=np.float32) * np.float32(0.01)
            else:
                data = rng.standard_normal(n, dtype=np.float32) * np.float32(0.01)
            if script:
                data = _script_patch(name, ne, kind, data, hp)
            nb = name.encode()
            f.write(struct.pack("<3i", len(ne), len(nb), 1 if is_f16 else 0))
            f.write(struct.pack("<%di" % len(ne), *ne))
            f.write(nb)
            f.write(data.astype("<f2" if is_f16 else "<f4").tobytes())
    os.replace(tmp, path)
    return hp


CALIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "script_calib.npz")


def write_script_model(path: str, base: str, seed: int = 1234, stage: int = 2, calib: dict | None = None, sparse: bool = False):
    """Write the scripted variant of model `base`.  stage 0: no centring (calibration pass 1), 1: encoder centred (pass 2),
    2: final model — needs the calibration entries of (base, seed) in script_calib.npz (or `calib`)."""
    global SC_CENTER, SC_GAIN, SC_ENC_CENTER, SC_ENC_GAIN, SC_SPARSE
    if calib is None and stage > 0:
        if not os.path.exists(CALIB_PATH):
            raise RuntimeError("no %s: run tools/calibrate_script.py (needs oracle/_ref)" % CALIB_PATH)
        z = np.load(CALIB_PATH)
        key = "%s_%d" % (base, seed)
        if key + "_enc" not in z:
            raise RuntimeError("scripted model %s (seed %d) has no calibration entry: run tools/calibrate_script.py %s" % (base, seed, base))
        calib = {"enc": z[key + "_enc"], "dec": z[key + "_dec"], "var": float(z[key + "_var"])}
    SC_ENC_CENTER, SC_ENC_GAIN = (calib["enc"], SC_ENC_GAIN_CALIBRATED) if stage >= 1 else (None, 1.0)
    if stage >= 2:
        # gain such that the variable ("noise") part of the logits has rms ~SC_NOISE_LOGIT_RMS: branch margins of a few units against
        # code margins of ~10.  noise logit rms = (emb_scale / sqrt(d)) * |variable part of z| * gamma
        d = MODELS[base].n_text_state
        SC_CENTER, SC_GAIN = calib["dec"], SC_NOISE_LOGIT_RMS * np.sqrt(d) / (3.0 * SC_GAMMA_NOISE * calib["var"])
    else:
        SC_CENTER, SC_GAIN = None, 1.0
    SC_SPARSE = sparse
    try:
        return write_model(path, base, seed, script=True)
    finally:
        SC_CENTER, SC_GAIN, SC_ENC_CENTER, SC_ENC_GAIN, SC_SPARSE = None, 1.0, None, 1.0, False


def model_path(name: str, seed: int = 1234, cache_dir: str | None = None) -> str:
    """Return (creating on first use) the cached synthetic model file for `name`.  The default cache is per user under the system's
    temporary directory: on a shared host another user's cache would be unwritable, and its files not ours to trust."""
    cache_dir = cache_dir or os.environ.get("WSP_MODEL_CACHE") or os.path.join(tempfile.gettempdir(), "wsp_models-%d" % os.getuid())
    os.makedirs(cache_dir, exist_ok=True)
    p = os.path.join(cache_dir, "ggml-%s-synth%d%s.bin" % (name, seed, "-r2" if name.endswith(("-sc", "-sc1")) else ""))
    if not os.path.exists(p):
        if name.endswith("-sc"):
            write_script_model(p, name[:-3], seed)
        elif name.endswith("-sc1"):
            write_script_model(p, name[:-4], seed, sparse=True)
        elif name.endswith("-ts"):
            write_model(p, name[:-3], seed, ts_boost=1.3, eot_boost=2.2)
        elif name.endswith("-words"):
            write_model(p, name[:-6], seed, words=tokenizer_test_words)
        else:
            write_model(p, name, seed)
    return p


def lcg_u32(seed: int, n: int) -> np.ndarray:
    """x_{k+1} = x_k * 1664525 + 1013904223 (mod 2^32), vectorised by doubling.  Returns x_1..x_n."""
    A = np.array([1664525], np.uint64)
    C = np.array([1013904223], np.uint64)
    M = np.uint64(0xFFFFFFFF)
    while A.size < n:
        Am, Cm = A[-1], C[-1]
        A2 = (A * Am) & M
        C2 = ((A * Cm) & M) + C & M
        A = np.concatenate([A, A2])
        C = np.concatenate([C, C2 & M])
    A, C = A[:n], C[:n]
    x = ((A * np.uint64(seed & 0xFFFFFFFF)) & M) + C & M
    return x.astype(np.uint32)


def synth_pcm(chunk_id: int = 0, n_samples: int = 480000, seed: int = 12345) -> np.ndarray:
    """30 s of 16 kHz mono f32: 0.3*sin(2*pi*440*i/16000) + a slow chirp + 0.05*U(-0.5,0.5)  (SURVEY.md §8(d))."""
    i = np.arange(n_samples, dtype=np.float64)
    u = lcg_u32(seed + chunk_id, n_samples).astype(np.float64) / 4294967296.0 - 0.5
    # the tone / envelope parameters cycle with period 16 (+ a small drift per cycle) so that every chunk id stays inside the family of
    # clips the scripted models were calibrated on (tools/calibrate_script.py); the noise always differs
    k, cyc = chunk_id % 16, chunk_id // 16
    f2 = 180.0 + 40.0 * k + 7.0 * cyc
    x = 0.3 * np.sin(2 * np.pi * 440.0 * i / 16000.0) + 0.1 * np.sin(2 * np.pi * (f2 + i * (900.0 / n_samples)) * i / 16000.0) + 0.05 * u
    # amplitude envelope so frames differ (speech-like energy bursts)
    env = 0.55 + 0.45 * np.sin(2 * np.pi * i / 16000.0 * (0.7 + 0.13 * k + 0.011 * cyc))
    return (x * env).astype(np.float32)
