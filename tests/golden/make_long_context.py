#!/usr/bin/env python
"""Generate tests/golden/long_context.npz from oracle/_ref — the reference's own CPU implementation, as make_golden.py does for the
other fixtures (same model files, PCM chunks and sub-sampling).  About 15 s on a CPU; two runs write identical files.

    python tests/golden/make_long_context.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle.ref import RefOracle  # noqa: E402
from tests.golden.make_golden import HERE, logits_sample, save  # noqa: E402
from whisper_b200 import synth  # noqa: E402

# The decoder deep into its context (tests/test_decoder_depth.py, tests/test_gpu_decoder_depth.py): whisper_full carries up to
# n_text_ctx / 2 = 224 earlier tokens into a window's prompt and decodes on until the window ends, so the step kernel runs with up to
# 447 rows in the self-KV cache.  A fixed, teacher-forced token sequence (no decision needs a margin) on the chunk of micro_en_30s:
# logits at checkpoints on both sides of every multiple of 128 rows (one K/V ring slot of the d = 128 step kernel), last-row logits of
# long prompts, and self-KV rows.
LONG_MODEL = "micro.en-sc"
LONG_LEN = 447                    # tokens [sot] + 446: single steps at n_past 0 .. 446 fill the context but for its last row
LONG_THREADS = (1, 2, 4)
LONG_CHECKPOINTS = (0, 1, 2, 3, 126, 127, 128, 129, 130, 254, 255, 256, 257, 258, 382, 383, 384, 385, 386, 443, 444, 445, 446)
# (n_past, N), run in this order after the single steps: carried-over prompts (223 + 224 = 447 rows), then prompts at the start of the
# context.  No call reads a row an earlier prefill wrote: the rows before each one's n_past are those of the single steps.
LONG_PREFILLS = ((223, 224), (130, 100), (0, 129), (0, 224), (0, 256))


def long_tokens(n_vocab: int, n: int = LONG_LEN, seed: int = 2024) -> np.ndarray:
    """[sot] then n - 1 ids drawn by synth.lcg_u32: three in four from the scripted model's active tokens, the rest arbitrary text ids."""
    codes, _ = synth.script_tokens(n_vocab)
    active = np.array(sorted(codes), np.int64)
    eot = 50256 + (1 if n_vocab == 51865 else 0)
    x = synth.lcg_u32(seed, n - 1).astype(np.int64)
    pick = np.where(x % 4 != 0, active[(x >> 2) % active.size], (x >> 8) % eot)
    return np.concatenate([[eot + 1], pick]).astype(np.int32)


def make_long_context(threads_list=LONG_THREADS):
    path = synth.model_path(LONG_MODEL)
    chunk = int(np.load(os.path.join(HERE, "micro_en_30s.npz"))["chunk"])
    o = RefOracle(path, threads=1)
    mel = o.pcm_to_mel(synth.synth_pcm(chunk))
    toks = long_tokens(o.n_vocab)
    assert toks[0] == o.special["sot"]
    cps = np.array(LONG_CHECKPOINTS, np.int32)
    out = {"chunk": np.int32(chunk), "tokens": toks, "checkpoints": cps, "prefills": np.array(LONG_PREFILLS, np.int32)}
    for th in threads_list:
        oo = RefOracle(path, threads=th)
        oo.set_mel(mel)
        oo.encode(0)
        lg_cp, mx_cp = [], []
        for p in range(LONG_LEN):
            lg, _ = oo.decode(toks[p:p + 1], p)
            if p in LONG_CHECKPOINTS:
                lg_cp.append(logits_sample(lg[0]))
                mx_cp.append(lg[0].max())
        out["t%d_logits" % th] = np.stack(lg_cp)
        out["t%d_logits_max" % th] = np.array(mx_cp, np.float32)
        k, v = oo.self_kv()
        last = oo.n_text_layer - 1
        out["t%d_self_k" % th] = k[[0, last]][:, cps].astype(np.float16)      # [2][checkpoints][d], layers 0 and L-1
        out["t%d_self_v" % th] = v[[0, last]][:, cps].astype(np.float16)
        pre_lg, pre_mx = [], []
        for n_past, n in LONG_PREFILLS:
            lg, _ = oo.decode(toks[n_past:n_past + n], n_past)
            pre_lg.append(logits_sample(lg[-1]))
            pre_mx.append(lg[-1].max())
        out["t%d_prefill_logits" % th] = np.stack(pre_lg)
        out["t%d_prefill_logits_max" % th] = np.array(pre_mx, np.float32)
        print("  long/t%d: logits rms %.2f at n_past 446" % (th, float(np.sqrt((out["t%d_logits" % th][-1] ** 2).mean()))), flush=True)
    return out


if __name__ == "__main__":
    save("long_context", make_long_context())
