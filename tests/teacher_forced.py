"""Teacher-forced restatement of the decoder for whole token sequences (tests only).

oracle/whisper_np.NpDecoder steps one call at a time and walks the reference's f16 V^T*P chains key by key in Python: about a
minute for a 447-token sequence.  restate() evaluates every teacher-forced position of a layer together.  Everything but the chains
runs row by row through the very numpy calls NpDecoder makes for one row, so single steps come out bitwise equal to it
(tests/test_decoder_depth.py proves that); the chains walk the keys once for all rows, each row with its own key partition.

`bug` injects a plausible fault of the step kernel (decode_flow.cu) into the restatement, so that the tests can show their
comparisons would notice it:
  "lost_slot"   the oldest CR cached rows never reach self-attention once more than one ring slot is in use
  "last_round"  the last round of self-attention V rows is skipped when a part's key range takes several rounds
  "own_part"    this step's own V row goes to the part after its own (pOwn off by one): into another chain, or lost past the last part
  "pos_shift"   the positional embedding row of position n_past + 1 is added instead of n_past
"""
from __future__ import annotations

import numpy as np

from oracle import whisper_np as wn

F16, F32 = np.float16, np.float32


def ring_rows(d: int) -> int:
    """CR of decode_flow.cu's Cfg<D>: K/V rows per ring slot, 128 for d <= 1024 and 160 for d = 1280."""
    rs = 2 * d + 64
    slot = max(8 * rs, 16384)
    return (slot // 128) & ~7


def v_round_rows(d: int, threads: int) -> int:
    """RR of decode_flow.cu: V rows of one part per slot (the four 64-thread groups own PG consecutive parts each)."""
    ng = min(threads, 4)
    pg = (threads + ng - 1) // ng
    return ring_rows(d) // pg


def _chains(P, Vh, nk, dc, threads, skip=None, own_to=None):
    """The reference's V^T*P for R rows at once (whisper_np.pv_mad_f16 per row).  P [H][R][nkmax] (masked keys exactly 0),
    Vh [H][nkmax][64] f16 values, nk [R] keys of each row's call, dc [R] keys per part of each row.  skip [R][nkmax] bool: keys left
    out of the chain; own_to [R]: part whose chain the row's last key (its own) closes instead of the part it falls into."""
    H, R, nkmax = P.shape
    if R == 0:
        return np.zeros((H, 0, Vh.shape[2]), F32)
    parts = np.arange(threads)[:, None]
    y = np.zeros((H, threads, R, Vh.shape[2]), F32)
    rows = np.arange(R)
    own = None
    if own_to is not None:
        own = nk - 1
        skip = np.zeros((R, nkmax), bool) if skip is None else skip.copy()
        skip[rows, own] = True
    for t in range(int(dc.max())):
        j = parts * dc[None, :] + t                                          # [threads][R]
        valid = (t < dc)[None, :] & (j < nk[None, :])
        if skip is not None:
            valid &= ~skip[rows[None, :], np.minimum(j, nkmax - 1)]
        jj = np.minimum(j, nkmax - 1)
        Vj = Vh[:, jj, :]                                                    # [H][threads][R][64]
        Pj = P[:, rows[None, :], jj]                                         # [H][threads][R]
        acc = Vj.astype(np.float64) * Pj[..., None].astype(np.float64) + y.astype(np.float64)
        y = np.where(valid[None, :, :, None], acc.astype(F32).astype(F16).astype(F32), y)
    if own_to is not None:
        Vo = Vh[:, own, :]                                                   # [H][R][64]
        Po = P[:, rows, own]
        r = rows[own_to < threads]             # a part past the last one is not there: the row is lost
        to = own_to[r]
        acc = Vo[:, r].astype(np.float64) * Po[:, r, None].astype(np.float64) + y[:, to, r].astype(np.float64)
        y[:, to, r] = acc.astype(F32).astype(F16).astype(F32)
    out = y[:, 0]
    for p in range(1, threads):
        out = (out + y[:, p]).astype(F32)
    return out                                                               # [H][R][64]


def restate(m: wn.NpModel, ck, cv, tokens, threads: int, n_past: int = 0, prefix=None, prefill: bool = False,
            logit_rows=None, bug: str | None = None, attn_hook=None):
    """Decoder outputs for tokens[r] at position n_past + r, every earlier position teacher-forced.

    prefill=False: each row is its own single-token call (whisper_decode at n_past + r): keys per part ceil((n_past + r + 1) / threads).
    prefill=True:  the rows are one call of len(tokens) tokens: keys per part ceil((n_past + len(tokens)) / threads) for every row.
    prefix: (k, v) [L][>= n_past][d] cache rows of the earlier positions (required when n_past > 0).
    attn_hook(layer, "self" | "cross", A [H][rows][64]) may replace an attention output (a control's fault); rows are all R, or in
    the last layer only the logit rows.
    Returns (logits [len(logit_rows)][n_vocab], self_k [L][n_past + R][d], self_v)."""
    d, H, L = m.n_text_state, m.n_text_head, m.n_text_layer
    toks = np.asarray(tokens, np.int64)
    R = toks.size
    pos = n_past + np.arange(R)
    nk = pos + 1
    dc = np.full(R, (n_past + R + threads - 1) // threads) if prefill else (nk + threads - 1) // threads
    cr, rr = ring_rows(d), v_round_rows(d, threads)
    s = F32(np.power(64.0, -0.25))
    te = m["decoder.token_embedding.weight"]
    pe = m["decoder.positional_embedding"]
    shift = 1 if bug == "pos_shift" else 0
    x = [te[toks[r:r + 1]] + pe[pos[r] + shift:pos[r] + shift + 1] for r in range(R)]
    kc = np.zeros((L, n_past + R, d), F32)
    vc = np.zeros((L, n_past + R, d), F32)
    if n_past:
        kc[:, :n_past] = prefix[0][:, :n_past]
        vc[:, :n_past] = prefix[1][:, :n_past]
    skip = own_to = None
    nkmax = n_past + R
    if bug == "lost_slot":             # the ring's first slot (rows [0, CR)) lost whenever the cached rows need more than one
        skip = (np.arange(nkmax)[None, :] < cr) & ((nk - 1) > cr)[:, None]
    elif bug == "last_round":          # chain offsets in the last of several rounds never arrive (the own row still does)
        t = np.arange(nkmax)[None, :] - (np.arange(nkmax)[None, :] // dc[:, None]) * dc[:, None]
        rounds = (dc + rr - 1) // rr
        skip = (t >= ((rounds - 1) * rr)[:, None]) & (rounds > 1)[:, None] & (np.arange(nkmax)[None, :] < (nk - 1)[:, None])
    elif bug == "own_part":
        own_to = (nk - 1) // dc + 1
    for il in range(L):
        p = "decoder.blocks.%d." % il
        Qs = []
        for r in range(R):
            cur = wn.norm(x[r], m[p + "attn_ln.weight"], m[p + "attn_ln.bias"])
            Q = (wn.mul_mat(m[p + "attn.query.weight"], cur) + m[p + "attn.query.bias"]) * s
            K = wn.mul_mat(m[p + "attn.key.weight"], cur) * s
            V = wn.mul_mat(m[p + "attn.value.weight"], cur) + m[p + "attn.value.bias"]
            kc[il, pos[r]] = wn.r16(K)[0]
            vc[il, pos[r]] = wn.r16(V)[0]
            Qs.append(wn.r16(Q).reshape(1, H, 64).transpose(1, 0, 2))
        Vh_all = vc[il].reshape(nkmax, H, 64).transpose(1, 0, 2)
        # past the last layer's K/V rows only the rows whose logits are asked for matter
        act = np.arange(R) if il < L - 1 or logit_rows is None else np.array(sorted(set(int(r) for r in logit_rows)), np.int64)
        P = np.zeros((H, act.size, nkmax), F32)
        for a, r in enumerate(act):
            n = int(nk[r]) if not prefill else nkmax
            S = np.einsum("hqd,hkd->hqk", Qs[r], kc[il, :n].reshape(n, H, 64).transpose(1, 0, 2)).astype(F32)
            keep = np.arange(n) <= pos[r]
            if bug == "lost_slot":
                keep &= ~skip[r, :n]
            S = np.where(keep[None, None, :], S, -np.inf).astype(F32)
            P[:, a, :n] = wn.softmax_rows(S)[:, 0]
        A = _chains(P, Vh_all, np.full(act.size, nkmax) if prefill else nk[act], dc[act], threads,
                    skip=None if bug == "lost_slot" or skip is None else skip[act], own_to=None if own_to is None else own_to[act])
        if attn_hook is not None:
            A = attn_hook(il, "self", A)
        Tk = ck.shape[1]
        Kx = ck[il].reshape(Tk, H, 64).transpose(1, 0, 2)
        Vx = cv[il].reshape(Tk, H, 64).transpose(1, 0, 2)
        Px = np.zeros((H, act.size, Tk), F32)
        for a, r in enumerate(act):
            cur = A[:, a:a + 1].transpose(1, 0, 2).reshape(1, d)
            cur = wn.mul_mat(m[p + "attn.out.weight"], cur) + m[p + "attn.out.bias"]
            x[r] = cur + x[r]
            cur = wn.norm(x[r], m[p + "cross_attn_ln.weight"], m[p + "cross_attn_ln.bias"])
            Q = (wn.mul_mat(m[p + "cross_attn.query.weight"], cur) + m[p + "cross_attn.query.bias"]) * s
            Qh = wn.r16(Q).reshape(1, H, 64).transpose(1, 0, 2)
            Px[:, a, :] = wn.softmax_rows(np.einsum("hqd,hkd->hqk", Qh, Kx).astype(F32))[:, 0]
        Ax = _chains(Px, Vx, np.full(act.size, Tk), np.full(act.size, (Tk + threads - 1) // threads), threads)
        if attn_hook is not None:
            Ax = attn_hook(il, "cross", Ax)
        for a, r in enumerate(act):
            cur = Ax[:, a:a + 1].transpose(1, 0, 2).reshape(1, d)
            cur = wn.mul_mat(m[p + "cross_attn.out.weight"], cur) + m[p + "cross_attn.out.bias"]
            x[r] = cur + x[r]
            cur = wn.norm(x[r], m[p + "mlp_ln.weight"], m[p + "mlp_ln.bias"])
            cur = wn.gelu(wn.mul_mat(m[p + "mlp.0.weight"], cur) + m[p + "mlp.0.bias"])
            cur = wn.mul_mat(m[p + "mlp.2.weight"], cur) + m[p + "mlp.2.bias"]
            x[r] = cur + x[r]
    rows = range(R) if logit_rows is None else logit_rows
    lg = [wn.mul_mat(te, wn.norm(x[r], m["decoder.ln.weight"], m["decoder.ln.bias"]))[0] for r in rows]
    return (np.stack(lg) if lg else np.zeros((0, m.n_vocab), F32)), kc, vc
