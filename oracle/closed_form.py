"""fp64 numpy closed-form restatement with HAND-DERIVED gradients (TEST INFRASTRUCTURE).

``oracle/ref_port.py`` follows the reference op by op and gets gradients from autograd, like the
reference does.  This file states the same mathematics in closed form together with the analytic
backward chain that the CUDA kernels implement (SURVEY.md section 8 rows a4 and a9), so the chain
can be checked against autograd on the CPU before any kernel is trusted.  Parity is pinned through
``tests/test_oracle_golden.py`` (same golden vectors as ref_port).

Only tests / smoke / bench's CPU leg may import this module.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import numpy as np


def _softmax(x, axis):
    x = x - np.max(x, axis=axis, keepdims=True)
    e = np.exp(x)
    return e / e.sum(axis=axis, keepdims=True)


def _lse(x, axis):
    m = np.max(x, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return (m + np.log(np.exp(x - m).sum(axis=axis, keepdims=True))).squeeze(axis)


# ----------------------------------------------------------------------------------------------
# generator word attention, forward + backward                 networks/attention.py:25-79 (a3/a4)
# ----------------------------------------------------------------------------------------------
def word_attention_fwd(h, words, W, mask, scaled=True):
    """h [B,C,P], words [B,E,T], W [C,E], mask [B,T] -> ctx [B,C,P], attn [B,T,P], we [B,C,T]."""
    h, words, W = (np.asarray(a, np.float64) for a in (h, words, W))
    C = h.shape[1]
    sc = 1.0 / math.sqrt(C) if scaled else 1.0
    we = np.einsum("ce,bet->bct", W, words)
    s = np.einsum("bcp,bct->btp", h, we) * sc
    s = np.where((np.asarray(mask) == 0)[:, :, None], -np.inf, s)
    a = _softmax(s, axis=1)
    ctx = np.einsum("bct,btp->bcp", we, a)
    return ctx, a, we


def word_attention_bwd(h, words, W, mask, dctx, dattn=None, scaled=True):
    """Analytic gradients (SURVEY a4).  Returns dh [B,C,P], dwords [B,E,T], dW [C,E]."""
    h, words, W, dctx = (np.asarray(a, np.float64) for a in (h, words, W, dctx))
    C = h.shape[1]
    sc = 1.0 / math.sqrt(C) if scaled else 1.0
    _, a, we = word_attention_fwd(h, words, W, mask, scaled)
    g = np.einsum("bct,bcp->btp", we, dctx)
    if dattn is not None:
        g = g + np.asarray(dattn, np.float64)
    ds = a * (g - (a * g).sum(axis=1, keepdims=True))                      # softmax backward
    dh = sc * np.einsum("bct,btp->bcp", we, ds)
    dwe = np.einsum("bcp,btp->bct", dctx, a) + sc * np.einsum("bcp,btp->bct", h, ds)
    dW = np.einsum("bct,bet->ce", dwe, words)
    dwords = np.einsum("ce,bct->bet", W, dwe)
    return dh, dwords, dW


# ----------------------------------------------------------------------------------------------
# DAMSM words similarity, forward + backward                       losses/words_loss.py:43-86 (a8/a9)
# ----------------------------------------------------------------------------------------------
def _pair_block(c, w, gamma1):
    """c [Bi,D,R], w [D,L] -> s, alpha, beta [Bi,R,L], v [Bi,D,L]."""
    D = c.shape[1]
    s = np.einsum("bdr,dt->brt", c, w) / math.sqrt(D)
    alpha = _softmax(s, axis=2)
    e = np.exp(gamma1 * alpha)                       # gamma1*alpha in [0,gamma1]: no max needed
    beta = e / e.sum(axis=1, keepdims=True)
    v = np.einsum("bdr,brt->bdt", c, beta)
    return alpha, beta, v


def words_similarity_fwd(c, words, cap_lens, gamma1=4.0, gamma2=5.0, eps=1e-8):
    """c [Bi,D,R], words [Bc,D,T] -> m [Bi,Bc] (log-sum-exp of gamma2*cos; gamma3 NOT applied),
    cos list (per caption [Bi,L])."""
    c = np.asarray(c, np.float64)
    words = np.asarray(words, np.float64)
    Bi = c.shape[0]
    m = np.zeros((Bi, len(cap_lens)))
    for i, L in enumerate(int(x) for x in cap_lens):
        w = words[i, :, :L]
        _, _, v = _pair_block(c, w, gamma1)
        n = np.einsum("dt,bdt->bt", w, v)
        den = np.maximum(np.linalg.norm(w, axis=0)[None] * np.linalg.norm(v, axis=1), eps)
        m[:, i] = _lse(gamma2 * n / den, axis=1)
    return m


def words_similarity_bwd(c, words, cap_lens, dm, gamma1=4.0, gamma2=5.0, eps=1e-8):
    """dm [Bi,Bc] = dL/dm.  Returns dc [Bi,D,R], dwords [Bc,D,T] (zero for t >= L_i)."""
    c = np.asarray(c, np.float64)
    words = np.asarray(words, np.float64)
    dm = np.asarray(dm, np.float64)
    Bi, D, R = c.shape
    isd = 1.0 / math.sqrt(D)
    dc = np.zeros_like(c)
    dwords = np.zeros_like(words)
    for i, L in enumerate(int(x) for x in cap_lens):
        w = words[i, :, :L]
        alpha, beta, v = _pair_block(c, w, gamma1)
        n = np.einsum("dt,bdt->bt", w, v)
        p = np.linalg.norm(w, axis=0)[None]                      # [1,L]
        q = np.linalg.norm(v, axis=1)                            # [Bi,L]
        pq = p * q
        live = pq > eps
        den = np.maximum(pq, eps)
        cos = n / den
        dcos = dm[:, i:i + 1] * gamma2 * _softmax(gamma2 * cos, axis=1)
        dn = dcos / den
        with np.errstate(divide="ignore", invalid="ignore"):
            dp_over_p = np.where(live, -dcos * n / (den * p * p), 0.0)     # (dL/dp) / p
            dq_over_q = np.where(live, -dcos * n / (den * q * q), 0.0)     # (dL/dq) / q
        dv = dn[:, None, :] * w[None] + dq_over_q[:, None, :] * v          # [Bi,D,L]
        dw = np.einsum("bt,bdt->dt", dn, v) + dp_over_p.sum(0)[None] * w
        dc += np.einsum("bdt,brt->bdr", dv, beta)
        dbeta = np.einsum("bdr,bdt->brt", c, dv)
        dalpha = gamma1 * beta * (dbeta - (beta * dbeta).sum(axis=1, keepdims=True))
        ds = alpha * (dalpha - (alpha * dalpha).sum(axis=2, keepdims=True))
        dc += isd * np.einsum("brt,dt->bdr", ds, w)
        dw += isd * np.einsum("bdr,brt->dt", c, ds)
        dwords[i, :, :L] = dw
    return dc, dwords


def two_way_ce_fwd_bwd(sim, labels_row, labels_col=None, lam=1.0):
    """sim [Bi,Bc] (may contain -inf).  loss = lam * (mean_b CE(sim[b,:], labels_row[b]) +
    mean_i CE(sim[:,i], labels_col[i])).  Returns (loss, dsim)."""
    sim = np.asarray(sim, np.float64)
    Bi, Bc = sim.shape
    labels_row = np.asarray(labels_row)
    labels_col = labels_row if labels_col is None else np.asarray(labels_col)
    lse_r = _lse(sim, axis=1)
    lse_c = _lse(sim, axis=0)
    loss = (lse_r - sim[np.arange(Bi), labels_row]).mean() + \
           (lse_c - sim[labels_col, np.arange(Bc)]).mean()
    d = np.exp(sim - lse_r[:, None]) / Bi + np.exp(sim - lse_c[None, :]) / Bc
    d[np.arange(Bi), labels_row] -= 1.0 / Bi
    d[labels_col, np.arange(Bc)] -= 1.0 / Bc
    return lam * loss, lam * d


def class_mask(class_ids_rows, class_ids_cols=None, row_offset=0) -> Optional[np.ndarray]:
    if class_ids_rows is None:
        return None
    r = np.asarray(class_ids_rows)
    c = r if class_ids_cols is None else np.asarray(class_ids_cols)
    m = r[:, None] == c[None, :]
    idx = np.arange(len(r))
    m[idx, idx + row_offset] = False
    return m


def words_loss_fwd_bwd(c, words, labels, cap_lens, class_ids, gamma1=4.0, gamma2=5.0, gamma3=10.0,
                       lam=5.0, eps=1e-8):
    """Full WordsLoss value + analytic grads.  c [B,D,R], words [B,D,T]."""
    m = words_similarity_fwd(c, words, cap_lens, gamma1, gamma2, eps)
    sim = gamma3 * m
    cm = class_mask(class_ids)
    if cm is not None:
        sim = np.where(cm, -np.inf, sim)
    loss, dsim = two_way_ce_fwd_bwd(sim, labels, lam=lam)
    if cm is not None:
        dsim = np.where(cm, 0.0, dsim)
    dc, dwords = words_similarity_bwd(c, words, cap_lens, gamma3 * dsim, gamma1, gamma2, eps)
    return loss, sim, dc, dwords


def sentence_loss_fwd_bwd(cnn, rnn, labels, class_ids, gamma3=10.0, lam=5.0, eps=1e-8):
    """SentenceLoss value + analytic grads (sentence_loss.py:33-49)."""
    cnn = np.asarray(cnn, np.float64)
    rnn = np.asarray(rnn, np.float64)
    p = np.linalg.norm(cnn, axis=1)[:, None]
    q = np.linalg.norm(rnn, axis=1)[None, :]
    num = cnn @ rnn.T
    pq = p * q
    den = np.maximum(pq, eps)
    sc = gamma3 * num / den
    cm = class_mask(class_ids)
    if cm is not None:
        sc = np.where(cm, -np.inf, sc)
    loss, dsc = two_way_ce_fwd_bwd(sc, labels, lam=lam)
    if cm is not None:
        dsc = np.where(cm, 0.0, dsc)
    g = gamma3 * dsc / den                                     # dL/dnum
    live = pq > eps
    gn = np.where(live, g * num, 0.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        dcnn = g @ rnn - np.where(p > 0, gn.sum(1, keepdims=True) / (p * p), 0.0) * cnn
        drnn = g.T @ cnn - np.where(q.T > 0, gn.sum(0)[:, None] / (q.T * q.T), 0.0) * rnn
    return loss, sc, dcnn, drnn


def func_attention_fwd(query, context, gamma1=4.0, scaled=True):
    """query [B,D,L], context [B,D,R] -> wc [B,D,L], beta [B,L,R]."""
    q = np.asarray(query, np.float64)
    c = np.asarray(context, np.float64)
    D = q.shape[1]
    s = np.einsum("bdr,bdt->brt", c, q) * (1.0 / math.sqrt(D) if scaled else 1.0)
    alpha = _softmax(s, axis=2)
    beta = _softmax(gamma1 * alpha, axis=1)
    return np.einsum("bdr,brt->bdt", c, beta), beta.transpose(0, 2, 1)


def text_encoder_fwd(sd, captions, cap_lens):
    """the reference's RNNEncoder in eval mode (rnn_encoder.py:69-96: embedding -> dropout (identity) -> packed
    one-layer bidirectional LSTM -> zero-padded outputs), in fp64.  sd: its state dict (numpy arrays), captions
    [B,T] word indices, cap_lens [B].  Returns words [B,2H,max(cap_lens)], sentence [B,2H] = (last forward state,
    last backward state).  LSTM cell as torch.nn.LSTM: gates i, f, g, o stacked in the weight rows."""
    def sig(x):
        return 1.0 / (1.0 + np.exp(-x))

    emb = np.asarray(sd["embedding.weight"], np.float64)[np.asarray(captions)]          # [B,T,E]
    lens = [int(n) for n in cap_lens]
    B, Tm = emb.shape[0], max(lens)
    H = np.asarray(sd["rnn.weight_hh_l0"]).shape[1]
    words = np.zeros((B, 2 * H, Tm))
    sent = np.zeros((B, 2 * H))
    for d, sfx in enumerate(("", "_reverse")):
        wi, wh, bi, bh = (np.asarray(sd[f"rnn.{k}_l0{sfx}"], np.float64)
                          for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh"))
        for b in range(B):
            h, c = np.zeros(H), np.zeros(H)
            steps = range(lens[b]) if d == 0 else range(lens[b] - 1, -1, -1)
            for t in steps:
                z = wi @ emb[b, t] + bi + wh @ h + bh
                i, f, g, o = sig(z[:H]), sig(z[H:2 * H]), np.tanh(z[2 * H:3 * H]), sig(z[3 * H:])
                c = f * c + i * g
                h = o * np.tanh(c)
                words[b, d * H:(d + 1) * H, t] = h
            sent[b, d * H:(d + 1) * H] = h
    return words, sent
