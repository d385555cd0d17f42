"""CPU restatement of the reference's word-region attention hot path (TEST INFRASTRUCTURE).

This file is the *oracle*: a torch-CPU restatement of what ku222/Attention-GAN computes on the
hot path, written from the formulas, not from the source text.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import
it.  The product (``attention-gan_b200/``) never does.

Parity status: PINNED.  ``oracle/make_golden.py`` imports the unmodified reference from
``/root/reference`` in the build container and stores its outputs (values and autograd
gradients) for seeded inputs under ``tests/golden/``; ``tests/test_oracle_golden.py`` checks every
function here against those vectors.

Reference lines each function follows (paths relative to the reference root):

* ``word_attention``      -> networks/attention.py:25-79   (AttentionModule.forward)
* ``func_attention``      -> networks/attention.py:82-121
* ``words_similarity``    -> losses/words_loss.py:43-86    (the per-caption loop)
* ``words_loss``          -> losses/words_loss.py:29-102
* ``sentence_loss``       -> losses/sentence_loss.py:12-50
* ``class_mask``          -> losses/words_loss.py:44-47,88-91 / losses/sentence_loss.py:17-25

All functions are differentiable through torch autograd, which is exactly how the reference gets
its gradients (it has no hand-written backward).
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# ----------------------------------------------------------------------------------------------
# generator word-context attention                                    networks/attention.py:25-79
# ----------------------------------------------------------------------------------------------
def word_attention(images: Tensor, words: Tensor, conv_weight: Tensor, mask: Tensor,
                   scaled: bool = True) -> Tuple[Tensor, Tensor]:
    """images [B,C,H,W], words [B,E,T], conv_weight [C,E,1,1] (bias-free 1x1 conv), mask [B,T]
    (0 = ignore the word).  Returns (context [B,C,H,W], attn [B,T,H,W]).

    attention.py:50-52  word projection  we = W e
    attention.py:59-61  scores h.we, optionally / sqrt(C)
    attention.py:65-68  mask -> -inf, softmax over the T words
    attention.py:73     context = sum_t attn * we
    """
    B, C, H, W = images.shape
    T = words.shape[2]
    we = torch.einsum("ce,bet->bct", conv_weight.reshape(C, -1), words)        # [B,C,T]
    h = images.reshape(B, C, H * W)
    s = torch.einsum("bcp,bct->bpt", h, we)                                     # [B,HW,T]
    if scaled:
        s = s * (1.0 / math.sqrt(C))
    s = s.masked_fill((mask == 0)[:, None, :], float("-inf"))
    a = torch.softmax(s, dim=2)                                                 # over words
    ctx = torch.einsum("bct,bpt->bcp", we, a)
    return ctx.reshape(B, C, H, W), a.transpose(1, 2).reshape(B, T, H, W)


# ----------------------------------------------------------------------------------------------
# functional region-word attention                                   networks/attention.py:82-121
# ----------------------------------------------------------------------------------------------
def func_attention(query: Tensor, context: Tensor, gamma1: float = 4.0,
                   scaled: bool = True) -> Tuple[Tensor, Tensor]:
    """query [B,D,L] (words), context [B,D,ih,iw] (regions).
    Returns (weighted_context [B,D,L], attn [B,L,ih,iw]).

    attention.py:99-101   s[b,r,t] = <c_r, q_t> (/ sqrt(D))
    attention.py:104      alpha = softmax over the L words          (implicit dim=1 of [B*R, L])
    attention.py:111-112  beta  = softmax over the R regions of gamma1*alpha
    attention.py:119      wc[:,t] = sum_r c_r beta[t,r]
    """
    B, D, L = query.shape
    ih, iw = context.shape[2], context.shape[3]
    c = context.reshape(B, D, ih * iw)
    s = torch.einsum("bdr,bdt->brt", c, query)
    if scaled:
        s = s * (1.0 / math.sqrt(D))
    alpha = torch.softmax(s, dim=2)
    beta = torch.softmax(alpha * gamma1, dim=1)                                 # [B,R,L]
    wc = torch.einsum("bdr,brt->bdt", c, beta)
    return wc, beta.transpose(1, 2).reshape(B, L, ih, iw)


# ----------------------------------------------------------------------------------------------
# class-id mask                                  words_loss.py:44-47,88-91 / sentence_loss.py:17-25
# ----------------------------------------------------------------------------------------------
def class_mask(class_ids_rows, class_ids_cols=None, row_offset: int = 0) -> Optional[Tensor]:
    """Boolean [Brow, Bcol]: True where the two samples share a class id but are not the same
    sample (global index of row r is ``row_offset + r``; columns are global)."""
    if class_ids_rows is None:
        return None
    r = np.asarray(class_ids_rows)
    c = r if class_ids_cols is None else np.asarray(class_ids_cols)
    m = r[:, None] == c[None, :]
    idx = np.arange(len(r))
    m[idx, idx + row_offset] = False
    return torch.from_numpy(m)


# ----------------------------------------------------------------------------------------------
# DAMSM words similarity matrix                                        losses/words_loss.py:43-86
# ----------------------------------------------------------------------------------------------
def words_similarity(img_features: Tensor, words_emb: Tensor, cap_lens: Sequence[int],
                     gamma1: float = 4.0, gamma2: float = 5.0, eps: float = 1e-8,
                     want_maps: bool = False, map_offset: int = 0
                     ) -> Tuple[Tensor, List[Tensor]]:
    """img_features [Bi,D,ih,iw], words_emb [Bc,D,T], cap_lens[Bc].
    Returns (m [Bi,Bc] with m[b,i] = log sum_t exp(gamma2 * cos(w_it, wc_bit)), att_maps).
    With want_maps, att_maps holds beta [1,L_i,ih,iw] of every matched pair (caption i, local image
    i - map_offset) that falls inside this row block (words_loss.py:63); map_offset is the global
    index of the first image row (0 in a single process).  gamma3 is applied by the caller
    (words_loss.py:93).
    """
    Bi, D = img_features.shape[0], img_features.shape[1]
    ih, iw = img_features.shape[2], img_features.shape[3]
    c = img_features.reshape(Bi, D, ih * iw)
    cols, maps = [], []
    for i, L in enumerate(int(x) for x in cap_lens):
        w = words_emb[i, :, :L]                                                 # [D,L]
        s = torch.einsum("bdr,dt->brt", c, w) * (1.0 / math.sqrt(D))            # attention.py:99-101
        alpha = torch.softmax(s, dim=2)                                         # attention.py:104
        beta = torch.softmax(alpha * gamma1, dim=1)                             # attention.py:111-112
        wc = torch.einsum("bdr,brt->bdt", c, beta)                              # attention.py:119
        if want_maps:
            b = i - map_offset
            if 0 <= b < Bi:
                maps.append(beta[b].transpose(0, 1).reshape(1, L, ih, iw))
        num = (wc * w[None]).sum(1)                                             # words_loss.py:24
        den = (wc.norm(2, dim=1) * w.norm(2, dim=0)[None]).clamp(min=eps)       # words_loss.py:25-27
        cos = num / den                                                         # [Bi,L]
        cols.append(torch.log(torch.exp(cos * gamma2).sum(1, keepdim=True)))    # words_loss.py:77-79
    return torch.cat(cols, 1), maps


def two_way_ce(sim: Tensor, labels: Tensor) -> Tensor:
    """CE(sim, labels) + CE(sim^T, labels), mean reduction   (words_loss.py:96-99)."""
    return F.cross_entropy(sim, labels) + F.cross_entropy(sim.t(), labels)


def words_loss(img_features: Tensor, words_emb: Tensor, labels: Tensor, cap_lens, class_ids,
               gamma1: float = 4.0, gamma2: float = 5.0, gamma3: float = 10.0,
               wlambda: float = 5.0) -> Tuple[Tensor, List[Tensor]]:
    """losses/words_loss.py:29-102 (single process: Bi == Bc == B)."""
    lens = cap_lens.tolist() if torch.is_tensor(cap_lens) else list(cap_lens)
    m, maps = words_similarity(img_features, words_emb, lens, gamma1, gamma2, want_maps=True)
    sim = m * gamma3
    cm = class_mask(class_ids)
    if cm is not None:
        # the reference writes -inf through .data (words_loss.py:95): no autograd edge, and the
        # softmax weight of a -inf logit is 0 anyway, so an out-of-place fill has the same grads.
        sim = sim.masked_fill(cm.to(sim.device), float("-inf"))
    return two_way_ce(sim, labels) * wlambda, maps


# ----------------------------------------------------------------------------------------------
# DAMSM sentence loss                                                losses/sentence_loss.py:12-50
# ----------------------------------------------------------------------------------------------
def sentence_similarity(cnn_code: Tensor, rnn_code: Tensor, gamma3: float = 10.0,
                        eps: float = 1e-8) -> Tensor:
    """[Bi,D] x [Bc,D] -> gamma3 * cosine matrix [Bi,Bc]   (sentence_loss.py:33-38)."""
    num = cnn_code @ rnn_code.t()
    den = (cnn_code.norm(2, dim=1, keepdim=True) * rnn_code.norm(2, dim=1, keepdim=True).t())
    return num / den.clamp(min=eps) * gamma3


def sentence_loss(cnn_code: Tensor, rnn_code: Tensor, labels: Tensor, class_ids,
                  gamma3: float = 10.0, slambda: float = 5.0, eps: float = 1e-8) -> Tensor:
    sc = sentence_similarity(cnn_code, rnn_code, gamma3, eps)
    cm = class_mask(class_ids)
    if cm is not None:
        sc = sc.masked_fill(cm.to(sc.device), float("-inf"))
    return two_way_ce(sc, labels) * slambda


# ----------------------------------------------------------------------------------------------
# seeded synthetic inputs (SURVEY.md section 8d)
# ----------------------------------------------------------------------------------------------
def synth_damsm(B: int, T: int = 18, D: int = 256, hw: int = 17, seed: int = 0,
                full_len: bool = False, n_classes: Optional[int] = None, trained_like: bool = False,
                dtype=torch.float32):
    """img_features [B,D,hw,hw], words_emb [B,D,T] as a transposed view of [B,T,D]
    (rnn_encoder.py:92), cnn_code/rnn_code [B,D], labels arange, cap_lens U{2..T}, class_ids."""
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(B, D, hw, hw, generator=g, dtype=torch.float32)
    wrd = torch.randn(B, T, D, generator=g, dtype=torch.float32)
    cnn = torch.randn(B, D, generator=g, dtype=torch.float32)
    rnn = torch.randn(B, D, generator=g, dtype=torch.float32)
    if trained_like:
        # a shared per-sample direction on top of the noise, so matched pairs really are more
        # similar (a partly-trained encoder).  gamma2*gamma3 = 50 amplifies the cosine, so a
        # signal of ~0.15 already moves the loss from ~2 log B to well under 1.
        a = 0.15 if trained_like is True else float(trained_like)
        u = torch.randn(B, D, generator=g, dtype=torch.float32)
        img = a * u[:, :, None, None] + img
        wrd = a * u[:, None, :] + wrd
        cnn, rnn = a * u + cnn, a * u + rnn
    if full_len:
        lens = torch.full((B,), T, dtype=torch.int64)
    else:
        lens = torch.randint(2, T + 1, (B,), generator=g, dtype=torch.int64)
        lens[0] = T
    cls = None
    if n_classes is not None:
        cls = torch.randint(0, n_classes, (B,), generator=g, dtype=torch.int64).numpy()
    labels = torch.arange(B, dtype=torch.int64)
    return (img.to(dtype), wrd.to(dtype).transpose(1, 2), cnn.to(dtype), rnn.to(dtype),
            labels, lens, cls)


def synth_attention(B: int, C: int = 32, E: int = 256, T: int = 18, hw: int = 64, seed: int = 0,
                    dtype=torch.float32):
    """images [B,C,hw,hw], words [B,E,T] (transposed view), conv weight [C,E,1,1] (Conv2d default
    init: U(-1/sqrt(E), 1/sqrt(E))), lens U{2..T} with one == T, int64 mask [B,T]."""
    g = torch.Generator().manual_seed(seed)
    images = torch.randn(B, C, hw, hw, generator=g, dtype=torch.float32)
    words = torch.randn(B, T, E, generator=g, dtype=torch.float32)
    bound = 1.0 / math.sqrt(E)
    weight = (torch.rand(C, E, 1, 1, generator=g, dtype=torch.float32) * 2 - 1) * bound
    lens = torch.randint(min(2, T), T + 1, (B,), generator=g, dtype=torch.int64)
    lens[0] = T
    mask = (torch.arange(T)[None, :] < lens[:, None]).to(torch.int64)
    return images.to(dtype), words.to(dtype).transpose(1, 2), weight.to(dtype), mask, lens


def synth_text_encoder(vocab: int, embdim: int = 300, nhidden: int = 256, seed: int = 0):
    """seeded state dict of the reference's RNNEncoder (bidirectional, nhidden // 2 per direction): embedding
    U(-0.1, 0.1) (rnn_encoder.py:48-50), LSTM tensors U(-1/sqrt(h), 1/sqrt(h)) (torch.nn.LSTM's default init)."""
    g = torch.Generator().manual_seed(seed)
    h = nhidden // 2
    sd = {"embedding.weight": (torch.rand(vocab, embdim, generator=g) * 2 - 1) * 0.1}
    for sfx in ("", "_reverse"):
        for k, shape in (("weight_ih", (4 * h, embdim)), ("weight_hh", (4 * h, h)), ("bias_ih", (4 * h,)),
                         ("bias_hh", (4 * h,))):
            sd[f"rnn.{k}_l0{sfx}"] = (torch.rand(*shape, generator=g) * 2 - 1) / math.sqrt(h)
    return sd
