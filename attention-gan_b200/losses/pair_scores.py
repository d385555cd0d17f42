"""Differentiable DAMSM scores of any list of (image, caption) pairs.

``DAMSMScorer.words_pairs`` / ``sentence_pairs`` score a pair list for evaluation; these two functions return the
same values with a gradient, so that a loss over a chosen set of pairs (hard negatives, a K-way listwise loss over
each image's candidates, generated images against their own captions) costs only those pairs instead of the dense
N x Nc similarity matrix:

    m   = words_pair_scores(img_features, words_emb, cap_lens, image_idx, caption_idx)    # [P]
    cos = sentence_pair_scores(cnn_code, sent_emb, image_idx, caption_idx)                # [P]
    loss = F.cross_entropy(gamma3 * m.view(N, K), torch.zeros(N, dtype=torch.long, device=m.device))

Forward: agb_damsm_pairs_train_fwd / agb_sent_cos_pairs_fwd; backward: agb_damsm_pairs_bwd / agb_sent_cos_pairs_bwd
(INTEGRATION.md §8).  Under ``torch.compile`` they go through the ``agb::damsm_pairs_train_fwd`` and
``agb::sent_cos_pairs_train_fwd`` custom ops, whose registered backward calls the same kernels.
"""
from __future__ import annotations

import torch

from ..agb_native import native, ops, torch_ops
from .damsm_core import as_device_i32, chunk_pairs, pair_index

_PAIR_MATH = ("f16", "bf16", "f16x2")


class _WordsPairs(torch.autograd.Function):
    """one chunk of pairs: m [P]; the training workspace is kept for the backward"""

    @staticmethod
    def forward(ctx, img, words, lens, pi, pc, gamma1, gamma2, math):
        m, ws = ops.damsm_pairs_train_fwd(img, words, lens, pi, pc, gamma1, gamma2, math)
        ctx.save_for_backward(img, words, lens, pi, pc)
        ctx.ws = ws
        ctx.cfg = (gamma1, gamma2, math)
        return m

    @staticmethod
    def backward(ctx, dm):
        img, words, lens, pi, pc = ctx.saved_tensors
        need_img, need_words = ctx.needs_input_grad[:2]
        dimg = dwords = None
        if need_img or need_words:
            if ctx.ws is None:
                raise RuntimeError(_TWICE)
            dimg, dw = ops.damsm_pairs_bwd(img, words, lens, pi, pc, *ctx.cfg, dm.float().contiguous(), ctx.ws,
                                           need_dwords=need_words, need_dimg=need_img)
            dwords = dw.transpose(1, 2) if need_words else None           # [Nc,D,T] view like words
        ctx.ws = None                             # the saved vectors are not needed again: free them now
        return dimg, dwords, None, None, None, None, None, None


class _SentencePairs(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cnn, rnn, pi, pc, eps):
        ctx.save_for_backward(cnn, rnn, pi, pc)
        ctx.eps = eps
        return ops.sent_cos_pairs_fwd(cnn, rnn, pi, pc, eps)

    @staticmethod
    def backward(ctx, dcos):
        cnn, rnn, pi, pc = ctx.saved_tensors
        need_c, need_r = ctx.needs_input_grad[:2]
        dc, dr = ops.sent_cos_pairs_bwd(cnn, rnn, pi, pc, ctx.eps, dcos.float().contiguous(), need_c, need_r)
        return dc, dr, None, None, None


_TWICE = ("words_pair_scores: a second backward through the same scores is not supported (the first one released "
          "the training workspace); compute the scores again")


def _traced_train_workspace_bytes(*args) -> int:
    return torch_ops.host_query("agb_damsm_pairs_train_workspace_bytes", *args)


def _traced_score_workspace_bytes(*args) -> int:
    return torch_ops.host_query("agb_damsm_pairs_workspace_bytes", *args)


def words_pair_scores(img_features: torch.Tensor, words_emb: torch.Tensor, cap_lens, image_idx, caption_idx, *,
                      gamma1: float = 4.0, gamma2: float = 5.0, math: str = "f16x2",
                      workspace_bytes: int = 4 << 30) -> torch.Tensor:
    """The DAMSM word-level score m [P] of the pairs (image_idx[p], caption_idx[p]), differentiable with respect to
    img_features [N,D,h,w] or [N,D,R] and words_emb [Nc,D,T] (any strides, e.g. the text encoder's transposed
    view); cap_lens [Nc]; image_idx, caption_idx [P] (numpy, int64 or int32; any order, duplicates allowed).

    m is bit for bit ``DAMSMScorer.words_pairs``'s for the same pairs and math ("f16x2", "f16" or "bf16"; the
    tensor-core range D = 256, T <= 32, R <= 320).  A pair with an index out of range or a caption of length 0 gives
    NaN and contributes to no gradient.  Gradients reach only what requires grad; images and captions in no valid
    pair, and padded word slots, get exactly 0.  A list whose training workspace exceeds workspace_bytes runs in
    contiguous chunks of pairs, each one autograd node holding its workspace until its backward.  Without a
    gradient to compute (autograd disabled, or no input requiring grad) the scores come from the scoring forward,
    which saves nothing."""
    if math not in _PAIR_MATH:
        raise ValueError(f"math must be one of {_PAIR_MATH} (pair scores run on the tensor cores)")
    mt = native.MATH_NAMES[math]
    ops.require_cuda(img_features, words_emb)
    img = img_features.reshape(img_features.shape[0], img_features.shape[1], -1).float().contiguous()
    words = words_emb.float()
    N, D, R = img.shape
    Nc, _, T = words.shape
    lens = as_device_i32(cap_lens, img.device)
    pi, pc = pair_index(image_idx, caption_idx, img.device)
    P = pi.shape[0]
    g1, g2 = float(gamma1), float(gamma2)
    compiling = torch.compiler.is_compiling()
    train = torch.is_grad_enabled() and (img.requires_grad or words.requires_grad)
    if train:
        ws_bytes = _traced_train_workspace_bytes if compiling else ops.damsm_pairs_train_workspace_bytes
    else:
        ws_bytes = _traced_score_workspace_bytes if compiling else ops.damsm_pairs_workspace_bytes
    per = chunk_pairs(N, Nc, max(P, 1), T, D, R, mt, ws_bytes, int(workspace_bytes))
    score_ws = None if train or compiling else ops._ws(ws_bytes(N, Nc, per, T, D, R, mt), img.device)
    parts = []
    for s in range(0, max(P, 1), per):
        a, b = pi[s:s + per], pc[s:s + per]
        if train and compiling:
            parts.append(torch.ops.agb.damsm_pairs_train_fwd(img, words, lens, a, b, g1, g2, mt)[0])
        elif train:
            parts.append(_WordsPairs.apply(img, words, lens, a, b, g1, g2, mt))
        elif compiling:
            parts.append(torch.ops.agb.damsm_pairs_fwd(img, words, lens, a, b, g1, g2, False, mt)[0])
        else:
            parts.append(ops.damsm_pairs_fwd(img, words, lens, a, b, g1, g2, mt, ws=score_ws)[0])
    return parts[0] if len(parts) == 1 else torch.cat(parts)


def sentence_pair_scores(cnn_code: torch.Tensor, sent_emb: torch.Tensor, image_idx, caption_idx,
                         eps: float = 1e-8) -> torch.Tensor:
    """The sentence cosine [P] of the pairs, differentiable with respect to cnn_code [N,D] and sent_emb [Nc,D]; bit
    for bit ``DAMSMScorer.sentence_pairs``'s value.  A pair with an index out of range gives NaN and no gradient."""
    ops.require_cuda(cnn_code, sent_emb)
    cnn = cnn_code.float().contiguous()
    rnn = sent_emb.float().contiguous()
    pi, pc = pair_index(image_idx, caption_idx, cnn.device)
    if torch.compiler.is_compiling():
        return torch.ops.agb.sent_cos_pairs_train_fwd(cnn, rnn, pi, pc, float(eps))
    return _SentencePairs.apply(cnn, rnn, pi, pc, float(eps))
