"""The ``agb::`` operator library: the functions of ``ops.py`` as ``torch.library`` custom ops, so that
``torch.compile`` can trace the drop-ins without a graph break.

Every op body calls the matching ``ops.*`` function, i.e. the same native kernels the eager path launches, so a
compiled call computes what the eager call computes, bit for bit.  The drop-ins call these ops only while
``torch.compiler.is_compiling()``; eager calls keep going through their ``torch.autograd.Function``s and never
enter the dispatcher (DESIGN.md §1).

* Schemas take tensors and scalars only; an optional output that is not asked for comes back as an empty tensor.
* Every op has a fake kernel (shapes, dtypes, strides).  Workspace outputs are sized with the library's host
  queries, which are pure host code; registering the ops loads nothing (the library is opened at the first query).
* The differentiable forward ops (``word_attn_fwd``, ``word_attn_cat``, ``damsm_fwd``, ``contrastive``,
  ``sent_cos_fwd``, ``func_attention_fwd``, ``region_head_fwd``) are functional and carry their backward
  (``register_autograd``), which calls the matching backward op.  ``damsm_bwd`` and ``region_head_bwd`` write
  their staging into the workspace the forward returned and declare it mutated (``ws``); inductor reuses that
  buffer in place, it does not copy it.
* ``host_query`` is the library's host queries for code that ``torch.compile`` traces: it is evaluated once at
  trace time and its result is a constant of the graph.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import native as N
from . import ops

_LIB = "agb"


def _op(name: str, mutates_args=()):
    return torch.library.custom_op(f"{_LIB}::{name}", mutates_args=mutates_args, device_types="cuda")


def _none(t: Optional[Tensor], dev) -> Tensor:
    """an output that was not asked for: an empty tensor (custom ops return no None)"""
    return t if t is not None else torch.empty(0, dtype=torch.float32, device=dev)


def _opt(t: Tensor) -> Optional[Tensor]:
    return None if t.numel() == 0 else t


def _ws_like(nbytes: int, ref: Tensor) -> Tensor:
    return ref.new_empty((max(int(nbytes), 16),), dtype=torch.uint8)


@torch.compiler.assume_constant_result
def host_query(name: str, *args) -> int:
    """``native.lib().<name>(*args)`` as an int, for traced code (a constant of the graph)"""
    return int(getattr(N.lib(), name)(*args))


# ------------------------------------------------------------------------------------------------
# generator word-context attention
# ------------------------------------------------------------------------------------------------
@_op("word_attn_fwd")
def word_attn_fwd(images: Tensor, words: Tensor, weight: Tensor, mask: Tensor, scaled: bool,
                  want_attn: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """images [B,C,H,W] contiguous, words [B,E,T] fp32, weight [C,E] fp32 contiguous, mask [B,T] int64 ->
    (ctx [B,C,H,W], attn [B,T,H,W] (empty unless want_attn), we [B,C,T] fp32)"""
    ctx, attn, we = ops.word_attn_fwd(images, words, weight, mask, scaled, want_attn)
    return ctx, _none(attn, images.device), we


@word_attn_fwd.register_fake
def _(images, words, weight, mask, scaled, want_attn):
    B, C, H, W = images.shape
    T = words.shape[2]
    attn = images.new_empty((B, T, H, W)) if want_attn else images.new_empty((0,), dtype=torch.float32)
    return torch.empty_like(images), attn, images.new_empty((B, C, T), dtype=torch.float32)


@_op("word_attn_cat")
def word_attn_cat(images: Tensor, words: Tensor, weight: Tensor, mask: Tensor, scaled: bool,
                  want_attn: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """word_attn_fwd writing cat((images, ctx), 1): (out [B,2C,H,W], attn or empty, we); the kernel writes the
    context at channel offset C of the fresh buffer (AttentionModule.forward_into)"""
    B, C, H, W = images.shape
    out = images.new_empty((B, 2 * C, H, W))
    out[:, :C].copy_(images)
    _, attn, we = ops.word_attn_fwd(images, words, weight, mask, scaled, want_attn, ctx_out=out[:, C:])
    return out, _none(attn, images.device), we


@word_attn_cat.register_fake
def _(images, words, weight, mask, scaled, want_attn):
    B, C, H, W = images.shape
    T = words.shape[2]
    attn = images.new_empty((B, T, H, W)) if want_attn else images.new_empty((0,), dtype=torch.float32)
    return images.new_empty((B, 2 * C, H, W)), attn, images.new_empty((B, C, T), dtype=torch.float32)


@_op("word_attn_bwd")
def word_attn_bwd(images: Tensor, words: Tensor, weight: Tensor, mask: Tensor, we: Tensor, dctx: Tensor,
                  dattn: Optional[Tensor], scaled: bool, need_dwords: bool,
                  need_dweight: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """(dimages, dwords [B,E,T] fp32 or empty, dweight [C,E] fp32 or empty)"""
    di, dw, dwt = ops.word_attn_bwd(images, words, weight, mask, we, dctx, dattn, scaled, need_dwords, need_dweight)
    return di, _none(dw, images.device), _none(dwt, images.device)


@word_attn_bwd.register_fake
def _(images, words, weight, mask, we, dctx, dattn, scaled, need_dwords, need_dweight):
    B, C = images.shape[:2]
    E, T = words.shape[1], words.shape[2]
    f32 = dict(dtype=torch.float32)
    return (torch.empty_like(images), images.new_empty((B, E, T) if need_dwords else (0,), **f32),
            images.new_empty((C, E) if need_dweight else (0,), **f32))


def _word_attn_setup(ctx, inputs, output):
    images, words, weight, mask, scaled, want_attn = inputs
    ctx.save_for_backward(images, words, weight, mask, output[2])
    ctx.scaled = scaled
    ctx.mark_non_differentiable(output[2])
    if not want_attn:
        ctx.mark_non_differentiable(output[1])
    ctx.set_materialize_grads(False)


def _word_attn_backward(ctx, dctx, dattn, _dwe):
    images, words, weight, mask, we = ctx.saved_tensors
    need_img, need_words, need_w = ctx.needs_input_grad[:3]
    if dctx is None:
        dctx = torch.zeros_like(images)
    di, dw, dwt = torch.ops.agb.word_attn_bwd(images, words, weight, mask, we, dctx.to(images.dtype),
                                              None if dattn is None else dattn.to(images.dtype), ctx.scaled,
                                              need_words, need_w)
    return (di if need_img else None), (dw if need_words else None), (dwt if need_w else None), None, None, None


def _word_attn_cat_backward(ctx, dout, dattn, _dwe):
    images, words, weight, mask, we = ctx.saved_tensors
    need_img, need_words, need_w = ctx.needs_input_grad[:3]
    if dout is None:
        return None, None, None, None, None, None
    C = images.shape[1]
    dout = dout.to(images.dtype).contiguous()
    # d context is the second channel half of d out, read in place through its batch stride
    di, dw, dwt = torch.ops.agb.word_attn_bwd(images, words, weight, mask, we, dout[:, C:],
                                              None if dattn is None else dattn.to(images.dtype), ctx.scaled,
                                              need_words, need_w)
    di = di + dout[:, :C] if need_img else None                  # the identity half of the concatenation
    return di, (dw if need_words else None), (dwt if need_w else None), None, None, None


word_attn_fwd.register_autograd(_word_attn_backward, setup_context=_word_attn_setup)
word_attn_cat.register_autograd(_word_attn_cat_backward, setup_context=_word_attn_setup)


# ------------------------------------------------------------------------------------------------
# DAMSM word-region similarity, contrastive loss, sentence cosine
# ------------------------------------------------------------------------------------------------
def damsm_workspace_bytes(Bi: int, Bc: int, T: int, D: int, R: int, math: int) -> int:
    return int(N.lib().agb_damsm_workspace_bytes(Bi, Bc, T, D, R, math))


@_op("damsm_fwd")
def damsm_fwd(img: Tensor, words: Tensor, cap_lens: Tensor, cnn: Optional[Tensor], rnn: Optional[Tensor],
              gamma1: float, gamma2: float, eps: float, row_offset: int, want_att: bool, math: int,
              save: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """img [Bi,D,R] fp32 contiguous, words [Bc,D,T] fp32, cap_lens [Bc] int32 ->
    (m [Bi,Bc], att [Bi,T,R] or empty, scos [Bi,Bc] or empty (cnn/rnn given), ws uint8).  ws holds the packed
    operands (and with save=True the context vectors) that damsm_bwd reuses."""
    m, att, scos, ws = ops.damsm_fwd(img, words, cap_lens, gamma1, gamma2, eps, row_offset, want_att, math, cnn,
                                     rnn, keep_ws=True, save=save)
    return m, _none(att, img.device), _none(scos, img.device), ws


@damsm_fwd.register_fake
def _(img, words, cap_lens, cnn, rnn, gamma1, gamma2, eps, row_offset, want_att, math, save):
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    nbytes = damsm_workspace_bytes(Bi, Bc, T, D, R, math)
    if nbytes == 0:
        raise N.NativeError(f"DAMSM shape T={T} D={D} R={R} is unsupported for math mode {math}")
    f32 = dict(dtype=torch.float32)
    return (img.new_empty((Bi, Bc), **f32), img.new_empty((Bi, T, R) if want_att else (0,), **f32),
            img.new_empty((Bi, Bc) if cnn is not None else (0,), **f32), _ws_like(nbytes, img))


@_op("damsm_bwd", mutates_args=("ws",))
def damsm_bwd(img: Tensor, words: Tensor, cap_lens: Tensor, gamma1: float, gamma2: float, eps: float, dm: Tensor,
              gscale: Optional[Tensor], need_dwords: bool, math: int, m_fwd: Optional[Tensor],
              ws: Optional[Tensor], ws_saved: bool) -> Tuple[Tensor, Tensor]:
    """(dimg [Bi,D,R], dwords [Bc,T,D] word-major or empty).  ws: the workspace damsm_fwd returned, which this
    call overwrites with its staging (None: a workspace of its own)"""
    dimg, dwords = ops.damsm_bwd(img, words, cap_lens, gamma1, gamma2, eps, dm, gscale, need_dwords, math, m_fwd,
                                 ws, ws_saved)
    return dimg, _none(dwords, img.device)


@damsm_bwd.register_fake
def _(img, words, cap_lens, gamma1, gamma2, eps, dm, gscale, need_dwords, math, m_fwd, ws, ws_saved):
    Bc, D, T = words.shape
    return torch.empty_like(img), img.new_empty((Bc, T, D) if need_dwords else (0,), dtype=torch.float32)


def _damsm_setup(ctx, inputs, output):
    img, words, cap_lens, cnn, rnn, gamma1, gamma2, eps, row_offset, want_att, math, save = inputs
    m, att, scos, ws = output
    ctx.save_for_backward(img, words, cap_lens, m, cnn, rnn)
    # the fp32 kernels stage nothing worth keeping: their backward allocates its own workspace, as in eager mode
    ctx.ws = ws if math != N.AGB_MATH_FP32 else None
    ctx.cfg = (gamma1, gamma2, eps, math, save)
    ctx.mark_non_differentiable(att, ws)
    ctx.set_materialize_grads(False)


def _damsm_backward(ctx, dm, _datt, dscos, _dws):
    img, words, cap_lens, m, cnn, rnn = ctx.saved_tensors
    gamma1, gamma2, eps, math, save = ctx.cfg
    need_img, need_words = ctx.needs_input_grad[:2]
    dimg = dwords = dcnn = drnn = None
    if dm is not None and (need_img or need_words):
        dimg, dw = torch.ops.agb.damsm_bwd(img, words, cap_lens, gamma1, gamma2, eps, dm.contiguous(), None,
                                           need_words, math, m, ctx.ws, save and ctx.ws is not None)
        dwords = dw.transpose(1, 2) if need_words else None             # [Bc,D,T] view like words
        dimg = dimg if need_img else None
    ctx.ws = None
    if dscos is not None and any(ctx.needs_input_grad[3:5]):
        dc, dr = torch.ops.agb.sent_cos_bwd(cnn, rnn, eps, dscos.contiguous(), None, ctx.needs_input_grad[3],
                                            ctx.needs_input_grad[4])
        dcnn, drnn = _opt(dc), _opt(dr)
    return dimg, dwords, None, dcnn, drnn, None, None, None, None, None, None, None


damsm_fwd.register_autograd(_damsm_backward, setup_context=_damsm_setup)


@_op("contrastive")
def contrastive(raw: Tensor, class_ids: Optional[Tensor], labels: Tensor, gamma3: float, lam: float,
                row_begin: int, row_count: int, want_grad: bool) -> Tuple[Tensor, Tensor]:
    """raw [B,B] fp32, class_ids [B] int32 or None, labels [B] int64 -> (loss [1], draw [row_count,B] or empty)"""
    loss, draw = ops.contrastive(raw, class_ids, labels, gamma3, lam, row_begin, row_count, want_grad)
    return loss, _none(draw, raw.device)


@contrastive.register_fake
def _(raw, class_ids, labels, gamma3, lam, row_begin, row_count, want_grad):
    B = raw.shape[0]
    return raw.new_empty((1,), dtype=torch.float32), raw.new_empty((row_count, B) if want_grad else (0,),
                                                                    dtype=torch.float32)


def _contrastive_setup(ctx, inputs, output):
    raw, class_ids, labels, gamma3, lam, row_begin, row_count, want_grad = inputs
    ctx.save_for_backward(output[1])
    ctx.rows = (raw.shape[0], row_begin, row_count, want_grad)
    ctx.mark_non_differentiable(output[1])


def _contrastive_backward(ctx, dloss, _ddraw):
    (draw,) = ctx.saved_tensors
    B, row_begin, row_count, want_grad = ctx.rows
    if not want_grad:
        raise RuntimeError("agb::contrastive was called with want_grad=False and has no gradient")
    # draw * dloss rounds exactly as the backward kernels' own  dm * gscale  does (they take gscale = None here)
    d = draw * dloss.float().reshape(1, 1)
    if row_begin != 0 or row_count != B:
        d = torch.nn.functional.pad(d, (0, 0, row_begin, B - row_begin - row_count))
    return d, None, None, None, None, None, None, None


contrastive.register_autograd(_contrastive_backward, setup_context=_contrastive_setup)


@_op("sent_cos_fwd")
def sent_cos_fwd(cnn: Tensor, rnn: Tensor, eps: float) -> Tensor:
    """cnn [Bi,D], rnn [Bc,D] fp32 contiguous -> cosine [Bi,Bc]"""
    return ops.sent_cos_fwd(cnn, rnn, eps)


@sent_cos_fwd.register_fake
def _(cnn, rnn, eps):
    return cnn.new_empty((cnn.shape[0], rnn.shape[0]), dtype=torch.float32)


@_op("sent_cos_bwd")
def sent_cos_bwd(cnn: Tensor, rnn: Tensor, eps: float, dscos: Tensor, gscale: Optional[Tensor], need_dcnn: bool,
                 need_drnn: bool) -> Tuple[Tensor, Tensor]:
    """(dcnn or empty, drnn or empty)"""
    dcnn, drnn = ops.sent_cos_bwd(cnn, rnn, eps, dscos, gscale, need_dcnn, need_drnn)
    return _none(dcnn, cnn.device), _none(drnn, cnn.device)


@sent_cos_bwd.register_fake
def _(cnn, rnn, eps, dscos, gscale, need_dcnn, need_drnn):
    e = cnn.new_empty((0,), dtype=torch.float32)
    return (torch.empty_like(cnn) if need_dcnn else e), (torch.empty_like(rnn) if need_drnn else e.clone())


def _sent_cos_setup(ctx, inputs, output):
    cnn, rnn, eps = inputs
    ctx.save_for_backward(cnn, rnn)
    ctx.eps = eps


def _sent_cos_backward(ctx, dscos):
    cnn, rnn = ctx.saved_tensors
    need_c, need_r = ctx.needs_input_grad[:2]
    dc, dr = torch.ops.agb.sent_cos_bwd(cnn, rnn, ctx.eps, dscos.contiguous(), None, need_c, need_r)
    return (dc if need_c else None), (dr if need_r else None), None


sent_cos_fwd.register_autograd(_sent_cos_backward, setup_context=_sent_cos_setup)


@_op("damsm_cand_fwd")
def damsm_cand_fwd(img: Tensor, words: Tensor, cap_lens: Tensor, cand: Tensor, gamma1: float, gamma2: float,
                   math: int) -> Tensor:
    """m [Bi,K] of the candidate pairs cand [Bi,K] int32 (ops.damsm_cand_fwd; the workspace is allocated here)"""
    return ops.damsm_cand_fwd(img, words, cap_lens, cand, gamma1, gamma2, math)


@damsm_cand_fwd.register_fake
def _(img, words, cap_lens, cand, gamma1, gamma2, math):
    return img.new_empty((img.shape[0], cand.shape[1]), dtype=torch.float32)


@_op("sent_cos_cand_fwd")
def sent_cos_cand_fwd(cnn: Tensor, rnn: Tensor, cand: Tensor, eps: float) -> Tensor:
    """cosine [Bi,K] of the candidate pairs"""
    return ops.sent_cos_cand_fwd(cnn, rnn, cand, eps)


@sent_cos_cand_fwd.register_fake
def _(cnn, rnn, cand, eps):
    return cnn.new_empty((cnn.shape[0], cand.shape[1]), dtype=torch.float32)


@_op("damsm_pairs_fwd")
def damsm_pairs_fwd(img: Tensor, words: Tensor, cap_lens: Tensor, pair_img: Tensor, pair_cap: Tensor, gamma1: float,
                    gamma2: float, want_att: bool, math: int) -> Tuple[Tensor, Tensor]:
    """(m [P], att [P,T,R] or empty) of the pair list pair_img / pair_cap [P] int32 (ops.damsm_pairs_fwd; the
    workspace is allocated here)"""
    m, att = ops.damsm_pairs_fwd(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math, want_att)
    return m, _none(att, img.device)


@damsm_pairs_fwd.register_fake
def _(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, want_att, math):
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    P = pair_img.shape[0]
    if pair_cap.shape[0] != P:
        raise RuntimeError(f"pair_img has {P} entries, pair_cap {pair_cap.shape[0]}")
    if int(N.lib().agb_damsm_pairs_workspace_bytes(Bi, Bc, P, T, D, R, math)) == 0:
        raise N.NativeError(f"pair DAMSM shape Bi={Bi} Bc={Bc} P={P} T={T} D={D} R={R} is unsupported for math mode {math}")
    f32 = dict(dtype=torch.float32)
    return img.new_empty((P,), **f32), img.new_empty((P, T, R) if want_att else (0,), **f32)


@_op("sent_cos_pairs_fwd")
def sent_cos_pairs_fwd(cnn: Tensor, rnn: Tensor, pair_img: Tensor, pair_cap: Tensor, eps: float) -> Tensor:
    """cosine [P] of the pair list"""
    return ops.sent_cos_pairs_fwd(cnn, rnn, pair_img, pair_cap, eps)


@sent_cos_pairs_fwd.register_fake
def _(cnn, rnn, pair_img, pair_cap, eps):
    if pair_cap.shape[0] != pair_img.shape[0]:
        raise RuntimeError(f"pair_img has {pair_img.shape[0]} entries, pair_cap {pair_cap.shape[0]}")
    return cnn.new_empty((pair_img.shape[0],), dtype=torch.float32)


# the differentiable pair scores (losses/pair_scores.py): the training forward returns its workspace, which the
# backward reads and overwrites with its staging
@_op("damsm_pairs_train_fwd")
def damsm_pairs_train_fwd(img: Tensor, words: Tensor, cap_lens: Tensor, pair_img: Tensor, pair_cap: Tensor,
                          gamma1: float, gamma2: float, math: int) -> Tuple[Tensor, Tensor]:
    """(m [P], ws uint8) of the pair list (ops.damsm_pairs_train_fwd)"""
    return ops.damsm_pairs_train_fwd(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math)


@damsm_pairs_train_fwd.register_fake
def _(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math):
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    P = pair_img.shape[0]
    if pair_cap.shape[0] != P:
        raise RuntimeError(f"pair_img has {P} entries, pair_cap {pair_cap.shape[0]}")
    nbytes = int(N.lib().agb_damsm_pairs_train_workspace_bytes(Bi, Bc, P, T, D, R, math))
    if nbytes == 0:
        raise N.NativeError(f"pair DAMSM shape Bi={Bi} Bc={Bc} P={P} T={T} D={D} R={R} is unsupported for math mode {math}")
    return img.new_empty((P,), dtype=torch.float32), _ws_like(nbytes, img)


@_op("damsm_pairs_bwd", mutates_args=("ws",))
def damsm_pairs_bwd(img: Tensor, words: Tensor, cap_lens: Tensor, pair_img: Tensor, pair_cap: Tensor, gamma1: float,
                    gamma2: float, math: int, dm: Tensor, ws: Tensor, need_dimg: bool,
                    need_dwords: bool) -> Tuple[Tensor, Tensor]:
    """(dimg [Bi,D,R] or empty, dwords [Bc,T,D] word-major or empty) from the workspace damsm_pairs_train_fwd
    returned"""
    dimg, dwords = ops.damsm_pairs_bwd(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math, dm, ws,
                                       need_dwords, need_dimg)
    return _none(dimg, img.device), _none(dwords, img.device)


@damsm_pairs_bwd.register_fake
def _(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math, dm, ws, need_dimg, need_dwords):
    Bc, D, T = words.shape
    e = img.new_empty((0,), dtype=torch.float32)
    return (torch.empty_like(img) if need_dimg else e), (img.new_empty((Bc, T, D)) if need_dwords else e.clone())


def _damsm_pairs_setup(ctx, inputs, output):
    img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math = inputs
    ctx.save_for_backward(img, words, cap_lens, pair_img, pair_cap)
    ctx.ws = output[1]
    ctx.cfg = (gamma1, gamma2, math)
    ctx.mark_non_differentiable(output[1])
    ctx.set_materialize_grads(False)


def _damsm_pairs_backward(ctx, dm, _dws):
    img, words, cap_lens, pair_img, pair_cap = ctx.saved_tensors
    gamma1, gamma2, math = ctx.cfg
    need_img, need_words = ctx.needs_input_grad[:2]
    dimg = dwords = None
    if dm is not None and (need_img or need_words):
        if ctx.ws is None:
            raise RuntimeError("agb::damsm_pairs_train_fwd: a second backward is not supported (the first one "
                               "released the training workspace)")
        di, dw = torch.ops.agb.damsm_pairs_bwd(img, words, cap_lens, pair_img, pair_cap, gamma1, gamma2, math,
                                               dm.contiguous(), ctx.ws, need_img, need_words)
        dimg = di if need_img else None
        dwords = dw.transpose(1, 2) if need_words else None           # [Bc,D,T] view like words
    ctx.ws = None
    return dimg, dwords, None, None, None, None, None, None


damsm_pairs_train_fwd.register_autograd(_damsm_pairs_backward, setup_context=_damsm_pairs_setup)


@_op("sent_cos_pairs_train_fwd")
def sent_cos_pairs_train_fwd(cnn: Tensor, rnn: Tensor, pair_img: Tensor, pair_cap: Tensor, eps: float) -> Tensor:
    """cosine [P] of the pair list, the values of sent_cos_pairs_fwd, with a registered backward"""
    return ops.sent_cos_pairs_fwd(cnn, rnn, pair_img, pair_cap, eps)


@sent_cos_pairs_train_fwd.register_fake
def _(cnn, rnn, pair_img, pair_cap, eps):
    if pair_cap.shape[0] != pair_img.shape[0]:
        raise RuntimeError(f"pair_img has {pair_img.shape[0]} entries, pair_cap {pair_cap.shape[0]}")
    return cnn.new_empty((pair_img.shape[0],), dtype=torch.float32)


@_op("sent_cos_pairs_bwd")
def sent_cos_pairs_bwd(cnn: Tensor, rnn: Tensor, pair_img: Tensor, pair_cap: Tensor, eps: float, dscos: Tensor,
                       need_dcnn: bool, need_drnn: bool) -> Tuple[Tensor, Tensor]:
    """(dcnn or empty, drnn or empty)"""
    dcnn, drnn = ops.sent_cos_pairs_bwd(cnn, rnn, pair_img, pair_cap, eps, dscos, need_dcnn, need_drnn)
    return _none(dcnn, cnn.device), _none(drnn, cnn.device)


@sent_cos_pairs_bwd.register_fake
def _(cnn, rnn, pair_img, pair_cap, eps, dscos, need_dcnn, need_drnn):
    e = cnn.new_empty((0,), dtype=torch.float32)
    return (torch.empty_like(cnn) if need_dcnn else e), (torch.empty_like(rnn) if need_drnn else e.clone())


def _sent_cos_pairs_setup(ctx, inputs, output):
    cnn, rnn, pair_img, pair_cap, eps = inputs
    ctx.save_for_backward(cnn, rnn, pair_img, pair_cap)
    ctx.eps = eps


def _sent_cos_pairs_backward(ctx, dscos):
    cnn, rnn, pair_img, pair_cap = ctx.saved_tensors
    need_c, need_r = ctx.needs_input_grad[:2]
    dc, dr = torch.ops.agb.sent_cos_pairs_bwd(cnn, rnn, pair_img, pair_cap, ctx.eps, dscos.contiguous(), need_c,
                                              need_r)
    return (dc if need_c else None), (dr if need_r else None), None, None, None


sent_cos_pairs_train_fwd.register_autograd(_sent_cos_pairs_backward, setup_context=_sent_cos_pairs_setup)


# ------------------------------------------------------------------------------------------------
# functional region-word attention
# ------------------------------------------------------------------------------------------------
@_op("func_attention_fwd")
def func_attention_fwd(query: Tensor, context: Tensor, gamma1: float, scaled: bool) -> Tuple[Tensor, Tensor]:
    """query [B,D,L] fp32, context [B,D,R] fp32 contiguous -> (wc [B,D,L], attn [B,L,R])"""
    return ops.func_attention_fwd(query, context, gamma1, scaled)


@func_attention_fwd.register_fake
def _(query, context, gamma1, scaled):
    B, D, L = query.shape
    return query.new_empty((B, D, L), dtype=torch.float32), query.new_empty((B, L, context.shape[2]),
                                                                            dtype=torch.float32)


@_op("func_attention_bwd")
def func_attention_bwd(query: Tensor, context: Tensor, gamma1: float, scaled: bool, dwc: Tensor,
                       dattn: Optional[Tensor], need_dquery: bool, need_dcontext: bool) -> Tuple[Tensor, Tensor]:
    """(dquery [B,D,L] or empty, dcontext [B,D,R] or empty)"""
    dq, dc = ops.func_attention_bwd(query, context, gamma1, scaled, dwc, dattn, need_dquery, need_dcontext)
    return _none(dq, query.device), _none(dc, query.device)


@func_attention_bwd.register_fake
def _(query, context, gamma1, scaled, dwc, dattn, need_dquery, need_dcontext):
    B, D, L = query.shape
    f32 = dict(dtype=torch.float32)
    return (query.new_empty((B, D, L) if need_dquery else (0,), **f32),
            query.new_empty((B, D, context.shape[2]) if need_dcontext else (0,), **f32))


def _func_attention_setup(ctx, inputs, output):
    query, context, gamma1, scaled = inputs
    ctx.save_for_backward(query, context)
    ctx.cfg = (gamma1, scaled)
    ctx.set_materialize_grads(False)


def _func_attention_backward(ctx, dwc, dattn):
    query, context = ctx.saved_tensors
    gamma1, scaled = ctx.cfg
    need_q, need_c = ctx.needs_input_grad[:2]
    dwc = torch.zeros_like(query) if dwc is None else dwc
    dq, dc = torch.ops.agb.func_attention_bwd(query, context, gamma1, scaled, dwc.contiguous(),
                                              None if dattn is None else dattn.contiguous(), need_q, need_c)
    return (dq if need_q else None), (dc if need_c else None), None, None


func_attention_fwd.register_autograd(_func_attention_backward, setup_context=_func_attention_setup)


# ------------------------------------------------------------------------------------------------
# region-feature head of the image encoder
# ------------------------------------------------------------------------------------------------
def region_head_workspace_bytes(B: int, Cin: int, Cout: int, R: int) -> int:
    return int(N.lib().agb_region_head_workspace_bytes(B, Cin, Cout, R))


@_op("region_head_fwd")
def region_head_fwd(x: Tensor, weight: Tensor) -> Tuple[Tensor, Tensor]:
    """x [B,Cin,R] fp32 contiguous, weight [Cout,Cin] fp32 -> (feat [B,Cout,R] fp32, ws uint8 holding the 16-bit
    operand copies region_head_bwd reuses)"""
    return ops.region_head_fwd(x, weight, keep_ws=True)


@region_head_fwd.register_fake
def _(x, weight):
    B, Cin, R = x.shape
    Cout = weight.shape[0]
    nbytes = region_head_workspace_bytes(B, Cin, Cout, R)
    if nbytes == 0:
        raise N.NativeError(f"region head shape Cin={Cin} Cout={Cout} is unsupported (Cin % 64, Cout % 128)")
    return x.new_empty((B, Cout, R), dtype=torch.float32), _ws_like(nbytes, x)


@_op("region_head_bwd", mutates_args=("ws",))
def region_head_bwd(x: Tensor, weight: Tensor, dfeat: Tensor, need_dw: bool, need_dx: bool,
                    ws: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """(dweight [Cout,Cin] or empty, dx [B,Cin,R] or empty); ws: the workspace region_head_fwd returned, which
    this call overwrites with its staging (None: a workspace of its own)"""
    dw, dx = ops.region_head_bwd(x, weight, dfeat, need_dw, need_dx, ws)
    return _none(dw, x.device), _none(dx, x.device)


@region_head_bwd.register_fake
def _(x, weight, dfeat, need_dw, need_dx, ws):
    f32 = dict(dtype=torch.float32)
    return (x.new_empty(tuple(weight.shape) if need_dw else (0,), **f32),
            x.new_empty(tuple(x.shape) if need_dx else (0,), **f32))


def _region_head_setup(ctx, inputs, output):
    x, weight = inputs
    ctx.save_for_backward(x, weight, output[1])
    ctx.mark_non_differentiable(output[1])


def _region_head_backward(ctx, dfeat, _dws):
    x, weight, ws = ctx.saved_tensors
    need_x, need_w = ctx.needs_input_grad[:2]
    dw, dx = torch.ops.agb.region_head_bwd(x, weight, dfeat.contiguous(), need_w, need_x, ws)
    return (dx if need_x else None), (dw if need_w else None)


region_head_fwd.register_autograd(_region_head_backward, setup_context=_region_head_setup)

OPS = ("word_attn_fwd", "word_attn_cat", "word_attn_bwd", "damsm_fwd", "damsm_bwd", "contrastive", "sent_cos_fwd",
       "sent_cos_bwd", "func_attention_fwd", "func_attention_bwd", "region_head_fwd", "region_head_bwd",
       "damsm_cand_fwd", "sent_cos_cand_fwd")
# the pair-list scorers of the evaluation path (DAMSMScorer.words_pairs / sentence_pairs)
PAIR_OPS = ("damsm_pairs_fwd", "sent_cos_pairs_fwd")
# the differentiable pair scores (losses/pair_scores.py)
PAIR_TRAIN_OPS = ("damsm_pairs_train_fwd", "damsm_pairs_bwd", "sent_cos_pairs_train_fwd", "sent_cos_pairs_bwd")
