"""Tensor-level wrappers over the C ABI: raw data_ptr()s, explicit strides, the current stream.

Every function here launches hand-written sm_100a kernels from libattngan_b200.so.  Inputs must
live on a CUDA device; anything else raises (there is no CPU path).  torch is used only for
device memory and streams.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import native as N

_IO = {torch.float32: N.AGB_F32, torch.bfloat16: N.AGB_BF16, torch.float16: N.AGB_F16}


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


def require_cuda(*tensors: torch.Tensor) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "attngan_b200 runs only on a CUDA (sm_100a) device: got a tensor on "
                f"'{t.device}'. There is no CPU fallback.")


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# ------------------------------------------------------------------------------------------------
# generator word-context attention                       reference networks/attention.py:25-79
# ------------------------------------------------------------------------------------------------
def word_attn_fwd(images: torch.Tensor, words: torch.Tensor, weight: torch.Tensor, mask: torch.Tensor,
                  scaled: bool, want_attn: bool = True, ctx_out: Optional[torch.Tensor] = None
                  ) -> Tuple[torch.Tensor, Optional[torch.Tensor], torch.Tensor]:
    """images [B,C,H,W] contiguous (f32/bf16/f16), words [B,E,T] fp32 any strides, weight [C,E] fp32,
    mask [B,T] int64.  Returns (ctx [B,C,H,W], attn [B,T,H,W] or None, we [B,C,T] fp32).
    ctx_out: optional pre-allocated destination whose batch stride may exceed C*H*W (a channel
    slice of a concat buffer, generator_submodules.py:116)."""
    require_cuda(images, words, weight, mask)
    B, C, H, W = images.shape
    E, T = words.shape[1], words.shape[2]
    HW = H * W
    if not images.is_contiguous():
        raise RuntimeError("images must be contiguous NCHW (the reference .view()s it, attention.py:55)")
    ctx = ctx_out if ctx_out is not None else torch.empty_like(images)
    if ctx.stride(1) != HW or ctx.stride(3) != 1 or ctx.stride(2) != W:
        raise RuntimeError("ctx_out must be channel-contiguous NCHW")
    attn = torch.empty((B, T, H, W), dtype=images.dtype, device=images.device) if want_attn else None
    we = torch.empty((B, C, T), dtype=torch.float32, device=images.device)
    rc = N.lib().agb_word_attn_fwd(_p(images), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                   _p(weight), _p(mask), _p(ctx), ctx.stride(0), _p(attn), _p(we),
                                   B, C, HW, E, T, _IO[images.dtype], int(bool(scaled)), _stream(images))
    N.check(rc, "agb_word_attn_fwd")
    return ctx, attn, we


def word_attn_bwd(images, words, weight, mask, we, dctx, dattn, scaled: bool, need_dwords: bool,
                  need_dweight: bool):
    """Returns (dimages, dwords [B,E,T] fp32 or None, dweight [C,E] fp32 or None)."""
    require_cuda(images, words, weight, mask, we, dctx, dattn)
    B, C, H, W = images.shape
    E, T = words.shape[1], words.shape[2]
    HW = H * W
    if dctx.stride(1) != HW or dctx.stride(3) != 1 or dctx.stride(2) != W:
        dctx = dctx.contiguous()
    if dattn is not None:
        dattn = dattn.contiguous()
    dimages = torch.empty_like(images)
    dwords = torch.empty((B, E, T), dtype=torch.float32, device=images.device) if need_dwords else None
    dweight = torch.empty((C, E), dtype=torch.float32, device=images.device) if need_dweight else None
    nbytes = N.lib().agb_word_attn_bwd_workspace_bytes(B, C, HW, E, T)
    ws = _ws(nbytes, images.device)
    rc = N.lib().agb_word_attn_bwd(_p(images), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                   _p(weight), _p(mask), _p(we), _p(dctx), dctx.stride(0), _p(dattn),
                                   _p(dimages), _p(dwords), _p(dweight), _p(ws), ws.numel(),
                                   B, C, HW, E, T, _IO[images.dtype], int(bool(scaled)), _stream(images))
    N.check(rc, "agb_word_attn_bwd")
    return dimages, dwords, dweight


# ------------------------------------------------------------------------------------------------
# DAMSM word-region similarity       reference losses/words_loss.py:43-86 + attention.py:82-121
# ------------------------------------------------------------------------------------------------
def damsm_supported(T: int, D: int, R: int, math: int) -> bool:
    return bool(N.lib().agb_damsm_supported(T, D, R, math))


def damsm_fwd(img: torch.Tensor, words: torch.Tensor, cap_lens: torch.Tensor, gamma1: float,
              gamma2: float, eps: float = 1e-8, row_offset: int = 0, want_att: bool = True,
              math: int = N.AGB_MATH_FP32, cnn: Optional[torch.Tensor] = None,
              rnn: Optional[torch.Tensor] = None, keep_ws: bool = False, save: bool = False):
    """img [Bi,D,R] fp32 contiguous, words [Bc,D,T] fp32 (any strides), cap_lens [Bc] int32.
    Returns (m [Bi,Bc], att [Bi,T,R] or None, scos [Bi,Bc] or None); with keep_ws also the workspace
    tensor, whose packed operands damsm_bwd(ws=...) can reuse.  save (tensor-core math only): the
    training forward, which also leaves the normalised context vectors in the workspace so that
    damsm_bwd(ws=..., ws_saved=True) does not recompute them."""
    require_cuda(img, words, cap_lens, cnn, rnn)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    dev = img.device
    m = torch.empty((Bi, Bc), dtype=torch.float32, device=dev)
    # the fp32 pair kernel writes only the live word rows of the matched-pair maps; the tensor-core path's
    # diag_att_kernel writes every row (zeros for t >= L), so it needs no zero fill
    att = None
    if want_att:
        att = (torch.zeros if math == N.AGB_MATH_FP32 else torch.empty)((Bi, T, R), dtype=torch.float32, device=dev)
    scos = torch.empty((Bi, Bc), dtype=torch.float32, device=dev) if cnn is not None else None
    nbytes = N.lib().agb_damsm_workspace_bytes(Bi, Bc, T, D, R, math)
    if nbytes == 0:
        raise N.NativeError(f"DAMSM shape T={T} D={D} R={R} is unsupported for math mode {math}")
    ws = _ws(nbytes, dev)
    rc = N.lib().agb_damsm_fwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                               _p(cap_lens), Bi, Bc, T, D, R, gamma1, gamma2, eps, row_offset, _p(m),
                               _p(att), _p(cnn), _p(rnn), _p(scos), _p(ws), ws.numel(),
                               math | (N.AGB_MATH_SAVE if save else 0), _stream(img))
    N.check(rc, "agb_damsm_fwd")
    if keep_ws:
        return m, att, scos, ws
    return m, att, scos


def damsm_bwd(img, words, cap_lens, gamma1, gamma2, eps, dm, gscale, need_dwords: bool,
              math: int = N.AGB_MATH_FP32, m_fwd: Optional[torch.Tensor] = None,
              ws: Optional[torch.Tensor] = None, ws_saved: bool = False):
    """dm [Bi,Bc] = dLoss/dm, gscale: device scalar or None.  ws: the workspace of the matching damsm_fwd
    call (ws_saved: that call ran with save=True).
    Returns (dimg [Bi,D,R], dwords [Bc,T,D] word-major or None)."""
    require_cuda(img, words, cap_lens, dm, gscale)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    dev = img.device
    dimg = torch.empty_like(img)
    dwords = torch.empty((Bc, T, D), dtype=torch.float32, device=dev) if need_dwords else None
    from_fwd = (2 if ws_saved else 1) if ws is not None else 0
    if ws is None:
        ws = _ws(N.lib().agb_damsm_workspace_bytes(Bi, Bc, T, D, R, math), dev)
    rc = N.lib().agb_damsm_bwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                               _p(cap_lens), Bi, Bc, T, D, R, gamma1, gamma2, eps, _p(dm), _p(m_fwd), _p(gscale),
                               _p(dimg), _p(dwords), _p(ws), ws.numel(), from_fwd, math, _stream(img))
    N.check(rc, "agb_damsm_bwd")
    return dimg, dwords


def damsm_cand_workspace_bytes(Bi: int, K: int, T: int, D: int, R: int, math: int) -> int:
    """workspace of damsm_cand_fwd; 0 when the shapes are outside the candidate path's range"""
    return int(N.lib().agb_damsm_cand_workspace_bytes(Bi, K, T, D, R, math))


def damsm_cand_fwd(img: torch.Tensor, words: torch.Tensor, cap_lens: torch.Tensor, cand: torch.Tensor,
                   gamma1: float, gamma2: float, math: int, ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """m of candidate pairs: img [Bi,D,R] fp32 contiguous, words [Bc,D,T] fp32 (any strides), cap_lens [Bc] int32,
    cand [Bi,K] int32 contiguous.  Returns m [Bi,K] fp32, m[b,k] = damsm_fwd's m[b, cand[b,k]] bit for bit
    (NaN where cand[b,k] is outside [0,Bc)).  Tensor-core math only.  ws: a uint8 workspace of at least
    damsm_cand_workspace_bytes (allocated here when None)."""
    require_cuda(img, words, cap_lens, cand)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    K = cand.shape[1]
    if cand.dtype != torch.int32 or not cand.is_contiguous() or cand.shape[0] != Bi:
        raise RuntimeError("cand must be a contiguous int32 [Bi,K] tensor")
    nbytes = damsm_cand_workspace_bytes(Bi, K, T, D, R, math)
    if nbytes == 0:
        raise N.NativeError(f"candidate DAMSM shape Bi={Bi} K={K} T={T} D={D} R={R} is unsupported for math mode {math}")
    if ws is None:
        ws = _ws(nbytes, img.device)
    m = torch.empty((Bi, K), dtype=torch.float32, device=img.device)
    rc = N.lib().agb_damsm_cand_fwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                    _p(cap_lens), Bc, _p(cand), Bi, K, T, D, R, gamma1, gamma2, _p(m), _p(ws),
                                    ws.numel(), math, _stream(img))
    N.check(rc, "agb_damsm_cand_fwd")
    return m


def sent_cos_cand_fwd(cnn: torch.Tensor, rnn: torch.Tensor, cand: torch.Tensor, eps: float) -> torch.Tensor:
    """cnn [Bi,D], rnn [Bc,D] fp32 contiguous, cand [Bi,K] int32 contiguous -> cosine [Bi,K] of the candidate
    pairs (NaN where cand[b,k] is outside [0,Bc))"""
    require_cuda(cnn, rnn, cand)
    Bi, D = cnn.shape
    Bc = rnn.shape[0]
    if cand.dtype != torch.int32 or not cand.is_contiguous() or cand.shape[0] != Bi:
        raise RuntimeError("cand must be a contiguous int32 [Bi,K] tensor")
    K = cand.shape[1]
    scos = torch.empty((Bi, K), dtype=torch.float32, device=cnn.device)
    rc = N.lib().agb_sent_cos_cand_fwd(_p(cnn), _p(rnn), Bc, _p(cand), Bi, K, D, eps, _p(scos), _stream(cnn))
    N.check(rc, "agb_sent_cos_cand_fwd")
    return scos


def damsm_pairs_workspace_bytes(Bi: int, Bc: int, P: int, T: int, D: int, R: int, math: int) -> int:
    """workspace of damsm_pairs_fwd; 0 when the shapes are outside the pair path's range"""
    return int(N.lib().agb_damsm_pairs_workspace_bytes(Bi, Bc, P, T, D, R, math))


def _pair_index(t: torch.Tensor, name: str) -> None:
    if t.dtype != torch.int32 or t.dim() != 1 or not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous int32 [P] tensor")


def damsm_pairs_fwd(img: torch.Tensor, words: torch.Tensor, cap_lens: torch.Tensor, pair_img: torch.Tensor,
                    pair_cap: torch.Tensor, gamma1: float, gamma2: float, math: int, want_att: bool = False,
                    ws: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """m of a pair list: img [Bi,D,R] fp32 contiguous, words [Bc,D,T] fp32 (any strides), cap_lens [Bc] int32,
    pair_img / pair_cap [P] int32 contiguous.  Returns (m [P] fp32, att [P,T,R] fp32 or None): m[p] = damsm_fwd's
    m[pair_img[p], pair_cap[p]] bit for bit, att[p] the pair's beta maps; NaN for an index out of range or a caption
    of length 0.  Tensor-core math only.  ws: a uint8 workspace of at least damsm_pairs_workspace_bytes."""
    require_cuda(img, words, cap_lens, pair_img, pair_cap)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    _pair_index(pair_img, "pair_img")
    _pair_index(pair_cap, "pair_cap")
    P = pair_img.shape[0]
    if pair_cap.shape[0] != P:
        raise RuntimeError(f"pair_img has {P} entries, pair_cap {pair_cap.shape[0]}")
    nbytes = damsm_pairs_workspace_bytes(Bi, Bc, P, T, D, R, math)
    if nbytes == 0:
        raise N.NativeError(f"pair DAMSM shape Bi={Bi} Bc={Bc} P={P} T={T} D={D} R={R} is unsupported for math mode {math}")
    m = torch.empty((P,), dtype=torch.float32, device=img.device)
    att = torch.empty((P, T, R), dtype=torch.float32, device=img.device) if want_att else None
    if P == 0:
        return m, att
    if ws is None:
        ws = _ws(nbytes, img.device)
    rc = N.lib().agb_damsm_pairs_fwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                     _p(cap_lens), Bi, Bc, _p(pair_img), _p(pair_cap), P, T, D, R, gamma1, gamma2,
                                     _p(m), _p(att), _p(ws), ws.numel(), math, _stream(img))
    N.check(rc, "agb_damsm_pairs_fwd")
    return m, att


def sent_cos_pairs_fwd(cnn: torch.Tensor, rnn: torch.Tensor, pair_img: torch.Tensor, pair_cap: torch.Tensor,
                       eps: float) -> torch.Tensor:
    """cnn [Bi,D], rnn [Bc,D] fp32 contiguous, pair_img / pair_cap [P] int32 contiguous -> cosine [P] of the pairs
    (NaN where an index is out of range)"""
    require_cuda(cnn, rnn, pair_img, pair_cap)
    Bi, D = cnn.shape
    _pair_index(pair_img, "pair_img")
    _pair_index(pair_cap, "pair_cap")
    P = pair_img.shape[0]
    if pair_cap.shape[0] != P:
        raise RuntimeError(f"pair_img has {P} entries, pair_cap {pair_cap.shape[0]}")
    scos = torch.empty((P,), dtype=torch.float32, device=cnn.device)
    rc = N.lib().agb_sent_cos_pairs_fwd(_p(cnn), _p(rnn), Bi, rnn.shape[0], _p(pair_img), _p(pair_cap), P, D, eps,
                                        _p(scos), _stream(cnn))
    N.check(rc, "agb_sent_cos_pairs_fwd")
    return scos


def damsm_pairs_train_workspace_bytes(Bi: int, Bc: int, P: int, T: int, D: int, R: int, math: int) -> int:
    """workspace of damsm_pairs_train_fwd / damsm_pairs_bwd; 0 when the shapes are outside the pair path's range"""
    return int(N.lib().agb_damsm_pairs_train_workspace_bytes(Bi, Bc, P, T, D, R, math))


def _pair_list(pair_img: torch.Tensor, pair_cap: torch.Tensor) -> int:
    _pair_index(pair_img, "pair_img")
    _pair_index(pair_cap, "pair_cap")
    P = pair_img.shape[0]
    if pair_cap.shape[0] != P:
        raise RuntimeError(f"pair_img has {P} entries, pair_cap {pair_cap.shape[0]}")
    return P


def _pairs_train_ws(img, words, P: int, math: int, ws: Optional[torch.Tensor]) -> torch.Tensor:
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    nbytes = damsm_pairs_train_workspace_bytes(Bi, Bc, P, T, D, R, math)
    if nbytes == 0:
        raise N.NativeError(f"pair DAMSM shape Bi={Bi} Bc={Bc} P={P} T={T} D={D} R={R} is unsupported for math mode {math}")
    if ws is None:
        return _ws(nbytes, img.device)
    if ws.numel() < nbytes:
        raise RuntimeError(f"workspace of {ws.numel()} bytes is below the {nbytes} the pair list needs")
    return ws


def damsm_pairs_train_fwd(img: torch.Tensor, words: torch.Tensor, cap_lens: torch.Tensor, pair_img: torch.Tensor,
                          pair_cap: torch.Tensor, gamma1: float, gamma2: float, math: int,
                          ws: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """The training forward of a pair list: the arguments of damsm_pairs_fwd without the maps.  Returns (m [P], ws):
    m bit for bit damsm_pairs_fwd's, ws the workspace (of at least damsm_pairs_train_workspace_bytes, allocated here
    when None) that damsm_pairs_bwd reads."""
    require_cuda(img, words, cap_lens, pair_img, pair_cap)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    P = _pair_list(pair_img, pair_cap)
    ws = _pairs_train_ws(img, words, P, math, ws)
    m = torch.empty((P,), dtype=torch.float32, device=img.device)
    rc = N.lib().agb_damsm_pairs_train_fwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                           _p(cap_lens), Bi, Bc, _p(pair_img), _p(pair_cap), P, T, D, R, gamma1,
                                           gamma2, _p(m), _p(ws), ws.numel(), math, _stream(img))
    N.check(rc, "agb_damsm_pairs_train_fwd")
    return m, ws


def damsm_pairs_bwd(img: torch.Tensor, words: torch.Tensor, cap_lens: torch.Tensor, pair_img: torch.Tensor,
                    pair_cap: torch.Tensor, gamma1: float, gamma2: float, math: int, dm: torch.Tensor,
                    ws: torch.Tensor, need_dwords: bool = True, need_dimg: bool = True
                    ) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """dm [P] fp32 contiguous = dLoss/dm in list order, ws: the workspace of the matching damsm_pairs_train_fwd.
    Returns (dimg [Bi,D,R] or None, dwords [Bc,T,D] word-major or None)."""
    require_cuda(img, words, cap_lens, pair_img, pair_cap, dm, ws)
    Bi, D, R = img.shape
    Bc, _, T = words.shape
    P = _pair_list(pair_img, pair_cap)
    if dm.dtype != torch.float32 or dm.shape != (P,) or not dm.is_contiguous():
        raise RuntimeError(f"dm must be a contiguous fp32 [{P}] tensor")
    ws = _pairs_train_ws(img, words, P, math, ws)
    dimg = torch.empty((Bi, D, R), dtype=torch.float32, device=img.device) if need_dimg else None
    dwords = torch.empty((Bc, T, D), dtype=torch.float32, device=img.device) if need_dwords else None
    rc = N.lib().agb_damsm_pairs_bwd(_p(img), _p(words), words.stride(0), words.stride(1), words.stride(2),
                                     _p(cap_lens), Bi, Bc, _p(pair_img), _p(pair_cap), P, T, D, R, gamma1, gamma2,
                                     _p(dm), _p(dimg), _p(dwords), _p(ws), ws.numel(), math, _stream(img))
    N.check(rc, "agb_damsm_pairs_bwd")
    return dimg, dwords


def sent_cos_pairs_bwd_workspace_bytes(Bi: int, Bc: int, P: int, D: int) -> int:
    return int(N.lib().agb_sent_cos_pairs_bwd_workspace_bytes(Bi, Bc, P, D))


def sent_cos_pairs_bwd(cnn: torch.Tensor, rnn: torch.Tensor, pair_img: torch.Tensor, pair_cap: torch.Tensor,
                       eps: float, dscos: torch.Tensor, need_dcnn: bool = True, need_drnn: bool = True):
    """dscos [P] fp32 contiguous = dLoss/dcos in list order -> (dcnn [Bi,D] or None, drnn [Bc,D] or None)"""
    require_cuda(cnn, rnn, pair_img, pair_cap, dscos)
    Bi, D = cnn.shape
    Bc = rnn.shape[0]
    P = _pair_list(pair_img, pair_cap)
    if dscos.dtype != torch.float32 or dscos.shape != (P,) or not dscos.is_contiguous():
        raise RuntimeError(f"dscos must be a contiguous fp32 [{P}] tensor")
    dcnn = torch.empty_like(cnn) if need_dcnn else None
    drnn = torch.empty_like(rnn) if need_drnn else None
    nbytes = sent_cos_pairs_bwd_workspace_bytes(Bi, Bc, P, D)
    if nbytes == 0:
        raise N.NativeError(f"sentence pair shape Bi={Bi} Bc={Bc} P={P} D={D} is unsupported")
    ws = _ws(nbytes, cnn.device)
    rc = N.lib().agb_sent_cos_pairs_bwd(_p(cnn), _p(rnn), Bi, Bc, _p(pair_img), _p(pair_cap), P, D, eps, _p(dscos),
                                        _p(dcnn), _p(drnn), _p(ws), ws.numel(), _stream(cnn))
    N.check(rc, "agb_sent_cos_pairs_bwd")
    return dcnn, drnn


def contrastive(raw: torch.Tensor, class_ids: Optional[torch.Tensor], labels: torch.Tensor, gamma3: float,
                lam: float, row_begin: int, row_count: int, want_grad: bool = True):
    """raw [B,B] fp32 (all rows), class_ids [B] int32 or None, labels [B] int64.
    Returns (loss [1], draw [row_count,B] or None): words_loss.py:88-101 / sentence_loss.py:40-49."""
    require_cuda(raw, class_ids, labels)
    B = raw.shape[0]
    dev = raw.device
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    draw = torch.empty((row_count, B), dtype=torch.float32, device=dev) if want_grad else None
    ws = _ws(N.lib().agb_contrastive_workspace_bytes(B), dev)
    rc = N.lib().agb_contrastive_fwd(_p(raw), B, _p(class_ids), _p(labels), gamma3, lam, row_begin, row_count,
                                     _p(loss), _p(draw), _p(ws), ws.numel(), _stream(raw))
    N.check(rc, "agb_contrastive_fwd")
    return loss, draw


def sent_cos_fwd(cnn: torch.Tensor, rnn: torch.Tensor, eps: float) -> torch.Tensor:
    require_cuda(cnn, rnn)
    Bi, D = cnn.shape
    Bc = rnn.shape[0]
    scos = torch.empty((Bi, Bc), dtype=torch.float32, device=cnn.device)
    rc = N.lib().agb_sent_cos_fwd(_p(cnn), _p(rnn), Bi, Bc, D, eps, _p(scos), _stream(cnn))
    N.check(rc, "agb_sent_cos_fwd")
    return scos


def sent_cos_bwd(cnn, rnn, eps, dscos, gscale, need_dcnn: bool = True, need_drnn: bool = True):
    require_cuda(cnn, rnn, dscos, gscale)
    Bi, D = cnn.shape
    Bc = rnn.shape[0]
    dcnn = torch.empty_like(cnn) if need_dcnn else None
    drnn = torch.empty_like(rnn) if need_drnn else None
    ws = _ws(N.lib().agb_sent_cos_bwd_workspace_bytes(Bi, Bc), cnn.device)
    rc = N.lib().agb_sent_cos_bwd(_p(cnn), _p(rnn), Bi, Bc, D, eps, _p(dscos), _p(gscale), _p(dcnn), _p(drnn),
                                  _p(ws), ws.numel(), _stream(cnn))
    N.check(rc, "agb_sent_cos_bwd")
    return dcnn, drnn


# ------------------------------------------------------------------------------------------------
# functional region-word attention                     reference networks/attention.py:82-121
# ------------------------------------------------------------------------------------------------
def func_attention_fwd(query: torch.Tensor, context: torch.Tensor, gamma1: float, scaled: bool):
    """query [B,D,L] fp32 strided, context [B,D,R] fp32 contiguous -> (wc [B,D,L], attn [B,L,R])."""
    require_cuda(query, context)
    B, D, L = query.shape
    R = context.shape[2]
    wc = torch.empty((B, D, L), dtype=torch.float32, device=query.device)
    attn = torch.empty((B, L, R), dtype=torch.float32, device=query.device)
    ws = _ws(N.lib().agb_func_attention_workspace_bytes(B, L, R), query.device)
    rc = N.lib().agb_func_attention_fwd(_p(query), query.stride(0), query.stride(1), query.stride(2),
                                        _p(context), B, D, L, R, gamma1, int(bool(scaled)), _p(wc), _p(attn),
                                        _p(ws), ws.numel(), _stream(query))
    N.check(rc, "agb_func_attention_fwd")
    return wc, attn


def func_attention_bwd(query, context, gamma1, scaled, dwc, dattn, need_dquery=True, need_dcontext=True):
    require_cuda(query, context, dwc, dattn)
    B, D, L = query.shape
    R = context.shape[2]
    dq = torch.empty((B, D, L), dtype=torch.float32, device=query.device) if need_dquery else None
    dc = torch.empty((B, D, R), dtype=torch.float32, device=query.device) if need_dcontext else None
    ws = _ws(N.lib().agb_func_attention_workspace_bytes(B, L, R), query.device)
    rc = N.lib().agb_func_attention_bwd(_p(query), query.stride(0), query.stride(1), query.stride(2),
                                        _p(context), B, D, L, R, gamma1, int(bool(scaled)), _p(dwc),
                                        _p(dattn), _p(dq), _p(dc), _p(ws), ws.numel(), _stream(query))
    N.check(rc, "agb_func_attention_bwd")
    return dq, dc


# ------------------------------------------------------------------------------------------------
# region-feature head of the image encoder                reference networks/cnn_encoder.py:56,101
# ------------------------------------------------------------------------------------------------
def region_head_fwd(x: torch.Tensor, weight: torch.Tensor, keep_ws: bool = False):
    """x [B,Cin,R] fp32 contiguous, weight [Cout,Cin] fp32 -> feat [B,Cout,R] fp32 (tcgen05, split precision);
    with keep_ws also the workspace, whose 16-bit operand copies region_head_bwd(ws=...) reuses"""
    require_cuda(x, weight)
    B, Cin, R = x.shape
    Cout = weight.shape[0]
    nbytes = N.lib().agb_region_head_workspace_bytes(B, Cin, Cout, R)
    if nbytes == 0:
        raise N.NativeError(f"region head shape Cin={Cin} Cout={Cout} is unsupported (Cin % 64, Cout % 128)")
    ws = _ws(nbytes, x.device)
    feat = torch.empty((B, Cout, R), dtype=torch.float32, device=x.device)
    rc = N.lib().agb_region_head_fwd(_p(x), _p(weight), _p(feat), _p(ws), ws.numel(), B, Cin, Cout, R, _stream(x))
    N.check(rc, "agb_region_head_fwd")
    return (feat, ws) if keep_ws else feat


def region_head_bwd(x: torch.Tensor, weight: torch.Tensor, dfeat: torch.Tensor, need_dw: bool, need_dx: bool,
                    ws: Optional[torch.Tensor] = None):
    """Returns (dweight [Cout,Cin] or None, dx [B,Cin,R] or None); ws: the workspace of the matching forward"""
    require_cuda(x, weight, dfeat)
    B, Cin, R = x.shape
    Cout = weight.shape[0]
    from_fwd = 1 if ws is not None else 0
    if ws is None:
        ws = _ws(N.lib().agb_region_head_workspace_bytes(B, Cin, Cout, R), x.device)
    dw = torch.empty((Cout, Cin), dtype=torch.float32, device=x.device) if need_dw else None
    dx = torch.empty_like(x) if need_dx else None
    if not (need_dw or need_dx):
        return None, None
    rc = N.lib().agb_region_head_bwd(_p(x), _p(weight), _p(dfeat), _p(dw), _p(dx), _p(ws), ws.numel(), from_fwd,
                                     B, Cin, Cout, R, _stream(x))
    N.check(rc, "agb_region_head_bwd")
    return dw, dx
