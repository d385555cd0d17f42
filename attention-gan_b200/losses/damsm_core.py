"""Host-side orchestration of the DAMSM losses: argument normalisation, the sharded (multi-GPU)
exchange and the autograd glue around the native kernels.

Single process: one ``damsm_fwd`` launch group gives the B x B word-region similarity (and, when
asked, the sentence cosine matrix from the same call), one ``contrastive`` call gives the loss and
dLoss/dsimilarity, and backward is one ``damsm_bwd`` call.

Sharded over N ranks (one process per GPU, SURVEY.md section 8e): rank k owns images and captions
[k*Bl, (k+1)*Bl).  Word features (+ lengths, class ids, sentence codes) are all-gathered so the
negatives span the global batch; each rank computes its row block sim[Bl, B]; the blocks are
all-gathered (B*B floats) so every rank evaluates the same global loss; in backward the image
gradients are local and the word-feature gradients are reduce-scattered back to their owners.
The loss returned on every rank is the loss of the concatenated batch, and the gradients are its
exact gradients.

``ops`` is injectable so the exchange logic can be exercised on CPU (gloo) in the tests with a
stand-in compute backend; the product default is the native library and nothing else.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from ..agb_native import native
from ..agb_native import ops as native_ops
from ..agb_native import torch_ops


@dataclass
class DamsmConfig:
    gamma1: float = 4.0
    gamma2: float = 5.0
    gamma3: float = 10.0
    lam: float = 5.0
    eps: float = 1e-8
    math: int = native.AGB_MATH_FP32
    group: Any = None          # torch.distributed process group, or None for a single process
    ops: Any = native_ops
    want_att: bool = True
    # sharded runs only: the caption length every rank pads its word features to before the all-gather.  The
    # reference's RNN pads to the LOCAL batch's longest caption (rnn_encoder.py:89-92), so T may differ per rank;
    # None = agree on max(T) with one all-reduce per step (a host sync), an int = no sync (must be >= every T)
    max_words: Optional[int] = None


def resolve_math(math, img_features=None, words_emb=None, gamma1: float = 4.0) -> int:
    """name -> enum of include/attngan_b200.h.  "auto": the split-precision tensor-core path when the shapes are
    inside its compiled range (and gamma1 inside fp16's range), else the fp32 CUDA-core path.  Both are native
    kernels of this library; the choice is a host-side query (agb_damsm_supported), no data is touched."""
    if math != "auto":
        return native.MATH_NAMES[math]
    query = torch_ops.host_query if torch.compiler.is_compiling() else _host_query
    if img_features is None or words_emb is None or not query("agb_has_tcgen05") or gamma1 > 11.0:
        return native.AGB_MATH_FP32
    D, T = int(words_emb.shape[1]), int(words_emb.shape[2])
    R = int(img_features.shape[2]) * int(img_features.shape[3]) if img_features.dim() == 4 else int(img_features.shape[2])
    ok = query("agb_damsm_supported", T, D, R, native.AGB_MATH_TC_F16X2)
    return native.AGB_MATH_TC_F16X2 if ok else native.AGB_MATH_FP32


def _host_query(name: str, *args):
    return getattr(native.lib(), name)(*args)


def _world(group) -> int:
    return 1 if group is None else dist.get_world_size(group)


def _rank(group) -> int:
    return 0 if group is None else dist.get_rank(group)


def _gather_cat(t: torch.Tensor, group) -> torch.Tensor:
    """all_gather along dim 0 (equal shapes on every rank)"""
    t = t.contiguous()
    out = torch.empty((_world(group) * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t, group=group) if t.is_cuda else \
        dist.all_gather(list(out.chunk(_world(group), 0)), t, group=group)
    return out


def _reduce_scatter_sum(t: torch.Tensor, group) -> torch.Tensor:
    """sum over ranks of t [W*n, ...], rank k keeps rows [k*n, (k+1)*n)"""
    W, k = _world(group), _rank(group)
    n = t.shape[0] // W
    t = t.contiguous()
    if t.is_cuda:
        out = torch.empty((n,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        dist.reduce_scatter_tensor(out, t, op=dist.ReduceOp.SUM, group=group)
        return out
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)          # gloo has no reduce_scatter
    return t[k * n:(k + 1) * n].clone()


def _agree_on_words(T_local: int, cfg: "DamsmConfig", device) -> int:
    """the caption length all ranks pad to (see DamsmConfig.max_words)"""
    if cfg.max_words is not None:
        if T_local > cfg.max_words:
            raise RuntimeError(f"words_emb has T={T_local} > max_words={cfg.max_words}")
        return int(cfg.max_words)
    t = torch.tensor([T_local], dtype=torch.int64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=cfg.group)
    return int(t.item())


def as_device_i32(x, device) -> Optional[torch.Tensor]:
    """cap_lens arrive as a device tensor (words_loss.py:41), class_ids as numpy (words_loss.py:45)"""
    if x is None:
        return None
    if torch.is_tensor(x) and x.dtype == torch.int32 and x.device == torch.device(device) and x.is_contiguous():
        return x                                           # already resident (a step helper uploads it once)
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x.astype(np.int32)))
    elif not torch.is_tensor(x):
        x = torch.as_tensor(list(x), dtype=torch.int32)
    return x.to(device=device, dtype=torch.int32, non_blocking=True).contiguous()


class _Exchange:
    """what every rank needs about the global batch"""

    def __init__(self, cfg: DamsmConfig, n_local: int, labels, cap_lens, class_ids, device):
        self.W, self.k = _world(cfg.group), _rank(cfg.group)
        self.n_local = n_local
        self.row0 = self.k * n_local
        lens = as_device_i32(cap_lens, device)
        cls = as_device_i32(class_ids, device)
        labels = labels.to(device=device, dtype=torch.int64)
        if self.W > 1:
            lens = _gather_cat(lens, cfg.group) if lens is not None else None
            cls = _gather_cat(cls, cfg.group) if cls is not None else None
            labels = _gather_cat(labels + self.row0, cfg.group)
        self.lens, self.cls, self.labels = lens, cls, labels.contiguous()


class _WordsLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, words, cfg: DamsmConfig, ex: _Exchange, cnn, rnn):
        o = cfg.ops
        Bl, D = img.shape[0], img.shape[1]
        img3 = img.detach().float().reshape(Bl, D, -1).contiguous()
        w32 = words.detach().float()
        T_local = w32.shape[2]
        if ex.W > 1:
            T_all = _agree_on_words(T_local, cfg, w32.device)
            wt = w32.transpose(1, 2)                                             # [Bl,T,D]
            if T_all != T_local:                                                 # zero slots: cap_lens masks them
                wt = torch.nn.functional.pad(wt, (0, 0, 0, T_all - T_local))
            w32 = _gather_cat(wt, cfg.group).transpose(1, 2)                     # [B,D,T] view of [B,T,D]
        fuse_sent = cnn is not None
        if fuse_sent:
            cnn32 = cnn.detach().float().reshape(Bl, -1).contiguous()
            rnn32 = rnn.detach().float().reshape(rnn.shape[-2], -1).contiguous()
            if ex.W > 1:
                rnn32 = _gather_cat(rnn32, cfg.group)
        # the math mode was resolved from the LOCAL caption padding; after the exchange every rank sees the agreed T:
        # if that leaves the tensor-core range, all ranks fall back to the fp32 kernels together
        math = cfg.math
        if math != native.AGB_MATH_FP32 and hasattr(o, "damsm_supported") and \
                not o.damsm_supported(int(w32.shape[2]), D, int(img3.shape[2]), math):
            math = native.AGB_MATH_FP32
        ctx.math = math
        save = math != native.AGB_MATH_FP32 and any(ctx.needs_input_grad[:2])       # training forward
        m, att, scos, ws = o.damsm_fwd(img3, w32, ex.lens, cfg.gamma1, cfg.gamma2, cfg.eps, ex.row0, cfg.want_att,
                                       math, cnn32 if fuse_sent else None, rnn32 if fuse_sent else None, True,
                                       save)
        # packed 16-bit operands (and, after a training forward, the saved context vectors), reused by backward
        ctx.ws = ws if math != native.AGB_MATH_FP32 else None
        ctx.ws_saved = save
        m_all = _gather_cat(m, cfg.group) if ex.W > 1 else m
        loss, dm = o.contrastive(m_all, ex.cls, ex.labels, cfg.gamma3, cfg.lam, ex.row0, Bl)
        ctx.save_for_backward(img3, w32, dm, m)
        ctx.cfg, ctx.ex = cfg, ex
        ctx.meta = (img.shape, img.dtype, words.dtype, T_local)
        outs = [loss.reshape(())]
        if att is None:
            att = torch.empty(0, device=img.device)
        elif att.shape[1] != T_local:
            att = att[:, :T_local].contiguous()                                  # rows t >= L are zero anyway
        outs.append(att)
        if fuse_sent:
            outs.append(scos)
            ctx.mark_non_differentiable(att, scos)
        else:
            ctx.mark_non_differentiable(att)
        return tuple(outs)

    @staticmethod
    def backward(ctx, dloss, *unused):
        img3, w32, dm, m = ctx.saved_tensors
        cfg, ex = ctx.cfg, ctx.ex
        ishape, idt, wdt, T_local = ctx.meta
        need_w = ctx.needs_input_grad[1]
        gscale = dloss.detach().float().reshape(1).contiguous()
        dimg, dwords = cfg.ops.damsm_bwd(img3, w32, ex.lens, cfg.gamma1, cfg.gamma2, cfg.eps, dm, gscale, need_w,
                                         ctx.math, m, ctx.ws, ctx.ws_saved)
        ctx.ws = None
        if dwords is not None:
            if ex.W > 1:
                dwords = _reduce_scatter_sum(dwords, cfg.group)
            dwords = dwords[:, :T_local].transpose(1, 2).to(wdt)                 # [Bl,D,T] like words_emb
        dimg = dimg.reshape(ishape).to(idt) if ctx.needs_input_grad[0] else None
        return dimg, dwords, None, None, None, None


class _SentLossFn(torch.autograd.Function):
    """loss from the cosine matrix; scos_pre: matrix already produced by the fused DAMSM launch"""

    @staticmethod
    def forward(ctx, cnn, rnn, cfg: DamsmConfig, ex: _Exchange, scos_pre):
        o = cfg.ops
        D = cnn.shape[-1]
        cnn32 = cnn.detach().float().reshape(-1, D).contiguous()
        rnn32 = rnn.detach().float().reshape(-1, D).contiguous()
        if ex.W > 1:
            rnn32 = _gather_cat(rnn32, cfg.group)
        scos = scos_pre if scos_pre is not None else o.sent_cos_fwd(cnn32, rnn32, cfg.eps)
        s_all = _gather_cat(scos, cfg.group) if ex.W > 1 else scos
        loss, ds = o.contrastive(s_all, ex.cls, ex.labels, cfg.gamma3, cfg.lam, ex.row0, cnn32.shape[0])
        ctx.save_for_backward(cnn32, rnn32, ds)
        ctx.cfg, ctx.ex = cfg, ex
        ctx.meta = (cnn.shape, cnn.dtype, rnn.shape, rnn.dtype)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, dloss):
        cnn32, rnn32, ds = ctx.saved_tensors
        cfg, ex = ctx.cfg, ctx.ex
        cshape, cdt, rshape, rdt = ctx.meta
        gscale = dloss.detach().float().reshape(1).contiguous()
        dcnn, drnn = cfg.ops.sent_cos_bwd(cnn32, rnn32, cfg.eps, ds, gscale, ctx.needs_input_grad[0],
                                          ctx.needs_input_grad[1])
        if drnn is not None:
            if ex.W > 1:
                drnn = _reduce_scatter_sum(drnn, cfg.group)
            drnn = drnn.reshape(rshape).to(rdt)
        if dcnn is not None:
            dcnn = dcnn.reshape(cshape).to(cdt)
        return dcnn, drnn, None, None, None


# ------------------------------------------------------------------------------------------------
# the same losses while torch.compile traces: the agb:: ops (agb_native/torch_ops.py), single process only
# ------------------------------------------------------------------------------------------------
def _op_path(*cfgs: DamsmConfig) -> bool:
    """trace the agb:: ops: compiling, the native kernels (not an injected backend) and no process group (the
    NCCL exchange of a sharded loss stays eager, behind a graph break)"""
    return torch.compiler.is_compiling() and all(c.ops is native_ops and c.group is None for c in cfgs)


def _words_loss_op(img, words, cfg: DamsmConfig, ex: _Exchange):
    """_WordsLossFn of a single process as agb:: ops: (loss, packed att [Bl,T,R] or empty)"""
    Bl, D = img.shape[0], img.shape[1]
    img3 = img.float().reshape(Bl, D, -1).contiguous()
    w32 = words.float()
    math = cfg.math
    if math != native.AGB_MATH_FP32 and \
            not torch_ops.host_query("agb_damsm_supported", int(w32.shape[2]), D, int(img3.shape[2]), math):
        math = native.AGB_MATH_FP32
    save = math != native.AGB_MATH_FP32 and torch.is_grad_enabled() and (img.requires_grad or words.requires_grad)
    m, att, _, _ = torch.ops.agb.damsm_fwd(img3, w32, ex.lens, None, None, cfg.gamma1, cfg.gamma2, cfg.eps, 0,
                                           cfg.want_att, math, save)
    loss, _ = torch.ops.agb.contrastive(m, ex.cls, ex.labels, cfg.gamma3, cfg.lam, 0, Bl, True)
    return loss.reshape(()), att


def _sentence_loss_op(cnn, rnn, cfg: DamsmConfig, ex: _Exchange):
    """_SentLossFn of a single process as agb:: ops"""
    D = cnn.shape[-1]
    cnn32 = cnn.float().reshape(-1, D).contiguous()
    rnn32 = rnn.float().reshape(-1, D).contiguous()
    scos = torch.ops.agb.sent_cos_fwd(cnn32, rnn32, cfg.eps)
    loss, _ = torch.ops.agb.contrastive(scos, ex.cls, ex.labels, cfg.gamma3, cfg.lam, 0, cnn32.shape[0], True)
    return loss.reshape(())


def split_att_maps(att: torch.Tensor, cap_lens, ih: int, iw: int, row0: int = 0) -> List[torch.Tensor]:
    """packed beta [Bl,T,R] of the matched pairs -> the reference's list of [1, L_i, ih, iw]
    (words_loss.py:63).  Needs the caption lengths on the host, like the reference (:41)."""
    lens = cap_lens.tolist() if torch.is_tensor(cap_lens) else [int(x) for x in cap_lens]
    return [att[b, : int(lens[b])].reshape(1, int(lens[b]), ih, iw) for b in range(att.shape[0])]


def words_loss(img_features, words_emb, labels, cap_lens, class_ids, cfg: DamsmConfig):
    """(wloss, packed att [Bl,T,R] or None)"""
    cfg.ops.require_cuda(img_features, words_emb) if hasattr(cfg.ops, "require_cuda") else None
    ex = _Exchange(cfg, img_features.shape[0], labels, cap_lens, class_ids, img_features.device)
    if _op_path(cfg):
        loss, att = _words_loss_op(img_features, words_emb, cfg, ex)
    else:
        loss, att = _WordsLossFn.apply(img_features, words_emb, cfg, ex, None, None)
    return loss, (att if cfg.want_att else None)


def sentence_loss(cnn_code, rnn_code, labels, class_ids, cfg: DamsmConfig):
    cfg.ops.require_cuda(cnn_code, rnn_code) if hasattr(cfg.ops, "require_cuda") else None
    n_local = cnn_code.shape[-2]
    ex = _Exchange(cfg, n_local, labels, None, class_ids, cnn_code.device)
    if _op_path(cfg):
        return _sentence_loss_op(cnn_code, rnn_code, cfg, ex)
    return _SentLossFn.apply(cnn_code, rnn_code, cfg, ex, None)


def damsm_losses(img_features, cnn_code, words_emb, rnn_code, labels, cap_lens, class_ids,
                 wcfg: DamsmConfig, scfg: DamsmConfig):
    """Both losses of one DAMSM step (pretrain_damsm.py:128-129) with the sentence cosine matrix
    coming out of the same native call as the word-region similarity.
    Returns (wloss, sloss, packed att or None)."""
    wcfg.ops.require_cuda(img_features, words_emb, cnn_code, rnn_code) if hasattr(wcfg.ops, "require_cuda") else None
    ex = _Exchange(wcfg, img_features.shape[0], labels, cap_lens, class_ids, img_features.device)
    if _op_path(wcfg, scfg):
        # traced: the two losses one after the other on the current stream (the kernels are deterministic, so the
        # results are those of the forked-stream eager path)
        sloss = _sentence_loss_op(cnn_code, rnn_code, scfg, ex)
        wloss, att = _words_loss_op(img_features, words_emb, wcfg, ex)
        return wloss, sloss, (att if wcfg.want_att else None)
    if ex.W == 1 and img_features.is_cuda:
        # Single process: the sentence loss (cosine matrix, its contrastive CE and, in backward, its two
        # gradient kernels) is independent of the word-region kernels, so it runs on a forked stream beside
        # them.  Autograd replays each node's backward on its forward stream, so the overlap carries over
        # to the backward pass; the fork / join are events, i.e. capturable in a CUDA graph.
        main = torch.cuda.current_stream(img_features.device)
        side = _side_stream(img_features.device)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            sloss = _SentLossFn.apply(cnn_code, rnn_code, scfg, ex, None)
        wloss, att = _WordsLossFn.apply(img_features, words_emb, wcfg, ex, None, None)
        main.wait_stream(side)
        sloss.record_stream(main)
        return wloss, sloss, (att if wcfg.want_att else None)
    wloss, att, scos = _WordsLossFn.apply(img_features, words_emb, wcfg, ex, cnn_code, rnn_code)
    sloss = _SentLossFn.apply(cnn_code, rnn_code, scfg, ex, scos)
    return wloss, sloss, (att if wcfg.want_att else None)


_SIDE_STREAMS = {}


def _side_stream(device) -> "torch.cuda.Stream":
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    s = _SIDE_STREAMS.get(key)
    if s is None:
        s = _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return s


def pair_index(image_idx, caption_idx, device):
    """image_idx, caption_idx [P] (numpy, int64 or int32) -> two contiguous int32 device tensors"""
    pi = as_device_i32(image_idx, device).reshape(-1)
    pc = as_device_i32(caption_idx, device).reshape(-1)
    if pi.shape[0] != pc.shape[0]:
        raise ValueError(f"image_idx has {pi.shape[0]} entries, caption_idx {pc.shape[0]}")
    return pi, pc


def chunk_pairs(N: int, Nc: int, P: int, T: int, D: int, R: int, math: int, ws_bytes, budget: int) -> int:
    """the most pairs of a list whose workspace ws_bytes(N, Nc, pairs, T, D, R, math) fits budget (the size grows
    with the pair count); long lists run in contiguous chunks of that many pairs"""
    if ws_bytes(N, Nc, 1, T, D, R, math) == 0:
        raise native.NativeError(f"pair DAMSM shape N={N} Nc={Nc} T={T} D={D} R={R} is unsupported")
    lo, hi = 0, P
    while lo < hi:
        mid = (lo + hi + 1) // 2
        nb = ws_bytes(N, Nc, mid, T, D, R, math)
        if 0 < nb <= budget:
            lo = mid
        else:
            hi = mid - 1
    if lo == 0:
        need = ws_bytes(N, Nc, 1, T, D, R, math)
        raise native.NativeError(f"workspace_bytes={budget} is below the {need} bytes one pair against {N} images needs")
    return lo
