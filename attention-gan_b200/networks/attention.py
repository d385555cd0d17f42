"""Drop-in for the reference ``networks/attention.py`` (ku222/Attention-GAN), B200-native.

Same names, signatures and return conventions as the reference:

* ``AttentionModule(nc_in, emb_dim)`` with ``conv1`` (bias-free 1x1 ``Conv2d``, weight
  ``[nc_in, emb_dim, 1, 1]`` so ``Generator.pkl`` state dicts load unchanged), ``mask``,
  ``apply_mask(mask)`` and ``forward(images, words, scaled=True) -> (context, attn)``
  (reference networks/attention.py:15-79);
* ``func_attention(query, context, gamma1=4.0, scaled=True) -> (weightedContext, attn)``
  (reference networks/attention.py:82-121).

The arithmetic runs in hand-written sm_100a kernels behind the C ABI of libattngan_b200.so
(forward and backward); nothing here falls back to PyTorch ops, and CPU tensors are rejected.
"""
from __future__ import annotations

import torch
from torch import nn

from ..agb_native import ops
from ..agb_native import torch_ops  # noqa: F401  (registers torch.ops.agb, used while compiling)

GlobalAttention = None  # set below (BASELINE.json's name for AttentionModule)


class _WordAttention(torch.autograd.Function):
    """fused  W.e projection -> scores -> mask -> softmax over words -> context   (fwd + bwd)"""

    @staticmethod
    def forward(ctx, images, words, weight, mask, scaled):
        w32 = words if words.dtype == torch.float32 else words.float()
        wt = weight.reshape(weight.shape[0], -1)
        wt32 = (wt if wt.dtype == torch.float32 else wt.float()).contiguous()
        m64 = mask if mask.dtype == torch.int64 else mask.to(torch.int64)
        m64 = m64.to(images.device).contiguous()
        out, attn, we = ops.word_attn_fwd(images.detach(), w32.detach(), wt32.detach(), m64, scaled, True)
        ctx.save_for_backward(images, w32, wt32, m64, we)
        ctx.scaled = scaled
        ctx.words_dtype = words.dtype
        ctx.weight_dtype = weight.dtype
        ctx.weight_shape = weight.shape
        ctx.set_materialize_grads(False)
        return out, attn

    @staticmethod
    def backward(ctx, dctx, dattn):
        images, w32, wt32, m64, we = ctx.saved_tensors
        if dctx is None:
            dctx = torch.zeros_like(images)
        need_img, need_words, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        dimages, dwords, dweight = ops.word_attn_bwd(images, w32, wt32, m64, we, dctx.to(images.dtype),
                                                     None if dattn is None else dattn.to(images.dtype),
                                                     ctx.scaled, need_words, need_w)
        if dwords is not None:
            dwords = dwords.to(ctx.words_dtype)
        if dweight is not None:
            dweight = dweight.reshape(ctx.weight_shape).to(ctx.weight_dtype)
        return (dimages if need_img else None), dwords, dweight, None, None


class _WordAttentionInto(torch.autograd.Function):
    """the same fused attention, writing  cat((images, context), 1)  into a caller-owned [B, 2C, H, W] buffer:
    the context leaves the kernel at channel offset C (ctx batch stride 2C*H*W in the C ABI), so GenNextStage's
    torch.cat (generator_submodules.py:116) costs one copy of `images` instead of re-reading and re-writing both"""

    @staticmethod
    def forward(ctx, images, words, weight, mask, scaled, out, want_attn):
        B, C, H, W = images.shape
        if out.shape != (B, 2 * C, H, W) or out.dtype != images.dtype or not out.is_contiguous():
            raise RuntimeError("forward_into: `out` must be a contiguous [B, 2*C, H, W] tensor of the images' dtype")
        w32 = words if words.dtype == torch.float32 else words.float()
        wt = weight.reshape(weight.shape[0], -1)
        wt32 = (wt if wt.dtype == torch.float32 else wt.float()).contiguous()
        m64 = (mask if mask.dtype == torch.int64 else mask.to(torch.int64)).to(images.device).contiguous()
        out[:, :C].copy_(images.detach())
        _, attn, we = ops.word_attn_fwd(images.detach(), w32.detach(), wt32.detach(), m64, scaled, want_attn,
                                        ctx_out=out[:, C:])
        ctx.mark_dirty(out)
        ctx.save_for_backward(images, w32, wt32, m64, we)
        ctx.scaled = scaled
        ctx.meta = (words.dtype, weight.dtype, weight.shape, C)
        ctx.set_materialize_grads(False)
        if attn is None:
            attn = torch.empty(0, device=images.device, dtype=images.dtype)
            ctx.mark_non_differentiable(attn)
        return out, attn

    @staticmethod
    def backward(ctx, dout, dattn):
        images, w32, wt32, m64, we = ctx.saved_tensors
        wdt, wtdt, wshape, C = ctx.meta
        need_img, need_words, need_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2]
        if dout is None:
            return None, None, None, None, None, None, None
        dout = dout.to(images.dtype)
        if not dout.is_contiguous():
            dout = dout.contiguous()
        # d context is the second channel half of d out, read in place through its batch stride
        dimages, dwords, dweight = ops.word_attn_bwd(images, w32, wt32, m64, we, dout[:, C:],
                                                     None if dattn is None else dattn.to(images.dtype),
                                                     ctx.scaled, need_words, need_w)
        if need_img:
            dimages += dout[:, :C]                       # the identity half of the concatenation
        if dwords is not None:
            dwords = dwords.to(wdt)
        if dweight is not None:
            dweight = dweight.reshape(wshape).to(wtdt)
        return (dimages if need_img else None), dwords, dweight, None, None, None, None


def _word_attn_operands(images, words, weight, mask):
    """the operands the kernels take, built like _WordAttention.forward does (traced by torch.compile)"""
    w32 = words if words.dtype == torch.float32 else words.float()
    wt = weight.reshape(weight.shape[0], -1)
    wt32 = (wt if wt.dtype == torch.float32 else wt.float()).contiguous()
    m64 = (mask if mask.dtype == torch.int64 else mask.to(torch.int64)).to(images.device).contiguous()
    return w32, wt32, m64


class AttentionModule(nn.Module):
    """Word-context attention of the generator's refinement stages
    (reference networks/attention.py:15-79; called from generator_submodules.py:113-114)."""

    def __init__(self, nc_in: int, emb_dim: int):
        super().__init__()
        # utilities/layers.py:46-48: conv1x1 = Conv2d(k=1, stride=1, padding=0, bias=False)
        self.conv1 = nn.Conv2d(emb_dim, nc_in, kernel_size=1, stride=1, padding=0, bias=False)
        self.mask = None

    def apply_mask(self, mask):
        self.mask = mask

    def forward(self, images, words, scaled=True):
        """images [B, nc_in, H, W], words [B, emb_dim, T] -> (context [B, nc_in, H, W],
        attn [B, T, H, W])."""
        if self.mask is None:
            # the reference dereferences self.mask unconditionally (attention.py:47,65)
            raise AttributeError("AttentionModule.forward called before apply_mask(mask)")
        ops.require_cuda(images, words, self.conv1.weight)
        if torch.compiler.is_compiling():
            w32, wt32, m64 = _word_attn_operands(images, words, self.conv1.weight, self.mask)
            ctx, attn, _ = torch.ops.agb.word_attn_fwd(images, w32, wt32, m64, bool(scaled), True)
            return ctx, attn
        return _WordAttention.apply(images, words, self.conv1.weight, self.mask, bool(scaled))

    def forward_into(self, images, words, out, scaled=True, want_attn=True):
        """images [B, C, H, W], words [B, E, T], out [B, 2C, H, W] (pre-allocated, contiguous) ->
        (out, attn [B, T, H, W] or None) with  out == torch.cat((images, context), 1)  -- what GenNextStage builds
        right after the attention call (generator_submodules.py:113-116).  Not part of the reference API."""
        if self.mask is None:
            raise AttributeError("AttentionModule.forward_into called before apply_mask(mask)")
        ops.require_cuda(images, words, self.conv1.weight, out)
        if torch.compiler.is_compiling():
            # the op returns a fresh buffer (custom ops do not write into their inputs' storage): one extra copy
            B, C, H, W = images.shape
            if out.shape != (B, 2 * C, H, W) or out.dtype != images.dtype or not out.is_contiguous():
                raise RuntimeError("forward_into: `out` must be a contiguous [B, 2*C, H, W] tensor of the images' dtype")
            res, attn = self.forward_cat(images, words, scaled, want_attn)
            return out.copy_(res), attn
        res, attn = _WordAttentionInto.apply(images, words, self.conv1.weight, self.mask, bool(scaled), out,
                                             bool(want_attn))
        return res, (attn if want_attn else None)

    def forward_cat(self, images, words, scaled=True, want_attn=True):
        """images [B, C, H, W], words [B, E, T] -> (torch.cat((images, context), 1) [B, 2C, H, W], attn [B, T, H, W]
        or None): forward_into with a buffer of its own.  The spelling for code compiled with torch.compile, where
        the kernel writes the context straight into the fresh buffer.  Not part of the reference API."""
        if self.mask is None:
            raise AttributeError("AttentionModule.forward_cat called before apply_mask(mask)")
        ops.require_cuda(images, words, self.conv1.weight)
        if torch.compiler.is_compiling():
            w32, wt32, m64 = _word_attn_operands(images, words, self.conv1.weight, self.mask)
            out, attn, _ = torch.ops.agb.word_attn_cat(images, w32, wt32, m64, bool(scaled), bool(want_attn))
            return out, (attn if want_attn else None)
        B, C, H, W = images.shape
        out = torch.empty((B, 2 * C, H, W), dtype=images.dtype, device=images.device)
        return self.forward_into(images, words, out, scaled, want_attn)


GlobalAttention = AttentionModule


class _FuncAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, query, context, gamma1, scaled):
        B, D, L = query.shape
        ih, iw = context.shape[2], context.shape[3]
        q32 = query if query.dtype == torch.float32 else query.float()
        c32 = (context if context.dtype == torch.float32 else context.float()).reshape(B, D, ih * iw).contiguous()
        wc, attn = ops.func_attention_fwd(q32.detach(), c32.detach(), gamma1, scaled)
        ctx.save_for_backward(q32, c32)
        ctx.cfg = (gamma1, scaled, query.dtype, context.dtype, context.shape)
        ctx.set_materialize_grads(False)
        return wc.to(query.dtype), attn.reshape(B, L, ih, iw).to(query.dtype)

    @staticmethod
    def backward(ctx, dwc, dattn):
        q32, c32 = ctx.saved_tensors
        gamma1, scaled, qdt, cdt, cshape = ctx.cfg
        if dwc is None:
            dwc = torch.zeros_like(q32)
        dwc = dwc.float().contiguous()
        if dattn is not None:
            dattn = dattn.float().reshape(q32.shape[0], q32.shape[2], -1).contiguous()
        dq, dc = ops.func_attention_bwd(q32, c32, gamma1, scaled, dwc, dattn,
                                        ctx.needs_input_grad[0], ctx.needs_input_grad[1])
        if dq is not None:
            dq = dq.to(qdt)
        if dc is not None:
            dc = dc.reshape(cshape).to(cdt)
        return dq, dc, None, None


def func_attention(query, context, gamma1=4.0, scaled=True):
    """query [B, D, L] (words), context [B, D, ih, iw] (regions) ->
    (weightedContext [B, D, L], attn [B, L, ih, iw])        reference networks/attention.py:82-121"""
    ops.require_cuda(query, context)
    if torch.compiler.is_compiling():
        B, D, L = query.shape
        ih, iw = context.shape[2], context.shape[3]
        q32 = query if query.dtype == torch.float32 else query.float()
        c32 = (context if context.dtype == torch.float32 else context.float()).reshape(B, D, ih * iw).contiguous()
        wc, attn = torch.ops.agb.func_attention_fwd(q32, c32, float(gamma1), bool(scaled))
        return wc.to(query.dtype), attn.reshape(B, L, ih, iw).to(query.dtype)
    return _FuncAttention.apply(query, context, float(gamma1), bool(scaled))
