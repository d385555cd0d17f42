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
from ..agb_native import torch_ops

GlobalAttention = None  # set below (BASELINE.json's name for AttentionModule)


def _word_attn_operands(images, words, weight, mask):
    """the operands of agb::word_attn_fwd / word_attn_cat after images: words and weight [C,E] in fp32, mask int64"""
    wt32 = weight.reshape(weight.shape[0], -1).float().contiguous()
    return words.float(), wt32, mask.to(device=images.device, dtype=torch.int64).contiguous()


def _word_attn_grads(ctx, grads):
    """the gradients of torch_ops.word_attn_backward / word_attn_cat_backward in the dtypes and shapes of words and
    conv1.weight"""
    di, dw, dwt = grads[:3]
    words_dtype, weight_dtype, weight_shape = ctx.meta
    return (di, None if dw is None else dw.to(words_dtype),
            None if dwt is None else dwt.reshape(weight_shape).to(weight_dtype), None, None, None)


class _WordAttention(torch.autograd.Function):
    """fused  W.e projection -> scores -> mask -> softmax over words -> context   (fwd + bwd): agb::word_attn_fwd
    without the dispatcher, with the casts of words and conv1.weight inside the one autograd node"""

    @staticmethod
    def forward(ctx, images, words, weight, mask, scaled, want_attn):
        inputs = (images, *_word_attn_operands(images, words, weight, mask), scaled, want_attn)
        out = torch_ops.word_attn_fwd(*inputs)
        torch_ops.word_attn_setup(ctx, inputs, out, bwd=torch_ops.word_attn_bwd)
        ctx.meta = (words.dtype, weight.dtype, weight.shape)
        return out[0], out[1]

    @staticmethod
    def backward(ctx, dctx, dattn):
        return _word_attn_grads(ctx, torch_ops.word_attn_backward(ctx, dctx, dattn, None))


def _check_cat_out(images, out):
    """`out` of forward_into: [B, 2C, H, W], the images' dtype and memory format (contiguous or channels_last)"""
    B, C, H, W = images.shape
    fmt = ops.attn_memory_format(images)
    if out.shape != (B, 2 * C, H, W) or out.dtype != images.dtype or not out.is_contiguous(memory_format=fmt):
        if fmt == torch.channels_last:
            raise RuntimeError("forward_into: `out` must be a channels_last [B, 2*C, H, W] tensor of the images' "
                               "dtype (the images are channels_last)")
        raise RuntimeError("forward_into: `out` must be a contiguous [B, 2*C, H, W] tensor of the images' dtype")


class _WordAttentionInto(torch.autograd.Function):
    """the same fused attention, writing  cat((images, context), 1)  into a caller-owned [B, 2C, H, W] buffer:
    the context leaves the kernel at channel offset C (ctx batch stride 2C*H*W in the C ABI; for channels_last maps
    also pixel stride 2C), so GenNextStage's torch.cat (generator_submodules.py:116) costs one copy of `images`
    instead of re-reading and re-writing both"""

    @staticmethod
    def forward(ctx, images, words, weight, mask, scaled, want_attn, out):
        _check_cat_out(images, out)
        inputs = (images, *_word_attn_operands(images, words, weight, mask), scaled, want_attn)
        res = torch_ops.word_attn_into(out, *inputs)
        ctx.mark_dirty(out)
        torch_ops.word_attn_setup(ctx, inputs, res, bwd=torch_ops.word_attn_bwd)
        ctx.meta = (words.dtype, weight.dtype, weight.shape)
        return res[0], res[1]

    @staticmethod
    def backward(ctx, dout, dattn):
        return _word_attn_grads(ctx, torch_ops.word_attn_cat_backward(ctx, dout, dattn, None)) + (None,)


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
        attn [B, T, H, W]).  images may be contiguous NCHW or channels_last; the outputs (and the gradient of
        images) take its memory format."""
        if self.mask is None:
            # the reference dereferences self.mask unconditionally (attention.py:47,65)
            raise AttributeError("AttentionModule.forward called before apply_mask(mask)")
        ops.require_cuda(images, words, self.conv1.weight)
        if torch.compiler.is_compiling():
            w32, wt32, m64 = _word_attn_operands(images, words, self.conv1.weight, self.mask)
            ctx, attn, _ = torch.ops.agb.word_attn_fwd(images, w32, wt32, m64, bool(scaled), True)
            return ctx, attn
        return _WordAttention.apply(images, words, self.conv1.weight, self.mask, bool(scaled), True)

    def forward_into(self, images, words, out, scaled=True, want_attn=True):
        """images [B, C, H, W], words [B, E, T], out [B, 2C, H, W] (pre-allocated, in the memory format of images:
        contiguous, or channels_last for channels_last images) ->
        (out, attn [B, T, H, W] or None) with  out == torch.cat((images, context), 1)  -- what GenNextStage builds
        right after the attention call (generator_submodules.py:113-116).  Not part of the reference API."""
        if self.mask is None:
            raise AttributeError("AttentionModule.forward_into called before apply_mask(mask)")
        ops.require_cuda(images, words, self.conv1.weight, out)
        if torch.compiler.is_compiling():
            # the op returns a fresh buffer (custom ops do not write into their inputs' storage): one extra copy
            _check_cat_out(images, out)
            res, attn = self.forward_cat(images, words, scaled, want_attn)
            return out.copy_(res), attn
        res, attn = _WordAttentionInto.apply(images, words, self.conv1.weight, self.mask, bool(scaled),
                                             bool(want_attn), out)
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
        out = torch.empty((B, 2 * C, H, W), dtype=images.dtype, device=images.device,
                          memory_format=ops.attn_memory_format(images))
        return self.forward_into(images, words, out, scaled, want_attn)


GlobalAttention = AttentionModule


def _func_attention_operands(query, context):
    """query [B,D,L] and context [B,D,ih,iw] -> the operands of agb::func_attention_fwd: fp32, context [B,D,R]"""
    return query.float(), context.float().reshape(context.shape[0], context.shape[1], -1).contiguous()


class _FuncAttention(torch.autograd.Function):
    """agb::func_attention_fwd without the dispatcher, with the casts and reshapes inside the one autograd node"""

    @staticmethod
    def forward(ctx, query, context, gamma1, scaled):
        inputs = (*_func_attention_operands(query, context), gamma1, scaled)
        wc, attn = torch_ops.func_attention_fwd(*inputs)
        torch_ops.func_attention_setup(ctx, inputs, (wc, attn), bwd=torch_ops.func_attention_bwd)
        ctx.meta = (query.dtype, context.dtype, context.shape)
        return wc.to(query.dtype), attn.reshape(*attn.shape[:2], *context.shape[2:]).to(query.dtype)

    @staticmethod
    def backward(ctx, dwc, dattn):
        qdt, cdt, cshape = ctx.meta
        dq, dc, _, _ = torch_ops.func_attention_backward(ctx, None if dwc is None else dwc.float(),
                                                         None if dattn is None else dattn.float().flatten(2))
        return (None if dq is None else dq.to(qdt)), (None if dc is None else dc.reshape(cshape).to(cdt)), None, None


def func_attention(query, context, gamma1=4.0, scaled=True):
    """query [B, D, L] (words), context [B, D, ih, iw] (regions) ->
    (weightedContext [B, D, L], attn [B, L, ih, iw])        reference networks/attention.py:82-121"""
    ops.require_cuda(query, context)
    if torch.compiler.is_compiling():
        wc, attn = torch.ops.agb.func_attention_fwd(*_func_attention_operands(query, context), float(gamma1),
                                                    bool(scaled))
        return wc.to(query.dtype), attn.reshape(*attn.shape[:2], *context.shape[2:]).to(query.dtype)
    return _FuncAttention.apply(query, context, float(gamma1), bool(scaled))
