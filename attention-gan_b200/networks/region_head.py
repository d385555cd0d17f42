"""B200-native region-feature head of the image encoder (SURVEY.md section 8, row f3).

``RegionFeatureHead(out_dim)`` is the ``emb_features`` 1x1 convolution of the reference's ``CNNEncoder``
(networks/cnn_encoder.py:56,101: ``Layers.conv1x1(768, out_dim)``, no bias) with the same parameter name and
shape (``emb_features.weight [out_dim, 768, 1, 1]``), so the head entries of ``CNNEncoder.pkl`` load unchanged.
Forward and backward run on tcgen05 through the C ABI (``agb_region_head_fwd/bwd``): the forward with split
bf16 operands (features within ~1e-5 of fp32 arithmetic; cuDNN's default for this convolution is TF32, 5e-4),
the backward with plain bf16 operands.
"""
from __future__ import annotations

import torch
from torch import nn

from ..agb_native import ops
from ..agb_native import torch_ops  # noqa: F401  (registers torch.ops.agb, used while compiling)


class _RegionHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight):
        B, Cin, H, W = x.shape
        x3 = (x if x.dtype == torch.float32 else x.float()).reshape(B, Cin, H * W).contiguous()
        w2 = weight.reshape(weight.shape[0], Cin)
        w2 = (w2 if w2.dtype == torch.float32 else w2.float()).contiguous()
        feat, ws = ops.region_head_fwd(x3.detach(), w2.detach(), keep_ws=True)
        ctx.save_for_backward(x3, w2)
        ctx.ws = ws if any(ctx.needs_input_grad) else None        # bf16 copies of x and W, reused by backward
        ctx.meta = (x.shape, x.dtype, weight.shape, weight.dtype)
        return feat.reshape(B, weight.shape[0], H, W).to(x.dtype)

    @staticmethod
    def backward(ctx, dfeat):
        x3, w2 = ctx.saved_tensors
        xshape, xdt, wshape, wdt = ctx.meta
        d3 = dfeat.float().reshape(x3.shape[0], w2.shape[0], -1).contiguous()
        dw, dx = ops.region_head_bwd(x3, w2, d3, ctx.needs_input_grad[1], ctx.needs_input_grad[0], ctx.ws)
        ctx.ws = None
        if dw is not None:
            dw = dw.reshape(wshape).to(wdt)
        if dx is not None:
            dx = dx.reshape(xshape).to(xdt)
        return dx, dw


def region_head(x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """x [B, Cin, H, W], weight [Cout, Cin, 1, 1] -> [B, Cout, H, W]: _RegionHead, or agb::region_head_fwd while
    torch.compile traces (same kernels, same operands)"""
    if torch.compiler.is_compiling():
        B, Cin, H, W = x.shape
        x3 = (x if x.dtype == torch.float32 else x.float()).reshape(B, Cin, H * W).contiguous()
        w2 = weight.reshape(weight.shape[0], Cin)
        w2 = (w2 if w2.dtype == torch.float32 else w2.float()).contiguous()
        feat, _ = torch.ops.agb.region_head_fwd(x3, w2)
        return feat.reshape(B, weight.shape[0], H, W).to(x.dtype)
    return _RegionHead.apply(x, weight)


class RegionFeatureHead(nn.Module):
    def __init__(self, out_dim: int = 256, in_dim: int = 768):
        super().__init__()
        self.emb_features = nn.Conv2d(in_dim, out_dim, kernel_size=1, stride=1, padding=0, bias=False)
        self.emb_features.weight.data.uniform_(-0.1, 0.1)            # cnn_encoder.py:60-63

    def forward(self, mixed_6e: torch.Tensor) -> torch.Tensor:
        """mixed_6e [B, 768, 17, 17] -> region features [B, out_dim, 17, 17]"""
        ops.require_cuda(mixed_6e, self.emb_features.weight)
        return region_head(mixed_6e, self.emb_features.weight)
