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
from ..agb_native import torch_ops


def _region_head_operands(x, weight):
    """x [B,Cin,H,W], weight [Cout,Cin,1,1] -> the operands of agb::region_head_fwd: x [B,Cin,H*W] and weight
    [Cout,Cin], fp32 contiguous"""
    B, Cin = x.shape[:2]
    return x.float().reshape(B, Cin, -1).contiguous(), weight.reshape(weight.shape[0], Cin).float().contiguous()


class _RegionHead(torch.autograd.Function):
    """agb::region_head_fwd without the dispatcher, with the casts and reshapes inside the one autograd node"""

    @staticmethod
    def forward(ctx, x, weight):
        inputs = _region_head_operands(x, weight)
        feat, ws = torch_ops.region_head_fwd(*inputs)
        torch_ops.region_head_setup(ctx, inputs, (feat, ws), bwd=torch_ops.region_head_bwd)
        ctx.meta = (x.shape, x.dtype, weight.shape, weight.dtype)
        return feat.reshape(*feat.shape[:2], *x.shape[2:]).to(x.dtype)

    @staticmethod
    def backward(ctx, dfeat):
        xshape, xdt, wshape, wdt = ctx.meta
        dx, dw = torch_ops.region_head_backward(ctx, dfeat.float().flatten(2), None)
        return ((None if dx is None else dx.reshape(xshape).to(xdt)),
                (None if dw is None else dw.reshape(wshape).to(wdt)))


def region_head(x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    """x [B, Cin, H, W], weight [Cout, Cin, 1, 1] -> [B, Cout, H, W]: _RegionHead, or agb::region_head_fwd while
    torch.compile traces (same kernels, same operands)"""
    if torch.compiler.is_compiling():
        feat, _ = torch.ops.agb.region_head_fwd(*_region_head_operands(x, weight))
        return feat.reshape(*feat.shape[:2], *x.shape[2:]).to(x.dtype)
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
