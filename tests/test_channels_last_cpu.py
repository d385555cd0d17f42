"""Channels_last word attention without a GPU: the layout rule, fake-kernel strides, the new C exports and the
refusal of CPU tensors and of other stride patterns."""
import subprocess

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

CL = torch.channels_last
NEW_EXPORTS = ("agb_word_attn_fwd_nhwc", "agb_word_attn_bwd_nhwc")


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


def test_new_exports_exist(agb):
    lib = agb.native.lib()
    for name in NEW_EXPORTS:
        assert hasattr(lib, name) and name in agb.native.SIGNATURES
    r = subprocess.run(["nm", "-D", "--defined-only", lib._name], capture_output=True, text=True)
    if r.returncode == 0:
        for name in NEW_EXPORTS:
            assert name in r.stdout


def test_layout_rule(agb):
    ops = agb.ops
    x = torch.empty(2, 8, 4, 5)
    assert ops.attn_layout_nhwc(x) is False
    assert ops.attn_layout_nhwc(x.contiguous(memory_format=CL)) is True
    # both NCHW- and channels_last-contiguous: the NCHW path
    for y in (torch.empty(2, 1, 4, 5).contiguous(memory_format=CL), torch.empty(2, 8, 1, 1).contiguous(memory_format=CL)):
        assert ops.attn_layout_nhwc(y) is False
        assert ops.attn_memory_format(y) == torch.contiguous_format
    for bad in (x[:, :, ::2], x.permute(0, 1, 3, 2), torch.empty(8, 2, 4, 5).transpose(0, 1)):
        with pytest.raises(RuntimeError, match="contiguous NCHW or channels_last"):
            ops.attn_layout_nhwc(bad)


def test_pixel_stride_of_concat_slice(agb):
    buf = torch.empty(2, 16, 4, 5).contiguous(memory_format=CL)
    assert agb.ops._nhwc_pixel_stride(buf[:, 8:]) == 16
    assert agb.ops._nhwc_pixel_stride(buf) == 16
    assert agb.ops._nhwc_pixel_stride(torch.empty(2, 8, 4, 5)) is None


def test_fake_kernels_take_the_images_memory_format(agb):
    with FakeTensorMode(allow_non_fake_inputs=False):
        for fmt in (torch.contiguous_format, CL):
            im = torch.empty(2, 32, 8, 8, device="cuda", dtype=torch.bfloat16).contiguous(memory_format=fmt)
            words = torch.empty(2, 64, 18, device="cuda")
            weight = torch.empty(32, 64, device="cuda")
            mask = torch.empty(2, 18, dtype=torch.int64, device="cuda")
            ctx, attn, we = torch.ops.agb.word_attn_fwd(im, words, weight, mask, True, True)
            assert ctx.shape == im.shape and attn.shape == (2, 18, 8, 8) and we.shape == (2, 32, 18)
            assert ctx.is_contiguous(memory_format=fmt) and attn.is_contiguous(memory_format=fmt)
            out, attn2, _ = torch.ops.agb.word_attn_cat(im, words, weight, mask, True, True)
            assert out.shape == (2, 64, 8, 8) and out.is_contiguous(memory_format=fmt)
            assert attn2.is_contiguous(memory_format=fmt)
            di, dw, dwt = torch.ops.agb.word_attn_bwd(im, words, weight, mask, we, ctx, attn, True, True, True)
            assert di.shape == im.shape and di.is_contiguous(memory_format=fmt)
            assert dw.shape == (2, 64, 18) and dwt.shape == (32, 64)
        if fmt == CL:
            assert not ctx.is_contiguous()


def test_cpu_tensors_and_other_layouts_are_refused(agb):
    mod = agb.AttentionModule(8, 16)
    mod.apply_mask(torch.ones(2, 5, dtype=torch.int64))
    im = torch.randn(2, 8, 4, 4).contiguous(memory_format=CL)
    with pytest.raises(RuntimeError, match="CUDA"):
        mod(im, torch.randn(2, 16, 5))
    with pytest.raises(RuntimeError, match="CUDA"):
        agb.ops.word_attn_fwd(im, torch.randn(2, 16, 5), torch.randn(8, 16), torch.ones(2, 5, dtype=torch.int64),
                              True)


def test_module_to_channels_last_keeps_the_weight_usable(agb):
    mod = agb.AttentionModule(8, 16).to(memory_format=CL)
    w = mod.conv1.weight
    assert w.shape == (8, 16, 1, 1)
    wt = w.reshape(8, -1)
    assert wt.is_contiguous() and wt.data_ptr() == w.data_ptr()
