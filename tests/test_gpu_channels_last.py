"""Generator word attention on channels_last feature maps (the NHWC kernels) on the GPU.

The NHWC path must compute exactly what the NCHW path computes: the same per-pixel arithmetic, the same tiles and
summation orders, only the addresses differ.  So every output and gradient is compared bit for bit with the NCHW
result of the same inputs, over the case grid of test_gpu_attention_tc.py and the attention cases of
test_gpu_parity.py (CUDA-core and tensor-core kernels, ragged and aligned HW, partial and all-masked captions).
The rest covers the oracle, output layouts, the concat buffer of forward_into, gradients that arrive in the other
layout, memory (no hidden copy of the images), kernel selection, torch.compile and CUDA-graph capture.
"""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_port as rp

pytestmark = pytest.mark.gpu
DEV = "cuda"
CL = torch.channels_last


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    assert pkg.native.lib().agb_version() >= 100
    return pkg


def _bits(t):
    t = t.detach().contiguous()
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def assert_bitwise(a, b, what=""):
    """equal bit for bit, NaN included (both NaN at the same places; other values identical)"""
    assert a.shape == b.shape and a.dtype == b.dtype, what
    na, nb = torch.isnan(a.detach()), torch.isnan(b.detach())
    assert torch.equal(na, nb), f"{what}: NaN positions differ"
    ia, ib = _bits(a), _bits(b)
    keep = ~na.contiguous()
    assert torch.equal(ia[keep], ib[keep]), f"{what}: values differ"


def _inputs(B, C, E, T, hw, dtype, seed, all_masked=False):
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=seed)
    if all_masked and B > 1:
        mask[1] = 0
    return (images.to(DEV, dtype), words.to(DEV), weight.reshape(C, E).contiguous().to(DEV), mask.to(DEV))


def _both_layouts(agb, images, words, weight, mask, scaled, with_dattn, need_dw, seed):
    """(NCHW results, NHWC results): ctx, attn, dimages, dwords, dweight"""
    B, C, H, W = images.shape
    T = words.shape[2]
    g = torch.Generator().manual_seed(seed)
    dctx = torch.randn(B, C, H, W, generator=g).to(DEV, images.dtype)
    dattn = torch.randn(B, T, H, W, generator=g).to(DEV, images.dtype) if with_dattn else None
    out = []
    for fmt in (torch.contiguous_format, CL):
        im = images.contiguous(memory_format=fmt)
        ctx, attn, we = agb.ops.word_attn_fwd(im, words, weight, mask, scaled, True)
        di, dw, dwt = agb.ops.word_attn_bwd(im, words, weight, mask, we, dctx.contiguous(memory_format=fmt),
                                            None if dattn is None else dattn.contiguous(memory_format=fmt),
                                            scaled, need_dw, need_dw)
        out.append((ctx, attn, di, dw, dwt))
    return out


# the dtype x C x T grid; each case runs a ragged HW (not a multiple of 8: CUDA-core kernels for every dtype) and
# an aligned one (tensor cores for 16-bit maps with C % 16 == 0)
GRID_C = [1, 3, 16, 32, 48, 64]
GRID_T = [1, 18, 32, 40, 64]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C", GRID_C)
@pytest.mark.parametrize("T", GRID_T)
def test_nhwc_equals_nchw_bitwise(agb, dtype, C, T):
    k = GRID_C.index(C) * len(GRID_T) + GRID_T.index(T)
    for hw, B in ((10, 3), (24, 4)):             # HW = 100 (ragged), 576 (4.5 tiles of 128)
        scaled = (k + hw) % 2 == 0
        with_dattn = k % 3 == 0
        need_dw = k % 4 != 1
        inp = _inputs(B, C, 40, T, hw, dtype, seed=100 * k + hw, all_masked=True)
        (c0, a0, d0, w0, t0), (c1, a1, d1, w1, t1) = _both_layouts(agb, *inp, scaled, with_dattn, need_dw, seed=k)
        tag = f"{dtype} C={C} T={T} hw={hw}"
        if C > 1:
            assert c1.is_contiguous(memory_format=CL) and a1.is_contiguous(memory_format=CL)
            assert d1.is_contiguous(memory_format=CL)
        assert torch.isnan(c1[1]).all() and torch.isnan(d1[1]).all()        # the all-masked sample
        assert_bitwise(c0, c1, "ctx " + tag)
        assert_bitwise(a0, a1, "attn " + tag)
        assert_bitwise(d0, d1, "d images " + tag)
        if need_dw:
            assert_bitwise(w0, w1, "d words " + tag)
            assert_bitwise(t0, t1, "d weight " + tag)
        else:
            assert w1 is None and t1 is None


PERSISTENT = [  # B, hw, T, C, dattn -- the persistent-kernel cases of test_gpu_attention_tc.py
    (40, 64, 18, 32, False), (600, 16, 18, 32, False), (5, 48, 32, 16, True), (3, 40, 7, 32, True),
    (2, 24, 64, 32, False), (3, 32, 40, 32, True), (20, 16, 50, 16, False), (2, 64, 64, 32, True),
    (7, 32, 18, 64, False)]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,hw,T,C,with_dattn", PERSISTENT)
def test_nhwc_equals_nchw_persistent_kernels(agb, dtype, B, hw, T, C, with_dattn):
    inp = _inputs(B, C, 64, T, hw, dtype, seed=7 * B + hw)
    r0, r1 = _both_layouts(agb, *inp, True, with_dattn, True, seed=B)
    for name, x, y in zip(("ctx", "attn", "d images", "d words", "d weight"), r0, r1):
        assert_bitwise(x, y, f"{name} {dtype} B={B} hw={hw} T={T} C={C}")


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-4), (torch.bfloat16, 1e-3 + 2.0 ** -8),
                                       (torch.float16, 1e-3 + 2.0 ** -11)])
def test_channels_last_module_matches_oracle(agb, dtype, tol):
    B, C, E, T, hw = 3, 32, 64, 18, 16
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=11)
    images = images.to(dtype)
    mod = agb.AttentionModule(C, E).to(DEV).to(memory_format=CL)
    with torch.no_grad():
        mod.conv1.weight.copy_(weight.to(DEV))
    mod.apply_mask(mask.to(DEV))
    im = images.to(DEV).contiguous(memory_format=CL).requires_grad_(True)
    ctx, attn = mod(im, words.to(DEV))
    g = torch.Generator().manual_seed(1)
    dctx = torch.randn(B, C, hw, hw, generator=g)
    ctx.backward(dctx.to(DEV, dtype).contiguous(memory_format=CL))
    h64 = images.double().numpy().reshape(B, C, -1)
    W64 = weight.reshape(C, E).double().numpy()
    rc, ra, _ = cf.word_attention_fwd(h64, words.double().numpy(), W64, mask.numpy(), True)
    dd = dctx.to(dtype).double().numpy().reshape(B, C, -1)
    dh, _, _ = cf.word_attention_bwd(h64, words.double().numpy(), W64, mask.numpy(), dd, None, True)

    def rel(x, ref):
        x = x.detach().double().cpu().numpy()
        return np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-30)
    assert rel(ctx, rc.reshape(ctx.shape)) < 2 * tol
    assert rel(attn, ra.reshape(attn.shape)) < 2 * tol
    assert rel(im.grad, dh.reshape(im.shape)) < 2 * tol
    assert im.grad.is_contiguous(memory_format=CL)


def _module(agb, dtype, C=32, E=64, T=18, hw=16, B=3, seed=5):
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=seed)
    mod = agb.AttentionModule(C, E).to(DEV)
    with torch.no_grad():
        mod.conv1.weight.copy_(weight.to(DEV))
    mod.apply_mask(mask.to(DEV))
    return mod, images.to(DEV, dtype), words.to(DEV)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_forward_into_channels_last_buffer_equals_cat(agb, dtype):
    mod, images, words = _module(agb, dtype)
    B, C, H, W = images.shape
    g = torch.Generator().manual_seed(3)
    dout = torch.randn(B, 2 * C, H, W, generator=g).to(DEV, dtype).contiguous(memory_format=CL)
    im0 = images.contiguous(memory_format=CL).requires_grad_(True)
    ctx, attn0 = mod(im0, words)
    ref = torch.cat((im0, ctx), 1)
    ref.backward(dout)
    im1 = images.contiguous(memory_format=CL).requires_grad_(True)
    buf = torch.empty(B, 2 * C, H, W, dtype=dtype, device=DEV, memory_format=CL)
    out, attn1 = mod.forward_into(im1, words, buf)
    assert out.data_ptr() == buf.data_ptr() and out.is_contiguous(memory_format=CL)
    out.backward(dout)
    assert_bitwise(ref, out, "forward_into out")
    assert_bitwise(attn0, attn1, "forward_into attn")
    assert_bitwise(im0.grad, im1.grad, "forward_into d images")
    # an NCHW gradient of out is converted once and gives the same result
    im2 = images.contiguous(memory_format=CL).requires_grad_(True)
    out2, _ = mod.forward_cat(im2, words)
    assert out2.is_contiguous(memory_format=CL)
    out2.backward(dout.contiguous())
    assert_bitwise(im0.grad, im2.grad, "forward_cat d images (NCHW gradient)")
    with pytest.raises(RuntimeError, match="channels_last"):
        mod.forward_into(images.contiguous(memory_format=CL), words, torch.empty(B, 2 * C, H, W, dtype=dtype,
                                                                                  device=DEV))


def test_gradient_in_the_other_layout(agb):
    mod, images, words = _module(agb, torch.bfloat16)
    g = torch.Generator().manual_seed(4)
    dctx = torch.randn(images.shape, generator=g).to(DEV, torch.bfloat16)
    dattn = torch.randn(3, 18, 16, 16, generator=g).to(DEV, torch.bfloat16)
    grads = []
    for dfmt in (CL, torch.contiguous_format):
        im = images.contiguous(memory_format=CL).requires_grad_(True)
        ctx, attn = mod(im, words)
        torch.autograd.backward((ctx, attn), (dctx.contiguous(memory_format=dfmt),
                                              dattn.contiguous(memory_format=dfmt)))
        grads.append((im.grad, mod.conv1.weight.grad.clone()))
        mod.conv1.weight.grad = None
    assert_bitwise(grads[0][0], grads[1][0], "d images")
    assert_bitwise(grads[0][1], grads[1][1], "d weight")
    # a broadcast gradient (strides 0) is accepted too
    im = images.contiguous(memory_format=CL).requires_grad_(True)
    mod(im, words)[0].sum().backward()
    assert im.grad.is_contiguous(memory_format=CL) and torch.isfinite(im.grad.float()).all()


def test_other_layouts_raise(agb):
    mod, images, words = _module(agb, torch.bfloat16)
    for bad in (images[:, :, ::2], images.permute(0, 1, 3, 2), images.transpose(0, 1).contiguous().transpose(0, 1)):
        with pytest.raises(RuntimeError, match="channels_last"):
            mod(bad, words)


def test_channels_last_forward_and_backward_allocate_no_copy_of_images(agb):
    B, C, T, hw, E = 16, 32, 18, 128, 256
    mod, images, words = _module(agb, torch.bfloat16, C=C, E=E, T=T, hw=hw, B=B)
    im = images.contiguous(memory_format=CL)
    es = im.element_size()
    img_bytes = im.numel() * es
    out_bytes = img_bytes + B * T * hw * hw * es + B * C * T * 4      # ctx + attn + W.e
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        ctx, attn, we = agb.ops.word_attn_fwd(im, words, mod.conv1.weight.reshape(C, E), mod.mask, True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < out_bytes + (4 << 20), (peak, out_bytes)          # a copy of images would add 16 MiB
    dctx = torch.randn_like(ctx)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    ws = agb.native.lib().agb_word_attn_bwd_workspace_bytes(B, C, hw * hw, E, T)
    di, _, _ = agb.ops.word_attn_bwd(im, words, mod.conv1.weight.reshape(C, E), mod.mask, we, dctx, None, True,
                                     True, True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < img_bytes + ws + (4 << 20), (peak, img_bytes + ws)
    assert di.is_contiguous(memory_format=CL)


@pytest.mark.parametrize("dtype,T", [(torch.bfloat16, 18), (torch.float16, 18), (torch.bfloat16, 40)])
def test_tensor_core_kernels_are_used(agb, dtype, T):
    lib = agb.native.lib()
    mod, images, words = _module(agb, dtype, T=T, hw=32, B=4)
    counts, names = [], []
    for fmt in (torch.contiguous_format, CL):
        im = images.contiguous(memory_format=fmt).requires_grad_(True)
        torch.cuda.synchronize()
        n0 = lib.agb_launch_count()
        ctx, attn = mod(im, words)
        ctx.backward(torch.ones_like(ctx))
        torch.cuda.synchronize()
        counts.append(lib.agb_launch_count() - n0)
    assert counts[0] == counts[1]
    im = images.contiguous(memory_format=CL).requires_grad_(True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ctx, attn = mod(im, words)
        ctx.backward(torch.ones_like(ctx))
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    for kern in ("word_attn_fwd_tc_kernel", "word_attn_bwd_tc_kernel"):
        hits = [n for n in names if kern in n]
        assert hits and all("true>" in n or ", 1>" in n for n in hits), (kern, hits)


def _block(agb, hw=32, B=8):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from scripts.time_compile import block_inputs
    block, h, w = block_inputs(hw, B=B)
    block = block.to(memory_format=CL)
    h = h.detach().contiguous(memory_format=CL).requires_grad_(True)
    return block, h, w


def test_channels_last_block_eager_and_compiled(agb):
    block, h, w = _block(agb)
    block.eval()                                          # fixed BatchNorm statistics for both runs
    img, att = block(h, w)
    assert img.is_contiguous(memory_format=CL) and att.is_contiguous(memory_format=CL)
    (img.float().square().mean() + att.float().mean()).backward()
    assert h.grad.is_contiguous(memory_format=CL)
    # the attention under torch.compile(fullgraph=True): no graph break, outputs and gradients equal eager bit for bit
    att_mod = block.attention
    f = lambda a, b: att_mod.forward_cat(a, b)            # noqa: E731
    torch._dynamo.reset()
    assert torch._dynamo.explain(f)(h, w).graph_break_count == 0
    assert torch._dynamo.explain(lambda a, b: block(a, b))(h, w).graph_break_count == 0
    res = []
    for fn in (f, torch.compile(f, fullgraph=True)):
        hh = h.detach().clone(memory_format=CL).requires_grad_(True)
        att_mod.conv1.weight.grad = None
        out, at = fn(hh, w)
        torch.autograd.backward((out, at), (torch.ones_like(out), torch.ones_like(at)))
        res.append((out, at, hh.grad, att_mod.conv1.weight.grad.clone()))
    for name, x, y in zip(("out", "attn", "d images", "d weight"), *res):
        assert_bitwise(x, y, "compiled " + name)
    assert res[1][0].is_contiguous(memory_format=CL) and res[1][2].is_contiguous(memory_format=CL)
    cb = torch.compile(lambda a, b: block(a, b), fullgraph=True)
    hh = h.detach().clone(memory_format=CL).requires_grad_(True)
    img_c, att_c = cb(hh, w)
    (img_c.float().square().mean() + att_c.float().mean()).backward()
    assert_bitwise(att, att_c, "compiled block attention maps")
    assert hh.grad is not None and torch.isfinite(hh.grad.float()).all()


def test_opcheck_channels_last(agb):
    images, words, weight, mask = _inputs(2, 32, 64, 18, 8, torch.bfloat16, seed=5)
    im = images.contiguous(memory_format=CL)
    _, _, we = agb.ops.word_attn_fwd(im, words, weight, mask, True)
    g = torch.Generator().manual_seed(9)
    dctx = torch.randn(2, 32, 8, 8, generator=g).to(DEV, torch.bfloat16).contiguous(memory_format=CL)
    dattn = torch.randn(2, 18, 8, 8, generator=g).to(DEV, torch.bfloat16).contiguous(memory_format=CL)
    every = ("test_schema", "test_autograd_registration", "test_faketensor", "test_aot_dispatch_static")
    ops = torch.ops.agb
    torch.library.opcheck(ops.word_attn_fwd.default, (im.clone().requires_grad_(), words.clone().requires_grad_(),
                                                      weight.clone().requires_grad_(), mask, True, True),
                          test_utils=every)
    torch.library.opcheck(ops.word_attn_cat.default, (im.clone().requires_grad_(), words.clone().requires_grad_(),
                                                      weight.clone().requires_grad_(), mask, True, False),
                          test_utils=every)
    torch.library.opcheck(ops.word_attn_bwd.default, (im, words, weight, mask, we, dctx, dattn, True, True, True),
                          test_utils=every)


def test_graphed_channels_last_step(agb):
    from attention_gan_b200.agb_native.graph import GraphedStep
    mod, images, words = _module(agb, torch.bfloat16, hw=32, B=4)
    im = images.contiguous(memory_format=CL).requires_grad_(True)
    C = images.shape[1]
    buf = torch.empty(4, 2 * C, 32, 32, dtype=torch.bfloat16, device=DEV, memory_format=CL)

    def step():
        out, attn = mod.forward_into(im, words, buf.detach())      # a fresh view: no history from the last step
        gi, gw = torch.autograd.grad(out, (im, mod.conv1.weight), torch.ones_like(out))
        return out, attn, gi, gw

    ref = [t.detach().clone() for t in step()]            # keeps no autograd graph (and its leaves' nodes) alive
    gs = GraphedStep(step)
    gs.replay()
    torch.cuda.synchronize()
    for x, y in zip(ref, gs.outputs):
        assert_bitwise(x, y, "graph replay")
