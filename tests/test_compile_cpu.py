"""CPU tests of the agb:: operator library (agb_native/torch_ops.py): registration, fake kernels (shapes, dtypes and
workspace sizes under FakeTensorMode with fake CUDA tensors), lazy loading of the library, and forward_cat's refusal
of CPU tensors."""
import os
import subprocess
import sys

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


def _fake():
    return FakeTensorMode(allow_non_fake_inputs=False)


def test_every_op_is_registered_with_a_fake_kernel(agb):
    T = agb.agb_native.torch_ops
    assert len(T.OPS) == 14
    for name in T.OPS:
        op = getattr(torch.ops.agb, name).default
        assert torch._C._dispatch_has_kernel_for_dispatch_key(op.name(), "CUDA"), name
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(op.name(), "CPU"), name
        assert torch._library.simple_registry.singleton.find(op.name()).fake_impl.kernel is not None, name
    mutated = {n: [a.name for a in getattr(torch.ops.agb, n).default._schema.arguments
                   if a.alias_info is not None and a.alias_info.is_write] for n in T.OPS}
    assert mutated.pop("damsm_bwd") == ["ws"] and mutated.pop("region_head_bwd") == ["ws"]
    assert not any(mutated.values()), mutated


def test_importing_the_package_does_not_load_the_library():
    code = ("import attention_gan_b200 as p, torch; assert p.native._lib is None; "
            "assert hasattr(torch.ops.agb, 'damsm_fwd'); print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr


def test_fake_word_attention(agb):
    B, C, E, T, H = 4, 32, 256, 18, 16
    with _fake():
        for dt in (torch.float32, torch.bfloat16):
            im = torch.empty(B, C, H, H, dtype=dt, device="cuda")
            w = torch.empty(B, E, T, device="cuda")
            wt = torch.empty(C, E, device="cuda")
            mask = torch.empty(B, T, dtype=torch.int64, device="cuda")
            ctx, attn, we = torch.ops.agb.word_attn_fwd(im, w, wt, mask, True, True)
            assert ctx.shape == im.shape and ctx.dtype == dt and ctx.is_cuda
            assert attn.shape == (B, T, H, H) and attn.dtype == dt
            assert we.shape == (B, C, T) and we.dtype == torch.float32
            out, attn, we = torch.ops.agb.word_attn_cat(im, w, wt, mask, True, False)
            assert out.shape == (B, 2 * C, H, H) and out.dtype == dt and out.is_contiguous() and attn.numel() == 0
            di, dw, dwt = torch.ops.agb.word_attn_bwd(im, w, wt, mask, we, ctx, None, True, True, False)
            assert di.shape == im.shape and di.dtype == dt
            assert dw.shape == (B, E, T) and dw.dtype == torch.float32 and dwt.numel() == 0


@pytest.mark.parametrize("math", ["fp32", "f16", "f16x2"])
def test_fake_damsm(agb, math):
    N = agb.native
    mm = N.MATH_NAMES[math]
    Bi, Bc, T, D, R = 8, 8, 18, 256, 289
    with _fake():
        img = torch.empty(Bi, D, R, device="cuda")
        words = torch.empty(Bc, T, D, device="cuda").transpose(1, 2)
        lens = torch.empty(Bc, dtype=torch.int32, device="cuda")
        m, att, scos, ws = torch.ops.agb.damsm_fwd(img, words, lens, None, None, 4.0, 5.0, 1e-8, 0, True, mm,
                                                   math != "fp32")
        assert m.shape == (Bi, Bc) and att.shape == (Bi, T, R) and scos.numel() == 0
        assert ws.dtype == torch.uint8 and ws.numel() == max(N.lib().agb_damsm_workspace_bytes(Bi, Bc, T, D, R, mm), 16)
        cnn = torch.empty(Bi, D, device="cuda")
        _, att, scos, _ = torch.ops.agb.damsm_fwd(img, words, lens, cnn, cnn, 4.0, 5.0, 1e-8, 0, False, mm, False)
        assert att.numel() == 0 and scos.shape == (Bi, Bc) and scos.dtype == torch.float32
        dimg, dwords = torch.ops.agb.damsm_bwd(img, words, lens, 4.0, 5.0, 1e-8, m, None, True, mm, m, ws, True)
        assert dimg.shape == img.shape and dwords.shape == (Bc, T, D)
        _, dwords = torch.ops.agb.damsm_bwd(img, words, lens, 4.0, 5.0, 1e-8, m, None, False, mm, None, None, False)
        assert dwords.numel() == 0
        labels = torch.empty(Bi, dtype=torch.int64, device="cuda")
        loss, draw = torch.ops.agb.contrastive(m, None, labels, 10.0, 5.0, 0, Bi, True)
        assert loss.shape == (1,) and draw.shape == (Bi, Bc)
        s = torch.ops.agb.sent_cos_fwd(cnn, cnn[:6], 1e-8)
        assert s.shape == (Bi, 6)
        dc, dr = torch.ops.agb.sent_cos_bwd(cnn, cnn[:6].clone(), 1e-8, s, None, True, False)
        assert dc.shape == cnn.shape and dr.numel() == 0


def test_fake_unsupported_damsm_shape_raises(agb):
    with _fake():
        img = torch.empty(4, 256, 289, device="cuda")
        words = torch.empty(4, 256, 40, device="cuda")                # T = 40 > 32: no tensor-core kernel
        lens = torch.empty(4, dtype=torch.int32, device="cuda")
        with pytest.raises(agb.native.NativeError):
            torch.ops.agb.damsm_fwd(img, words, lens, None, None, 4.0, 5.0, 1e-8, 0, True, agb.native.AGB_MATH_TC_F16,
                                    False)


def test_fake_func_attention_region_head_candidates(agb):
    N = agb.native
    with _fake():
        q = torch.empty(3, 256, 12, device="cuda")
        c = torch.empty(3, 256, 289, device="cuda")
        wc, attn = torch.ops.agb.func_attention_fwd(q, c, 4.0, True)
        assert wc.shape == (3, 256, 12) and attn.shape == (3, 12, 289)
        dq, dc = torch.ops.agb.func_attention_bwd(q, c, 4.0, True, wc, None, False, True)
        assert dq.numel() == 0 and dc.shape == c.shape
        x = torch.empty(4, 768, 289, device="cuda")
        w = torch.empty(256, 768, device="cuda")
        feat, ws = torch.ops.agb.region_head_fwd(x, w)
        assert feat.shape == (4, 256, 289) and feat.dtype == torch.float32
        assert ws.dtype == torch.uint8 and ws.numel() == N.lib().agb_region_head_workspace_bytes(4, 768, 256, 289)
        dw, dx = torch.ops.agb.region_head_bwd(x, w, feat, True, True, ws)
        assert dw.shape == w.shape and dx.shape == x.shape
        cand = torch.empty(6, 100, dtype=torch.int32, device="cuda")
        m = torch.ops.agb.damsm_cand_fwd(torch.empty(6, 256, 289, device="cuda"), torch.empty(9, 256, 18, device="cuda"),
                                         torch.empty(9, dtype=torch.int32, device="cuda"), cand, 4.0, 5.0,
                                         N.AGB_MATH_TC_F16)
        assert m.shape == (6, 100) and m.dtype == torch.float32
        s = torch.ops.agb.sent_cos_cand_fwd(torch.empty(6, 256, device="cuda"), torch.empty(9, 256, device="cuda"),
                                            cand, 1e-8)
        assert s.shape == (6, 100)


def test_host_query_is_a_trace_time_constant(agb):
    T = agb.agb_native.torch_ops
    assert getattr(T.host_query, "_dynamo_marked_constant", False)
    assert T.host_query("agb_damsm_workspace_bytes", 8, 8, 18, 256, 289, 1) == \
        agb.native.lib().agb_damsm_workspace_bytes(8, 8, 18, 256, 289, 1)


def test_forward_cat_rejects_cpu_tensors(agb):
    mod = agb.AttentionModule(32, 256)
    mod.apply_mask(torch.zeros(2, 18, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mod.forward_cat(torch.zeros(2, 32, 8, 8), torch.zeros(2, 256, 18))
    with pytest.raises(AttributeError):
        agb.AttentionModule(32, 256).forward_cat(torch.zeros(2, 32, 8, 8), torch.zeros(2, 256, 18))


def test_compiled_drop_ins_reject_cpu_tensors(agb):
    mod = agb.AttentionModule(32, 256)
    mod.apply_mask(torch.zeros(2, 18, dtype=torch.int64))
    torch._dynamo.reset()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        torch.compile(mod.forward_cat)(torch.zeros(2, 32, 8, 8), torch.zeros(2, 256, 18))
    loss = agb.SentenceLoss("cpu")
    torch._dynamo.reset()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        torch.compile(loss.get_loss)(torch.zeros(4, 256), torch.zeros(4, 256), torch.arange(4), None)
