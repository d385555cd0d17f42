"""torch.compile through the agb:: op library (agb_native/torch_ops.py), on the GPU.

* opcheck of every op (schema incl. the declared workspace mutation, fake kernel, autograd registration, AOT dispatch)
* no graph breaks, and compiled outputs and input gradients equal to eager bit for bit: AttentionModule (forward,
  forward_cat, forward_into), func_attention, the DAMSM losses (f16, f16x2, fp32; saved-context, multi-chunk and
  frozen-words backward), RegionFeatureHead / RegionHeads, DAMSMScorer
* a GenNextStage-shaped block, reduce-overhead replays, the memory of the compiled DAMSM step, and that the eager
  drop-ins never enter the op library
"""
import numpy as np
import pytest
import torch

from oracle import ref_port as rp

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


@pytest.fixture
def chunk_budget(agb):
    def set_mb(mb):
        agb.native.set_option("damsm_chunk_mb", mb)
    yield set_mb
    agb.native.set_option("damsm_chunk_mb", 16384)


def _compile(fn, **kw):
    torch._dynamo.reset()
    return torch.compile(fn, fullgraph=True, **kw)


def _breaks(fn, *args):
    torch._dynamo.reset()
    ex = torch._dynamo.explain(fn)(*args)
    return ex.graph_break_count, [str(r.reason)[:200] for r in ex.break_reasons]


def _run(fn, inputs, needs_grad, params=(), seed=0):
    """outputs of fn(*inputs) and the gradients of a seeded random weighting of its differentiable outputs with
    respect to every input that needs one and every parameter"""
    xs = [x.detach().clone().requires_grad_(bool(g)) if torch.is_tensor(x) else x for x, g in zip(inputs, needs_grad)]
    for p in params:
        p.grad = None
    outs = fn(*xs)
    outs = [o for o in (outs if isinstance(outs, (tuple, list)) else (outs,)) if torch.is_tensor(o)]
    res = [o.detach().clone() for o in outs]
    gen = torch.Generator(device=DEV).manual_seed(seed)
    diff = [o for o in outs if o.requires_grad]
    if diff:
        loss = sum((o.float() * torch.randn(o.shape, generator=gen, device=DEV)).sum() for o in diff)
        loss.backward()
    none = torch.empty(0, device=DEV)                                   # stands for "no gradient"
    res += [none if x.grad is None else x.grad for x, g in zip(xs, needs_grad) if g]
    res += [none if p.grad is None else p.grad.clone() for p in params]
    return res


def _assert_bitwise(a, b, what):
    assert len(a) == len(b), what
    for i, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and x.dtype == y.dtype, (what, i, x.shape, y.shape)
        assert torch.equal(x, y), (what, i, (x.float() - y.float()).abs().max().item())


def _eager_vs_compiled(fn, inputs, needs_grad, params=(), what=""):
    n, reasons = _breaks(fn, *inputs)
    assert n == 0, (what, reasons)
    ref = _run(fn, inputs, needs_grad, params)
    got = _run(_compile(fn), inputs, needs_grad, params)
    _assert_bitwise(ref, got, what)
    return ref


# ------------------------------------------------------------------------------------------------
# opcheck
# ------------------------------------------------------------------------------------------------
def _op_cases(agb):
    N = agb.native
    g = torch.Generator().manual_seed(7)

    def r(*shape, grad=False):
        return torch.randn(*shape, generator=g).to(DEV).requires_grad_(grad)
    images, words, weight, mask, _ = rp.synth_attention(2, 32, 256, 18, 8, seed=5)
    im, wd, wt, mk = images.to(DEV), words.to(DEV), weight.reshape(32, 256).contiguous().to(DEV), mask.to(DEV)
    _, _, we = agb.ops.word_attn_fwd(im, wd, wt, mk, True)
    img, wrd, cnn, rnn, labels, lens, cls = rp.synth_damsm(4, seed=6, n_classes=2)
    img3 = img.reshape(4, 256, -1).contiguous().to(DEV)
    w3, lens32 = wrd.to(DEV), lens.to(DEV, torch.int32)
    f16 = N.AGB_MATH_TC_F16
    m, _, _, ws = agb.ops.damsm_fwd(img3, w3, lens32, 4.0, 5.0, 1e-8, 0, True, f16, keep_ws=True, save=True)
    x, hw = r(2, 768, 289), r(256, 768)
    _, hws = agb.ops.region_head_fwd(x, hw, keep_ws=True)
    q, c = r(2, 256, 12), r(2, 256, 289)
    cand = torch.tensor([[0, 1, 2, 3, 3], [3, 2, 1, 0, 0], [1, 1, 1, 1, 1], [2, 3, 0, 1, 2]], dtype=torch.int32,
                        device=DEV)
    cls32 = torch.from_numpy(cls).to(DEV, torch.int32)
    gs = torch.full((1,), 0.75, device=DEV)
    no_aot = ("test_schema", "test_autograd_registration", "test_faketensor")
    return {
        "word_attn_fwd": ((im.clone().requires_grad_(), wd.clone().requires_grad_(), wt.clone().requires_grad_(), mk,
                           True, True), None),
        "word_attn_cat": ((im.clone().requires_grad_(), wd.clone().requires_grad_(), wt.clone().requires_grad_(), mk,
                           True, False), None),
        "word_attn_bwd": ((im, wd, wt, mk, we, r(*im.shape), r(2, 18, 8, 8), True, True, True), None),
        # the workspace output holds bytes the kernels never write (padding): compared by the compiled tests instead
        "damsm_fwd": ((img3.clone().requires_grad_(), w3.clone().requires_grad_(), lens32, None, None, 4.0, 5.0,
                       1e-8, 0, True, f16, True), no_aot),
        "damsm_bwd": ((img3, w3, lens32, 4.0, 5.0, 1e-8, r(4, 4), gs, True, f16, m, ws, True), None),
        "contrastive": ((m.clone().requires_grad_(), cls32, labels.to(DEV), 10.0, 5.0, 0, 4, True), None),
        "sent_cos_fwd": ((cnn.to(DEV).requires_grad_(), rnn.to(DEV).requires_grad_(), 1e-8), None),
        "sent_cos_bwd": ((cnn.to(DEV), rnn.to(DEV), 1e-8, r(4, 4), gs, True, True), None),
        "func_attention_fwd": ((q.clone().requires_grad_(), c.clone().requires_grad_(), 4.0, True), None),
        "func_attention_bwd": ((q, c, 4.0, True, r(2, 256, 12), r(2, 12, 289), True, True), None),
        "region_head_fwd": ((x.clone().requires_grad_(), hw.clone().requires_grad_()), no_aot),
        "region_head_bwd": ((x, hw, r(2, 256, 289), True, True, hws), None),
        "damsm_cand_fwd": ((img3, w3, lens32, cand, 4.0, 5.0, f16), None),
        "sent_cos_cand_fwd": ((cnn.to(DEV), rnn.to(DEV), cand, 1e-8), None),
    }


def test_opcheck_every_op(agb):
    cases = _op_cases(agb)
    assert set(cases) == set(agb.agb_native.torch_ops.OPS)
    every = ("test_schema", "test_autograd_registration", "test_faketensor", "test_aot_dispatch_static")
    for name, (args, utils) in cases.items():
        torch.library.opcheck(getattr(torch.ops.agb, name).default, args, test_utils=utils or every)


# ------------------------------------------------------------------------------------------------
# generator attention
# ------------------------------------------------------------------------------------------------
def _attention(agb, dt, T, hw, seed=1, B=4, C=32, E=256):
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=seed)
    mod = agb.AttentionModule(C, E).to(DEV)
    with torch.no_grad():
        mod.conv1.weight.copy_(weight.to(DEV))
    mod.apply_mask(mask.to(DEV))
    return mod, images.to(dt).to(DEV), words.to(DEV)


@pytest.mark.parametrize("dt,T,hw", [(torch.float32, 18, 16), (torch.bfloat16, 18, 32), (torch.float32, 64, 16),
                                     (torch.bfloat16, 64, 32)])
def test_attention_compiles_bit_for_bit(agb, dt, T, hw):
    mod, im, w = _attention(agb, dt, T, hw)
    params = [mod.conv1.weight]
    _eager_vs_compiled(lambda a, b: mod(a, b), (im, w), (True, True), params, "forward")
    _eager_vs_compiled(lambda a, b: mod.forward_cat(a, b), (im, w), (True, True), params, "forward_cat")
    _eager_vs_compiled(lambda a, b: mod.forward_cat(a, b, want_attn=False)[0], (im, w), (True, True), params,
                       "forward_cat without attn")
    _eager_vs_compiled(lambda a, b: mod(a, b)[0], (im, w), (True, False), params, "frozen words, attn unused")


def test_forward_into_keeps_its_contract_under_compile(agb):
    mod, im, w = _attention(agb, torch.bfloat16, 18, 32)
    B, C, H, W = im.shape

    def f(a, b, out):
        res, att = mod.forward_into(a, b, out)
        return res, att
    out_e = torch.empty(B, 2 * C, H, W, dtype=im.dtype, device=DEV)
    out_c = torch.empty_like(out_e)
    ref = f(im, w, out_e)
    got = _compile(f)(im, w, out_c)
    assert torch.equal(out_c, out_e) and torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    assert torch.equal(out_c[:, :C], im)


def test_func_attention_compiles_bit_for_bit(agb):
    g = torch.Generator().manual_seed(3)
    q = torch.randn(3, 256, 12, generator=g).to(DEV)
    c = torch.randn(3, 256, 17, 17, generator=g).to(DEV)
    _eager_vs_compiled(lambda a, b: agb.func_attention(a, b, 4.0), (q, c), (True, True), (), "func_attention")


# ------------------------------------------------------------------------------------------------
# DAMSM losses
# ------------------------------------------------------------------------------------------------
def _damsm(B=48, seed=11):
    img, wrd, cnn, rnn, labels, lens, cls = rp.synth_damsm(B, seed=seed, n_classes=B // 4)
    return (img.to(DEV), cnn.to(DEV), wrd.to(DEV), rnn.to(DEV), labels.to(DEV), lens.to(DEV),
            torch.from_numpy(cls).to(DEV, torch.int32))


@pytest.mark.parametrize("math", ["f16", "f16x2", "fp32", "auto"])
def test_damsm_losses_compile_bit_for_bit(agb, math):
    img, cnn, wrd, rnn, labels, lens, cls = _damsm()
    wl = agb.WordsLoss(DEV, math=math, att_maps="packed")
    sl = agb.SentenceLoss(DEV)
    dl = agb.DAMSMLoss(DEV, math=math, att_maps="packed")
    args = (img, cnn, wrd, rnn, labels, lens, cls)
    trainable = (True, True, True, True, False, False, False)
    _eager_vs_compiled(lambda i, c, w, r, lb, ln, cl: wl.get_loss(i, w, lb, ln, cl), args, trainable, (), "WordsLoss")
    _eager_vs_compiled(lambda i, c, w, r, lb, ln, cl: sl.get_loss(c, r, lb, cl), args, trainable, (), "SentenceLoss")
    _eager_vs_compiled(lambda *a: dl.get_losses(*a), args, trainable, (), "DAMSMLoss")
    frozen = (True, True, False, False, False, False, False)                       # text encoder frozen: no d words
    _eager_vs_compiled(lambda *a: dl.get_losses(*a), args, frozen, (), "DAMSMLoss, frozen words")
    no_att = agb.DAMSMLoss(DEV, math=math, att_maps=None)
    _eager_vs_compiled(lambda *a: no_att.get_losses(*a)[:2], args, trainable, (), "DAMSMLoss, no maps")


def test_damsm_multi_chunk_backward_compiles_bit_for_bit(agb, chunk_budget):
    img, cnn, wrd, rnn, labels, lens, cls = _damsm(B=64, seed=641)
    chunk_budget(11)                                               # several backward chunks at B = 64 (f16)
    wl = agb.WordsLoss(DEV, math="f16", att_maps="packed")
    f = lambda i, w, lb, ln, cl: wl.get_loss(i, w, lb, ln, cl)          # noqa: E731
    _eager_vs_compiled(f, (img, wrd, labels, lens, cls), (True, True, False, False, False), (), "multi-chunk")
    _eager_vs_compiled(f, (img, wrd, labels, lens, cls), (True, False, False, False, False), (), "multi-chunk frozen")


def test_damsm_graph_breaks_that_stay(agb):
    """att_maps="list" needs the caption lengths on the host, numpy class ids leave the graph: documented breaks"""
    img, cnn, wrd, rnn, labels, lens, cls = _damsm()
    as_list = agb.WordsLoss(DEV, math="f16", att_maps="list")
    n, _ = _breaks(lambda i, w, lb, ln, cl: as_list.get_loss(i, w, lb, ln, cl)[0], img, wrd, labels, lens, cls)
    assert n >= 1
    packed = agb.WordsLoss(DEV, math="f16", att_maps="packed")
    cls_np = cls.cpu().numpy()
    loss_e, _ = packed.get_loss(img, wrd, labels, lens, cls_np)
    torch._dynamo.reset()
    loss_c, _ = torch.compile(lambda i, w, lb, ln: packed.get_loss(i, w, lb, ln, cls_np))(img, wrd, labels, lens)
    assert torch.equal(loss_e, loss_c)


# ------------------------------------------------------------------------------------------------
# region heads, scorer
# ------------------------------------------------------------------------------------------------
def test_region_heads_compile_bit_for_bit(agb):
    from attention_gan_b200.pretrain import RegionHeads
    torch.manual_seed(0)
    heads = RegionHeads(256).to(DEV)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(8, 768, 17, 17, generator=g).to(DEV)
    pooled = torch.randn(8, 2048, generator=g).to(DEV)
    # the region features and their gradients come from the native head; cnn_code is an nn.Linear, whose compiled
    # bias gradient inductor may sum in another order, so only the native half is held to bit equality
    _eager_vs_compiled(lambda a, b: heads(a, b)[0], (x, pooled), (True, False), [heads.emb_features.weight],
                       "RegionHeads")
    head = agb.RegionFeatureHead(256).to(DEV)
    _eager_vs_compiled(lambda a: head(a), (x,), (False,), list(head.parameters()), "RegionFeatureHead")


@pytest.mark.parametrize("math", ["f16", "f16x2"])
def test_scorer_compiles_bit_for_bit(agb, math):
    img, cnn, wrd, rnn, labels, lens, cls = _damsm(B=64, seed=21)
    cands = torch.from_numpy(agb.mismatched_candidates(None, n_mismatched=15, n=64, seed=2)).to(DEV)
    scorer = agb.DAMSMScorer(DEV, math=math, workspace_bytes=4 << 20)          # a small budget: several chunks
    for f, args in ((lambda i, w, ln, cd: scorer.words(i, w, ln, cd), (img, wrd, lens, cands)),
                    (lambda c, r, cd: scorer.sentence(c, r, cd), (cnn, rnn, cands))):
        n, reasons = _breaks(f, *args)
        assert n == 0, reasons
        torch.testing.assert_close(_compile(f)(*args), f(*args), rtol=0, atol=0, equal_nan=True)


# ------------------------------------------------------------------------------------------------
# a compiled generator block, CUDA graphs, memory, the eager path
# ------------------------------------------------------------------------------------------------
def test_mixed_block_matches_eager(agb):
    from scripts.time_compile import block_inputs
    block, h, w = block_inputs(32, B=8)
    f = lambda a, b: block(a, b)                                        # noqa: E731
    assert _breaks(f, h, w)[0] == 0
    params = list(block.parameters())
    block.eval()                                                        # fixed BatchNorm statistics for both runs
    ref = _run(f, (h, w), (True, False), params)
    got = _run(_compile(f), (h, w), (True, False), params)
    for x, y in zip(ref, got):
        scale = max(x.float().abs().max().item(), 1e-6)
        assert (x.float() - y.float()).abs().max().item() <= 3e-2 * scale


def test_reduce_overhead_replays_match_eager(agb):
    img, cnn, wrd, rnn, labels, lens, cls = _damsm()
    dl = agb.DAMSMLoss(DEV, math="f16", att_maps="packed")
    args = (img, cnn, wrd, rnn, labels, lens, cls)
    grads = (True, True, True, True, False, False, False)
    ref = _run(lambda *a: dl.get_losses(*a), args, grads)
    torch._dynamo.reset()
    f = torch.compile(lambda *a: dl.get_losses(*a), mode="reduce-overhead")
    for _ in range(4):                                                  # warm-up, recording, replays
        torch.compiler.cudagraph_mark_step_begin()
        _assert_bitwise(ref, _run(f, args, grads), "reduce-overhead")
    mod, im, w = _attention(agb, torch.bfloat16, 18, 32)
    ref = _run(lambda a, b: mod.forward_cat(a, b), (im, w), (True, True), [mod.conv1.weight])
    torch._dynamo.reset()
    f = torch.compile(lambda a, b: mod.forward_cat(a, b), mode="reduce-overhead")
    for _ in range(4):
        torch.compiler.cudagraph_mark_step_begin()
        _assert_bitwise(ref, _run(f, (im, w), (True, True), [mod.conv1.weight]), "reduce-overhead attention")


def test_compiled_damsm_step_does_not_copy_the_workspace(agb):
    """Bi = Bc = 512 in f16: the forward's workspace (~10 GiB) is handed to the backward, which writes its staging
    into it; the compiled step must reuse it in place, so its peak memory matches eager's"""
    img, cnn, wrd, rnn, labels, lens, cls = _damsm(B=512, seed=512)
    ws = agb.native.lib().agb_damsm_workspace_bytes(512, 512, 18, 256, 289, agb.native.AGB_MATH_TC_F16)
    assert ws > 8 << 30
    dl = agb.DAMSMLoss(DEV, math="f16", att_maps="packed")
    xs = [t.clone().requires_grad_(True) for t in (img, cnn, wrd, rnn)]

    def step(fn):
        for t in xs:
            t.grad = None
        wl, sl, _ = fn(*xs, labels, lens, cls)
        (wl + sl).backward()
        torch.cuda.synchronize()

    def peak(fn):
        step(fn)                                                        # warm-up / compile
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        step(fn)
        return torch.cuda.max_memory_allocated()
    eager = peak(dl.get_losses)
    compiled = peak(_compile(lambda *a: dl.get_losses(*a)))
    assert compiled <= 1.05 * eager, (compiled / 2**30, eager / 2**30)


def test_eager_drop_ins_never_enter_the_op_library(agb, monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("the eager path called torch.ops.agb")
    for name in agb.agb_native.torch_ops.OPS:
        monkeypatch.setattr(torch.ops.agb, name, refuse)
    with pytest.raises(AssertionError):
        torch.ops.agb.damsm_fwd()
    mod, im, w = _attention(agb, torch.bfloat16, 18, 32)
    im.requires_grad_(True)
    c, a = mod(im, w)
    o, a2 = mod.forward_cat(im, w)
    (c.float().sum() + a.float().sum() + o.float().sum()).backward()
    agb.func_attention(torch.randn(2, 256, 12, device=DEV, requires_grad=True),
                       torch.randn(2, 256, 17, 17, device=DEV))[0].sum().backward()
    img, cnn, wrd, rnn, labels, lens, cls = _damsm()
    xs = [t.clone().requires_grad_(True) for t in (img, cnn, wrd, rnn)]
    wl, sl, _ = agb.DAMSMLoss(DEV, math="f16", att_maps="packed").get_losses(*xs, labels, lens, cls)
    wl2, _ = agb.WordsLoss(DEV).get_loss(xs[0], xs[2], labels, lens, cls)
    sl2 = agb.SentenceLoss(DEV).get_loss(xs[1], xs[3], labels, cls)
    (wl + sl + wl2 + sl2).backward()
    agb.RegionFeatureHead(256).to(DEV)(torch.randn(2, 768, 17, 17, device=DEV, requires_grad=True)).sum().backward()
    cands = agb.mismatched_candidates(None, n_mismatched=3, n=48)
    scorer = agb.DAMSMScorer(DEV, math="f16")
    assert np.isfinite(scorer.words(img, wrd, lens, cands).cpu().numpy()).all()
    assert np.isfinite(scorer.sentence(cnn, rnn, cands).cpu().numpy()).all()
    torch.cuda.synchronize()
