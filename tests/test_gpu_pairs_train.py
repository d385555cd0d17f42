"""GPU tests of training on pair lists (words_pair_scores / sentence_pair_scores over agb_damsm_pairs_train_fwd,
agb_damsm_pairs_bwd and agb_sent_cos_pairs_bwd): the scores equal the scorer's bit for bit, the gradients agree with
the fp64 oracle and with the dense tensor-core backward on dLoss/dm scattered into [N, Nc], invalid pairs contribute
nothing, unused rows get exactly 0, and the results are deterministic, chunk-independent, capturable and
compilable."""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import closed_form as cf
from oracle import ref_port as rp

pytestmark = pytest.mark.gpu

G1, G2 = 4.0, 5.0
NAN = float("nan")
GTOL = {"f16": 5e-3, "f16x2": 5e-3, "bf16": 2e-2}     # the suite's tensor-core gradient tolerances


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


def _inputs(Bc, T=18, seed=0, trained_like=False):
    img, wrd, cnn, rnn, _, lens, cls = rp.synth_damsm(Bc, T=T, seed=seed, trained_like=trained_like, n_classes=50)
    return img.reshape(Bc, 256, -1), wrd, cnn, rnn, lens, cls


def _rel(x, ref):
    x = x.detach().double().cpu().numpy() if torch.is_tensor(x) else np.asarray(x, np.float64)
    ref = ref.detach().double().cpu().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    return np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-30)


def _assert_same_bits(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    a, b = a.reshape(-1), b.reshape(-1)
    same = (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
    assert bool(same.all()), f"{int((~same).sum())} entries differ"


def _list(case, Bi, Bc):
    """(pair_img, pair_cap) int32 on the host"""
    g = torch.Generator().manual_seed(sum(map(ord, case)))

    def rnd(n, hi):
        return torch.randint(0, hi, (n,), generator=g, dtype=torch.int32)
    if case == "random":
        return rnd(997, Bi), rnd(997, Bc)
    if case == "shuffled":                                       # a K-way candidate list in random order
        pi = torch.arange(Bi, dtype=torch.int32).repeat_interleave(12)
        pc = rnd(pi.shape[0], Bc)
        perm = torch.randperm(pi.shape[0], generator=g)
        return pi[perm], pc[perm]
    if case == "duplicates":
        pi, pc = rnd(300, Bi), rnd(300, Bc)
        return torch.cat([pi, pi[:100], pi[5:6].repeat(40)]), torch.cat([pc, pc[:100], pc[5:6].repeat(40)])
    if case == "sparse":                                         # only a few images and captions have pairs
        return rnd(60, Bi // 4) * 4 + 1, rnd(60, Bc // 8) * 8
    if case == "p1":
        return torch.tensor([Bi - 1], dtype=torch.int32), torch.tensor([3], dtype=torch.int32)
    if case == "one_image":                                      # 10^5 pairs, all on one image
        return torch.full((10 ** 5,), 17, dtype=torch.int32), rnd(10 ** 5, Bc)
    if case == "len1_len32":
        pi, pc = rnd(500, Bi), rnd(500, Bc)
        pc[::3], pc[1::3] = 3, 4
        return pi, pc
    if case == "invalid":                                        # out-of-range indices and length-0 captions
        pi, pc = rnd(600, Bi), rnd(600, Bc)
        pi[::7], pi[3::11] = -1, Bi
        pc[1::9], pc[2::13] = -5, Bc
        pi[5], pc[5] = 70000, 2 ** 31 - 1
        pc[4::10] = 6                                            # caption 6 gets length 0 below
        return pi, pc
    raise ValueError(case)


def _valid(pi, pc, Bi, Bc, lens):
    ok = (pi >= 0) & (pi < Bi) & (pc >= 0) & (pc < Bc)
    ok[ok.clone()] &= lens[pc[ok].long()] > 0
    return ok


def _scatter(dm, pi, pc, ok, Bi, Bc):
    """dLoss/dm of the list scattered into [Bi, Bc], duplicates summed (fp64)"""
    d = np.zeros((Bi, Bc))
    np.add.at(d, (pi[ok].long().numpy(), pc[ok].long().numpy()), dm[ok].double().numpy())
    return d


def _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name, **kw):
    im = img.detach().clone().cuda().requires_grad_(True)
    wd = wrd.detach().clone().cuda().requires_grad_(True)
    m = agb.words_pair_scores(im, wd, lens.cuda(), pi.cuda(), pc.cuda(), gamma1=G1, gamma2=G2, math=math_name, **kw)
    m.backward(dm.cuda())
    return m.detach(), im.grad, wd.grad


def _dense_tc_grads(agb, img, wrd, lens, dm_dense, math_name):
    """the dense tensor-core backward (save forward, then damsm_bwd) on a [Bi, Bc] dLoss/dm"""
    mt = agb.native.MATH_NAMES[math_name]
    im, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda().to(torch.int32)
    m, _, _, ws = agb.ops.damsm_fwd(im, wd, ln, G1, G2, 1e-8, 0, False, mt, keep_ws=True, save=True)
    dimg, dw = agb.ops.damsm_bwd(im, wd, ln, G1, G2, 1e-8, torch.from_numpy(dm_dense).float().cuda(), None, True, mt,
                                 m, ws, True)
    return dimg, dw.transpose(1, 2)


CASES = ["random", "shuffled", "duplicates", "sparse", "p1", "one_image", "len1_len32", "invalid"]


@pytest.mark.parametrize("math_name", ["f16", "bf16", "f16x2"])
@pytest.mark.parametrize("case", CASES)
def test_pair_gradients(agb, case, math_name):
    T = 32 if case == "len1_len32" else 18
    Bi, Bc = 40, 64
    img, wrd, _, _, lens, _ = _inputs(Bc, T=T, seed=21)
    img = img[:Bi].contiguous()
    if case == "len1_len32":
        lens[3], lens[4] = 1, 32
    if case == "invalid":
        lens[6] = 0
    pi, pc = _list(case, Bi, Bc)
    ok = _valid(pi, pc, Bi, Bc, lens)
    dm = torch.randn(pi.shape[0], generator=torch.Generator().manual_seed(3)) * 0.05
    dm[~ok] = NAN                                                # an invalid pair's dLoss/dm reaches nothing
    m, gi, gw = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name)
    _assert_same_bits(m, scorer.words_pairs(img.cuda(), wrd.cuda(), lens.cuda(), pi.cuda(), pc.cuda()))
    assert bool(torch.isfinite(gi).all()) and bool(torch.isfinite(gw).all())
    # exact zeros: images and captions in no valid pair, padded word slots
    used_i = torch.zeros(Bi, dtype=torch.bool)
    used_i[pi[ok].long()] = True
    used_c = torch.zeros(Bc, dtype=torch.bool)
    used_c[pc[ok].long()] = True
    assert bool((gi[~used_i.cuda()] == 0).all()) and bool((gw[~used_c.cuda()] == 0).all())
    pad = torch.arange(T)[None, :] >= lens[:, None]
    assert bool((gw.transpose(1, 2)[pad.cuda()] == 0).all())
    if case in ("p1", "sparse"):
        assert int((~used_i).sum()) > 0 and int((~used_c).sum()) > 0
    dmd = _scatter(dm, pi, pc, ok, Bi, Bc)
    lens_o = lens.clone()
    lens_o[lens_o == 0] = 1                                      # such captions have no valid pair (dm column 0)
    dc0, dw0 = cf.words_similarity_bwd(img.numpy(), wrd.numpy(), lens_o.numpy(), dmd, G1, G2)
    tol = GTOL[math_name]
    e_img, e_wrd = _rel(gi, dc0), _rel(gw, dw0)
    assert e_img < tol and e_wrd < tol, (e_img, e_wrd)
    di, dw = _dense_tc_grads(agb, img, wrd, lens_o, dmd, math_name)
    d_img, d_wrd = _rel(gi, di), _rel(gw, dw)
    print(f"{case} {math_name}: oracle {e_img:.2e} / {e_wrd:.2e}, dense tensor-core backward {d_img:.2e} / {d_wrd:.2e}")
    assert d_img < tol and d_wrd < tol, (d_img, d_wrd)


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_invalid_pairs_change_nothing(agb, math_name):
    """a list with invalid pairs gives the gradients of the list without them (within tolerance: the packing
    differs), and two runs give bit-identical gradients"""
    Bi, Bc = 40, 64
    img, wrd, _, _, lens, _ = _inputs(Bc, seed=8)
    img = img[:Bi].contiguous()
    lens[6] = 0
    pi, pc = _list("invalid", Bi, Bc)
    ok = _valid(pi, pc, Bi, Bc, lens)
    dm = torch.randn(pi.shape[0], generator=torch.Generator().manual_seed(1)) * 0.05
    _, gi, gw = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name)
    _, gi2, gw2 = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name)
    assert torch.equal(gi, gi2) and torch.equal(gw, gw2)
    _, hi, hw = _pair_grads(agb, img, wrd, lens, pi[ok], pc[ok], dm[ok], math_name)
    assert _rel(gi, hi) < GTOL[math_name] and _rel(gw, hw) < GTOL[math_name]


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_chunked_lists_and_staging(agb, math_name, chunk_budget):
    """a small workspace_bytes runs the list in >= 3 chunks of pairs, a small staging budget runs the backward in
    many chunks of word tiles: m is bit-identical, gradients agree with one chunk"""
    Bi, Bc = 48, 96
    img, wrd, _, _, lens, _ = _inputs(Bc, seed=12)
    img = img[:Bi].contiguous()
    pi, pc = _list("shuffled", Bi, Bc)
    P = pi.shape[0]
    dm = torch.randn(P, generator=torch.Generator().manual_seed(2)) * 0.05
    m, gi, gw = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name)
    mt = agb.native.MATH_NAMES[math_name]
    q = agb.ops.damsm_pairs_train_workspace_bytes
    budget = q(Bi, Bc, P // 3, 18, 256, 289, mt)
    m3, gi3, gw3 = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name, workspace_bytes=budget)
    assert q(Bi, Bc, P, 18, 256, 289, mt) > budget
    _assert_same_bits(m3, m)
    assert _rel(gi3, gi) < GTOL[math_name] and _rel(gw3, gw) < GTOL[math_name]
    chunk_budget(1)                                              # 1 MiB of staging: 3 word tiles per chunk
    ms, gis, gws = _pair_grads(agb, img, wrd, lens, pi, pc, dm, math_name)
    chunk_budget(16384)
    _assert_same_bits(ms, m)
    assert _rel(gis, gi) < GTOL[math_name] and _rel(gws, gw) < GTOL[math_name]


def test_frozen_inputs_and_empty_list(agb):
    Bi, Bc = 12, 20
    img, wrd, _, _, lens, _ = _inputs(Bc, seed=4)
    img = img[:Bi].contiguous()
    pi, pc = _list("random", Bi, Bc)
    im = img.cuda().requires_grad_(True)
    wd = wrd.cuda()                                              # frozen text encoder
    m = agb.words_pair_scores(im, wd, lens.cuda(), pi, pc, math="f16")
    m.sum().backward()
    assert im.grad is not None and wd.grad is None
    im.grad = None
    e = np.zeros(0, np.int64)
    wd.requires_grad_(True)
    m0 = agb.words_pair_scores(im, wd, lens.cuda(), e, e, math="f16")
    assert m0.shape == (0,)
    m0.sum().backward()
    assert bool((im.grad == 0).all()) and bool((wd.grad == 0).all())


def test_workspace_release_and_scoring_forward(agb, monkeypatch):
    """the backward frees the training workspace (a second backward raises instead of reading freed state), and
    without a gradient to compute the scoring forward runs: the same m, no training forward"""
    Bi, Bc = 16, 24
    img, wrd, _, _, lens, _ = _inputs(Bc, seed=11)
    img = img[:Bi].contiguous()
    pi, pc = _list("random", Bi, Bc)
    im = img.cuda().requires_grad_(True)
    m = agb.words_pair_scores(im, wrd.cuda(), lens, pi, pc, math="f16")
    node = m.grad_fn
    m.sum().backward(retain_graph=True)
    assert node.ws is None
    with pytest.raises(RuntimeError, match="second backward"):
        m.sum().backward()
    ref = m.detach()

    def no_training_forward(*a, **k):
        raise AssertionError("training forward without a gradient to compute")
    monkeypatch.setattr(agb.ops, "damsm_pairs_train_fwd", no_training_forward)
    with torch.no_grad():
        _assert_same_bits(agb.words_pair_scores(im, wrd.cuda(), lens, pi, pc, math="f16"), ref)
    _assert_same_bits(agb.words_pair_scores(im.detach(), wrd.cuda(), lens, pi, pc, math="f16", workspace_bytes=
                                            agb.ops.damsm_pairs_workspace_bytes(Bi, Bc, 300, 18, 256, 289,
                                                                                agb.native.AGB_MATH_TC_F16)), ref)


def test_sentence_pair_gradients(agb):
    N, Nc = 30, 50
    _, _, cnn, rnn, _, _ = _inputs(Nc, seed=3)
    cnn = cnn[:N].contiguous()
    pi, pc = _list("invalid", N, Nc)
    pi[pi == 3], pc[pc == 7] = -1, Nc                            # image 3 and caption 7 in no valid pair
    ok = (pi >= 0) & (pi < N) & (pc >= 0) & (pc < Nc)
    dg = torch.randn(pi.shape[0], generator=torch.Generator().manual_seed(5))
    dg[~ok] = NAN
    c = cnn.cuda().requires_grad_(True)
    r = rnn.cuda().requires_grad_(True)
    cos = agb.sentence_pair_scores(c, r, pi, pc)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16")
    _assert_same_bits(cos, scorer.sentence_pairs(cnn.cuda(), rnn.cuda(), pi, pc))
    cos.backward(dg.cuda())
    d = _scatter(dg, pi, pc, ok, N, Nc)
    cc, rr = cnn.double().numpy(), rnn.double().numpy()       # fp64 statement of the dense sentence backward
    p, q = np.linalg.norm(cc, axis=1)[:, None], np.linalg.norm(rr, axis=1)[None]
    gg = d / np.maximum(p * q, 1e-8)
    gn = np.where(p * q > 1e-8, gg * (cc @ rr.T), 0.0)
    dc0 = gg @ rr - gn.sum(1, keepdims=True) / (p * p) * cc
    dr0 = gg.T @ cc - gn.sum(0)[:, None] / (q.T * q.T) * rr
    assert _rel(c.grad, dc0) < 1e-5 and _rel(r.grad, dr0) < 1e-5
    used_c = torch.zeros(Nc, dtype=torch.bool)
    used_c[pc[ok].long()] = True
    used_i = torch.zeros(N, dtype=torch.bool)
    used_i[pi[ok].long()] = True
    assert int((~used_i).sum()) > 0 and int((~used_c).sum()) > 0
    assert bool((r.grad[~used_c.cuda()] == 0).all()) and bool((c.grad[~used_i.cuda()] == 0).all())
    c2 = cnn.cuda().requires_grad_(True)
    r2 = rnn.cuda().requires_grad_(True)
    agb.sentence_pair_scores(c2, r2, pi, pc).backward(dg.cuda())
    assert torch.equal(c.grad, c2.grad) and torch.equal(r.grad, r2.grad)


def test_graph_capture_equals_eager(agb):
    Bi, Bc = 40, 64
    img, wrd, cnn, rnn, lens, _ = _inputs(Bc, seed=6)
    pi, pc = (t.cuda() for t in _list("duplicates", Bi, Bc))
    im = img[:Bi].contiguous().cuda().requires_grad_(True)
    wd = wrd.cuda().requires_grad_(True)
    c = cnn[:Bi].contiguous().cuda().requires_grad_(True)
    r = rnn.cuda().requires_grad_(True)
    ln = lens.cuda().to(torch.int32)
    dm = (torch.randn(pi.shape[0], generator=torch.Generator().manual_seed(9)) * 0.05).cuda()

    def step():
        m = agb.words_pair_scores(im, wd, ln, pi, pc, math="f16x2")
        cos = agb.sentence_pair_scores(c, r, pi, pc)
        return (m, cos) + torch.autograd.grad((m, cos), (im, wd, c, r), (dm, dm))
    ref = [t.detach().clone() for t in step()]              # keeps no autograd graph (and its leaves' nodes) alive
    g = agb.GraphedStep(step)
    g.replay()
    out = g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, ref):
        _assert_same_bits(a, b)


def test_compiled_equals_eager(agb):
    Bi, Bc = 24, 40
    img, wrd, cnn, rnn, lens, _ = _inputs(Bc, seed=7)
    pi, pc = (t.cuda() for t in _list("random", Bi, Bc))
    ln = lens.cuda().to(torch.int32)
    dm = (torch.randn(pi.shape[0], generator=torch.Generator().manual_seed(4)) * 0.05).cuda()

    def fn(im, wd, c, r):
        m = agb.words_pair_scores(im, wd, ln, pi, pc, math="f16x2", workspace_bytes=1 << 30)
        return m, agb.sentence_pair_scores(c, r, pi, pc)

    def run(f):
        xs = [img[:Bi].contiguous().cuda(), wrd.cuda(), cnn[:Bi].contiguous().cuda(), rnn.cuda()]
        xs = [x.detach().clone().requires_grad_(True) for x in xs]
        m, cos = f(*xs)
        torch.autograd.backward((m, cos), (dm, dm))
        return [m.detach(), cos.detach()] + [x.grad for x in xs]
    torch._dynamo.reset()
    ex = torch._dynamo.explain(fn)(img[:Bi].contiguous().cuda(), wrd.cuda(), cnn[:Bi].contiguous().cuda(),
                                   rnn.cuda())
    assert ex.graph_break_count == 0, [str(b.reason)[:200] for b in ex.break_reasons]
    ref = run(fn)
    torch._dynamo.reset()
    got = run(torch.compile(fn, fullgraph=True))
    for a, b in zip(ref, got):
        assert torch.equal(a, b), (a - b).abs().max().item()


def test_opcheck_pair_train_ops(agb):
    N = agb.native
    img, wrd, cnn, rnn, _, lens, _ = rp.synth_damsm(6, seed=6)
    img3 = img.reshape(6, 256, -1).contiguous().cuda()
    w3, l32 = wrd.cuda(), lens.cuda().to(torch.int32)
    pi = torch.tensor([0, 5, 2, 2, 9, 1, 3], dtype=torch.int32, device="cuda")
    pc = torch.tensor([1, 0, 2, 2, 3, -1, 5], dtype=torch.int32, device="cuda")
    f16 = N.AGB_MATH_TC_F16
    m, ws = agb.ops.damsm_pairs_train_fwd(img3, w3, l32, pi, pc, G1, G2, f16)
    dm = torch.randn(7, device="cuda")
    no_aot = ("test_schema", "test_autograd_registration", "test_faketensor")
    every = no_aot + ("test_aot_dispatch_static",)
    # the workspace output holds bytes the kernels never write (padding): not compared by the AOT check
    torch.library.opcheck(torch.ops.agb.damsm_pairs_train_fwd.default,
                          (img3.clone().requires_grad_(), w3.clone().requires_grad_(), l32, pi, pc, G1, G2, f16),
                          test_utils=no_aot)
    torch.library.opcheck(torch.ops.agb.damsm_pairs_bwd.default,
                          (img3, w3, l32, pi, pc, G1, G2, f16, dm, ws, True, True), test_utils=every)
    # in-range pairs for the cosine: the AOT check compares outputs without equating NaNs
    c, r = cnn.cuda(), rnn.cuda()
    si, sc = pi.clamp(0, 5), pc.clamp(0, 5)
    torch.library.opcheck(torch.ops.agb.sent_cos_pairs_train_fwd.default,
                          (c.clone().requires_grad_(), r.clone().requires_grad_(), si, sc, 1e-8), test_utils=every)
    torch.library.opcheck(torch.ops.agb.sent_cos_pairs_bwd.default, (c, r, pi, pc, 1e-8, dm, True, True),
                          test_utils=every)


def test_listwise_loss_end_to_end(agb):
    """the docs example at N = 256, K = 100: gradients of the K-way listwise loss through words_pair_scores equal
    those of the same loss through the dense backward (dLoss/dm scattered into [N, N])"""
    N, K, gamma3 = 256, 100, 10.0
    img, wrd, _, _, lens, cls = _inputs(N, seed=17, trained_like=0.06)
    cands = agb.mismatched_candidates(cls, n_mismatched=K - 1, seed=0)
    pi, pc = np.repeat(np.arange(N), K), cands.reshape(-1)
    im = img.cuda().requires_grad_(True)
    wd = wrd.cuda().requires_grad_(True)
    m = agb.words_pair_scores(im, wd, lens, pi, pc, math="f16x2").view(N, K)
    loss = F.cross_entropy(gamma3 * m, torch.zeros(N, dtype=torch.long, device=m.device))
    dm = torch.autograd.grad(loss, m, retain_graph=True)[0]
    loss.backward()
    dmd = _scatter(dm.reshape(-1).cpu(), torch.from_numpy(pi), torch.from_numpy(pc),
                   torch.ones(N * K, dtype=torch.bool), N, N)
    di, dw = _dense_tc_grads(agb, img, wrd, lens, dmd, "f16x2")
    e_img, e_wrd = _rel(im.grad, di.reshape(img.shape)), _rel(wd.grad, dw)
    print(f"listwise N={N} K={K}: rel. difference to the dense backward {e_img:.2e} / {e_wrd:.2e}")
    assert e_img < 5e-3 and e_wrd < 5e-3
