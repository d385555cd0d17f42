"""GPU tests of pair-list scoring (agb_damsm_pairs_fwd, agb_sent_cos_pairs_fwd, DAMSMScorer.words_pairs /
sentence_pairs / by="caption"): pair m equals the dense similarity matrix gathered, bit for bit, in any list order,
and pair maps equal the loss's matched maps; both agree with the fp64 oracle."""

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_port as rp

pytestmark = pytest.mark.gpu

G1, G2 = 4.0, 5.0
NAN = float("nan")


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


def _inputs(Bc, T=18, seed=0, trained_like=False):
    img, wrd, cnn, rnn, _, lens, cls = rp.synth_damsm(Bc, T=T, seed=seed, trained_like=trained_like, n_classes=50)
    return img.reshape(Bc, 256, -1), wrd, cnn, rnn, lens, cls


def _dense_gathered(agb, img, wrd, lens, pi, pc, math_name):
    """the dense inference forward, then the gather at (pi, pc); NaN where either index is out of range"""
    lens = lens.to(torch.int32)                               # ops.damsm_fwd reads cap_lens as int32
    m, _, _ = agb.ops.damsm_fwd(img, wrd, lens, G1, G2, 1e-8, 0, False, agb.native.MATH_NAMES[math_name])
    i, j = pi.long(), pc.long()
    ok = (i >= 0) & (i < m.shape[0]) & (j >= 0) & (j < m.shape[1])
    g = m[i.clamp(0, m.shape[0] - 1), j.clamp(0, m.shape[1] - 1)]
    return torch.where(ok, g, torch.full_like(g, NAN))


def _assert_same_bits(a, b):
    assert a.shape == b.shape, (a.shape, b.shape)
    a, b = a.reshape(-1), b.reshape(-1)
    same = (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
    if not bool(same.all()):
        idx = torch.nonzero(~same)[:5, 0].tolist()
        raise AssertionError(f"{int((~same).sum())} entries differ, e.g. at {idx}: "
                             f"{[(a[i].item(), b[i].item()) for i in idx]}")


def _list(case, Bi, Bc, lens):
    """(pair_img, pair_cap) int32 on the host"""
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    if case == "random":
        P = 997
        return (torch.randint(0, Bi, (P,), generator=g, dtype=torch.int32),
                torch.randint(0, Bc, (P,), generator=g, dtype=torch.int32))
    if case == "duplicates":
        pi = torch.randint(0, Bi, (300,), generator=g, dtype=torch.int32)
        pc = torch.randint(0, Bc, (300,), generator=g, dtype=torch.int32)
        return torch.cat([pi, pi[:100], pi[5:6].repeat(40)]), torch.cat([pc, pc[:100], pc[5:6].repeat(40)])
    if case == "empty_images":                                   # only the odd images and image 0 have pairs
        pi = torch.randint(0, Bi // 2, (400,), generator=g, dtype=torch.int32) * 2 + 1
        pi[::50] = 0
        return pi, torch.randint(0, Bc, (400,), generator=g, dtype=torch.int32)
    if case == "p1":
        return torch.tensor([Bi - 1], dtype=torch.int32), torch.tensor([3], dtype=torch.int32)
    if case == "skewed":                                         # every pair on one image
        P = 10 ** 5
        return torch.full((P,), 17, dtype=torch.int32), torch.randint(0, Bc, (P,), generator=g, dtype=torch.int32)
    if case == "len1_len32":
        pi = torch.randint(0, Bi, (500,), generator=g, dtype=torch.int32)
        pc = torch.randint(0, Bc, (500,), generator=g, dtype=torch.int32)
        pc[::3], pc[1::3] = 3, 4
        return pi, pc
    if case == "out_of_range":
        pi = torch.randint(0, Bi, (600,), generator=g, dtype=torch.int32)
        pc = torch.randint(0, Bc, (600,), generator=g, dtype=torch.int32)
        pi[::7], pi[3::11] = -1, Bi
        pc[1::9], pc[2::13] = -5, Bc
        pi[5], pc[5] = 70000, 2 ** 31 - 1
        return pi, pc
    raise ValueError(case)


CASES = ["random", "duplicates", "empty_images", "p1", "skewed", "len1_len32", "out_of_range"]


@pytest.mark.parametrize("math_name,tol", [("f16", 2e-3), ("bf16", 2e-2), ("f16x2", 2e-5)])
@pytest.mark.parametrize("case", CASES)
def test_pairs_equal_dense_gathered_and_oracle(agb, case, math_name, tol):
    T = 32 if case == "len1_len32" else 18
    img, wrd, _, _, lens, _ = _inputs(64, T=T, seed=21)
    if case == "len1_len32":
        lens[3], lens[4] = 1, 32
    Bi = 40
    pi, pc = _list(case, Bi, 64, lens)
    img_d, wd, ln = img[:Bi].cuda().contiguous(), wrd.cuda(), lens.cuda().to(torch.int32)
    m = agb.DAMSMScorer("cuda", G1, G2, math=math_name).words_pairs(img_d, wd, ln, pi.cuda(), pc.cuda())
    _assert_same_bits(m, _dense_gathered(agb, img_d, wd, ln, pi.cuda(), pc.cuda(), math_name))
    bad = ((pi < 0) | (pi >= Bi) | (pc < 0) | (pc >= 64)).cuda()
    assert bool(torch.isnan(m[bad]).all()) and bool(torch.isfinite(m[~bad]).all())
    if case == "out_of_range":
        assert int(bad.sum()) > 150
    ok = ~bad.cpu()
    ref = cf.words_similarity_fwd(img[:Bi].numpy(), wrd.numpy(), lens.numpy(), G1, G2)
    err = np.abs(m.cpu()[ok].double().numpy() - ref[pi[ok].long().numpy(), pc[ok].long().numpy()]).max()
    assert err < tol, f"max |m - oracle| = {err:.3e}"


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_image_to_text_candidates_as_pairs(agb, math_name):
    """the candidate list as pairs, in candidate order and shuffled, equals words(candidates) bit for bit"""
    img, wrd, _, _, lens, cls = _inputs(120, seed=5)
    cand = torch.from_numpy(agb.mismatched_candidates(cls, n_mismatched=29, seed=1)).to(torch.int32)
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda()
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name)
    ref = scorer.words(img_d, wd, ln, cand.cuda()).reshape(-1)
    pi = torch.arange(120, dtype=torch.int32).repeat_interleave(30)
    pc = cand.reshape(-1)
    _assert_same_bits(scorer.words_pairs(img_d, wd, ln, pi, pc), ref)
    perm = torch.randperm(pi.shape[0], generator=torch.Generator().manual_seed(4))
    m = scorer.words_pairs(img_d, wd, ln, pi[perm].cuda(), pc[perm].cuda())
    _assert_same_bits(m, ref[perm.cuda()])


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_text_to_image_by_caption(agb, math_name):
    img, wrd, cnn, rnn, lens, cls = _inputs(96, seed=9)
    cand = torch.from_numpy(agb.mismatched_candidates(cls, n_mismatched=19, seed=4)).to(torch.int32)   # images
    cand[3, 2], cand[7, 0] = -1, 96
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda()
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name)
    m = scorer.words(img_d, wd, ln, cand.cuda(), by="caption")
    assert m.shape == (96, 20)
    caps = torch.arange(96, dtype=torch.int32)[:, None].expand(96, 20)
    _assert_same_bits(m, _dense_gathered(agb, img_d, wd, ln, cand.cuda(), caps.cuda(), math_name))
    # sentence: equal to the candidate cosine of the same pairs (image-major lists of one pair each), and within
    # 1e-6 of the dense cosine gathered
    c, r = cnn.cuda(), rnn.cuda()
    s = scorer.sentence(c, r, cand.numpy(), by="caption")
    sp = scorer.sentence_pairs(c, r, cand.reshape(-1), caps.reshape(-1))
    _assert_same_bits(sp, s.reshape(-1))
    bad = ((cand < 0) | (cand >= 96)).cuda()
    # the candidate cosine of image b with caption j, as agb_sent_cos_cand_fwd computes it
    cand_cos = agb.ops.sent_cos_cand_fwd(c, r, torch.arange(96, dtype=torch.int32, device="cuda")[None].expand(96, 96)
                                         .contiguous(), 1e-8)
    ci = cand.long().cuda().clamp(0, 95)
    ref = cand_cos[ci, torch.arange(96, device="cuda")[:, None].expand(96, 20)]
    _assert_same_bits(s, torch.where(bad, torch.full_like(ref, NAN), ref))
    dense = agb.ops.sent_cos_fwd(c, r, 1e-8)[ci, torch.arange(96, device="cuda")[:, None].expand(96, 20)]
    rel = ((s - dense).abs() / dense.abs().clamp_min(1e-30))[~bad].max().item()
    assert rel < 1e-6, f"relative difference {rel:.2e}"
    assert bool(torch.isnan(s[bad]).all())
    agb.r_precision(m)                                           # the [Nc, K] result ranks unchanged


@pytest.mark.parametrize("math_name", ["f16", "bf16", "f16x2"])
def test_pair_maps(agb, math_name):
    B = 24
    img, wrd, _, _, lens, _ = _inputs(B, seed=13)
    lens[2] = 1
    img4 = img.reshape(B, 256, 17, 17).cuda()
    wd, ln = wrd.cuda(), lens.cuda().to(torch.int32)
    _, packed = agb.WordsLoss("cuda", G1, G2, math=math_name, att_maps="packed").get_loss(
        img4, wd, torch.arange(B, device="cuda"), ln, None)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name)
    diag = torch.arange(B, dtype=torch.int32, device="cuda")
    m, maps = scorer.words_pairs(img4, wd, ln, diag, diag, att_maps=True)
    assert maps.shape == (B, 18, 17, 17)
    _assert_same_bits(maps, packed)
    _assert_same_bits(m, scorer.words_pairs(img4, wd, ln, diag, diag))      # maps do not change m
    g = torch.Generator().manual_seed(2)
    pi = torch.randint(0, B, (60,), generator=g, dtype=torch.int32)
    pc = torch.randint(0, B, (60,), generator=g, dtype=torch.int32)
    pi[7], pc[9], pc[11] = B, -1, B
    _, maps = scorer.words_pairs(img4, wd, ln, pi.cuda(), pc.cuda(), att_maps=True)
    maps = maps.reshape(60, 18, 289).cpu()
    for p in range(60):
        b, j = int(pi[p]), int(pc[p])
        if not (0 <= b < B and 0 <= j < B):
            assert bool(torch.isnan(maps[p]).all()), p
            continue
        L = int(lens[j])
        _, beta = cf.func_attention_fwd(wrd[j:j + 1, :, :L].numpy(), img[b:b + 1].numpy(), G1)
        assert np.abs(maps[p, :L].double().numpy() - beta[0]).max() < 1e-5, p
        assert bool((maps[p, L:] == 0).all()), p


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_chunking_does_not_change_results(agb, math_name):
    img, wrd, _, _, lens, _ = _inputs(80, seed=6)
    g = torch.Generator().manual_seed(8)
    P = 3000
    pi = torch.randint(0, 80, (P,), generator=g, dtype=torch.int32).cuda()
    pc = torch.randint(0, 80, (P,), generator=g, dtype=torch.int32).cuda()
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda()
    m1, a1 = agb.DAMSMScorer("cuda", G1, G2, math=math_name).words_pairs(img_d, wd, ln, pi, pc, att_maps=True)
    mt = agb.native.MATH_NAMES[math_name]
    small = agb.ops.damsm_pairs_workspace_bytes(80, 80, P // 4, 18, 256, img.shape[2], mt)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name, workspace_bytes=small)
    assert scorer._chunk_pairs(80, 80, P, 18, 256, img.shape[2], agb.ops.damsm_pairs_workspace_bytes) <= P // 4
    m2, a2 = scorer.words_pairs(img_d, wd, ln, pi, pc, att_maps=True)
    _assert_same_bits(m2, m1)
    _assert_same_bits(a2, a1)


def test_deterministic_and_graph_capture(agb):
    img, wrd, _, _, lens, _ = _inputs(96, seed=8)
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda().to(torch.int32)
    g = torch.Generator().manual_seed(5)
    pi = torch.randint(0, 96, (2000,), generator=g, dtype=torch.int32).cuda()
    pc = torch.randint(0, 96, (2000,), generator=g, dtype=torch.int32).cuda()
    pi[:500] = 3                                                  # a skewed head
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16x2")
    m1, a1 = scorer.words_pairs(img_d, wd, ln, pi, pc, att_maps=True)
    m2, a2 = scorer.words_pairs(img_d, wd, ln, pi, pc, att_maps=True)
    _assert_same_bits(m1, m2)
    _assert_same_bits(a1, a2)
    step = agb.GraphedStep(lambda: scorer.words_pairs(img_d, wd, ln, pi, pc, att_maps=True))
    out = step.replay()
    out = step.replay()
    torch.cuda.synchronize()
    _assert_same_bits(out[0], m1)
    _assert_same_bits(out[1], a1)


def test_end_to_end_text_to_image_r_precision(agb):
    N = 256
    img, wrd, cnn, rnn, lens, cls = _inputs(N, seed=17, trained_like=0.06)
    cand = agb.mismatched_candidates(cls, n_mismatched=49, seed=0)          # images per caption (shared classes)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16x2")
    m = scorer.words(img.cuda().contiguous(), wrd.cuda(), lens.cuda(), cand, by="caption")
    c64, w64 = img.double().numpy(), wrd.double().numpy()
    ref = np.empty(cand.shape)
    for i in range(N):                                                       # caption i against its image list
        ref[i] = cf.words_similarity_fwd(c64[cand[i]], w64[i:i + 1], [int(lens[i])], G1, G2)[:, 0]
    ref = torch.from_numpy(ref)
    hits, ref_hits = agb.r_precision(m).cpu(), agb.r_precision(ref)
    margin = (ref[:, 0] - ref[:, 1:].max(dim=1).values).abs()
    near = margin < 1e-4
    assert bool((hits == ref_hits)[~near].all()), f"{int((hits != ref_hits)[~near].sum())} hits differ"
    assert 0.0 < hits.float().mean().item() < 1.0
    s = scorer.sentence(cnn.cuda(), rnn.cuda(), cand, by="caption")
    cn, rn = cnn.double().numpy()[cand], rnn.double().numpy()              # [N, K, D], [N, D]
    num = np.einsum("nkd,nd->nk", cn, rn)
    den = np.maximum(np.linalg.norm(cn, axis=2) * np.linalg.norm(rn, axis=1)[:, None], 1e-8)
    assert torch.equal(agb.r_precision(s).cpu(), agb.r_precision(torch.from_numpy(num / den)))


def test_compiled_pair_scorers(agb):
    torch._dynamo.reset()
    img, wrd, cnn, rnn, lens, cls = _inputs(64, seed=3)
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda().to(torch.int32)
    c, r = cnn.cuda(), rnn.cuda()
    g = torch.Generator().manual_seed(1)
    pi = torch.randint(0, 64, (700,), generator=g, dtype=torch.int32).cuda()
    pc = torch.randint(0, 64, (700,), generator=g, dtype=torch.int32).cuda()
    cand = torch.from_numpy(agb.mismatched_candidates(cls, n_mismatched=9, seed=2)).to(torch.int32).cuda()
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16x2")

    def f(img_d, wd, ln, pi, pc, c, r, cand):
        m, maps = scorer.words_pairs(img_d, wd, ln, pi, pc, att_maps=True)
        return (m, maps, scorer.sentence_pairs(c, r, pi, pc), scorer.words(img_d, wd, ln, cand, by="caption"),
                scorer.sentence(c, r, cand, by="caption"))

    args = (img_d, wd, ln, pi, pc, c, r, cand)
    eager = f(*args)
    explained = torch._dynamo.explain(f)(*args)
    assert explained.graph_break_count == 0, explained.break_reasons
    torch._dynamo.reset()
    compiled = torch.compile(f, fullgraph=True)(*args)
    for a, b in zip(compiled, eager):
        _assert_same_bits(a, b)


def test_pair_ops_opcheck(agb):
    img, wrd, cnn, rnn, lens, _ = _inputs(16, seed=4)
    g = torch.Generator().manual_seed(3)
    # valid indices only: opcheck compares outputs with assert_close, which treats NaN as unequal
    pi = torch.randint(0, 16, (50,), generator=g, dtype=torch.int32).cuda()
    pc = torch.randint(0, 16, (50,), generator=g, dtype=torch.int32).cuda()
    args = (img.cuda().contiguous(), wrd.cuda(), lens.cuda().to(torch.int32), pi, pc, G1, G2, True,
            agb.native.AGB_MATH_TC_F16)
    every = ("test_schema", "test_autograd_registration", "test_faketensor", "test_aot_dispatch_static")
    torch.library.opcheck(torch.ops.agb.damsm_pairs_fwd.default, args, test_utils=every)
    torch.library.opcheck(torch.ops.agb.sent_cos_pairs_fwd.default, (cnn.cuda(), rnn.cuda(), pi, pc, 1e-8),
                          test_utils=every)
