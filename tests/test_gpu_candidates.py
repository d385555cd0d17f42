"""GPU tests of candidate scoring (agb_damsm_cand_fwd, agb_sent_cos_cand_fwd, attention_gan_b200.evaluation):
candidate m equals the dense similarity matrix gathered, bit for bit, and both agree with the fp64 oracle."""
import math

import numpy as np
import pytest
import torch

from oracle import closed_form as cf
from oracle import ref_port as rp

pytestmark = pytest.mark.gpu

G1, G2 = 4.0, 5.0


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


def _inputs(Bc, T=18, seed=0, trained_like=False):
    img, wrd, cnn, rnn, _, lens, cls = rp.synth_damsm(Bc, T=T, seed=seed, trained_like=trained_like, n_classes=50)
    return img.reshape(Bc, 256, -1), wrd, cnn, rnn, lens, cls


def _dense_gathered(agb, img, wrd, lens, cand, math_name):
    """what a user computes without candidate mode: the dense inference forward, then the gather"""
    m, _, _ = agb.ops.damsm_fwd(img, wrd, lens, G1, G2, 1e-8, 0, False, agb.native.MATH_NAMES[math_name])
    c = cand.long()
    ok = (c >= 0) & (c < m.shape[1])
    return torch.where(ok, m.gather(1, c.clamp(0, m.shape[1] - 1)), torch.full_like(c, float("nan"), dtype=m.dtype))


def _assert_same_bits(a, b):
    assert a.shape == b.shape
    same = (a.view(torch.int32) == b.view(torch.int32)) | (torch.isnan(a) & torch.isnan(b))
    if not bool(same.all()):
        idx = torch.nonzero(~same)[:5].tolist()
        raise AssertionError(f"{int((~same).sum())} entries differ, e.g. at {idx}: "
                             f"{[(a[i, j].item(), b[i, j].item()) for i, j in idx]}")


@pytest.mark.parametrize("math_name,tol", [("f16", 2e-3), ("bf16", 2e-2), ("f16x2", 2e-5)])
def test_candidates_equal_dense_gathered_and_oracle(agb, math_name, tol):
    """Bi = 40 images against lists drawn from Bc = 96 captions with ragged lengths and duplicates in a list"""
    img, wrd, _, _, lens, _ = _inputs(96, seed=11)
    img40 = img[:40].cuda().contiguous()
    wd, ln = wrd.cuda(), lens.cuda().to(torch.int32)
    g = torch.Generator().manual_seed(3)
    cand = torch.randint(0, 96, (40, 37), generator=g, dtype=torch.int32)
    cand[:, 5] = cand[:, 4]                                   # duplicates inside every list
    cand[:, 0] = torch.arange(40)
    cand_d = cand.cuda()
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name)
    m = scorer.words(img40, wd, ln, cand_d)
    _assert_same_bits(m, _dense_gathered(agb, img40, wd, ln, cand_d, math_name))
    ref = cf.words_similarity_fwd(img[:40].numpy(), wrd.numpy(), lens.numpy(), G1, G2)
    ref_c = np.take_along_axis(ref, cand.long().numpy(), axis=1)
    err = np.abs(m.double().cpu().numpy() - ref_c).max()
    assert err < tol, f"max |m - oracle| = {err:.3e}"


def _edge_case(case):
    """(img [Bi,256,R], words [Bc,256,T], lens [Bc], cand [Bi,K]) on the host"""
    g = torch.Generator().manual_seed(sum(map(ord, case)))
    T = 32 if case == "len1_len32" else 18
    img, wrd, _, _, lens, _ = _inputs(64, T=T, seed=21)
    Bi = 1 if case == "bi1" else 24
    K = {"k1": 1, "k300": 300}.get(case, 40)
    cand = torch.randint(0, 64, (Bi, K), generator=g, dtype=torch.int32)
    if case == "repeated":
        cand[:] = 7
    if case == "len1_len32":
        lens[3], lens[4] = 1, 32
        cand[:, ::3] = 3
        cand[:, 1::3] = 4
    if case == "out_of_range":
        cand[:, 2] = -1
        cand[:, 9] = 64
        cand[5, :] = -1                                       # an image with no valid candidate at all
    return img[:Bi].contiguous(), wrd, lens, cand


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
@pytest.mark.parametrize("case", ["k1", "k300", "repeated", "len1_len32", "bi1", "out_of_range"])
def test_candidate_edge_cases(agb, case, math_name):
    img, wrd, lens, cand = _edge_case(case)
    img, wd, ln, cd = img.cuda(), wrd.cuda(), lens.cuda().to(torch.int32), cand.cuda()
    m = agb.DAMSMScorer("cuda", G1, G2, math=math_name).words(img, wd, ln, cd)
    _assert_same_bits(m, _dense_gathered(agb, img, wd, ln, cd, math_name))
    bad = ((cand < 0) | (cand >= wrd.shape[0])).cuda()
    assert bool(torch.isnan(m[bad]).all()) and bool(torch.isfinite(m[~bad]).all())
    if case == "out_of_range":
        assert int(bad.sum()) > 40


def test_caption_length_33_is_refused(agb):
    img, wrd, _, _, lens, _ = _inputs(8, T=33, seed=2)
    with pytest.raises(agb.native.NativeError):
        agb.DAMSMScorer("cuda", math="f16").words(img.cuda(), wrd.cuda(), lens.cuda(), np.zeros((8, 4), np.int64))


@pytest.mark.parametrize("math_name", ["f16", "f16x2"])
def test_chunking_does_not_change_results(agb, math_name):
    img, wrd, _, _, lens, cls = _inputs(200, seed=5)
    cand = agb.mismatched_candidates(cls, n_mismatched=49, seed=1)
    img, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda()
    m1 = agb.DAMSMScorer("cuda", G1, G2, math=math_name).words(img, wd, ln, cand)
    mt = agb.native.MATH_NAMES[math_name]
    small = agb.ops.damsm_cand_workspace_bytes(200 // 3, 50, 18, 256, img.shape[2], mt)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math=math_name, workspace_bytes=small)
    assert math.ceil(200 / scorer._chunk_images(200, 50, 18, 256, img.shape[2])) >= 3
    _assert_same_bits(scorer.words(img, wd, ln, cand), m1)


def test_words_capture_in_a_cuda_graph(agb):
    img, wrd, _, _, lens, cls = _inputs(96, seed=8)
    img, wd = img.cuda().contiguous(), wrd.cuda()
    ln = lens.cuda().to(torch.int32)
    cand = torch.from_numpy(agb.mismatched_candidates(cls, n_mismatched=29, seed=2)).to(torch.int32).cuda()
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16x2")
    eager = scorer.words(img, wd, ln, cand)
    step = agb.GraphedStep(lambda: scorer.words(img, wd, ln, cand))
    out = step.replay()
    torch.cuda.synchronize()
    _assert_same_bits(out, eager)


def test_sentence_scores(agb):
    _, _, cnn, rnn, _, cls = _inputs(96, seed=9)
    cand = torch.from_numpy(agb.mismatched_candidates(cls, n_mismatched=19, seed=4)).to(torch.int32)
    cand[3, 2], cand[7, 0] = -1, 96
    c, r = cnn[:40].cuda(), rnn.cuda()
    s = agb.DAMSMScorer("cuda").sentence(c, r, cand[:40].numpy())
    dense = agb.ops.sent_cos_fwd(c, r, 1e-8)
    cd = cand[:40].long().cuda()
    bad = (cd < 0) | (cd >= 96)
    ref = dense.gather(1, cd.clamp(0, 95))
    assert bool(torch.isnan(s[bad]).all()) and bool(torch.isfinite(s[~bad]).all())
    rel = ((s - ref).abs() / ref.abs().clamp_min(1e-30))[~bad].max().item()
    assert rel < 1e-6, f"relative difference {rel:.2e}"


def _oracle_cand_m(img, wrd, lens, cand):
    """fp64 m of the candidate pairs, the closed form of oracle/closed_form.words_similarity_fwd evaluated in torch
    (on the GPU: 512 x 100 pairs are too many for the numpy loop)"""
    c = img.double()
    N, D, R = c.shape
    T = wrd.shape[2]
    out = torch.empty(cand.shape, dtype=torch.float64, device=c.device)
    t = torch.arange(T, device=c.device)
    for k in range(cand.shape[1]):
        j = cand[:, k].long()
        w = wrd[j].double()                                   # [N, D, T]
        live = t[None, :] < lens[j].long()[:, None]           # [N, T]
        s = torch.einsum("bdr,bdt->brt", c, w) / math.sqrt(D)
        alpha = torch.softmax(s.masked_fill(~live[:, None, :], -math.inf), dim=2)
        e = torch.exp(G1 * alpha)
        beta = e / e.sum(dim=1, keepdim=True)
        v = torch.einsum("bdr,brt->bdt", c, beta)
        n = (w * v).sum(dim=1)
        den = torch.clamp(w.norm(dim=1) * v.norm(dim=1), min=1e-8)
        out[:, k] = torch.logsumexp((G2 * n / den).masked_fill(~live, -math.inf), dim=1)
    return out


def test_end_to_end_r_precision(agb):
    N = 512
    img, wrd, cnn, rnn, lens, cls = _inputs(N, seed=17, trained_like=0.06)
    cand = agb.mismatched_candidates(cls, n_mismatched=99, seed=0)
    scorer = agb.DAMSMScorer("cuda", G1, G2, math="f16x2")
    img_d, wd, ln = img.cuda().contiguous(), wrd.cuda(), lens.cuda()
    cand_d = torch.from_numpy(cand).cuda()
    m = scorer.words(img_d, wd, ln, cand)
    ref = _oracle_cand_m(img_d, wd, ln, cand_d)
    # the torch statement of the oracle agrees with the numpy one (3 images, all of their candidates)
    np_ref = cf.words_similarity_fwd(img[:3].numpy(), wrd.numpy(), lens.numpy(), G1, G2)
    np.testing.assert_allclose(ref[:3].cpu().numpy(), np.take_along_axis(np_ref, cand[:3], axis=1), rtol=1e-10, atol=1e-10)
    hits = agb.r_precision(m)
    ref_hits = agb.r_precision(ref)
    margin = (ref[:, 0] - ref[:, 1:].max(dim=1).values).abs()
    near = margin < 1e-4
    assert bool((hits == ref_hits)[~near].all()), f"{int((hits != ref_hits)[~near].sum())} word-level hits differ"
    assert int(near.sum()) <= 5, f"{int(near.sum())} images within 1e-4 of a tie"
    assert 0.0 < hits.float().mean().item() < 1.0        # the synthetic signal leaves both hits and misses
    # sentence score: the fp32 kernel ranks exactly as an fp64 numpy computation does
    s = scorer.sentence(cnn.cuda(), rnn.cuda(), cand)
    c64, r64 = cnn.double().numpy(), rnn.double().numpy()[cand]               # [N, D], [N, K, D]
    num = np.einsum("nd,nkd->nk", c64, r64)
    den = np.maximum(np.linalg.norm(c64, axis=1)[:, None] * np.linalg.norm(r64, axis=2), 1e-8)
    s_ref = torch.from_numpy(num / den)
    assert torch.equal(agb.r_precision(s).cpu(), agb.r_precision(s_ref))
    for r in (1, 2, 5):
        assert torch.equal(agb.r_precision(s, r=r).cpu(), agb.r_precision(s_ref, r=r))
