"""CPU tests of the R-precision evaluation (attention_gan_b200.evaluation): the candidate sampling, the ranking rule,
the refusal of CPU tensors and the host-side queries of the candidate entry points."""
import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def ev():
    import attention_gan_b200 as pkg
    return pkg


def test_mismatched_candidates_protocol(ev):
    rng = np.random.default_rng(5)
    cls = rng.integers(0, 7, size=300)
    c = ev.mismatched_candidates(cls, n_mismatched=99, seed=3)
    assert c.shape == (300, 100) and c.dtype == np.int64
    np.testing.assert_array_equal(c[:, 0], np.arange(300))
    assert c.min() >= 0 and c.max() < 300
    assert not (cls[c[:, 1:]] == cls[:, None]).any(), "a mismatched caption has the image's own class"
    # every other-class caption is reachable, and the draw is uniform over them (with replacement)
    big = ev.mismatched_candidates(np.array([0] * 3 + [1] * 5 + [2] * 2), n_mismatched=20000, seed=1)
    counts = np.bincount(big[0, 1:], minlength=10)
    assert (counts[:3] == 0).all() and (counts[3:] > 0).all()
    assert np.abs(counts[3:] / 20000 - 1 / 7).max() < 0.015
    # deterministic per seed, different across seeds; torch tensors and lists are accepted
    np.testing.assert_array_equal(c, ev.mismatched_candidates(torch.from_numpy(cls), n_mismatched=99, seed=3))
    np.testing.assert_array_equal(c, ev.mismatched_candidates(list(cls), n_mismatched=99, seed=3))
    assert not np.array_equal(c, ev.mismatched_candidates(cls, n_mismatched=99, seed=4))


def test_mismatched_candidates_without_classes(ev):
    c = ev.mismatched_candidates(None, n_mismatched=50, seed=0, n=40)
    assert c.shape == (40, 51)
    np.testing.assert_array_equal(c[:, 0], np.arange(40))
    assert not (c[:, 1:] == np.arange(40)[:, None]).any()
    assert set(np.unique(c[:, 1:])) == set(range(40))
    np.testing.assert_array_equal(c, ev.mismatched_candidates(None, n_mismatched=50, seed=0, n=40))
    with pytest.raises(ValueError):
        ev.mismatched_candidates(None, n_mismatched=5)


def test_mismatched_candidates_impossible(ev):
    with pytest.raises(ValueError, match="no caption of another class"):
        ev.mismatched_candidates(np.array([4, 4, 4]), n_mismatched=2)
    with pytest.raises(ValueError):
        ev.mismatched_candidates(None, n_mismatched=2, n=1)


def test_r_precision_ranking_rule(ev):
    nan = float("nan")
    s = torch.tensor([[0.9, 0.1, 0.2, 0.3],      # own caption first: hit
                      [0.5, 0.5, 0.1, 0.0],      # tie with a mismatch: miss at r = 1
                      [0.2, 0.3, 0.1, 0.0],      # second: miss at r = 1, hit at r = 2
                      [0.2, 0.3, 0.4, 0.1],      # third
                      [nan, 0.1, 0.2, 0.3],      # own score NaN: always a miss
                      [0.9, nan, 0.1, 0.2],      # a NaN competitor counts against the own caption
                      [0.9, 0.9, 0.9, 0.9]])     # all tied
    np.testing.assert_array_equal(ev.r_precision(s, r=1).numpy(), [1, 0, 0, 0, 0, 0, 0])
    np.testing.assert_array_equal(ev.r_precision(s, r=2).numpy(), [1, 1, 1, 0, 0, 1, 0])
    np.testing.assert_array_equal(ev.r_precision(s, r=3).numpy(), [1, 1, 1, 1, 0, 1, 0])
    np.testing.assert_array_equal(ev.r_precision(s, r=4).numpy(), [1, 1, 1, 1, 0, 1, 1])
    assert ev.r_precision(s).dtype == torch.bool and ev.r_precision(s).device == s.device
    # a list of one caption is always a hit unless its score is NaN
    np.testing.assert_array_equal(ev.r_precision(torch.tensor([[1.0], [nan]])).numpy(), [1, 0])


def test_scorer_refuses_cpu_tensors(ev):
    scorer = ev.DAMSMScorer("cpu", math="f16")
    cands = ev.mismatched_candidates(None, n_mismatched=3, n=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.words(torch.zeros(4, 256, 17, 17), torch.zeros(4, 256, 18), torch.full((4,), 18), cands)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.sentence(torch.zeros(4, 256), torch.zeros(4, 256), cands)
    with pytest.raises(ValueError):
        ev.DAMSMScorer("cpu", math="fp32")


def test_candidate_entry_points_host_side(ev):
    """the new symbols are declared, exported and bound (the header <-> exports <-> ctypes test covers them too);
    the workspace query is pure host code and follows the documented limits"""
    lib = ev.native.lib()
    N = ev.native
    for name in ("agb_damsm_cand_workspace_bytes", "agb_damsm_cand_fwd", "agb_sent_cos_cand_fwd"):
        assert hasattr(lib, name) and name in N.SIGNATURES
    f16 = lib.agb_damsm_cand_workspace_bytes(2048, 100, 18, 256, 289, N.AGB_MATH_TC_F16)
    x2 = lib.agb_damsm_cand_workspace_bytes(2048, 100, 18, 256, 289, N.AGB_MATH_TC_F16X2)
    assert 0 < f16 < x2
    assert lib.agb_damsm_cand_workspace_bytes(4096, 100, 18, 256, 289, N.AGB_MATH_TC_F16) > f16
    assert lib.agb_damsm_cand_workspace_bytes(2048, 100, 33, 256, 289, N.AGB_MATH_TC_F16) == 0     # T > 32
    assert lib.agb_damsm_cand_workspace_bytes(2048, 100, 18, 256, 289, N.AGB_MATH_FP32) == 0
    assert lib.agb_damsm_cand_workspace_bytes(2048, 100, 18, 256, 289, N.AGB_MATH_TC_F16 | N.AGB_MATH_SAVE) == 0
    assert lib.agb_damsm_cand_workspace_bytes(65536, 1, 18, 256, 289, N.AGB_MATH_TC_F16) == 0      # Bi > 65535
    assert lib.agb_damsm_cand_workspace_bytes(65535, 40000, 18, 256, 289, N.AGB_MATH_TC_F16) == 0  # Bi*K >= 2^31
    rc = lib.agb_damsm_cand_fwd(None, None, 0, 0, 0, None, 1, None, 1, 1, 18, 256, 289, 4.0, 5.0, None, None, 0,
                                N.AGB_MATH_TC_F16, None)
    assert rc == -1 and b"null" in lib.agb_last_error()
    rc = lib.agb_sent_cos_cand_fwd(None, None, 4, None, 4, 3, 256, 1e-8, None, None)
    assert rc == -1 and b"null" in lib.agb_last_error()
