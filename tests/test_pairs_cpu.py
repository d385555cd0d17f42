"""CPU tests of pair-list scoring (agb_damsm_pairs_fwd, agb_sent_cos_pairs_fwd, DAMSMScorer.words_pairs /
sentence_pairs / by="caption"): the workspace query, argument checks, refusal of CPU tensors, fake kernels and lazy
loading of the library."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def agb():
    import attention_gan_b200 as pkg
    return pkg


def test_pairs_workspace_query(agb):
    N = agb.native
    lib = N.lib()
    for name in ("agb_damsm_pairs_workspace_bytes", "agb_damsm_pairs_fwd", "agb_sent_cos_pairs_fwd"):
        assert hasattr(lib, name) and name in N.SIGNATURES
    q = lib.agb_damsm_pairs_workspace_bytes
    f16 = q(2048, 2048, 204800, 18, 256, 289, N.AGB_MATH_TC_F16)
    assert 0 < f16 < q(2048, 2048, 204800, 18, 256, 289, N.AGB_MATH_TC_F16X2)
    assert q(2048, 2048, 204800, 18, 256, 289, N.AGB_MATH_TC_BF16) > 0
    assert q(2048, 2048, 100, 33, 256, 289, N.AGB_MATH_TC_F16) == 0       # T > 32
    assert q(2048, 2048, 100, 18, 128, 289, N.AGB_MATH_TC_F16) == 0       # D != 256
    assert q(2048, 2048, 100, 18, 256, 361, N.AGB_MATH_TC_F16) == 0       # R > 320
    assert q(2048, 2048, 100, 18, 256, 289, N.AGB_MATH_FP32) == 0
    assert q(2048, 2048, 100, 18, 256, 289, N.AGB_MATH_TC_F16 | N.AGB_MATH_SAVE) == 0
    assert q(65536, 8, 100, 18, 256, 289, N.AGB_MATH_TC_F16) == 0        # Bi > 65535
    assert q(8, 8, 2 ** 31, 18, 256, 289, N.AGB_MATH_TC_F16) == 0        # P >= 2^31
    for mt in (N.AGB_MATH_TC_F16, N.AGB_MATH_TC_F16X2):
        sizes = [q(300, 500, P, 18, 256, 289, mt) for P in (0, 1, 2, 7, 100, 1000, 10 ** 5, 10 ** 6)]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes), sizes
        # the size depends on (Bi, Bc, P, T, math) only: R changes nothing
        assert q(300, 500, 1000, 18, 256, 100, mt) == q(300, 500, 1000, 18, 256, 289, mt)


def test_pair_entry_points_reject_bad_arguments(agb):
    N = agb.native
    lib = N.lib()
    rc = lib.agb_damsm_pairs_fwd(None, None, 0, 0, 0, None, 4, 4, None, None, 3, 18, 256, 289, 4.0, 5.0, None, None,
                                 None, 0, N.AGB_MATH_TC_F16, None)
    assert rc == -1 and b"null" in lib.agb_last_error()
    rc = lib.agb_damsm_pairs_fwd(None, None, 0, 0, 0, None, 4, 4, None, None, 3, 18, 256, 289, 4.0, 5.0, None, None,
                                 None, 0, N.AGB_MATH_TC_F16 | N.AGB_MATH_SAVE, None)
    assert rc != 0
    # P = 0 is a successful no-op that touches nothing
    assert lib.agb_damsm_pairs_fwd(None, None, 0, 0, 0, None, 4, 4, None, None, 0, 18, 256, 289, 4.0, 5.0, None, None,
                                   None, 0, N.AGB_MATH_TC_F16, None) == 0
    assert lib.agb_sent_cos_pairs_fwd(None, None, 4, 4, None, None, 0, 256, 1e-8, None, None) == 0
    rc = lib.agb_sent_cos_pairs_fwd(None, None, 4, 4, None, None, 3, 256, 1e-8, None, None)
    assert rc == -1 and b"null" in lib.agb_last_error()


def test_pair_scorers_refuse_cpu_tensors(agb):
    scorer = agb.DAMSMScorer("cpu", math="f16")
    idx = np.arange(4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.words_pairs(torch.zeros(4, 256, 17, 17), torch.zeros(4, 256, 18), torch.full((4,), 18), idx, idx)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.sentence_pairs(torch.zeros(4, 256), torch.zeros(4, 256), idx, idx)
    cands = agb.mismatched_candidates(None, n_mismatched=3, n=4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.words(torch.zeros(4, 256, 17, 17), torch.zeros(4, 256, 18), torch.full((4,), 18), cands, by="caption")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        scorer.sentence(torch.zeros(4, 256), torch.zeros(4, 256), cands, by="caption")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agb.ops.sent_cos_pairs_fwd(torch.zeros(4, 256), torch.zeros(4, 256), torch.zeros(4, dtype=torch.int32),
                                   torch.zeros(4, dtype=torch.int32), 1e-8)


def test_pair_index_and_shape_checks(agb):
    """checked before anything reaches a device (the index lists are host arrays here)"""
    scorer = agb.DAMSMScorer("cpu", math="f16")
    S = agb.DAMSMScorer
    with pytest.raises(ValueError, match="entries"):
        S._pairs(np.arange(5), np.arange(4), "cpu")
    with pytest.raises(ValueError, match="caption"):
        S._by_caption(np.zeros((3, 4), np.int64), 4, "cpu")           # Nc rows expected
    with pytest.raises(ValueError, match="caption"):
        S._by_caption(np.zeros(12, np.int64), 4, "cpu")               # not [Nc, K]
    pi, pc, K = S._by_caption(np.array([[0, 2], [1, 0], [2, 1]]), 3, "cpu")
    assert K == 2 and pi.tolist() == [0, 2, 1, 0, 2, 1] and pc.tolist() == [0, 0, 1, 1, 2, 2]
    assert pi.dtype == torch.int32 and pc.dtype == torch.int32
    with pytest.raises(ValueError, match="by"):
        scorer.words(torch.zeros(4, 256, 17, 17), torch.zeros(4, 256, 18), torch.full((4,), 18), np.zeros((4, 2)),
                     by="pairs")
    with pytest.raises(ValueError, match="by"):
        scorer.sentence(torch.zeros(4, 256), torch.zeros(4, 256), np.zeros((4, 2)), by="text")


def test_fake_pair_ops(agb):
    N = agb.native
    with FakeTensorMode(allow_non_fake_inputs=False):
        img = torch.empty(6, 256, 289, device="cuda")
        wrd = torch.empty(9, 256, 18, device="cuda")
        lens = torch.empty(9, dtype=torch.int32, device="cuda")
        pi = torch.empty(37, dtype=torch.int32, device="cuda")
        pc = torch.empty(37, dtype=torch.int32, device="cuda")
        m, att = torch.ops.agb.damsm_pairs_fwd(img, wrd, lens, pi, pc, 4.0, 5.0, False, N.AGB_MATH_TC_F16)
        assert m.shape == (37,) and m.dtype == torch.float32 and m.is_cuda and att.numel() == 0
        m, att = torch.ops.agb.damsm_pairs_fwd(img, wrd, lens, pi, pc, 4.0, 5.0, True, N.AGB_MATH_TC_F16X2)
        assert m.shape == (37,) and att.shape == (37, 18, 289) and att.dtype == torch.float32
        with pytest.raises(N.NativeError):
            torch.ops.agb.damsm_pairs_fwd(img, torch.empty(9, 256, 33, device="cuda"), lens, pi, pc, 4.0, 5.0, False,
                                          N.AGB_MATH_TC_F16)
        with pytest.raises(RuntimeError, match="entries"):
            torch.ops.agb.damsm_pairs_fwd(img, wrd, lens, pi, pc[:5], 4.0, 5.0, False, N.AGB_MATH_TC_F16)
        s = torch.ops.agb.sent_cos_pairs_fwd(torch.empty(6, 256, device="cuda"), torch.empty(9, 256, device="cuda"),
                                             pi, pc, 1e-8)
        assert s.shape == (37,) and s.dtype == torch.float32


def test_pair_ops_registered_without_loading_the_library():
    code = ("import attention_gan_b200 as p, torch; assert p.native._lib is None; "
            "T = p.agb_native.torch_ops; "
            "assert all(hasattr(torch.ops.agb, n) for n in T.PAIR_OPS); "
            "assert p.native._lib is None; print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr
