"""CPU tests of training on pair lists (agb_damsm_pairs_train_fwd / agb_damsm_pairs_bwd / agb_sent_cos_pairs_bwd,
words_pair_scores / sentence_pair_scores): workspace queries from shapes, argument checks, refusal of CPU tensors,
the C exports, fake kernels and lazy registration of the ops."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_EXPORTS = ("agb_damsm_pairs_train_workspace_bytes", "agb_damsm_pairs_train_fwd", "agb_damsm_pairs_bwd",
               "agb_sent_cos_pairs_bwd_workspace_bytes", "agb_sent_cos_pairs_bwd")


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


def test_train_workspace_query(agb):
    N = agb.native
    q = N.lib().agb_damsm_pairs_train_workspace_bytes
    fwd = N.lib().agb_damsm_pairs_workspace_bytes
    for mt in (N.AGB_MATH_TC_F16, N.AGB_MATH_TC_BF16, N.AGB_MATH_TC_F16X2):
        big = q(2048, 2048, 204800, 18, 256, 289, mt)
        # the training workspace holds the scoring one plus the saved rows (>= 512 B per packed row) and the staging
        assert big > fwd(2048, 2048, 204800, 18, 256, 289, mt) + 204800 // 6 * 128 * 512
        sizes = [q(300, 500, P, 18, 256, 289, mt) for P in (0, 1, 2, 7, 100, 1000, 10 ** 5, 10 ** 6)]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes), sizes
        assert q(300, 500, 1000, 18, 256, 100, mt) == q(300, 500, 1000, 18, 256, 289, mt)
    assert q(2048, 2048, 100, 33, 256, 289, N.AGB_MATH_TC_F16) == 0       # T > 32
    assert q(2048, 2048, 100, 18, 128, 289, N.AGB_MATH_TC_F16) == 0       # D != 256
    assert q(2048, 2048, 100, 18, 256, 321, N.AGB_MATH_TC_F16) == 0       # R > 320
    assert q(2048, 2048, 100, 18, 256, 289, N.AGB_MATH_FP32) == 0
    assert q(65536, 8, 100, 18, 256, 289, N.AGB_MATH_TC_F16) == 0        # Bi > 65535
    assert q(8, 8, 2 ** 31, 18, 256, 289, N.AGB_MATH_TC_F16) == 0        # P >= 2^31
    assert q(8, 8, -1, 18, 256, 289, N.AGB_MATH_TC_F16) == 0             # P < 0
    s = N.lib().agb_sent_cos_pairs_bwd_workspace_bytes
    assert 0 < s(4, 4, 0, 256) < s(4, 4, 100, 256) < s(4, 4, 10 ** 6, 256)
    assert s(4, 4, -1, 256) == 0 and s(0, 4, 10, 256) == 0 and s(4, 4, 2 ** 31, 256) == 0


def test_train_entry_points_reject_bad_arguments(agb):
    N = agb.native
    lib = N.lib()
    f16 = N.AGB_MATH_TC_F16

    def train(Bi, P, ptr=None, math=f16):
        return lib.agb_damsm_pairs_train_fwd(ptr, ptr, 0, 0, 0, ptr, Bi, 4, ptr, ptr, P, 18, 256, 289, 4.0, 5.0, ptr,
                                             ptr, 1 << 40, math, None)

    def bwd(Bi, P, ptr=None, math=f16):
        return lib.agb_damsm_pairs_bwd(ptr, ptr, 0, 0, 0, ptr, Bi, 4, ptr, ptr, P, 18, 256, 289, 4.0, 5.0, ptr, ptr,
                                       ptr, ptr, 1 << 40, math, None)

    for call in (train, bwd):
        assert call(4, 3) == -1 and b"null" in lib.agb_last_error()
        fake = 1 << 20                          # never dereferenced: the size checks come first
        assert call(4, -1, fake) != 0
        assert call(65536, 3, fake) != 0 and b"65535" in lib.agb_last_error()
        assert call(4, 2 ** 31, fake) != 0
        assert call(4, 3, fake, N.AGB_MATH_FP32) != 0
        assert call(4, 3, fake, f16 | N.AGB_MATH_SAVE) != 0
    assert train(4, 0) == 0                     # P = 0: a no-op that touches nothing
    rc = lib.agb_sent_cos_pairs_bwd(None, None, 4, 4, None, None, 3, 256, 1e-8, None, None, None, None, 0, None)
    assert rc == -1 and b"null" in lib.agb_last_error()
    fake = 1 << 20
    assert lib.agb_sent_cos_pairs_bwd(fake, fake, 4, 4, fake, fake, -1, 256, 1e-8, fake, None, None, fake, 0, None) != 0


def test_python_argument_checks(agb):
    """length mismatch, P < 0 via a bad list, Bi > 65535: raised before anything reaches a device"""
    from attention_gan_b200.losses.damsm_core import chunk_pairs, pair_index
    with pytest.raises(ValueError, match="entries"):
        pair_index(np.arange(5), np.arange(4), "cpu")
    q = agb.ops.damsm_pairs_train_workspace_bytes
    with pytest.raises(agb.native.NativeError, match="unsupported"):
        chunk_pairs(65536, 8, 10, 18, 256, 289, agb.native.AGB_MATH_TC_F16, q, 4 << 30)
    with pytest.raises(agb.native.NativeError, match="below"):
        chunk_pairs(8, 8, 10, 18, 256, 289, agb.native.AGB_MATH_TC_F16, q, 1024)
    per = chunk_pairs(64, 64, 10 ** 6, 18, 256, 289, agb.native.AGB_MATH_TC_F16, q, 1 << 30)
    assert 0 < per < 10 ** 6
    assert q(64, 64, per, 18, 256, 289, agb.native.AGB_MATH_TC_F16) <= 1 << 30 < q(64, 64, per + 1, 18, 256, 289,
                                                                                 agb.native.AGB_MATH_TC_F16)
    with pytest.raises(ValueError, match="math"):
        agb.words_pair_scores(torch.zeros(4, 256, 17, 17), torch.zeros(4, 256, 18), torch.full((4,), 18),
                              np.arange(4), np.arange(4), math="fp32")


@pytest.mark.parametrize("compiling", [False, True])
def test_pair_scores_refuse_cpu_tensors(agb, compiling, monkeypatch):
    if compiling:
        monkeypatch.setattr(torch.compiler, "is_compiling", lambda: True)
    idx = np.arange(4)
    img = torch.zeros(4, 256, 17, 17, requires_grad=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agb.words_pair_scores(img, torch.zeros(4, 256, 18), torch.full((4,), 18), idx, idx)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agb.sentence_pair_scores(torch.zeros(4, 256, requires_grad=True), torch.zeros(4, 256), idx, idx)
    z = torch.zeros(4, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agb.ops.damsm_pairs_train_fwd(torch.zeros(4, 256, 289), torch.zeros(4, 256, 18), z, z, z, 4.0, 5.0,
                                      agb.native.AGB_MATH_TC_F16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agb.ops.sent_cos_pairs_bwd(torch.zeros(4, 256), torch.zeros(4, 256), z, z, 1e-8, torch.zeros(4))


def test_fake_pair_train_ops(agb):
    N = agb.native
    lib = N.lib()
    with FakeTensorMode(allow_non_fake_inputs=False):
        img = torch.empty(6, 256, 289, device="cuda")
        wrd = torch.empty(9, 256, 18, device="cuda")
        lens = torch.empty(9, dtype=torch.int32, device="cuda")
        pi = torch.empty(37, dtype=torch.int32, device="cuda")
        pc = torch.empty(37, dtype=torch.int32, device="cuda")
        for mt in (N.AGB_MATH_TC_F16, N.AGB_MATH_TC_BF16, N.AGB_MATH_TC_F16X2):
            m, ws = torch.ops.agb.damsm_pairs_train_fwd(img, wrd, lens, pi, pc, 4.0, 5.0, mt)
            assert m.shape == (37,) and m.dtype == torch.float32 and m.is_cuda
            assert ws.dtype == torch.uint8 and ws.shape == (lib.agb_damsm_pairs_train_workspace_bytes(6, 9, 37, 18,
                                                                                                      256, 289, mt),)
            dimg, dw = torch.ops.agb.damsm_pairs_bwd(img, wrd, lens, pi, pc, 4.0, 5.0, mt, m, ws, True, True)
            assert dimg.shape == (6, 256, 289) and dw.shape == (9, 18, 256)
            dimg, dw = torch.ops.agb.damsm_pairs_bwd(img, wrd, lens, pi, pc, 4.0, 5.0, mt, m, ws, False, False)
            assert dimg.numel() == 0 and dw.numel() == 0
        with pytest.raises(N.NativeError):
            torch.ops.agb.damsm_pairs_train_fwd(img, torch.empty(9, 256, 33, device="cuda"), lens, pi, pc, 4.0, 5.0,
                                                N.AGB_MATH_TC_F16)
        with pytest.raises(RuntimeError, match="entries"):
            torch.ops.agb.damsm_pairs_train_fwd(img, wrd, lens, pi, pc[:5], 4.0, 5.0, N.AGB_MATH_TC_F16)
        cnn, rnn = torch.empty(6, 256, device="cuda"), torch.empty(9, 256, device="cuda")
        s = torch.ops.agb.sent_cos_pairs_train_fwd(cnn, rnn, pi, pc, 1e-8)
        assert s.shape == (37,) and s.dtype == torch.float32
        dc, dr = torch.ops.agb.sent_cos_pairs_bwd(cnn, rnn, pi, pc, 1e-8, s, True, False)
        assert dc.shape == (6, 256) and dr.numel() == 0


def test_pair_train_ops_registered_without_loading_the_library():
    code = ("import attention_gan_b200 as p, torch; assert p.native._lib is None; "
            "T = p.agb_native.torch_ops; "
            "assert all(hasattr(torch.ops.agb, n) for n in T.PAIR_TRAIN_OPS); "
            "assert p.native._lib is None; print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr
