"""CPU tests (no GPU): the C-ABI library loads and exports every symbol the header declares, the
drop-in modules keep the reference's interface and refuse CPU tensors, and the host-side sharding
logic (world_size 2, gloo) reproduces the single-process loss and gradients."""
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "attngan_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(agb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import attention_gan_b200 as pkg
    lib = pkg.native.lib()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/attngan_b200.h but not exported"
        assert s in pkg.native.SIGNATURES, f"{s} has no ctypes signature"
    assert set(pkg.native.SIGNATURES) == set(syms)
    assert lib.agb_version() == 100
    # pure host queries work without a GPU
    assert lib.agb_contrastive_workspace_bytes(48) == 4 * 48 * 4
    assert lib.agb_damsm_supported(18, 256, 289, pkg.native.AGB_MATH_FP32) == 1
    assert lib.agb_damsm_supported(65, 256, 289, pkg.native.AGB_MATH_FP32) == 0
    assert lib.agb_damsm_workspace_bytes(48, 48, 18, 256, 289, 0) > 0
    assert lib.agb_word_attn_bwd_workspace_bytes(2, 32, 4096, 256, 18) > 0


def test_argument_errors_are_reported_without_a_gpu():
    import attention_gan_b200 as pkg
    lib = pkg.native.lib()
    rc = lib.agb_contrastive_fwd(None, 4, None, None, 10.0, 5.0, 0, 4, None, None, None, 0, None)
    assert rc == -1 and b"null" in lib.agb_last_error()
    rc = lib.agb_word_attn_fwd(None, None, 0, 0, 0, None, None, None, 0, None, None, 1, 1, 1, 1, 65, 0, 1, None)
    assert rc == -2 and b"T=65" in lib.agb_last_error()


def test_dropin_interface_matches_reference_signatures():
    import inspect
    import attention_gan_b200 as pkg
    m = pkg.AttentionModule(nc_in=32, emb_dim=256)
    assert list(m.state_dict().keys()) == ["conv1.weight"]            # Generator.pkl compatibility
    assert tuple(m.conv1.weight.shape) == (32, 256, 1, 1) and m.conv1.bias is None
    assert m.mask is None
    assert list(inspect.signature(m.forward).parameters) == ["images", "words", "scaled"]
    assert list(inspect.signature(pkg.func_attention).parameters) == ["query", "context", "gamma1", "scaled"]
    wl = pkg.WordsLoss(torch.device("cpu"))
    assert (wl.gamma1, wl.gamma2, wl.gamma3, wl.wlambda) == (4.0, 5.0, 10.0, 5.0)
    assert list(inspect.signature(wl.get_loss).parameters) == ["img_features", "words_emb", "labels", "cap_lens", "class_ids"]
    sl = pkg.SentenceLoss(torch.device("cpu"))
    assert (sl.gamma3, sl.slambda) == (10.0, 5.0)
    assert list(inspect.signature(sl.get_loss).parameters) == ["cnn_code", "rnn_code", "labels", "class_ids", "eps"]
    x1, x2 = torch.randn(5, 7), torch.randn(5, 7)
    torch.testing.assert_close(wl.cosine_similarity(x1, x2), torch.nn.functional.cosine_similarity(x1, x2))
    # importing the package does not shadow the reference's top-level packages
    assert not any(p.rstrip("/").endswith("attention-gan_b200") for p in sys.path)


_INSTALL_CHILD = r'''
import os, sys
ref = sys.argv[1]
order = sys.argv[2]
sys.path.insert(0, ref)
sys.path.insert(0, sys.argv[3])
if order == "after":                      # the reference's modules are imported first, install() rebinds them
    import networks.generator_submodules as gs
    import losses.words_loss as ref_wl
    from losses.words_loss import WordsLoss as RefWordsLoss
import attention_gan_b200 as agb
agb.install()
from networks.attention import AttentionModule, func_attention
from losses.words_loss import WordsLoss
from losses.sentence_loss import SentenceLoss
assert AttentionModule is agb.AttentionModule and func_attention is agb.func_attention
assert WordsLoss is agb.WordsLoss and SentenceLoss is agb.SentenceLoss
# the rest of the reference's packages still resolve to the reference
import networks.generator_submodules as gs
import losses.gen_loss, losses.KL_loss, networks.rnn_encoder
assert os.path.realpath(gs.__file__).startswith(os.path.realpath(ref))
assert os.path.realpath(losses.gen_loss.__file__).startswith(os.path.realpath(ref))
assert gs.AttentionModule is agb.AttentionModule, "GenNextStage would still build the reference attention"
import networks, losses
assert networks.attention.AttentionModule is agb.AttentionModule and losses.words_loss.WordsLoss is agb.WordsLoss
print("install ok", order)
'''


def _fake_reference(tmp):
    """a miniature tree with the reference's package layout and import lines (generator_submodules.py:10,
    train.py:17,23-24)"""
    files = {
        "networks/__init__.py": "",
        "networks/attention.py": "class AttentionModule: pass\ndef func_attention(*a): raise RuntimeError('reference')\n",
        "networks/generator_submodules.py": "from .attention import AttentionModule\nclass GenNextStage: pass\n",
        "networks/rnn_encoder.py": "class RNNEncoder: pass\n",
        "losses/__init__.py": "",
        "losses/words_loss.py": "from networks.attention import func_attention\nclass WordsLoss: pass\n",
        "losses/sentence_loss.py": "class SentenceLoss: pass\n",
        "losses/gen_loss.py": "class GenLoss: pass\n",
        "losses/KL_loss.py": "class KLLoss: pass\n",
    }
    for rel, text in files.items():
        path = os.path.join(tmp, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            fh.write(text)
    return tmp


@pytest.mark.parametrize("order", ["before", "after"])
@pytest.mark.parametrize("tree", ["fake", "real"])
def test_install_routes_reference_imports_without_shadowing(tmp_path, order, tree):
    """ADVICE r1: the drop-ins must not shadow the reference's `networks` / `losses` packages.  install() swaps
    exactly the three hot-path modules; everything else of the reference stays importable."""
    import subprocess
    if tree == "real":
        # the original package tree cannot be stored here, so this case runs only against a checkout named by
        # AGB_REFERENCE_ROOT; the "fake" case carries the reference's import lines that install() has to reroute
        ref = os.environ.get("AGB_REFERENCE_ROOT", "")
        if not ref or not os.path.isdir(os.path.join(ref, "networks")):
            pytest.skip("needs AGB_REFERENCE_ROOT: a checkout of the original project")
    else:
        ref = _fake_reference(str(tmp_path))
    r = subprocess.run([sys.executable, "-c", _INSTALL_CHILD, ref, order, ROOT], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "install ok" in r.stdout, r.stdout + r.stderr


def test_no_cpu_fallback():
    import attention_gan_b200 as pkg
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.func_attention(torch.zeros(1, 4, 2), torch.zeros(1, 4, 2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.WordsLoss("cpu").get_loss(torch.zeros(2, 4, 2, 2), torch.zeros(2, 4, 3), torch.arange(2),
                                      torch.tensor([3, 3]), None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.SentenceLoss("cpu").get_loss(torch.zeros(2, 4), torch.zeros(2, 4), torch.arange(2), None)


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.join(ROOT, "attention-gan_b200")
    for base, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(base, f)).read()
                assert "oracle" not in src.replace("oracle_ops", ""), f"{f} mentions the oracle"


# ---- world_size-2 gloo test of the sharded exchange ------------------------------------------
def _single_process_reference(seed, ragged=False):
    sys.path.insert(0, ROOT)
    from oracle import closed_form as cf
    from oracle import ref_port as rp
    img, wrd, cnn, rnn, labels, lens, cls = rp.synth_damsm(6, T=5, D=16, hw=3, seed=seed, n_classes=3)
    if ragged:                      # the second rank's captions are all shorter than T: its RNN pads to T - 1 only
        lens[3:] = torch.clamp(lens[3:], max=4)
    B, D = img.shape[:2]
    wl, _, dc, dw = cf.words_loss_fwd_bwd(img.numpy().reshape(B, D, -1), wrd.numpy(), labels.numpy(), lens.numpy(), cls)
    sl, _, dcnn, drnn = cf.sentence_loss_fwd_bwd(cnn.numpy(), rnn.numpy(), labels.numpy(), cls)
    return (img, wrd, cnn, rnn, labels, lens, cls), (wl, sl, dc.reshape(img.shape), dw, dcnn, drnn)


def _worker(rank, world, port, seed, fused, out, ragged=False):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sys.path.insert(0, ROOT)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_ops
        from attention_gan_b200.losses import damsm_core as core
        (img, wrd, cnn, rnn, labels, lens, cls), _ = _single_process_reference(seed, ragged)
        n = img.shape[0] // world
        sl = slice(rank * n, rank * n + n)
        im = img[sl].clone().requires_grad_(True)
        wd = wrd[sl].clone()
        if ragged and rank == 1:
            wd = wd[:, :, :4].clone()                     # T differs per rank (rnn_encoder.py:89-92)
        wd.requires_grad_(True)
        cn = cnn[sl].clone().requires_grad_(True)
        rn = rnn[sl].clone().requires_grad_(True)
        loc_labels = torch.arange(n)
        wcfg = core.DamsmConfig(group=dist.group.WORLD, ops=oracle_ops)
        scfg = core.DamsmConfig(group=dist.group.WORLD, ops=oracle_ops)
        if fused:
            wl, sls, att = core.damsm_losses(im, cn, wd, rn, loc_labels, lens[sl], cls[sl], wcfg, scfg)
        else:
            wl, att = core.words_loss(im, wd, loc_labels, lens[sl], cls[sl], wcfg)
            sls = core.sentence_loss(cn, rn, loc_labels, cls[sl], scfg)
        (wl + sls).backward()
        assert att.shape[1] == wd.shape[2]
        maps = core.split_att_maps(att, lens[sl], 3, 3)
        out[rank] = dict(wl=wl.item(), sl=sls.item(), dimg=im.grad.numpy(), dwords=wd.grad.numpy(),
                         dcnn=cn.grad.numpy(), drnn=rn.grad.numpy(), maps=[m.numpy() for m in maps])
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("fused", [False, True])
def test_sharded_losses_equal_single_process(fused):
    world, seed = 2, 11
    port = 29500 + (os.getpid() % 2000) + (7 if fused else 0)
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, seed, fused, out), nprocs=world, join=True)
    (img, wrd, cnn, rnn, labels, lens, cls), (wl0, sl0, dc0, dw0, dcnn0, drnn0) = _single_process_reference(seed)
    n = img.shape[0] // world
    sys.path.insert(0, ROOT)
    from oracle import ref_port as rp
    _, ref_maps = rp.words_loss(img.double(), wrd.double(), labels, lens, cls)
    for r in range(world):
        o = out[r]
        sl = slice(r * n, r * n + n)
        assert abs(o["wl"] - wl0) < 1e-5 * abs(wl0) and abs(o["sl"] - sl0) < 1e-5 * abs(sl0)
        np.testing.assert_allclose(o["dimg"], dc0[sl], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(o["dwords"], dw0[sl], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(o["dcnn"], dcnn0[sl], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(o["drnn"], drnn0[sl], rtol=1e-4, atol=1e-6)
        for j, m in enumerate(o["maps"]):
            np.testing.assert_allclose(m, ref_maps[r * n + j].numpy(), rtol=1e-5, atol=1e-7)


def test_sharded_losses_with_different_caption_padding_per_rank():
    """ADVICE r1: the reference's RNN pads to the LOCAL batch's longest caption, so T can differ per rank; the
    exchange pads to the agreed maximum and slices the word gradients back"""
    world, seed = 2, 13
    port = 29500 + (os.getpid() % 2000) + 19
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, seed, True, out, True), nprocs=world, join=True)
    (img, wrd, cnn, rnn, labels, lens, cls), (wl0, sl0, dc0, dw0, dcnn0, drnn0) = _single_process_reference(seed, True)
    n = img.shape[0] // world
    for r in range(world):
        o = out[r]
        sl = slice(r * n, r * n + n)
        assert abs(o["wl"] - wl0) < 1e-5 * abs(wl0) and abs(o["sl"] - sl0) < 1e-5 * abs(sl0)
        np.testing.assert_allclose(o["dimg"], dc0[sl], rtol=1e-4, atol=1e-6)
        T_r = 4 if r == 1 else 5
        assert o["dwords"].shape[2] == T_r
        np.testing.assert_allclose(o["dwords"], dw0[sl][:, :, :T_r], rtol=1e-4, atol=1e-6)


def test_options_and_helpers_without_a_gpu():
    """agb_set_option validates names on the host; the graph / prefetch helpers refuse to run without CUDA"""
    import attention_gan_b200 as pkg
    lib = pkg.native.lib()
    assert lib.agb_set_option(b"damsm_chunk_mb", 16384) == 0
    assert lib.agb_set_option(b"no_such_option", 1) == -1 and b"unknown option" in lib.agb_last_error()
    with pytest.raises(pkg.native.NativeError):
        pkg.native.set_option("no_such_option", 1)
    # workspace sizes follow the staging budget (the tests force the multi-chunk path this way)
    big = lib.agb_damsm_workspace_bytes(64, 64, 18, 256, 289, pkg.native.AGB_MATH_TC_F16)
    pkg.native.set_option("damsm_chunk_mb", 11)
    small = lib.agb_damsm_workspace_bytes(64, 64, 18, 256, 289, pkg.native.AGB_MATH_TC_F16)
    pkg.native.set_option("damsm_chunk_mb", 16384)
    assert 0 < small < big
    # split precision needs the lo operand copies
    assert lib.agb_damsm_workspace_bytes(64, 64, 18, 256, 289, pkg.native.AGB_MATH_TC_F16X2) > big
    assert lib.agb_damsm_supported(18, 256, 289, pkg.native.AGB_MATH_TC_F16X2) == 1
    assert lib.agb_region_head_workspace_bytes(4, 768, 256, 289) > 0
    assert lib.agb_region_head_workspace_bytes(4, 100, 96, 289) == 0
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            pkg.GraphedStep(lambda: None)
        with pytest.raises(RuntimeError, match="CUDA"):
            pkg.HostPrefetcher("cuda")
