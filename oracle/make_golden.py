"""Generate tests/golden/*.npz by running the UNMODIFIED reference (TEST INFRASTRUCTURE).

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    python oracle/make_golden.py

It imports ``networks.attention``, ``losses.words_loss`` and ``losses.sentence_loss`` from
``/root/reference`` and records, for seeded inputs, the values and the autograd gradients the
reference produces.  The one shim: torch 2.11 rejects the uint8 ``torch.ByteTensor`` masks the
reference builds for ``class_ids`` (words_loss.py:90,95; sentence_loss.py:24,43), so those two
modules see a ``torch`` proxy whose ``ByteTensor(a)`` returns a bool tensor.  Nothing under
/root/reference is modified or copied.

Each fixture stores inputs (fp32-representable values), reference outputs computed in fp64 (the
"exact" answer for those inputs) and the loss computed by the reference in its native fp32.
"""
from __future__ import annotations

import os
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("AGB_REFERENCE_ROOT", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")

sys.path.insert(0, ROOT)
from oracle import ref_port  # noqa: E402  (input generators only)


def load_reference():
    sys.path.insert(0, REF)
    warnings.filterwarnings("ignore", message="Implicit dimension choice")
    import networks.attention as ratt          # noqa
    import losses.words_loss as rwl            # noqa
    import losses.sentence_loss as rsl         # noqa

    class _TorchProxy(types.ModuleType):
        def __getattr__(self, name):
            return getattr(torch, name)

        @staticmethod
        def ByteTensor(a):
            return torch.from_numpy(np.ascontiguousarray(a)).bool()

    proxy = _TorchProxy("torch_proxy")
    rwl.torch = proxy
    rsl.torch = proxy
    return ratt, rwl, rsl


def npy(t):
    """numpy copy; large fp64 arrays are stored as fp32 to keep the fixtures small (the small
    cases keep full fp64 so the oracle can be pinned to 1e-12 there)."""
    a = t.detach().cpu().numpy()
    if a.dtype == np.float64 and a.size > 20000:
        a = a.astype(np.float32)
    return a


def golden_attention(ratt, name, B, C, E, T, hw, seed, scaled):
    images, words, weight, mask, lens = ref_port.synth_attention(B, C, E, T, hw, seed)
    g = torch.Generator().manual_seed(seed + 1000)
    dctx = torch.randn(B, C, hw, hw, generator=g)
    dattn = torch.randn(B, T, hw, hw, generator=g) * 0.1
    out = {}
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        mod = ratt.AttentionModule(nc_in=C, emb_dim=E).to(dt)
        with torch.no_grad():
            mod.conv1.weight.copy_(weight.to(dt))
        im = images.to(dt).clone().requires_grad_(True)
        wd = words.to(dt).clone().requires_grad_(True)
        mod.apply_mask(mask)
        ctx, attn = mod(im, wd, scaled=scaled)
        (ctx * dctx.to(dt)).sum().add((attn * dattn.to(dt)).sum()).backward()
        out[f"ctx_{tag}"] = npy(ctx)
        out[f"attn_{tag}"] = npy(attn)
        if tag == "f64":
            out["dimages"] = npy(im.grad)
            out["dwords"] = npy(wd.grad)
            out["dweight"] = npy(mod.conv1.weight.grad)
    np.savez_compressed(os.path.join(OUT, name + ".npz"),
                        images=npy(images), words=npy(words.contiguous()), weight=npy(weight),
                        mask=npy(mask), dctx=npy(dctx), dattn=npy(dattn),
                        scaled=np.array(scaled), **out)


def golden_func_attention(ratt, name, B, D, L, hw, seed, gamma1):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(B, D, L, generator=g)
    c = torch.randn(B, D, hw, hw, generator=g)
    dwc = torch.randn(B, D, L, generator=g)
    q64 = q.double().requires_grad_(True)
    c64 = c.double().requires_grad_(True)
    wc, attn = ratt.func_attention(q64, c64, gamma1=gamma1)
    (wc * dwc.double()).sum().backward()
    np.savez_compressed(os.path.join(OUT, name + ".npz"), query=npy(q), context=npy(c), dwc=npy(dwc),
                        gamma1=np.array(gamma1), wc=npy(wc), attn=npy(attn),
                        dquery=npy(q64.grad), dcontext=npy(c64.grad))


def golden_damsm(rwl, rsl, name, B, T, D, hw, seed, n_classes, full_len=False, trained_like=False,
                 gammas=(4.0, 5.0, 10.0), lambdas=(5.0, 5.0)):
    img, wrd, cnn, rnn, labels, lens, cls = ref_port.synth_damsm(
        B, T, D, hw, seed, full_len=full_len, n_classes=n_classes, trained_like=trained_like)
    dev = torch.device("cpu")
    out = {}
    for tag, dt in (("f64", torch.float64), ("f32", torch.float32)):
        im = img.to(dt).clone().requires_grad_(True)
        wd = wrd.to(dt).clone().requires_grad_(True)
        cn = cnn.to(dt).clone().requires_grad_(True)
        rn = rnn.to(dt).clone().requires_grad_(True)
        WL = rwl.WordsLoss(dev, gamma1=gammas[0], gamma2=gammas[1], gamma3=gammas[2], wlambda=lambdas[0])
        SL = rsl.SentenceLoss(dev, gamma3=gammas[2], slambda=lambdas[1])
        wloss, maps = WL.get_loss(im, wd, labels, lens, cls)
        sloss = SL.get_loss(cn, rn, labels, cls)
        (wloss + sloss).backward()
        out[f"wloss_{tag}"] = npy(wloss)
        out[f"sloss_{tag}"] = npy(sloss)
        if tag == "f64":
            assert len(maps) == B and maps[0].shape == (1, int(lens[0]), hw, hw)
            packed = np.zeros((B, T, hw, hw), np.float32 if B * T * hw * hw > 20000 else np.float64)
            for i, m in enumerate(maps):
                packed[i, : int(lens[i])] = npy(m)[0]
            out["att_maps"] = packed
            out["dimg"] = npy(im.grad)
            out["dwords"] = npy(wd.grad)
            out["dcnn"] = npy(cn.grad)
            out["drnn"] = npy(rn.grad)
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"), img=npy(img), words=npy(wrd.contiguous()), cnn=npy(cnn),
        rnn=npy(rnn), labels=npy(labels), cap_lens=npy(lens),
        class_ids=(np.array([-1]) if cls is None else cls), has_class_ids=np.array(cls is not None),
        gammas=np.array(gammas), lambdas=np.array(lambdas), **out)


def golden_text_encoder(name, seed):
    """the text encoder's fixture.  The reference's RNNEncoder is stated in fp64 by oracle/closed_form.py
    (text_encoder_fwd) on seeded weights (ref_port.synth_text_encoder); no reference import is needed, so
    ``python oracle/make_golden.py text_encoder`` writes only this file.  tests/test_pretrain_cpu.py checks the
    reference itself against it whenever AGB_REFERENCE_ROOT names a checkout."""
    from attention_gan_b200.pretrain import SyntheticBedroomCaptions
    from oracle import closed_form
    d = SyntheticBedroomCaptions(64, seed=1)
    caps, lens, _ = d.batch(0, 8)
    ragged = torch.tensor([7, 3, 5, 2, 7, 6, 4, 2])
    sd = ref_port.synth_text_encoder(d.vocab_size, seed=seed)
    sd64 = {k: v.numpy() for k, v in sd.items()}
    out = {}
    for tag, ln in (("full", lens), ("ragged", ragged)):
        out[f"words_{tag}"], out[f"sent_{tag}"] = closed_form.text_encoder_fwd(sd64, caps.numpy(), ln.numpy())
    np.savez_compressed(os.path.join(OUT, name + ".npz"), captions=caps.numpy(), cap_lens=lens.numpy(),
                        cap_lens_ragged=ragged.numpy(), vocab=np.array(d.vocab_size), seed=np.array(seed),
                        weight_abs_sums=np.array([float(v.double().abs().sum()) for v in sd.values()]), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    if sys.argv[1:] == ["text_encoder"]:
        golden_text_encoder("text_encoder", seed=1)
        return
    ratt, rwl, rsl = load_reference()
    # generator attention (a3/a4)
    golden_attention(ratt, "attn_small_scaled", B=3, C=8, E=16, T=5, hw=6, seed=1, scaled=True)
    golden_attention(ratt, "attn_small_unscaled", B=3, C=8, E=16, T=5, hw=6, seed=2, scaled=False)
    golden_attention(ratt, "attn_cfg1_slice", B=2, C=32, E=256, T=18, hw=16, seed=3, scaled=True)
    golden_attention(ratt, "attn_odd", B=2, C=12, E=40, T=23, hw=7, seed=4, scaled=True)
    # functional attention (a5)
    golden_func_attention(ratt, "func_small", B=3, D=16, L=5, hw=4, seed=5, gamma1=4.0)
    golden_func_attention(ratt, "func_real", B=1, D=256, L=18, hw=17, seed=6, gamma1=4.0)
    # DAMSM losses (a8/a9/a10)
    golden_damsm(rwl, rsl, "damsm_small", B=6, T=7, D=32, hw=5, seed=7, n_classes=None)
    golden_damsm(rwl, rsl, "damsm_small_cls", B=6, T=7, D=32, hw=5, seed=8, n_classes=3)
    golden_damsm(rwl, rsl, "damsm_real_cls", B=3, T=18, D=256, hw=17, seed=9, n_classes=2)
    golden_damsm(rwl, rsl, "damsm_real_trained", B=3, T=18, D=256, hw=17, seed=10, n_classes=None,
                 trained_like=0.12)
    golden_damsm(rwl, rsl, "damsm_gammas", B=5, T=6, D=64, hw=4, seed=11, n_classes=4,
                 gammas=(2.0, 3.0, 7.0), lambdas=(1.5, 0.5), full_len=True)
    golden_text_encoder("text_encoder", seed=1)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
