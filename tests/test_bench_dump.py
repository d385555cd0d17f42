"""bench.py --dump-outputs: the outputs of the last timed step, within the size budget, sampled at the same positions
on every run, and equal to the oracle on the benchmark's own inputs."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_host_outputs_budget_dtypes_and_fixed_sample():
    outs = {"big": torch.arange(12 << 20, dtype=torch.float64).reshape(3, -1), "mid": torch.randn(1 << 20),
            "loss": torch.tensor(2.5), "half": torch.randn(3, 5).bfloat16()}
    a, b = bench.host_outputs(outs), bench.host_outputs(outs)
    assert list(a) == list(outs)
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_BYTES
    big = a["big"]                                                       # element i holds i: the sampled positions
    assert big.dtype == np.float64 and big.ndim == 1 and (12 << 20) // 3 < big.size < 12 << 20
    assert (np.diff(big) > 0).all() and big[-1] < 12 << 20               # distinct, in order, of the output
    assert all(np.array_equal(a[k], b[k]) for k in outs)                 # the same positions every time
    assert a["mid"].dtype == np.float32 and np.array_equal(a["mid"], outs["mid"].numpy())   # within budget: whole
    assert a["loss"].shape == () and a["loss"] == np.float32(2.5)
    assert a["half"].dtype == np.float32 and np.array_equal(a["half"], outs["half"].float().numpy())


def rel(x, ref):
    return np.abs(x - ref).max() / np.abs(ref).max()


def dump(tmp_path, *args):
    """bench.py ... --dump-outputs: {name: array}"""
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--no-secondary", "--dump-outputs", str(out), *args],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return {f[:-4]: np.load(out / f) for f in os.listdir(out)}


@pytest.mark.gpu
def test_dumped_cfg2_outputs_match_the_oracle(tmp_path):
    """the DAMSM step, replayed from a CUDA graph"""
    from oracle import closed_form as cf
    d = dump(tmp_path, "--workload", "cfg2")
    assert set(d) == {"words_loss", "sentence_loss", "att_maps", "d_img_features", "d_words_emb", "d_cnn_code",
                      "d_rnn_code"}
    B = 48
    img, wrd, cnn, rnn, lens, cls = bench.damsm_inputs(B)
    labels = np.arange(B)
    wl0, _, dc0, dw0 = cf.words_loss_fwd_bwd(img.numpy().reshape(B, 256, -1), wrd.numpy().transpose(0, 2, 1), labels,
                                             lens.numpy(), cls.numpy())
    sl0, _, dcnn0, drnn0 = cf.sentence_loss_fwd_bwd(cnn.numpy(), rnn.numpy(), labels, cls.numpy())
    assert abs(d["words_loss"] - wl0) <= 1e-4 * abs(wl0)                # tensor-core default math at batch 48
    assert abs(d["sentence_loss"] - sl0) <= 1e-5 * abs(sl0)
    assert d["att_maps"].shape == (B, 18, 17, 17)
    assert rel(d["d_img_features"], dc0.reshape(B, 256, 17, 17)) < 5e-3
    assert rel(d["d_words_emb"], dw0.transpose(0, 2, 1)) < 5e-3
    assert rel(d["d_cnn_code"], dcnn0) < 1e-4 and rel(d["d_rnn_code"], drnn0) < 1e-4


@pytest.mark.gpu
def test_dumped_cfg1_outputs_match_the_oracle(tmp_path):
    """the attention step, timed eagerly (--no-graph): the outputs of its last eager step"""
    from oracle import closed_form as cf
    from oracle import ref_port as rp
    d = dump(tmp_path, "--workload", "cfg1", "--no-graph")
    assert set(d) == {"ctx_64", "attn_64", "d_images_64", "d_weight_64", "d_words"}
    B, C, E, T, hw = 16, 32, 256, 18, 64
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=0)      # bench.py's inputs
    dctx = torch.randn(B, C, hw, hw, generator=torch.Generator().manual_seed(1))
    h, w, W, m = images.numpy().reshape(B, C, -1), words.numpy(), weight.numpy().reshape(C, E), mask.numpy()
    ctx0, attn0, _ = cf.word_attention_fwd(h, w, W, m, True)
    dh0, dw0, dW0 = cf.word_attention_bwd(h, w, W, m, dctx.numpy().reshape(B, C, -1), None, True)
    assert rel(d["ctx_64"], ctx0.reshape(B, C, hw, hw)) < 1e-4
    assert rel(d["attn_64"], attn0.reshape(B, T, hw, hw)) < 1e-4
    assert rel(d["d_images_64"], dh0.reshape(B, C, hw, hw)) < 1e-4
    assert rel(d["d_words"], dw0.transpose(0, 2, 1)) < 1e-4
    assert rel(d["d_weight_64"], dW0.reshape(C, E, 1, 1)) < 1e-4


@pytest.mark.gpu
def test_dumped_pretrain_step_outputs(tmp_path):
    """the whole pretraining step: its loss and every trainable parameter after the last step"""
    from attention_gan_b200.pretrain import RegionHeads, TextEncoder
    d = dump(tmp_path, "--workload", "cfg4step", "--batch", "64")
    shapes = {f"RNNEncoder.{k}": tuple(v.shape) for k, v in TextEncoder(vocabsize=1, nhidden=256).state_dict().items()}
    shapes.update({f"CNNEncoder.{k}": tuple(v.shape) for k, v in RegionHeads(256).state_dict().items()})
    assert set(d) == {"loss"} | set(shapes)
    for k, shape in shapes.items():
        assert d[k].shape[1:] == shape[1:] and np.isfinite(d[k]).all(), k    # the embedding's rows: the vocabulary
    assert d["loss"].shape == () and np.isfinite(d["loss"]) and d["loss"] > 0
    torch.manual_seed(0)                                                 # DamsmPretrainStep's seed: its initial weights
    init = TextEncoder(vocabsize=d["RNNEncoder.embedding.weight"].shape[0], nhidden=256).state_dict()
    for k, v in init.items():                                            # Adam (lr 2e-3) moved them, a little
        assert 0 < np.abs(d[f"RNNEncoder.{k}"] - v.numpy()).max() < 0.5, k
