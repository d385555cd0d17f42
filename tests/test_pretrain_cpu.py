"""CPU tests of the DAMSM pretraining harness (SURVEY 8 f4): the synthetic caption generator has the structure of the
reference's hierarchical-cluster captions (data/bedrooms.py:241-304) and the encoder modules keep the reference's
state-dict names and arithmetic (networks/rnn_encoder.py, networks/cnn_encoder.py:54-64)."""
import os
import sys

import numpy as np
import pytest
import torch

from attention_gan_b200.pretrain import RegionHeads, SyntheticBedroomCaptions, TextEncoder, hierarchical_k_values
from conftest import load_golden
from oracle import ref_port as rp

# a checkout of the original project (as for oracle/make_golden.py); the live comparison with it skips without one
REF = os.environ.get("AGB_REFERENCE_ROOT", "")


def test_k_values_follow_the_reference_recipe():
    # pretrain_damsm.py:57: max_vocab_size=1000, min_clusters=5 -> 7 levels, 990 words at most
    assert hierarchical_k_values(1000, 5) == [7, 15, 31, 62, 125, 250, 500]
    assert sum(hierarchical_k_values(1000, 5)) == 990
    assert hierarchical_k_values(600, 5) == [9, 18, 37, 75, 150, 300]          # the method's own defaults


def test_synthetic_captions_have_the_reference_structure():
    d = SyntheticBedroomCaptions(5000, seed=3)
    ks = d.k_values
    assert d.captions.shape == (5000, 7) and d.captions.dtype == torch.int64
    assert torch.all(d.lengths == 7)                                            # fixed 7-token captions
    assert d.vocab_size <= 990 and int(d.captions.max()) == d.vocab_size - 1
    assert int(d.class_ids.max()) < 500 and int(d.class_ids.min()) == 0
    lab = d.cluster_labels
    for l, k in enumerate(ks):
        assert lab[:, l].min() >= 0 and lab[:, l].max() < k
    # nested: the finest cluster determines every coarser one (cuts of one dendrogram)
    for l in range(len(ks) - 1, 0, -1):
        pairs = set(zip(lab[:, l].tolist(), lab[:, l - 1].tolist()))
        assert len(pairs) == len(set(lab[:, l].tolist()))
    # class id <-> finest cluster is a bijection; same class => same caption
    caps = d.captions.numpy()
    by_class = {}
    for c, row in zip(d.class_ids.tolist(), caps):
        assert by_class.setdefault(c, tuple(row)) == tuple(row)
    # word indices in order of first occurrence (Vocab._addWord, bedrooms.py:94-99)
    assert caps[0].tolist() == list(range(7))
    seen = -1
    for v in caps.reshape(-1):
        assert v <= seen + 1
        seen = max(seen, int(v))
    # seeded
    assert torch.equal(SyntheticBedroomCaptions(64, seed=5).captions, SyntheticBedroomCaptions(64, seed=5).captions)
    assert not torch.equal(SyntheticBedroomCaptions(64, seed=5).captions, SyntheticBedroomCaptions(64, seed=6).captions)


def test_encoder_state_dicts_keep_the_reference_names():
    t = TextEncoder(vocabsize=990, nhidden=256)
    assert list(t.state_dict().keys()) == [
        "embedding.weight", "rnn.weight_ih_l0", "rnn.weight_hh_l0", "rnn.bias_ih_l0", "rnn.bias_hh_l0",
        "rnn.weight_ih_l0_reverse", "rnn.weight_hh_l0_reverse", "rnn.bias_ih_l0_reverse", "rnn.bias_hh_l0_reverse"]
    assert tuple(t.embedding.weight.shape) == (990, 300) and tuple(t.rnn.weight_ih_l0.shape) == (512, 300)
    assert float(t.embedding.weight.abs().max()) <= 0.1
    h = RegionHeads(256)
    sd = h.state_dict()
    assert list(sd.keys()) == ["emb_features.weight", "emb_cnn_code.weight", "emb_cnn_code.bias"]
    assert tuple(sd["emb_features.weight"].shape) == (256, 768, 1, 1) and tuple(sd["emb_cnn_code.weight"].shape) == (256, 2048)
    f, c = h(torch.randn(2, 768, 17, 17), torch.randn(2, 2048))
    assert f.shape == (2, 256, 17, 17) and c.shape == (2, 256)


def test_text_encoder_matches_the_reference_fixture():
    """TextEncoder == tests/golden/text_encoder.npz: the reference's RNNEncoder stated in fp64 on seeded weights
    (oracle/closed_form.py text_encoder_fwd, written by oracle/make_golden.py); full-length captions through the
    packed and the fixed-length path, ragged lengths through the packed path"""
    g = load_golden("text_encoder")
    sd = rp.synth_text_encoder(int(g["vocab"]), seed=int(g["seed"]))
    np.testing.assert_allclose([float(v.double().abs().sum()) for v in sd.values()], g["weight_abs_sums"], rtol=1e-12)
    mine = TextEncoder(vocabsize=int(g["vocab"]), nhidden=256).eval()
    assert list(mine.state_dict().keys()) == list(sd.keys())
    mine.load_state_dict(sd)
    caps = torch.from_numpy(g["captions"])
    cases = [("full", g["cap_lens"], False), ("full", g["cap_lens"], True), ("ragged", g["cap_lens_ragged"], False)]
    with torch.no_grad():
        for tag, lens, fixed in cases:
            w, s = mine(caps, torch.from_numpy(lens), fixed_length=fixed)
            assert w.shape == g[f"words_{tag}"].shape == (8, 256, 7)
            np.testing.assert_allclose(w.numpy(), g[f"words_{tag}"], rtol=0, atol=1e-6)
            np.testing.assert_allclose(s.numpy(), g[f"sent_{tag}"], rtol=0, atol=1e-6)


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "networks")),
                    reason="needs AGB_REFERENCE_ROOT: a checkout of the original project")
def test_text_encoder_equals_the_reference_rnn_encoder():
    import subprocess
    code = r'''
import sys, warnings, torch
warnings.filterwarnings("ignore")
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
from networks.rnn_encoder import RNNEncoder
from attention_gan_b200.pretrain import TextEncoder, SyntheticBedroomCaptions
d = SyntheticBedroomCaptions(64, seed=1)
ref = RNNEncoder(vocabsize=d.vocab_size, nhidden=256).eval()
mine = TextEncoder(vocabsize=d.vocab_size, nhidden=256).eval()
assert list(ref.state_dict().keys()) == list(mine.state_dict().keys())
mine.load_state_dict(ref.state_dict())
caps, lens, _ = d.batch(0, 8)
w0, s0 = ref(caps, lens)
for fixed in (False, True):
    w1, s1 = mine(caps, lens, fixed_length=fixed)
    assert w1.shape == w0.shape == (8, 256, 7) and (w1 - w0).abs().max() < 1e-6 and (s1 - s0).abs().max() < 1e-6
# ragged lengths through the packed path, like a real caption batch
lens2 = torch.tensor([7, 3, 5, 2, 7, 6, 4, 2])
w0, s0 = ref(caps, lens2); w1, s1 = mine(caps, lens2)
assert (w1 - w0).abs().max() < 1e-6 and (s1 - s0).abs().max() < 1e-6
# the reference on the stored fixture's weights and captions reproduces it
import numpy as np
from oracle import ref_port as rp
g = np.load(sys.argv[3])
ref = RNNEncoder(vocabsize=int(g["vocab"]), nhidden=256).eval()
ref.load_state_dict(rp.synth_text_encoder(int(g["vocab"]), seed=int(g["seed"])))
for tag in ("full", "ragged"):
    lens = g["cap_lens" if tag == "full" else "cap_lens_ragged"]
    w0, s0 = ref(torch.from_numpy(g["captions"]), torch.from_numpy(lens))
    assert np.abs(w0.detach().numpy() - g["words_" + tag]).max() < 1e-6
    assert np.abs(s0.detach().numpy() - g["sent_" + tag]).max() < 1e-6
print("encoder ok")
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    fixture = os.path.join(root, "tests", "golden", "text_encoder.npz")
    r = subprocess.run([sys.executable, "-c", code, REF, root, fixture], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "encoder ok" in r.stdout, r.stdout + r.stderr
