"""Importable name of the ``attention-gan_b200/`` tree (a hyphen is not a legal module name).

The sub-packages of ``attention-gan_b200/`` are served as ``attention_gan_b200.agb_native``,
``attention_gan_b200.networks``, ``attention_gan_b200.losses`` and ``attention_gan_b200.evaluation`` (this package's
``__path__`` points there).
Nothing is put on ``sys.path``: the reference's own top-level ``networks`` / ``losses`` packages stay importable
next to the drop-ins (its generator, discriminators, encoders, GAN losses are NOT replaced).

    from attention_gan_b200 import AttentionModule, func_attention, WordsLoss, SentenceLoss

To make the reference's own import lines (``from networks.attention import AttentionModule``,
``from losses.words_loss import WordsLoss`` ...; train.py:17,23-24, pretrain_damsm.py:19,25-26,
generator_submodules.py:10) resolve to the B200-native implementations, call ``install()`` once, before or after
the reference's modules are imported; see INTEGRATION.md.
"""
import importlib
import os
import sys

PACKAGE_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "attention-gan_b200")
__path__.append(PACKAGE_DIR)

from .agb_native import native, ops  # noqa: E402,F401
from .agb_native.graph import GraphedStep  # noqa: E402,F401
from .agb_native.pipeline import HostPrefetcher  # noqa: E402,F401
from .networks.attention import AttentionModule, GlobalAttention, func_attention  # noqa: E402,F401
from .networks.region_head import RegionFeatureHead  # noqa: E402,F401
from .losses.words_loss import WordsLoss  # noqa: E402,F401
from .losses.sentence_loss import SentenceLoss  # noqa: E402,F401
from .losses.damsm_loss import DAMSMLoss  # noqa: E402,F401
from .evaluation import DAMSMScorer, mismatched_candidates, r_precision  # noqa: E402,F401
from .losses.pair_scores import sentence_pair_scores, words_pair_scores  # noqa: E402,F401

# reference module -> (native module, names it provides)
_REPLACED = {
    "networks.attention": ("attention_gan_b200.networks.attention", ("AttentionModule", "func_attention")),
    "losses.words_loss": ("attention_gan_b200.losses.words_loss", ("WordsLoss",)),
    "losses.sentence_loss": ("attention_gan_b200.losses.sentence_loss", ("SentenceLoss",)),
}


def install(rebind_loaded: bool = True) -> None:
    """Route the reference's three hot-path modules to the native drop-ins WITHOUT shadowing its packages.

    ``sys.modules['networks.attention']``, ``['losses.words_loss']`` and ``['losses.sentence_loss']`` are pointed at
    the native modules (and set as attributes of the reference's ``networks`` / ``losses`` packages when those are
    importable), so every later ``from networks.attention import AttentionModule`` / ``from .attention import ...``
    gets the native class while ``networks.generator``, ``losses.gen_loss`` etc. still come from the reference.
    With ``rebind_loaded`` the names already imported into loaded modules (``from x import Name`` copies) are
    rebound too, so calling this after ``import train``-style imports also works."""
    old = {}
    for ref_name, (native_name, names) in _REPLACED.items():
        mod = importlib.import_module(native_name)
        prev = sys.modules.get(ref_name)
        if prev is not None and prev is not mod:
            for n in names:
                if hasattr(prev, n):
                    old[id(getattr(prev, n))] = getattr(mod, n)
        sys.modules[ref_name] = mod
        parent_name, _, leaf = ref_name.rpartition(".")
        parent = sys.modules.get(parent_name)
        if parent is None:
            try:
                parent = importlib.import_module(parent_name)
            except ImportError:
                parent = None          # the reference is not on sys.path (yet): the sys.modules entry is enough
        if parent is not None:
            setattr(parent, leaf, mod)
    if rebind_loaded and old:
        for m in list(sys.modules.values()):
            d = getattr(m, "__dict__", None)
            if not d or getattr(m, "__name__", "").startswith("attention_gan_b200"):
                continue
            for k, v in list(d.items()):
                if id(v) in old:
                    d[k] = old[id(v)]
