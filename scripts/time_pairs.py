"""Times pair-list scoring (DAMSMScorer.words_pairs / words(by="caption")) against the fixed-K candidate call and
against what a user does without it.

    python scripts/time_pairs.py [--n 2048] [--k 100] [--iters 20] [--warmup 3] [--out FILE]

Seeded synthetic inputs as in scripts/time_candidates.py: N images = N captions (T = 18, lengths U{2..18},
17 x 17 regions, words in the text encoder's transposed layout), class ids U{0..499}, K = 100 candidates from
mismatched_candidates.  For each math mode ("f16", "f16x2"), every result is checked bit for bit before it is timed:
  (a) words_pairs on the image -> text candidate list (P = N K pairs in candidate order) against words on the same
      candidates: the cost of grouping the pairs by image and scattering m back;
  (b) words(by="caption") (text -> image: each caption against K images) against the dense N x N forward gathered;
  (c) the same P pairs shuffled, and P pairs that all name one image;
  (d) words_pairs with att_maps=True on the list of (a).
The scorer's workspace budget holds every call in one launch.  CUDA events around every iteration, the L2 flushed
between iterations outside the events (a 256 MiB write).  Prints one JSON line; GPU name, power limit and SM clock
come from read-only nvidia-smi queries in the same run.  Needs a CUDA device: there is no fallback.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from time_candidates import gpu_context  # noqa: E402

L2_FLUSH_BYTES = 256 << 20
G1, G2 = 4.0, 5.0
D, T, HW = 256, 18, 17


def same_bits(a, b):
    return a.shape == b.shape and bool(((a.view(torch.int32) == b.view(torch.int32)) |
                                        (torch.isnan(a) & torch.isnan(b))).all())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2048)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_pairs.py needs a CUDA device (B200); there is no CPU fallback")
    if args.iters < 20:
        sys.exit("--iters must be at least 20")
    import attention_gan_b200 as pkg
    lib = pkg.native.lib()
    dev = torch.device("cuda")
    N, K = args.n, args.k
    P = N * K

    g = torch.Generator().manual_seed(0)
    img = torch.randn(N, D, HW * HW, generator=g).to(dev)
    words = torch.randn(N, T, D, generator=g).to(dev).transpose(1, 2)          # [N, D, T] view, RNN layout
    lens = torch.randint(2, T + 1, (N,), generator=g, dtype=torch.int32).to(dev)
    cls = np.random.default_rng(0).integers(0, 500, size=N)
    cand = torch.from_numpy(pkg.mismatched_candidates(cls, n_mismatched=K - 1, seed=0)).to(torch.int32).to(dev)
    # image -> text list in candidate order, the same list shuffled, and P pairs on image 0
    pi = torch.arange(N, dtype=torch.int32, device=dev).repeat_interleave(K)
    pc = cand.reshape(-1)
    perm = torch.randperm(P, generator=g).to(dev)
    pi_s, pc_s = pi[perm].contiguous(), pc[perm].contiguous()
    pi_1 = torch.zeros(P, dtype=torch.int32, device=dev)
    pc_1 = torch.randint(0, N, (P,), generator=g, dtype=torch.int32).to(dev)
    caps = torch.arange(N, device=dev)[:, None].expand(N, K)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def timed(fn, tags=()):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.iters)]
        for a, b in ev:
            flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        ms = sorted(a.elapsed_time(b) for a, b in ev)
        res = {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1]}
        if tags:                                  # kernel times in a separate pass: event recording perturbs timing
            lib.agb_prof_enable(1)
            for t in tags:
                lib.agb_prof_read(t, ctypes.byref(ctypes.c_double()), ctypes.byref(ctypes.c_longlong()))
            for _ in range(args.iters):
                flush.zero_()
                fn()
            torch.cuda.synchronize()
            for t in tags:
                tot, n = ctypes.c_double(0.0), ctypes.c_longlong(0)
                lib.agb_prof_read(t, ctypes.byref(tot), ctypes.byref(n))
                res[f"tag{t}_ms"] = tot.value / args.iters
            lib.agb_prof_enable(0)
        return res

    out = {"what": "pair-list DAMSM scoring, N images = N captions, K per list", "N": N, "K": K, "P": P, "T": T,
           "R": HW * HW, "iters": args.iters, "warmup": args.warmup, "l2_flush_bytes": L2_FLUSH_BYTES}
    out.update(gpu_context())
    for name in ("f16", "f16x2"):
        mt = pkg.native.MATH_NAMES[name]
        scorer = pkg.DAMSMScorer(dev, G1, G2, math=name, workspace_bytes=64 << 30)

        def fixed_k():
            return scorer.words(img, words, lens, cand)

        def pairs():
            return scorer.words_pairs(img, words, lens, pi, pc)

        def by_caption():
            return scorer.words(img, words, lens, cand, by="caption")

        def dense_t2i():
            m, _, _ = pkg.ops.damsm_fwd(img, words, lens, G1, G2, 1e-8, 0, False, mt)
            return m[cand.long(), caps]

        def shuffled():
            return scorer.words_pairs(img, words, lens, pi_s, pc_s)

        def one_image():
            return scorer.words_pairs(img, words, lens, pi_1, pc_1)

        def with_maps():
            return scorer.words_pairs(img, words, lens, pi, pc, att_maps=True)

        ref = fixed_k().reshape(-1)
        dense_full, _, _ = pkg.ops.damsm_fwd(img, words, lens, G1, G2, 1e-8, 0, False, mt)
        checks = {"pairs_eq_fixed_k": same_bits(pairs(), ref),
                  "by_caption_eq_dense_gathered": same_bits(by_caption(), dense_t2i()),
                  "shuffled_eq_fixed_k": same_bits(shuffled(), ref[perm]),
                  "one_image_eq_dense_gathered": same_bits(one_image(), dense_full[0, pc_1.long()]),
                  "maps_m_eq_fixed_k": same_bits(with_maps()[0], ref)}
        del dense_full
        torch.cuda.synchronize()
        if not all(checks.values()):
            sys.exit(f"{name}: results differ: {checks}")
        t_fixed = timed(fixed_k, tags=(9,))
        t_pairs = timed(pairs, tags=(9,))
        t_cap = timed(by_caption, tags=(9,))
        t_dense = timed(dense_t2i, tags=(2,))
        t_shuf = timed(shuffled, tags=(9,))
        t_one = timed(one_image, tags=(9,))
        t_maps = timed(with_maps, tags=(9,))
        out[name] = {
            "bit_exact": checks,
            "a_fixed_k_words": t_fixed, "a_words_pairs": t_pairs,
            "a_pairs_over_fixed_k": t_pairs["ms_median"] / t_fixed["ms_median"],
            "b_words_by_caption": t_cap, "b_dense_then_gather": t_dense,
            "b_speedup_vs_dense_then_gather": t_dense["ms_median"] / t_cap["ms_median"],
            "c_shuffled": t_shuf, "c_one_image": t_one,
            "c_shuffled_over_fixed_k": t_shuf["ms_median"] / t_fixed["ms_median"],
            "c_one_image_over_fixed_k": t_one["ms_median"] / t_fixed["ms_median"],
            "d_words_pairs_att_maps": t_maps,
            "d_maps_over_pairs": t_maps["ms_median"] / t_pairs["ms_median"],
        }
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
