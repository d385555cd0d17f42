"""Times training on a pair list (words_pair_scores forward + backward) against what a user does without it.

    python scripts/time_pairs_train.py [--n 2048] [--k 100] [--iters 20] [--warmup 3] [--out FILE]

Seeded synthetic inputs as in scripts/time_pairs.py: N images = N captions (T = 18, lengths U{2..18}, 17 x 17
regions, words in the text encoder's transposed layout), class ids U{0..499}, K = 100 candidates per image from
mismatched_candidates, i.e. P = N K pairs.  For each math mode ("f16", "f16x2"):
  (a) the K-way listwise loss of INTEGRATION.md §8, forward + backward through words_pair_scores;
  (b) the same loss the way it is done without pair training: the dense N x N training forward (AGB_MATH_SAVE),
      the gather, and the dense backward with dLoss/dm zero outside the list;
  (c) the forward alone, as DAMSMScorer.words_pairs scores it;
  (d) agb_damsm_pairs_bwd alone and (e) the dense agb_damsm_bwd alone, for the per-pair rate of the two backwards;
  (f) forward + backward of P pairs that all name one image, and (g) of P pairs that all name one caption: the
      lists on which the per-image d img GEMM and the per-caption d words reduction have the most work per row.
Before timing, m of (a) is checked bit for bit against (c) and the gradients of (a) against those of (b) (largest
difference relative to the tensor's scale, bound 5e-3).  The variants alternate inside every iteration; CUDA events
around every call, the L2 flushed before every call outside the events (a 256 MiB write); medians of --iters
(>= 20) iterations after --warmup.  Prints one JSON line; GPU name, power limit and SM clock come from read-only
nvidia-smi queries in the same run.  Needs a CUDA device: there is no fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from time_candidates import gpu_context  # noqa: E402

L2_FLUSH_BYTES = 256 << 20
G1, G2, G3 = 4.0, 5.0, 10.0
D, T, HW = 256, 18, 17


def rel(x, ref):
    return ((x - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2048)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_pairs_train.py needs a CUDA device (B200); there is no CPU fallback")
    if args.iters < 20:
        sys.exit("--iters must be at least 20")
    import attention_gan_b200 as pkg
    ops = pkg.ops
    dev = torch.device("cuda")
    N, K = args.n, args.k
    P = N * K

    g = torch.Generator().manual_seed(0)
    img = torch.randn(N, D, HW * HW, generator=g).to(dev).requires_grad_(True)
    words = torch.randn(N, T, D, generator=g).to(dev).transpose(1, 2).detach().requires_grad_(True)   # [N, D, T]
    lens = torch.randint(2, T + 1, (N,), generator=g, dtype=torch.int32).to(dev)
    cls = np.random.default_rng(0).integers(0, 500, size=N)
    cand = torch.from_numpy(pkg.mismatched_candidates(cls, n_mismatched=K - 1, seed=0)).to(torch.int32).to(dev)
    pi = torch.arange(N, dtype=torch.int32, device=dev).repeat_interleave(K)
    pc = cand.reshape(-1).contiguous()
    pil, pcl = pi.long(), pc.long()
    target = torch.zeros(N, dtype=torch.long, device=dev)
    skew = torch.randint(0, N, (P,), generator=g, dtype=torch.int32).to(dev)
    one = torch.full((P,), 17, dtype=torch.int32, device=dev)
    dm_skew = (torch.randn(P, generator=g) * 1e-4).to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def listwise(m):
        return F.cross_entropy(G3 * m.view(N, K), target)

    out = {"what": "K-way listwise DAMSM loss on a pair list, forward + backward; N images = N captions",
           "N": N, "K": K, "P": P, "T": T, "R": HW * HW, "iters": args.iters, "warmup": args.warmup,
           "l2_flush_bytes": L2_FLUSH_BYTES}
    out.update(gpu_context())
    for name in ("f16", "f16x2"):
        mt = pkg.native.MATH_NAMES[name]
        scorer = pkg.DAMSMScorer(dev, G1, G2, math=name, workspace_bytes=64 << 30)

        def a_pairs():
            m = pkg.words_pair_scores(img, words, lens, pi, pc, gamma1=G1, gamma2=G2, math=name,
                                      workspace_bytes=64 << 30)
            return (m,) + torch.autograd.grad(listwise(m), (img, words))

        def b_dense():
            m, _, _, ws = ops.damsm_fwd(img.detach(), words.detach(), lens, G1, G2, 1e-8, 0, False, mt, keep_ws=True,
                                        save=True)
            ml = m.detach().requires_grad_(True)
            dm = torch.autograd.grad(listwise(ml[pil, pcl]), ml)[0]
            dimg, dw = ops.damsm_bwd(img.detach(), words.detach(), lens, G1, G2, 1e-8, dm, None, True, mt, m, ws, True)
            return dimg, dw.transpose(1, 2)

        def c_forward():
            return scorer.words_pairs(img, words, lens, pi, pc)

        # the backwards alone, on the saved workspaces of one training forward each
        m_p, ws_p = ops.damsm_pairs_train_fwd(img.detach(), words.detach(), lens, pi, pc, G1, G2, mt)
        dm_p = torch.randn(P, generator=g).to(dev) * 1e-4
        m_d, _, _, ws_d = ops.damsm_fwd(img.detach(), words.detach(), lens, G1, G2, 1e-8, 0, False, mt, keep_ws=True,
                                        save=True)
        dm_d = torch.zeros(N, N, device=dev)
        dm_d.index_put_((pil, pcl), dm_p, accumulate=True)

        def d_pair_bwd():
            return ops.damsm_pairs_bwd(img.detach(), words.detach(), lens, pi, pc, G1, G2, mt, dm_p, ws_p)

        def e_dense_bwd():
            return ops.damsm_bwd(img.detach(), words.detach(), lens, G1, G2, 1e-8, dm_d, None, True, mt, m_d, ws_d,
                                 True)

        def f_one_image():
            m = pkg.words_pair_scores(img, words, lens, one, skew, gamma1=G1, gamma2=G2, math=name,
                                      workspace_bytes=64 << 30)
            return (m,) + torch.autograd.grad(m, (img, words), dm_skew)

        def g_one_caption():
            m = pkg.words_pair_scores(img, words, lens, skew, one, gamma1=G1, gamma2=G2, math=name,
                                      workspace_bytes=64 << 30)
            return (m,) + torch.autograd.grad(m, (img, words), dm_skew)

        ra, rb, rc = a_pairs(), b_dense(), c_forward()
        rd, re = d_pair_bwd(), e_dense_bwd()
        checks = {"m_eq_words_pairs": bool(torch.equal(ra[0].view(torch.int32), rc.view(torch.int32))),
                  "train_fwd_m_eq_words_pairs": bool(torch.equal(m_p.view(torch.int32), rc.view(torch.int32))),
                  "rel_dimg_vs_dense": rel(ra[1], rb[0]), "rel_dwords_vs_dense": rel(ra[2], rb[1]),
                  "rel_pair_bwd_dimg_vs_dense": rel(rd[0], re[0]),
                  "rel_pair_bwd_dwords_vs_dense": rel(rd[1], re[1]),
                  "one_image_m_eq_words_pairs": bool(torch.equal(
                      f_one_image()[0].view(torch.int32), scorer.words_pairs(img, words, lens, one, skew).view(torch.int32))),
                  "one_caption_m_eq_words_pairs": bool(torch.equal(
                      g_one_caption()[0].view(torch.int32), scorer.words_pairs(img, words, lens, skew, one).view(torch.int32)))}
        del ra, rb, rc, rd, re
        if not (checks["m_eq_words_pairs"] and checks["train_fwd_m_eq_words_pairs"]
                and checks["one_image_m_eq_words_pairs"] and checks["one_caption_m_eq_words_pairs"]
                and max(v for k, v in checks.items() if k.startswith("rel")) < 5e-3):
            sys.exit(f"{name}: results differ: {checks}")
        variants = {"a_pairs_fwd_bwd": a_pairs, "b_dense_fwd_bwd": b_dense, "c_pairs_forward": c_forward,
                    "d_pair_backward": d_pair_bwd, "e_dense_backward": e_dense_bwd,
                    "f_one_image_fwd_bwd": f_one_image, "g_one_caption_fwd_bwd": g_one_caption}
        for fn in variants.values():
            for _ in range(args.warmup):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in variants}
        for _ in range(args.iters):
            evs = []
            for k, fn in variants.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                flush.zero_()
                a.record()
                fn()
                b.record()
                evs.append((k, a, b))
            torch.cuda.synchronize()
            for k, a, b in evs:
                times[k].append(a.elapsed_time(b))
        res = {"checks": checks}
        for k, ms in times.items():
            ms = sorted(ms)
            res[k] = {"ms_median": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1]}
        med = {k: res[k]["ms_median"] for k in variants}
        res["a_speedup_vs_b"] = med["b_dense_fwd_bwd"] / med["a_pairs_fwd_bwd"]
        res["a_over_c"] = med["a_pairs_fwd_bwd"] / med["c_pairs_forward"]
        res["f_over_a"] = med["f_one_image_fwd_bwd"] / med["a_pairs_fwd_bwd"]
        res["g_over_a"] = med["g_one_caption_fwd_bwd"] / med["a_pairs_fwd_bwd"]
        res["backward_speedup_pair_vs_dense"] = med["e_dense_backward"] / med["d_pair_backward"]
        # pairs per ms of each backward; the dense backward computes all N x N pairs
        res["pair_backward_rate_over_dense"] = (P / med["d_pair_backward"]) / (N * N / med["e_dense_backward"])
        out[name] = res
        del ws_p, ws_d, m_d, dm_d
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
