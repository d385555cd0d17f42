"""Times R-precision scoring (attention_gan_b200.evaluation) against what a user does without candidate mode.

    python scripts/time_candidates.py [--n 2048] [--k 100] [--iters 20] [--warmup 3] [--out FILE]

Seeded synthetic inputs: N images = N captions (T = 18, lengths U{2..18}, 17 x 17 regions, words in the text
encoder's transposed [N, T, D] layout), class ids U{0..499}, K = 100 candidates per image from
mismatched_candidates.  For each math mode ("f16", "f16x2"):
  * candidate m is checked bit for bit against the dense forward gathered, at the timed size, before timing;
  * DAMSMScorer.words (packing + pair kernel; the pair kernel alone is profiling tag 9);
  * the dense inference forward ops.damsm_fwd at N x N (pair kernel: tag 2) followed by the gather.
Then DAMSMScorer.sentence.  CUDA events around every iteration, the L2 flushed between iterations outside the
events (a 256 MiB write, as bench.py does).  Prints one JSON line; GPU name, power limit and SM clock come from
read-only nvidia-smi queries in the same run.  Needs a CUDA device: there is no fallback.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_FLUSH_BYTES = 256 << 20
G1, G2 = 4.0, 5.0
D, T, HW = 256, 18, 17


def gpu_context():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        idx = torch.cuda.current_device()
        name, power, sm, sm_max = [x.strip() for x in out[idx].split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock": sm, "sm_clock_max": sm_max}
    except Exception as e:  # the numbers stay valid without the context; say it is missing
        return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": f"unavailable ({type(e).__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=2048)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_candidates.py needs a CUDA device (B200); there is no CPU fallback")
    if args.iters < 20:
        sys.exit("--iters must be at least 20")
    import attention_gan_b200 as pkg
    lib = pkg.native.lib()
    dev = torch.device("cuda")
    N, K = args.n, args.k

    g = torch.Generator().manual_seed(0)
    img = torch.randn(N, D, HW * HW, generator=g).to(dev)
    words = torch.randn(N, T, D, generator=g).to(dev).transpose(1, 2)          # [N, D, T] view, RNN layout
    lens = torch.randint(2, T + 1, (N,), generator=g, dtype=torch.int32).to(dev)
    cnn = torch.randn(N, D, generator=g).to(dev)
    rnn = torch.randn(N, D, generator=g).to(dev)
    cls = np.random.default_rng(0).integers(0, 500, size=N)
    cand_np = pkg.mismatched_candidates(cls, n_mismatched=K - 1, seed=0)
    cand = torch.from_numpy(cand_np).to(torch.int32).to(dev)
    cand_long = cand.long()
    lens_h = lens.cpu().numpy()
    lbar_cand = float(lens_h[cand_np].mean())
    lbar_dense = float(lens_h.mean())
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
                res[f"tag{t}_ms"] = tot.value / args.iters             # per call (a call may launch it more than once)
                res[f"tag{t}_launches_per_call"] = n.value / args.iters
            lib.agb_prof_enable(0)
        return res

    out = {"what": "R-precision scoring, N images x K candidates", "N": N, "K": K, "T": T, "R": HW * HW,
           "lbar_candidates": lbar_cand, "lbar_dense": lbar_dense, "iters": args.iters, "warmup": args.warmup,
           "l2_flush_bytes": L2_FLUSH_BYTES}
    out.update(gpu_context())
    pairs_c, pairs_d = N * K, N * N
    for name in ("f16", "f16x2"):
        mt = pkg.native.MATH_NAMES[name]
        scorer = pkg.DAMSMScorer(dev, G1, G2, math=name)

        def dense():
            m, _, _ = pkg.ops.damsm_fwd(img, words, lens, G1, G2, 1e-8, 0, False, mt)
            return m.gather(1, cand_long)

        def cand_words():
            return scorer.words(img, words, lens, cand)

        mc = cand_words()
        md = dense()
        torch.cuda.synchronize()
        same = bool(((mc.view(torch.int32) == md.view(torch.int32)) | (torch.isnan(mc) & torch.isnan(md))).all())
        if not same:
            sys.exit(f"{name}: candidate m differs from the dense result gathered")
        tc = timed(cand_words, tags=(9,))
        td = timed(dense, tags=(2,))
        flop_c = 4.0 * HW * HW * lbar_cand * D * pairs_c
        flop_d = 4.0 * HW * HW * lbar_dense * D * pairs_d
        k9, k2 = tc["tag9_ms"], td["tag2_ms"]
        out[name] = {
            "bit_exact_vs_dense_gathered": same,
            "candidates": {**tc, "pack_ms": tc["ms_median"] - k9, "pairs_per_s": pairs_c / tc["ms_median"] * 1e3,
                           "pair_kernel_pairs_per_s": pairs_c / k9 * 1e3,
                           "algorithmic_tflops": flop_c / tc["ms_median"] / 1e9,
                           "pair_kernel_algorithmic_tflops": flop_c / k9 / 1e9},
            "dense_then_gather": {**td, "pairs_per_s": pairs_d / td["ms_median"] * 1e3,
                                  "pair_kernel_pairs_per_s": pairs_d / k2 * 1e3,
                                  "algorithmic_tflops": flop_d / td["ms_median"] / 1e9,
                                  "pair_kernel_algorithmic_tflops": flop_d / k2 / 1e9},
            # per-pair throughput of candidate mode over the dense forward's, whole call and pair kernel alone
            "per_pair_rel_dense": (pairs_c / tc["ms_median"]) / (pairs_d / td["ms_median"]),
            "per_pair_rel_dense_pair_kernel": (pairs_c / k9) / (pairs_d / k2),
            "speedup_vs_dense_then_gather": td["ms_median"] / tc["ms_median"],
        }
    scorer = pkg.DAMSMScorer(dev)
    ts = timed(lambda: scorer.sentence(cnn, rnn, cand))
    td = timed(lambda: pkg.ops.sent_cos_fwd(cnn, rnn, 1e-8).gather(1, cand_long))
    out["sentence"] = {"candidates": ts, "dense_then_gather": td,
                       "speedup_vs_dense_then_gather": td["ms_median"] / ts["ms_median"]}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
