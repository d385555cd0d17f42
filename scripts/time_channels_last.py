"""Generator word attention on channels_last feature maps: NHWC kernels against NCHW and against the workaround.

At cfg3 shapes (B = 64, C = 32, T = 18, bf16; 64x64, 128x128 and 256x256 maps) it measures
  kernel   the attention forward and backward kernels alone (the library's per-launch CUDA events), NHWC against
           NCHW, with achieved GB/s on the algorithmic bytes (fwd es*(2C+T), bwd es*3C per pixel, DESIGN.md)
  call     one ops.word_attn_fwd + ops.word_attn_bwd call on channels_last maps (CUDA events around the calls): the
           NHWC kernels, the NCHW kernels on NCHW maps, and today's workaround for channels_last maps (.contiguous()
           in, .contiguous(memory_format=torch.channels_last) out, and the same for the gradients)
  block    the GenNextStage-shaped NextStageBlock of scripts/time_compile.py, forward + backward, in channels_last
           against NCHW, eager and torch.compile'd, as ms per step (64x64 and 128x128)
The results of the variants are checked bit for bit against each other before anything is timed.  The L2 cache
(126 MB; cfg3's 128x128 maps are 67 MB) is overwritten before every timed kernel and call; the variants alternate
inside every iteration and the JSON keeps medians, with the GPU's name and power limit.  Needs a CUDA device.

    python scripts/time_channels_last.py --out profiles/time_channels_last.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import attention_gan_b200 as agb  # noqa: E402
from oracle import ref_port as rp  # noqa: E402
from scripts.time_compile import block_inputs, gpu_info, make_step, time_steps  # noqa: E402

CL = torch.channels_last
PROF_ATTN_FWD, PROF_ATTN_BWD = 4, 5


def prof_ms(lib, tag) -> float:
    ms, n = ctypes.c_double(0.0), ctypes.c_longlong(0)
    rc = lib.agb_prof_read(tag, ctypes.byref(ms), ctypes.byref(n))
    if rc != 0 or n.value != 1:
        raise RuntimeError(f"agb_prof_read(tag={tag}) gave rc={rc}, {n.value} launches")
    return ms.value


class Flush:
    """overwrites the L2 cache (256 MB of writes)"""

    def __init__(self):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self):
        self.buf.zero_()


def attention_case(hw, B=64, C=32, E=256, T=18, dtype=torch.bfloat16):
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=hw)
    images = images.to("cuda", dtype)
    g = torch.Generator().manual_seed(1)
    dctx = torch.randn(B, C, hw, hw, generator=g).to("cuda", dtype)
    return images, words.to("cuda"), weight.reshape(C, E).contiguous().to("cuda"), mask.to("cuda"), dctx


def run_nchw(im, words, weight, mask, dctx):
    ctx, attn, we = agb.ops.word_attn_fwd(im, words, weight, mask, True)
    di, dw, dwt = agb.ops.word_attn_bwd(im, words, weight, mask, we, dctx, None, True, True, True)
    return ctx, attn, di, dw, dwt


def run_workaround(im, words, weight, mask, dctx):
    """channels_last in and out through the NCHW kernels, as a user has to write it without the NHWC path"""
    ctx, attn, we = agb.ops.word_attn_fwd(im.contiguous(), words, weight, mask, True)
    ctx, attn = ctx.contiguous(memory_format=CL), attn.contiguous(memory_format=CL)
    di, dw, dwt = agb.ops.word_attn_bwd(im.contiguous(), words, weight, mask, we, dctx.contiguous(), None, True,
                                        True, True)
    return ctx, attn, di.contiguous(memory_format=CL), dw, dwt


def bitwise_equal(a, b) -> bool:
    return all(torch.equal(x.contiguous().view(torch.int16 if x.dtype != torch.float32 else torch.int32),
                           y.contiguous().view(torch.int16 if y.dtype != torch.float32 else torch.int32))
               for x, y in zip(a, b))


def time_attention(hw, iters, flush, lib):
    images, words, weight, mask, dctx = attention_case(hw)
    B, C, H, W = images.shape
    T = words.shape[2]
    es = images.element_size()
    inputs = {"nchw": (images, dctx), "nhwc": (images.contiguous(memory_format=CL), dctx.contiguous(memory_format=CL))}
    ref = run_nchw(images, words, weight, mask, dctx)
    got = run_nchw(*inputs["nhwc"][:1], words, weight, mask, inputs["nhwc"][1])
    wa = run_workaround(*inputs["nhwc"][:1], words, weight, mask, inputs["nhwc"][1])
    checked = bitwise_equal(ref, got) and bitwise_equal(ref, wa)
    if not checked:
        raise SystemExit(f"hw={hw}: NHWC results differ from NCHW; nothing timed")
    del ref, got, wa
    calls = {"nchw": lambda: run_nchw(images, words, weight, mask, dctx),
             "nhwc": lambda: run_nchw(inputs["nhwc"][0], words, weight, mask, inputs["nhwc"][1]),
             "workaround": lambda: run_workaround(inputs["nhwc"][0], words, weight, mask, inputs["nhwc"][1])}
    for f in calls.values():                     # warm-up: module load, tensor maps, allocator
        f()
    kern = {v: {"fwd": [], "bwd": []} for v in ("nchw", "nhwc")}
    call = {v: [] for v in calls}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(iters):
        for v, f in calls.items():
            flush()
            lib.agb_prof_enable(1)
            ev0.record()
            f()
            ev1.record()
            ev1.synchronize()
            call[v].append(ev0.elapsed_time(ev1))
            if v in kern:
                kern[v]["fwd"].append(prof_ms(lib, PROF_ATTN_FWD))
                kern[v]["bwd"].append(prof_ms(lib, PROF_ATTN_BWD))
            lib.agb_prof_enable(0)
    px = B * H * W
    nbytes = {"fwd": px * es * (2 * C + T), "bwd": px * es * 3 * C}
    res = {"B": B, "C": C, "T": T, "hw": hw, "dtype": str(images.dtype), "checked_bitwise": checked, "kernel": {}}
    for v in kern:
        res["kernel"][v] = {d: {"ms_median": statistics.median(kern[v][d]),
                                "GB_per_s": nbytes[d] / statistics.median(kern[v][d]) / 1e6} for d in ("fwd", "bwd")}
    for d in ("fwd", "bwd"):
        res["kernel"][f"nhwc_over_nchw_{d}"] = res["kernel"]["nhwc"][d]["ms_median"] / res["kernel"]["nchw"][d]["ms_median"]
    res["call_ms_median"] = {v: statistics.median(t) for v, t in call.items()}
    res["call_workaround_over_nhwc"] = res["call_ms_median"]["workaround"] / res["call_ms_median"]["nhwc"]
    return res


def time_block(hw, steps, rounds, warmup):
    """the same block and inputs twice: once NCHW, once converted with .to(memory_format=torch.channels_last)"""
    variants = {}
    for name in ("nchw", "channels_last"):
        block, h, w = block_inputs(hw)
        if name == "channels_last":
            block = block.to(memory_format=CL)
            h = h.detach().contiguous(memory_format=CL).requires_grad_(True)

        def fwd(a, b, block=block):
            img, att = block(a, b)
            return img.float().square().mean() + att.float().mean()
        grads = [h, *block.parameters()]
        variants[f"{name}_eager"] = make_step(fwd, (h, w), grads, False)
        variants[f"{name}_compile"] = make_step(torch.compile(fwd), (h, w), grads, False)
    for step in variants.values():
        for _ in range(warmup):
            step()
    torch.cuda.synchronize()
    ms = {k: [] for k in variants}
    for _ in range(rounds):
        for k, step in variants.items():
            ms[k].append(time_steps(step, steps))
    return {k: {"ms_per_step_median": statistics.median(t), "ms_per_step_min": min(t), "ms_per_step_max": max(t)}
            for k, t in ms.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_channels_last.json"))
    ap.add_argument("--iters", type=int, default=30, help="alternating iterations of the attention variants")
    ap.add_argument("--sizes", default="64,128,256")
    ap.add_argument("--block-sizes", default="64,128")
    ap.add_argument("--steps", type=int, default=10, help="block steps per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds of the block variants")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_channels_last.py needs a CUDA device")
    lib = agb.native.lib()
    flush = Flush()
    result = {"gpu": gpu_info(), "iters": args.iters, "attention": {}, "block": {}}
    for hw in (int(s) for s in args.sizes.split(",") if s):
        result["attention"][str(hw)] = r = time_attention(hw, args.iters, flush, lib)
        print("attention", hw, json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    for hw in (int(s) for s in args.block_sizes.split(",") if s):
        result["block"][str(hw)] = r = time_block(hw, args.steps, args.rounds, args.warmup)
        print("block", hw, json.dumps(r), flush=True)
        torch._dynamo.reset()
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
