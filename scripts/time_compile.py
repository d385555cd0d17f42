"""Eager vs torch.compile vs torch.compile(mode="reduce-overhead") on two workloads that use the drop-ins:

  block   a GenNextStage-shaped block (generator_submodules.py:95-120) at cfg3 shapes: AttentionModule.forward_cat
          (attention + concat), two residual blocks and an upsampling block from torch.nn; batch 64, C = 32, T = 18,
          bf16, at 64x64 and 128x128; one step = forward + backward
  damsm   the cfg2 DAMSM loss step: DAMSMLoss (words + sentence loss, att_maps="packed", device class ids) forward +
          backward at batch 48, R = 289, T = 18, math f16

For every variant it records the graph breaks torch._dynamo.explain reports and ms/step from CUDA events.  Every
shape and variant is warmed up (compiled, CUDA graphs recorded) before timing; the variants then alternate within
one run, `--rounds` times, and the JSON keeps the median, min and max over the rounds, with the GPU's name and power
limit.  Needs a CUDA device; there is no CPU fallback.

    python scripts/time_compile.py --out profiles/time_compile_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import attention_gan_b200 as agb  # noqa: E402
from oracle import ref_port as rp  # noqa: E402


class GLU(nn.Module):
    def forward(self, x):
        nc = x.size(1) // 2
        return x[:, :nc] * torch.sigmoid(x[:, nc:])


def conv3x3(cin, cout):
    return nn.Conv2d(cin, cout, kernel_size=3, stride=1, padding=1, bias=False)


class ResBlock(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.block = nn.Sequential(conv3x3(c, 2 * c), nn.BatchNorm2d(2 * c), GLU(), conv3x3(c, c), nn.BatchNorm2d(c))

    def forward(self, x):
        return x + self.block(x)


class NextStageBlock(nn.Module):
    """attention + concat + two residual blocks + upsample, the layout of GenNextStage"""

    def __init__(self, ngf: int = 32, nef: int = 256):
        super().__init__()
        self.attention = agb.AttentionModule(ngf, nef)
        self.residual = nn.Sequential(ResBlock(2 * ngf), ResBlock(2 * ngf))
        self.upsample = nn.Sequential(nn.Upsample(scale_factor=2, mode="nearest"), conv3x3(2 * ngf, 2 * ngf),
                                      nn.BatchNorm2d(2 * ngf), GLU())

    def forward(self, h_code, word_embs):
        h_c_code, att = self.attention.forward_cat(h_code, word_embs)
        return self.upsample(self.residual(h_c_code)), att


def block_inputs(hw: int, B: int = 64, C: int = 32, E: int = 256, T: int = 18, dtype=torch.bfloat16, seed: int = 0,
                 device="cuda"):
    """a NextStageBlock in `dtype` with the attention weight and mask of rp.synth_attention, and its inputs"""
    torch.manual_seed(seed)
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=seed)
    block = NextStageBlock(C, E).to(device=device, dtype=dtype)
    with torch.no_grad():
        block.attention.conv1.weight.copy_(weight)
    block.attention.apply_mask(mask.to(device))
    h = images.to(device=device, dtype=dtype).requires_grad_(True)
    return block, h, words.to(device)


def damsm_inputs(B: int = 48, math: str = "f16", seed: int = 0, device="cuda"):
    img, wrd, cnn, rnn, labels, lens, cls = rp.synth_damsm(B, seed=seed, n_classes=500)
    loss = agb.DAMSMLoss(device, math=math, att_maps="packed")
    args = [img.to(device).requires_grad_(True), cnn.to(device).requires_grad_(True),
            wrd.to(device).requires_grad_(True), rnn.to(device).requires_grad_(True), labels.to(device),
            lens.to(device), torch.from_numpy(cls).to(device=device, dtype=torch.int32)]
    return loss, args


def workloads(device="cuda"):
    """name -> (forward function returning a scalar loss, its arguments, the tensors whose .grad a step sets)"""
    out = {}
    for hw in (64, 128):
        block, h, w = block_inputs(hw, device=device)

        def fwd(h, w, block=block):
            img, att = block(h, w)
            return img.float().square().mean() + att.float().mean()
        out[f"block_{hw}"] = (fwd, (h, w), [h, *block.parameters()])
    loss, args = damsm_inputs(device=device)

    def fwd_damsm(*a, loss=loss):
        wl, sl, _ = loss.get_losses(*a)
        return wl + sl
    out["damsm_cfg2"] = (fwd_damsm, tuple(args), [a for a in args if a.requires_grad])
    return out


def graph_breaks(fn, args) -> int:
    torch._dynamo.reset()
    return int(torch._dynamo.explain(fn)(*args).graph_break_count)


def make_step(fn, args, grads, graphs: bool):
    def step():
        for t in grads:
            t.grad = None
        if graphs:
            torch.compiler.cudagraph_mark_step_begin()
        fn(*args).backward()
    return step


def time_steps(step, steps: int) -> float:
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        step()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / steps


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0), "torch": torch.__version__}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else None
    except (OSError, subprocess.SubprocessError, IndexError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_compile_b200.json"))
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds of all variants")
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_compile.py needs a CUDA device")
    result = {"gpu": gpu_info(), "steps": args.steps, "rounds": args.rounds, "workloads": {}}
    for name, (fn, fargs, grads) in workloads().items():
        breaks = graph_breaks(fn, fargs)
        torch._dynamo.reset()
        variants = {"eager": make_step(fn, fargs, grads, False),
                    "compile": make_step(torch.compile(fn), fargs, grads, False),
                    "reduce-overhead": make_step(torch.compile(fn, mode="reduce-overhead"), fargs, grads, True)}
        for step in variants.values():
            for _ in range(args.warmup):
                step()
        torch.cuda.synchronize()
        ms = {v: [] for v in variants}
        for _ in range(args.rounds):
            for v, step in variants.items():
                ms[v].append(time_steps(step, args.steps))
        result["workloads"][name] = {
            v: {"graph_breaks": None if v == "eager" else breaks, "ms_per_step_median": statistics.median(t),
                "ms_per_step_min": min(t), "ms_per_step_max": max(t)} for v, t in ms.items()}
        print(name, json.dumps(result["workloads"][name]), flush=True)
        torch._dynamo.reset()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
