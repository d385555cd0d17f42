#!/usr/bin/env python
"""Benchmark of the word-region attention hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference]
                    [--workload cfg4|cfg2|cfg3|cfg5|cfg1] [--math fp32|f16|bf16] [--batch B] [--no-secondary]
                    [--dump-outputs DIR]

One "step" is one pass of the hot path over one batch of synthetic input.  The DEFAULT workload, at every N, is
BASELINE.json configs[3] -- the configuration the headline metric is quoted on:

  cfg4   DAMSM WordsLoss + SentenceLoss forward+backward at GLOBAL batch 2048 (17x17 regions, T=18, D=256; grads
         w.r.t. region features, word embeddings and both sentence codes), sharded over the N ranks with the word
         features all-gathered over NCCL so the negatives span the global batch.  Strong scaling: N=1 computes all
         2048 x 2048 pairs on one GPU, so the driver's 1/2/4/8 curve is ONE workload.
  cfg2   the same step at batch 48 (configs[1])
  cfg3   generator word attention forward+backward, bf16, batch 64, stages 64x64 + 128x128 + 256x256 (configs[2])
  cfg5   long-caption stress: T=64 words, 256x256, bf16, batch 256 split over the ranks (configs[4]; 32 per GPU)
  cfg1   attention fp32, batch 16, 64x64 (configs[0])
  cfg4step  the WHOLE pretraining step of configs[3] (reference pretrain_damsm.py:110-134): synthetic 7-token bedroom
         captions -> LSTM text encoder + the two trainable CNN heads (on synthetic Inception features) -> both
         losses -> backward -> clip_grad_norm_(RNN, 0.25) -> Adam; global batch 2048 sharded over the ranks
         (attention-gan_b200/pretrain/); at N=1 a batch-256 version runs as a secondary measurement

At N=1 the default run also measures cfg2, cfg3 and one GPU's share of cfg5 and reports them under "secondary"
in the same JSON line (pairs/s, pixels/s, HBM fraction).

Metric: pairs/s (image-caption pairs) for the DAMSM step, pixels/s for the attention workloads.
`value`   inputs resident in HBM; the whole step replayed from a CUDA graph in a single process (the product's
          GraphedStep helper), eager launches under torchrun; `eager` gives the un-graphed time next to it.
`e2e`     the same step through the public drop-in API from pinned HOST inputs: host->device copies of every input
          and the device->host read of the losses inside the timed region (`e2e_eager`: without the graph).
`roofline` per kernel, timed live with CUDA events on the launching stream (agb_prof_* hooks) in an eager pass:
          algorithmic flops (or bytes) of the launches / their summed duration; nothing is summed across
          concurrently running kernels.
`cpu_baseline` / `--impl reference`: the oracle port of the reference (the reference is Python under /root/reference,
          which does not exist on the GPU box) on the host cores, on a bounded sample of the same workload;
`torch_eager_gpu`: the same op-by-op port on cuda:0 (PyTorch ATen/cuBLAS eager), the second baseline of SURVEY 8d.
Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes what the last timed step of `value` handed back to its caller (losses, attention maps,
gradients w.r.t. every input; for cfg4step the loss and the updated parameters), rank 0's shard, as DIR/<name>.npy
in float32 (float64 stays float64).  The inputs are seeded, so two builds run with the same arguments can be compared
array for array.  The files total at most 60 MiB: an output above its share of that is written as a fixed, seeded
sample of its flattened elements (the same positions on every run with the same arguments).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

R_, T_, D_ = 289, 18, 256
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 60 << 20                   # --dump-outputs: under 64 MB with the .npy headers
CFG_BATCH = {"cfg2": 48, "cfg4": 2048}
METRIC_DAMSM = "damsm_words_sentence_loss_fwd_bwd_pairs_per_sec"
METRIC_ATTN = "word_attention_fwd_bwd_pixels_per_sec"
# algorithmic GEMM units (2*R*L*D flop each) per (image, caption) pair and kernel, SURVEY 8d / DESIGN.md section 4
DAMSM_KERNELS = {2: ("damsm_fwd2_kernel (scores + context, both softmaxes, cosine, LSE)", 2),
                 3: ("damsm_bwd3_kernel (d beta GEMM + both softmax backwards)", 1),
                 6: ("tc_gemm_kernel d img (dC via beta + dC via ds)", 2),
                 7: ("tc_gemm_kernel d words (dW via ds)", 1)}


def workload_name(wl, Bg=None, world=1):
    if wl in ("cfg2", "cfg4"):
        Bg = Bg or CFG_BATCH[wl]
        return (f"{wl}: DAMSM WordsLoss+SentenceLoss fwd+bwd, global batch {Bg}, R=289, T=18 (cap_lens U{{2..18}}), "
                f"D=256, class_ids U{{0..499}}")
    if wl == "cfg3":
        return "cfg3: AttentionModule fwd+bwd, batch 64, feature maps 64x64 + 128x128 + 256x256, T=18, C=32, E=256, bf16 I/O"
    if wl == "cfg5":
        return "cfg5: AttentionModule fwd+bwd, long captions T=64, 256x256, C=32, E=256, bf16 I/O, global batch 256"
    return "cfg1: AttentionModule fwd+bwd, batch 16, 64x64, T=18, C=32, E=256, fp32 I/O"


def load_traffic(key):
    """measured DRAM bytes per launch of the dominant kernel (committed ncu --set full capture), or None"""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                d = json.load(fh)
            if key in d:
                return d[key].get("bytes_per_launch", d[key].get("bytes_per_step"))
        except Exception:
            continue
    return None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]),
                    tf_sust=float(p["bf16_tflops_sustained"]), source="MEASURED_PEAKS.json")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="B200_PROFILING.md fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic inputs: ONE recipe for both arms (the reference arm takes the first rows of the same global batch)
# ------------------------------------------------------------------------------------------------
def damsm_inputs(Bg):
    """the global batch of cfg2 / cfg4 from one seed (SURVEY 8d): features ~ N(0,1), cap_lens ~ U{2..18} with one
    caption of full length, class_ids ~ U{0..499} (k = 500 finest clusters, data/bedrooms.py:291-304)"""
    import torch
    g = torch.Generator().manual_seed(0)
    img = torch.randn(Bg, D_, 17, 17, generator=g)
    wrd = torch.randn(Bg, T_, D_, generator=g)                      # physical [B,T,D] (rnn_encoder.py:91-92)
    cnn = torch.randn(Bg, D_, generator=g)
    rnn = torch.randn(Bg, D_, generator=g)
    lens = torch.randint(2, T_ + 1, (Bg,), generator=g, dtype=torch.int64)
    lens[0] = T_
    cls = torch.randint(0, 500, (Bg,), generator=g, dtype=torch.int64)
    return img, wrd, cnn, rnn, lens, cls


def ref_damsm_step(B, Bg, device="cpu"):
    """WordsLoss + SentenceLoss fwd+bwd of the op-by-op port on the first B samples of the global batch"""
    import torch
    from oracle import ref_port as rp
    img, wrd, cnn, rnn, lens, cls = damsm_inputs(Bg)
    img = img[:B].to(device).requires_grad_(True)
    wrd = wrd[:B].to(device).transpose(1, 2).detach().requires_grad_(True)
    cnn = cnn[:B].to(device).requires_grad_(True)
    rnn = rnn[:B].to(device).requires_grad_(True)
    lens, cls = lens[:B], cls[:B].numpy()
    labels = torch.arange(B, device=device)

    def step():
        for t in (img, wrd, cnn, rnn):
            t.grad = None
        wl, _ = rp.words_loss(img, wrd, labels, lens, cls)
        sl = rp.sentence_loss(cnn, rnn, labels, cls)
        (wl + sl).backward()
        return float(wl.detach()) + float(sl.detach())
    return step, B * B


def ref_attn_step(B, C, E, T, hw, device="cpu"):
    import torch
    from oracle import ref_port as rp
    images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, 0)
    images = images.to(device).requires_grad_(True)
    words = words.to(device).detach().clone().requires_grad_(True)
    weight = weight.to(device).requires_grad_(True)
    mask = mask.to(device)
    dctx = torch.randn(B, C, hw, hw, generator=torch.Generator().manual_seed(1)).to(device)

    def step():
        for t in (images, words, weight):
            t.grad = None
        ctx, _ = rp.word_attention(images, words, weight, mask)
        ctx.backward(dctx)
        return 0.0
    return step, B * hw * hw


def time_host(step, steps, warmup, sync=None):
    for _ in range(warmup):
        step()
    if sync:
        sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    if sync:
        sync()
    return (time.perf_counter() - t0) / steps


def host_outputs(outputs):
    """name -> device tensor  =>  name -> float32 / float64 numpy array, DUMP_BYTES in all.  Smallest first, each
    output gets an equal share of what the smaller ones left; one above its share keeps a sorted sample of its
    flattened elements drawn from a fixed seed"""
    import torch
    def elem_bytes(t):
        return 8 if t.dtype == torch.float64 else 4
    left, host = DUMP_BYTES, {}
    order = sorted(outputs, key=lambda k: outputs[k].numel() * elem_bytes(outputs[k]))
    for i, name in enumerate(order):
        t = outputs[name].detach()
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        keep = left // (len(order) - i) // elem_bytes(t)
        if t.numel() > keep:
            idx = torch.randint(t.numel(), (keep,), generator=torch.Generator().manual_seed(0)).unique()
            t = t.reshape(-1)[idx.to(t.device)]
        host[name] = t.to(dt).cpu().numpy()
        left -= host[name].nbytes
    return {k: host[k] for k in outputs}


def run_reference(args):
    """reference arm: the reference's CPU implementation of the path (oracle port) on the host cores, rank 0 only"""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    wl = args.workload
    if wl in ("cfg2", "cfg4", "cfg4step"):
        Bg = args.batch or CFG_BATCH.get(wl, 2048)
        B = min(Bg, 48 if wl == "cfg2" else 96)
        step, units = ref_damsm_step(B, Bg)
        metric, unit = METRIC_DAMSM, "pairs/s"
        sample = (f"oracle/ref_port.py (op-by-op torch-CPU port of the reference) WordsLoss+SentenceLoss fwd+bwd on the "
                  f"first {B} samples of the workload's global batch ({B}x{B} pairs per step), fp32, all host threads")
    else:
        if wl == "cfg1":
            B, C, E, T, hw = 16, 32, 256, 18, 64
        elif wl == "cfg5":
            B, C, E, T, hw = 1, 32, 256, 64, 256
        else:
            B, C, E, T, hw = 4, 32, 256, 18, 128
        step, units = ref_attn_step(B, C, E, T, hw)
        metric, unit = METRIC_ATTN, "pixels/s"
        sample = f"oracle/ref_port.py word_attention fwd+bwd, fp32, B={B}, {hw}x{hw}, T={T}, C={C}, all host threads"
    sec = time_host(step, args.steps, args.warmup)
    v = units / sec
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong" if wl in ("cfg4", "cfg5", "cfg4step") else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload_name("cfg4" if wl == "cfg4step" else wl, args.batch)},
            "cpu_baseline": {"value": v, "unit": unit, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": sample},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
class Env:
    """per-process measurement context: device, ranks, timing helpers"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py (native arm) needs a CUDA device"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD
        import attention_gan_b200 as pkg
        self.pkg = pkg
        self.lib = pkg.native.lib()
        self.flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=self.dev)

    def l2_flush(self):
        self.flush.zero_()                    # write a buffer larger than the 126 MB L2: evicts every input line

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, run, steps):
        """CUDA events around each of `steps` runs (L2 flushed between them, outside the events), barrier +
        synchronize on both sides, max over ranks; seconds per step"""
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        for a, b in ev:
            self.l2_flush()
            a.record()
            run()
            b.record()
        self.barrier()
        sec = sum(a.elapsed_time(b) for a, b in ev) / 1e3 / steps
        t = torch.tensor([sec], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def graphed(self, fn):
        if self.world > 1 or self.args.no_graph:
            return None
        from attention_gan_b200.agb_native.graph import try_graphed
        return try_graphed(fn)

    def prof_read(self, tag):
        ms, n = ctypes.c_double(0.0), ctypes.c_longlong(0)
        self.lib.agb_prof_read(tag, ctypes.byref(ms), ctypes.byref(n))
        return ms.value, n.value

    def measure(self, make_dev, step_dev, step_e2e, tags, steps, warmup, sample_clocks=False, e2e_pipe=None,
                keep_outputs=False):
        """the four timings of one workload + the per-kernel profile; all ranks call this together.
        step_dev returns its outputs as {name: tensor}; keep_outputs: host copies of those of the last timed step of
        `value` under out["outputs"]"""
        lib = self.lib
        ts = make_dev()
        for _ in range(warmup):
            step_dev(ts)
        self.barrier()
        prof_steps = min(steps, 5)
        lib.agb_prof_enable(1)
        n0 = lib.agb_launch_count()
        for _ in range(prof_steps):
            self.l2_flush()
            step_dev(ts)
        self.barrier()
        launches_per_step = (lib.agb_launch_count() - n0) // prof_steps
        prof = {t: self.prof_read(t) for t in tags}
        lib.agb_prof_enable(0)
        self.torch.cuda.empty_cache()
        out = {"prof": prof, "prof_steps": prof_steps, "launches_per_step": int(launches_per_step)}
        torch = self.torch
        sampler = ClockSampler(self.local) if (sample_clocks and self.rank == 0) else None
        g = self.graphed(lambda: step_dev(ts))
        if g is None and sampler:
            sampler.start()                       # no graph (torchrun / --no-graph): the eager timing IS the value
        step_dev(ts)                              # untimed: re-grows the allocator pool emptied above (cudaMalloc of the workspace)
        run_eager, last = (lambda: step_dev(ts)), {}
        if keep_outputs and g is None:            # the eager timing is `value`: hold on to its last step's outputs only
            done = [0]

            def run_eager():
                outs = step_dev(ts)
                done[0] += 1
                if done[0] == steps:
                    last["outputs"] = outs
        out["eager"] = self.timed(run_eager, steps)
        if g is not None:
            if sampler:
                sampler.start()
            out["value"] = self.timed(g.replay, steps)
        else:
            out["value"] = out["eager"]
        if keep_outputs:                          # a graph's static outputs hold what its last replay wrote
            out["outputs"] = host_outputs(g.outputs if g is not None else last.pop("outputs"))
        out["clocks"] = sampler.stop() if sampler else None
        out["graph"] = g is not None
        del g
        torch.cuda.empty_cache()                  # a captured step owns a private copy of the workspace
        for _ in range(max(1, warmup // 2)):
            step_e2e()
        self.barrier()
        out["e2e_eager"] = self.timed(step_e2e, steps)
        g2 = self.graphed(step_e2e)
        out["e2e"] = self.timed(g2.replay, steps) if g2 is not None else out["e2e_eager"]
        out["e2e_graph"] = g2 is not None
        del g2, ts
        torch.cuda.empty_cache()
        if e2e_pipe is not None:
            # the same end-to-end step with the product's HostPrefetcher: the H2D copy of step i+1 runs on a copy
            # stream under the kernels of step i (every step still copies all of its inputs inside the timed region)
            host, run_on = e2e_pipe
            for rep in range(2):                       # warm-up pass, then the timed pass
                n = 3 if rep == 0 else steps
                pf = self.pkg.HostPrefetcher(self.dev)
                state = {"i": 0}

                def run():
                    i = state["i"]
                    if i == 0:
                        pf.submit(host)
                    ts_ = pf.acquire()
                    if i + 1 < n:
                        pf.submit(host)
                    run_on(ts_)
                    pf.release()
                    state["i"] = i + 1
                sec = self.timed(run, n)
            out["e2e_pipelined"] = sec
        return out


def damsm_workload(env: Env, wl, Bg, math, steps, warmup, sample_clocks, keep_outputs=False):
    torch, pkg, dev, world, rank = env.torch, env.pkg, env.dev, env.world, env.rank
    assert Bg % world == 0
    Bl = Bg // world
    sl = slice(rank * Bl, rank * Bl + Bl)
    img, wrd, cnn, rnn, lens, cls = damsm_inputs(Bg)         # every rank: the same global batch, keeps its shard
    mean_len = float(lens.float().mean())
    img_h, wrd_h = img[sl].contiguous().pin_memory(), wrd[sl].contiguous().pin_memory()
    cnn_h, rnn_h = cnn[sl].contiguous().pin_memory(), rnn[sl].contiguous().pin_memory()
    lens_h = lens[sl].to(torch.int32).contiguous().pin_memory()
    cls_h = cls[sl].to(torch.int32).contiguous().pin_memory()
    del img, wrd, cnn, rnn
    labels = torch.arange(Bl, device=dev)
    loss_mod = pkg.DAMSMLoss(dev, math=math, process_group=env.group, att_maps="packed", max_words=T_)
    out_h = torch.empty(2, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (img_h, wrd_h, cnn_h, rnn_h, lens_h, cls_h))

    def make_dev():
        ts = [img_h.to(dev), wrd_h.to(dev), cnn_h.to(dev), rnn_h.to(dev)]
        for t in ts:
            t.requires_grad_(True)
        return ts + [lens_h.to(dev), cls_h.to(dev)]

    def step_dev(ts):
        im, wd, cn, rn, ln, cl = ts
        for t in (im, wd, cn, rn):
            t.grad = None
        wl_, sl_, maps = loss_mod.get_losses(im, cn, wd.transpose(1, 2), rn, labels, ln, cl)
        (wl_ + sl_).backward()
        return {"words_loss": wl_, "sentence_loss": sl_, "att_maps": maps, "d_img_features": im.grad,
                "d_words_emb": wd.grad, "d_cnn_code": cn.grad, "d_rnn_code": rn.grad}

    def step_e2e():
        im = img_h.to(dev, non_blocking=True).requires_grad_(True)
        wd = wrd_h.to(dev, non_blocking=True).requires_grad_(True)
        cn = cnn_h.to(dev, non_blocking=True).requires_grad_(True)
        rn = rnn_h.to(dev, non_blocking=True).requires_grad_(True)
        ln = lens_h.to(dev, non_blocking=True)
        cl = cls_h.to(dev, non_blocking=True)
        wl_, sl_, _ = loss_mod.get_losses(im, cn, wd.transpose(1, 2), rn, labels, ln, cl)
        (wl_ + sl_).backward()
        out_h[0:1].copy_(wl_.detach().reshape(1), non_blocking=True)
        out_h[1:2].copy_(sl_.detach().reshape(1), non_blocking=True)

    def run_on(ts):
        im, wd, cn, rn, ln, cl = ts
        for t in (im, wd, cn, rn):
            t.grad = None
            t.requires_grad_(True)
        wl_, sl_, _ = loss_mod.get_losses(im, cn, wd.transpose(1, 2), rn, labels, ln, cl)
        (wl_ + sl_).backward()
        out_h[0:1].copy_(wl_.detach().reshape(1), non_blocking=True)
        out_h[1:2].copy_(sl_.detach().reshape(1), non_blocking=True)

    tc = math != "fp32"
    tags = list(DAMSM_KERNELS) if tc else [1]
    m = env.measure(make_dev, step_dev, step_e2e, tags, steps, warmup, sample_clocks,
                    e2e_pipe=([img_h, wrd_h, cnn_h, rnn_h, lens_h, cls_h], run_on), keep_outputs=keep_outputs)
    m.update(units=Bl * Bg, total_units=Bg * Bg, h2d=int(h2d), d2h=8, mean_len=mean_len, tc=tc,
             flop_unit=2.0 * R_ * mean_len * D_, metric=METRIC_DAMSM, unit="pairs/s",
             dtype={"fp32": "f32", "f16": "f16", "bf16": "bf16", "f16x2": "f16"}[math], math=math)
    return m


def pretrain_workload(env: Env, Bg, math, steps, warmup, sample_clocks, keep_outputs=False):
    """the whole DAMSM pretraining step (SURVEY 8 f4) on synthetic bedroom captions + synthetic Inception features"""
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    from attention_gan_b200.pretrain import DamsmPretrainStep, SyntheticBedroomCaptions
    assert Bg % world == 0
    Bl = Bg // world
    sl = slice(rank * Bl, rank * Bl + Bl)
    data = SyntheticBedroomCaptions(Bg, seed=0)             # k = 7..500 hierarchy, 7-token captions, <= 990 words
    g = torch.Generator().manual_seed(0)
    caps_h = data.captions[sl].contiguous().pin_memory()
    lens_h = data.lengths[sl].to(torch.int32).contiguous().pin_memory()
    cls_h = data.class_ids[sl].to(torch.int32).contiguous().pin_memory()
    m6e_h = (torch.randn(Bg, 768, 17, 17, generator=g)[sl] * 0.5).contiguous().pin_memory()
    pool_h = (torch.randn(Bg, 2048, generator=g)[sl] * 0.5).contiguous().pin_memory()
    labels = torch.arange(Bl, device=dev)
    st = DamsmPretrainStep(data.vocab_size, dev, math=math, process_group=env.group, fixed_length=True, max_words=7)
    out_h = torch.empty(1, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (caps_h, lens_h, cls_h, m6e_h, pool_h))

    params = {f"{k}.{n}": p for k, mod in st.modules().items() for n, p in mod.named_parameters() if p.requires_grad}

    def make_dev():
        return [caps_h.to(dev), lens_h.to(dev), cls_h.to(dev), m6e_h.to(dev), pool_h.to(dev)]

    def step_dev(ts):
        return {"loss": st.step(ts[0], ts[1], ts[2], ts[3], ts[4], labels), **params}   # parameters: updated in place

    def step_e2e():
        ts = [t.to(dev, non_blocking=True) for t in (caps_h, lens_h, cls_h, m6e_h, pool_h)]
        loss = st.step(ts[0], ts[1], ts[2], ts[3], ts[4], labels)
        out_h.copy_(loss.reshape(1), non_blocking=True)

    def run_on(ts):
        loss = st.step(ts[0], ts[1], ts[2], ts[3], ts[4], labels)
        out_h.copy_(loss.reshape(1), non_blocking=True)

    tc = math != "fp32"
    m = env.measure(make_dev, step_dev, step_e2e, list(DAMSM_KERNELS) if tc else [1], steps, warmup, sample_clocks,
                    e2e_pipe=([caps_h, lens_h, cls_h, m6e_h, pool_h], run_on), keep_outputs=keep_outputs)
    m.update(units=Bl * Bg, total_units=Bg * Bg, h2d=int(h2d), d2h=4, mean_len=7.0, tc=tc,
             flop_unit=2.0 * R_ * 7.0 * D_, metric="damsm_pretrain_step_pairs_per_sec", unit="pairs/s",
             dtype={"fp32": "f32", "f16": "f16", "bf16": "bf16", "f16x2": "f16"}[math], math=math)
    return m


def attn_workload(env: Env, wl, batch, hw_only, steps, warmup, sample_clocks, local_share=False, keep_outputs=False):
    torch, pkg, dev, world, rank = env.torch, env.pkg, env.dev, env.world, env.rank
    from oracle import ref_port as rp          # seeded input generators only (never inside a timed region)
    if wl == "cfg1":
        B, C, E, T, hws, tdt = 16, 32, 256, 18, [64], torch.float32
    elif wl == "cfg5":
        B, C, E, T, hws, tdt = 256, 32, 256, 64, [256], torch.bfloat16
    else:
        B, C, E, T, hws, tdt = 64, 32, 256, 18, [64, 128, 256], torch.bfloat16
    if hw_only:
        hws = [hw_only]
    B = batch or B
    if local_share:                              # one GPU's share of an 8-GPU workload, measured on this GPU alone
        B = B // 8
        share, rk = 1, 0
    else:
        share, rk = world, rank
    assert B % share == 0
    Bl = B // share
    sl = slice(rk * Bl, rk * Bl + Bl)
    g = torch.Generator().manual_seed(1)
    img_h, dctx_h = [], []
    for hw in hws:
        images, words, weight, mask, _ = rp.synth_attention(B, C, E, T, hw, seed=0)
        img_h.append(images[sl].to(tdt).contiguous().pin_memory())
        dctx_h.append(torch.randn(B, C, hw, hw, generator=g)[sl].to(tdt).contiguous().pin_memory())
        del images
    wrd_h = words[sl].transpose(1, 2).contiguous().pin_memory()        # physical [B,T,E]
    mask_d = mask[sl].to(dev)
    mods = []
    for hw in hws:                                                      # one AttentionModule per stage
        mod = pkg.AttentionModule(C, E).to(dev)
        with torch.no_grad():
            mod.conv1.weight.copy_(weight.to(dev))
        mod.apply_mask(mask_d)
        mods.append(mod)
    out_h = torch.empty(256 * len(hws), dtype=tdt).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (*img_h, *dctx_h, wrd_h))
    d2h = out_h.numel() * out_h.element_size()

    def make_dev():
        return [[t.to(dev).requires_grad_(True) for t in img_h], wrd_h.to(dev).requires_grad_(True),
                [t.to(dev) for t in dctx_h]]

    def step_dev(ts):
        ims, wd, dctxs = ts
        wd.grad = None
        outs = {}
        for hw, mod, im, dctx in zip(hws, mods, ims, dctxs):
            im.grad = None
            mod.conv1.weight.grad = None
            ctx, attn = mod(im, wd.transpose(1, 2))
            ctx.backward(dctx)
            outs.update({f"ctx_{hw}": ctx, f"attn_{hw}": attn, f"d_images_{hw}": im.grad,
                         f"d_weight_{hw}": mod.conv1.weight.grad})
        outs["d_words"] = wd.grad                 # summed over the stages
        return outs

    def step_e2e():
        wd = wrd_h.to(dev, non_blocking=True).requires_grad_(True)
        for i, (mod, im_h, dc_h) in enumerate(zip(mods, img_h, dctx_h)):
            im = im_h.to(dev, non_blocking=True).requires_grad_(True)
            dctx = dc_h.to(dev, non_blocking=True)
            mod.conv1.weight.grad = None
            ctx, attn = mod(im, wd.transpose(1, 2))
            ctx.backward(dctx)
            out_h[256 * i:256 * (i + 1)].copy_(im.grad.reshape(-1)[:256], non_blocking=True)   # a slice of every stage's result

    def run_on(ts):
        n = len(hws)
        wd = ts[2 * n].requires_grad_(True)
        wd.grad = None
        for i, mod in enumerate(mods):
            im = ts[i].requires_grad_(True)
            im.grad = None
            mod.conv1.weight.grad = None
            ctx, attn = mod(im, wd.transpose(1, 2))
            ctx.backward(ts[n + i])
            out_h[256 * i:256 * (i + 1)].copy_(im.grad.reshape(-1)[:256], non_blocking=True)

    npix = sum(hw * hw for hw in hws)
    es = 4 if tdt == torch.float32 else 2
    m = env.measure(make_dev, step_dev, step_e2e, [4, 5], steps, warmup, sample_clocks,
                    e2e_pipe=([*img_h, *dctx_h, wrd_h], run_on), keep_outputs=keep_outputs)
    m.update(units=Bl * npix, total_units=B * npix, h2d=int(h2d), d2h=int(d2h), metric=METRIC_ATTN, unit="pixels/s",
             bytes_fwd=es * (2 * C + T), bytes_bwd=es * 3 * C, dtype="f32" if es == 4 else "bf16",
             io="fp32" if es == 4 else "bf16", B=B, T=T, C=C, hws=hws)
    return m


def damsm_roofline(m, peaks, long_step):
    """per-kernel tensor roofline of one DAMSM measurement (no sums over concurrently running kernels)"""
    pairs = m["units"] * m["prof_steps"]
    peak = peaks["tf_sust"] if long_step else peaks["tf_burst"]
    which = "sustained" if long_step else "burst"
    kernels = []
    if m["tc"]:
        for tag, (name, gemm_units) in DAMSM_KERNELS.items():
            ms, n = m["prof"][tag]
            if n == 0:
                continue
            tf = gemm_units * m["flop_unit"] * pairs / (ms * 1e-3) / 1e12
            kernels.append({"kernel": name, "launches": int(n), "avg_launch_ms": ms / n, "ms_per_step": ms / m["prof_steps"],
                            "algorithmic_gemm_units_per_pair": gemm_units, "achieved": tf, "frac": tf / peak})
    else:
        ms, n = m["prof"][1]
        tf = 6 * m["flop_unit"] * pairs / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        kernels.append({"kernel": "sgemm_strided_kernel (fp32 CUDA cores)", "launches": int(n),
                        "avg_launch_ms": ms / max(n, 1), "ms_per_step": ms / m["prof_steps"],
                        "algorithmic_gemm_units_per_pair": 6, "achieved": tf, "frac": tf / peak})
    dom = max(kernels, key=lambda k: k["ms_per_step"])
    step_tf = 6 * m["flop_unit"] * m["units"] / m["value"] / 1e12
    roof = {"bound": "tensor", "achieved": dom["achieved"], "peak": peak, "unit": "TFLOP/s", "frac": dom["frac"],
            "traffic": load_traffic("damsm_bwd3_kernel") if ("bwd3" in dom["kernel"]) else None,
            "kernel": dom["kernel"], "launches": dom["launches"], "avg_launch_ms": dom["avg_launch_ms"],
            "peak_source": f"{peaks['source']} dense bf16 {which} (kernel timed with CUDA events on its launching stream "
                           f"inside {'a long step' if long_step else 'a short step'})",
            "algorithmic": "GEMM unit = 2*R*mean(cap_len)*D flop per (image,caption) pair; fwd 2 units, d beta 1, "
                           "d img 2, d words 1 = 12*R*L*D per pair (recomputation is not counted)",
            "step": {"achieved": step_tf, "frac": step_tf / peak, "frac_of_burst": step_tf / peaks["tf_burst"],
                     "note": "all 12*R*L*D flop per pair of this rank / device-timed step"},
            "kernels": kernels,
            "concurrency_note": "the d img and d words GEMMs run concurrently on two streams: their event durations "
                                "overlap in time and are NOT additive (serialised under ncu the d words GEMM is ~4x "
                                "shorter, profiles/r2_launches_cfg4_n1.csv); the pair kernels run alone"}
    return roof


def attn_roofline(m, peaks):
    (ms_f, n_f), (ms_b, n_b) = m["prof"][4], m["prof"][5]
    px = m["units"] * m["prof_steps"]
    fwd = m["bytes_fwd"] * px / 1e9 / (ms_f * 1e-3) if ms_f > 0 else 0.0
    bwd = m["bytes_bwd"] * px / 1e9 / (ms_b * 1e-3) if ms_b > 0 else 0.0
    both = (m["bytes_fwd"] + m["bytes_bwd"]) * px / 1e9 / ((ms_f + ms_b) * 1e-3) if ms_f + ms_b > 0 else 0.0
    step = (m["bytes_fwd"] + m["bytes_bwd"]) * m["units"] / 1e9 / m["value"]
    dom_bwd = ms_b >= ms_f
    return {"bound": "hbm", "achieved": bwd if dom_bwd else fwd, "peak": peaks["hbm"], "unit": "GB/s",
            "frac": (bwd if dom_bwd else fwd) / peaks["hbm"], "traffic": None,
            "kernel": "word_attn_bwd_tc_kernel" if dom_bwd else "word_attn_fwd_tc_kernel",
            "launches": int(n_b if dom_bwd else n_f), "avg_launch_ms": (ms_b / max(n_b, 1)) if dom_bwd else (ms_f / max(n_f, 1)),
            "fwd_gbs": fwd, "bwd_gbs": bwd, "fwd_bwd_kernels_gbs": both, "fwd_bwd_kernels_frac": both / peaks["hbm"],
            "step": {"achieved": step, "frac": step / peaks["hbm"],
                     "note": "algorithmic bytes of all stages / device-timed step (projection + reduction kernels included)"},
            "peak_source": f"{peaks['source']} HBM copy", "algorithmic": "es*(2C+T) B/pixel fwd + es*3C B/pixel bwd"}


def summary(m, roof, name):
    """compact record of a secondary workload"""
    return {"workload": name, "metric": m["metric"], "unit": m["unit"], "value": m["total_units"] / m["value"],
            "ms_per_step": m["value"] * 1e3, "eager_ms_per_step": m["eager"] * 1e3,
            "e2e": {"value": m["total_units"] / m["e2e"], "ms_per_step": m["e2e"] * 1e3,
                    "eager_ms_per_step": m["e2e_eager"] * 1e3, "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
            "cuda_graph": m["graph"], "gpu_launches_per_step": m["launches_per_step"], "dtype": m["dtype"], "roofline": roof}


def run_native(args):
    env = Env(args)
    torch = env.torch
    peaks = load_peaks()
    wl = args.workload
    damsm = wl in ("cfg2", "cfg4", "cfg4step")
    keep = args.dump_outputs is not None
    if wl == "cfg4step":
        Bg = args.batch or 2048
        m = pretrain_workload(env, Bg, args.math, args.steps, args.warmup, True, keep_outputs=keep)
        roof = damsm_roofline(m, peaks, long_step=m["value"] > 2e-3)
        name = (f"cfg4step: DAMSM pretraining step (text LSTM + CNN heads + WordsLoss + SentenceLoss + backward + clip + "
                f"Adam), synthetic 7-token bedroom captions (k=7..500 hierarchy, <=990 words), global batch {Bg}")
    elif damsm:
        Bg = args.batch or CFG_BATCH[wl]
        m = damsm_workload(env, wl, Bg, args.math, args.steps, args.warmup, True, keep_outputs=keep)
        roof = damsm_roofline(m, peaks, long_step=m["value"] > 2e-3)
        name = workload_name(wl, Bg)
    else:
        m = attn_workload(env, wl, args.batch, args.hw, args.steps, args.warmup, True, keep_outputs=keep)
        roof = attn_roofline(m, peaks)
        name = workload_name(wl)
    if keep and env.rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, a in m.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), a)

    secondary = {}
    if env.world == 1 and args.secondary and not (args.batch or args.hw):
        ssteps, swarm = min(args.steps, 20), 3
        for w2 in ("cfg2", "cfg3", "cfg5", "cfg4_f16x2", "pretrain_step_b256"):
            if w2 == wl:
                continue
            try:
                if w2 == "cfg4_f16x2":
                    if wl != "cfg4" or args.math == "f16x2":
                        continue
                    m2 = damsm_workload(env, "cfg4", CFG_BATCH["cfg4"], "f16x2", 5, swarm, False)
                    secondary[w2] = summary(m2, damsm_roofline(m2, peaks, long_step=True),
                                            workload_name("cfg4") + "; math=f16x2 (split-precision forward: loss within "
                                            "1e-4 of the reference on every fixture)")
                elif w2 == "pretrain_step_b256":
                    m2 = pretrain_workload(env, 256, args.math, ssteps, swarm, False)
                    secondary[w2] = summary(m2, damsm_roofline(m2, peaks, long_step=False),
                                            "whole DAMSM pretraining step (pretrain_damsm.py:110-134), synthetic bedroom "
                                            "captions (7 tokens), batch 256 on one GPU")
                elif w2 == "cfg2":
                    m2 = damsm_workload(env, w2, CFG_BATCH[w2], args.math, ssteps, swarm, False)
                    secondary[w2] = summary(m2, damsm_roofline(m2, peaks, long_step=False), workload_name(w2))
                else:
                    m2 = attn_workload(env, w2, None, None, ssteps, swarm, False, local_share=(w2 == "cfg5"))
                    nm = workload_name(w2) + ("; ONE GPU's share (32 samples) measured on this GPU" if w2 == "cfg5" else "")
                    secondary[w2] = summary(m2, attn_roofline(m2, peaks), nm)
            except Exception as e:                 # a failing secondary must not take the headline down with it
                secondary[w2] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.synchronize()

    if env.rank != 0:
        if env.world > 1:
            env.dist.destroy_process_group()
        return

    # ---- baselines on this box (rank 0, N=1 only): the oracle port on the host cores and on the GPU (torch eager) ----
    cpu = gpu_eager = None
    if env.world == 1:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        if damsm:
            cstep, cunits = ref_damsm_step(48, CFG_BATCH["cfg4"] if wl != "cfg2" else 48)
            csample = ("oracle/ref_port.py WordsLoss+SentenceLoss fwd+bwd on the first 48 samples of the workload's batch "
                       "(48x48 pairs per step), fp32, 3 steps after 1 warm-up")
            gstep, gunits = ref_damsm_step(128, max(128, CFG_BATCH.get(wl, 128)), device=env.dev)
            gsample = "oracle/ref_port.py (torch eager: ATen + cuBLAS) on cuda:0, first 128 samples (128x128 pairs), fp32"
        else:
            cstep, cunits = ref_attn_step(16, 32, 256, 18, 64)
            csample = "oracle/ref_port.py word_attention fwd+bwd at B=16, 64x64 (cfg1 shape), fp32, 3 steps after 1 warm-up"
            gstep, gunits = ref_attn_step(16, 32, 256, 18, 128, device=env.dev)
            gsample = "oracle/ref_port.py word_attention (torch eager) on cuda:0, B=16, 128x128, fp32"
        csec = time_host(cstep, 3, 1)
        cpu = {"value": cunits / csec, "unit": m["unit"], "cores": torch.get_num_threads(), "kind": "port", "sample": csample}
        try:
            gsec = time_host(gstep, 5, 2, sync=torch.cuda.synchronize)
            gpu_eager = {"value": gunits / gsec, "unit": m["unit"], "sample": gsample,
                         "note": "per-unit rate of the reference's own op sequence on this B200; not the product"}
        except Exception as e:
            gpu_eager = {"error": f"{type(e).__name__}: {e}"}

    sec, sec2 = m["value"], m["e2e"]
    e2e_how = "graph replay, copies on the compute stream" if m["e2e_graph"] else "eager, copies on the compute stream"
    if m.get("e2e_pipelined") and m["e2e_pipelined"] < sec2:
        sec2 = m["e2e_pipelined"]
        e2e_how = "eager, HostPrefetcher: the copy of step i+1 overlaps the kernels of step i (attention-gan_b200/agb_native/pipeline.py)"
    line = {"metric": m["metric"], "value": m["total_units"] / sec, "unit": m["unit"], "n_gpus": env.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong" if wl in ("cfg4", "cfg5", "cfg4step") else "weak", "vs_baseline": None, "dtype": m["dtype"],
            "data": "synthetic", "config": {"workload": name},
            "method": {"math": args.math if damsm else None,
                       "l2": "256 MiB write between timed iterations (outside the events)",
                       "timing": "CUDA events per step on the current stream, barrier + synchronize on both sides, max over ranks",
                       "cuda_graph": {"value": m["graph"], "e2e": m["e2e_graph"]},
                       "sharding": ("rows [k*B/N,(k+1)*B/N) per rank, NCCL all-gather of word features + similarity blocks, "
                                    "reduce-scatter of d words" if env.world > 1 and damsm else
                                    ("batch split over the ranks, no collective" if env.world > 1 else "single process")),
                       "roofline_timing": f"library CUDA events around each kernel in an eager pass of {m['prof_steps']} steps"},
            "eager": {"value": m["total_units"] / m["eager"], "ms_per_step": m["eager"] * 1e3},
            "e2e": {"value": m["total_units"] / sec2, "unit": m["unit"], "h2d_bytes_per_step": m["h2d"],
                    "d2h_bytes_per_step": m["d2h"], "ms_per_step": sec2 * 1e3, "how": e2e_how},
            "e2e_eager": {"value": m["total_units"] / m["e2e_eager"], "ms_per_step": m["e2e_eager"] * 1e3,
                          "note": "copies on the compute stream, no graph"},
            "e2e_variants_ms": {"sequential_graph": m["e2e"] * 1e3 if m["e2e_graph"] else None,
                                "sequential_eager": m["e2e_eager"] * 1e3,
                                "pipelined_eager": m["e2e_pipelined"] * 1e3 if m.get("e2e_pipelined") else None},
            "gpu_launches": int(m["launches_per_step"] * args.steps), "gpu_launches_per_step": m["launches_per_step"],
            "roofline": roof, "cpu_baseline": cpu, "torch_eager_gpu": gpu_eager, "clocks": m["clocks"]}
    if secondary:
        line["secondary"] = secondary
    print(json.dumps(line), flush=True)
    if env.world > 1:
        env.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5", "cfg4step"])
    ap.add_argument("--math", default=None, choices=["fp32", "f16", "bf16", "f16x2"])
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--hw", type=int, default=None, help="attention workloads: a single feature-map side instead of the config's stages")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false",
                    help="N=1: skip the cfg2 / cfg3 / cfg5 measurements reported under 'secondary'")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy; 60 MiB in all, an output "
                         "above its share is written as a fixed, seeded sample of its elements")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs; it needs --impl native")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.math is None:
        import attention_gan_b200 as pkg
        args.math = "f16" if pkg.native.lib().agb_has_tcgen05() else "fp32"
    run_native(args)


if __name__ == "__main__":
    main()
