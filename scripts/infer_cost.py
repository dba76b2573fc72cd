#!/usr/bin/env python
"""Cost of sliding-window MM_Net prediction (mmunet_b200/infer.py) on one GPU -> JSON (default profiles/r4_inference.json).

  forward     MM_Net forward at 512x512, batch 16, bf16 autocast, channels-last: forward-only (no_grad: the Mamba Functions skip the
              scan-state stores and save nothing) against grad-saving (grad mode on, output kept), eager and as a CUDA-graph replay;
              median ms per forward and peak allocated memory (eager)
  predictor   SlidingWindowPredictor(roi 512, overlap 0.5, sw_batch_size 8, bf16, channels-last) images/s on 584x565 images
              (4 windows each), 1024x1024 images (9 windows) and one 2336x3504 image (117 windows), graph against eager
  stitch      the mmu_sw_stitch launch against the torch composition it replaces (per window: F.interpolate of the five heads,
              four adds, accumulate into the image and a count map; then one divide), on the same head maps

Variants of one measurement alternate round by round; every figure is the median over rounds of CUDA-event times.  The GPU's name
and power limit are read in the same run and stored with the numbers.

    python scripts/infer_cost.py [--out PATH] [--rounds R]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mm-unet_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def timed(fn, reps=1):
    """ms of `reps` calls of fn on the current stream (CUDA events)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def alternate(variants, rounds, reps=1):
    """{name: median ms}: one timed call of every variant per round, in turn."""
    for fn in variants.values():       # warm-up
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            times[k].append(timed(fn, reps))
    return {k: statistics.median(v) for k, v in times.items()}


def net_512(channels_last=True):
    from mmunet_b200.mm_net import MM_Net
    torch.manual_seed(50)
    net = MM_Net(num_classes=1).cuda().eval()
    return net.to(memory_format=torch.channels_last) if channels_last else net


def forward_cost(rounds):
    net = net_512()
    x = torch.randn(16, 3, 512, 512, device="cuda").contiguous(memory_format=torch.channels_last)

    def fwd(grad):
        with torch.set_grad_enabled(grad), torch.autocast("cuda", dtype=torch.bfloat16):
            return net(x)

    peak = {}
    for grad in (False, True, False, True):            # second pass of each: warm
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fwd(grad)
        torch.cuda.synchronize()
        peak["grad_saving" if grad else "forward_only"] = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
        del out
    graphs = {}
    for grad in (False, True):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fwd(grad)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            graphs[grad] = (g, fwd(grad))
    t = alternate({"eager_forward_only": lambda: fwd(False), "eager_grad_saving": lambda: fwd(True),
                   "graph_forward_only": graphs[False][0].replay, "graph_grad_saving": graphs[True][0].replay}, rounds)
    return {"shape": "B16 3x512x512 bf16 autocast channels-last, eval()", "ms": t, "peak_allocated_GiB_eager": peak}


def predictor_cost(rounds):
    from mmunet_b200.infer import SlidingWindowPredictor
    net = net_512()
    cases = {"drive_584x565_x8": torch.randn(8, 3, 584, 565, device="cuda"),
             "1024x1024_x4": torch.randn(4, 3, 1024, 1024, device="cuda"),
             "hrf_2336x3504_x1": torch.randn(1, 3, 2336, 3504, device="cuda")}
    preds = {g: SlidingWindowPredictor(net, roi_size=512, overlap=0.5, sw_batch_size=8, dtype="bf16", graph=g) for g in (False, True)}
    out = {}
    for name, x in cases.items():
        t = alternate({f"graph={g}": (lambda p=p: p.predict(x)) for g, p in preds.items()}, rounds)
        out[name] = {k: {"ms": v, "images_per_s": x.shape[0] * 1000.0 / v} for k, v in t.items()}
    return {"predictor": "roi 512, overlap 0.5, sw_batch_size 8, bf16 autocast, channels-last", "cases": out}


def torch_stitch(heads, H, W, roi, overlap):
    from mmunet_b200.infer import pad_for_roi, window_starts
    B = heads[0].shape[0]
    (pt, pb), (pl, pr) = pad_for_roi(H, roi), pad_for_roi(W, roi)
    nh, nw = H + pt + pb, W + pl + pr
    acc = torch.zeros(B, 1, nh, nw, device="cuda")
    cnt = torch.zeros(1, 1, nh, nw, device="cuda")
    wins = [(a, b) for a in window_starts(nh, roi, overlap) for b in window_starts(nw, roi, overlap)]
    for w, (a, b) in enumerate(wins):
        v = None
        for h in heads:
            up = F.interpolate(h[:, w:w + 1].float(), size=(roi, roi), mode="bilinear", align_corners=True)
            v = up if v is None else v + up
        acc[:, :, a:a + roi, b:b + roi] += v
        cnt[:, :, a:a + roi, b:b + roi] += 1
    return (acc / cnt)[:, :, pt:pt + H, pl:pl + W]


def stitch_cost(rounds):
    from mmunet_b200.infer import pad_for_roi, sw_stitch, window_starts
    out = {}
    for name, (B, H, W) in {"drive_584x565_x8": (8, 584, 565), "hrf_2336x3504_x1": (1, 2336, 3504)}.items():
        nwin = len(window_starts(H + sum(pad_for_roi(H, 512)), 512, .5)) * len(window_starts(W + sum(pad_for_roi(W, 512)), 512, .5))
        heads = [torch.randn(B, nwin, s, s, device="cuda").to(torch.bfloat16) for s in (256, 128, 64, 32, 256)]
        a, b = sw_stitch(heads, (H, W), 512, .5)[0], torch_stitch(heads, H, W, 512, .5)
        err = float((a - b).abs().max() / b.abs().max())
        t = alternate({"sw_stitch": lambda: sw_stitch(heads, (H, W), 512, .5), "torch": lambda: torch_stitch(heads, H, W, 512, .5)},
                      rounds, reps=5)
        out[name] = {"windows_per_image": nwin, "ms": t, "speedup": t["torch"] / t["sw_stitch"], "max_rel_diff": err}
    return {"heads": "bf16, 5 maps per window (256, 128, 64, 32, 256 squared)", "cases": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_inference.json"))
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("infer_cost.py measures on a CUDA device; none is available")
    res = {"gpu": gpu_info(), "rounds": a.rounds, "statistic": "median over alternating rounds, CUDA events",
           "stitch": stitch_cost(a.rounds), "forward": forward_cost(a.rounds), "predictor": predictor_cost(a.rounds)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
