"""Deterministic MM_Net training: which ops torch flags, what the mode costs per step, and the resize backward against ATen's.

  ops     one eager Trainer step (image 64, batch 2) under torch.use_deterministic_algorithms(True, warn_only=True), fp32 NCHW and
          bf16 channels-last: every "does not have a deterministic implementation" alert, with MM_Net's resizes on plain
          F.interpolate (as before ops.resize_bilinear) and as shipped; then the same step in strict mode (raises or not).
  step    512x512, batch 16, bf16 autocast, channels-last, whole-step CUDA graph: ms/step with the mode off and in strict mode, the two
          trainers alternating step by step (CUDA events around each replay).
  resize  the resize backward at each of MM_Net's resize shapes (batch 16, 512x512 input): ours (mmu_resize_bilinear_bwd_det) against
          ATen's atomic kernel, CUDA events over many launches; algorithmic bytes = read dout + write dx.
Usage: CUBLAS_WORKSPACE_CONFIG=:4096:8 python scripts/det_train_cost.py [--out profiles/r3_det_training.json] [--steps 20]"""
import argparse
import json
import os
import subprocess
import sys
import warnings

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "mm-unet_b200")]
from mmunet_b200 import mm_net, ops  # noqa: E402
from mmunet_b200.train import Trainer  # noqa: E402

DEV = "cuda"


def _plain_resize(x, size=None, scale_factor=None):
    return F.interpolate(x, size=size, scale_factor=scale_factor, mode="bilinear", align_corners=True)


def one_step(dtype, cl):
    tr = Trainer(image_size=64, batch_per_rank=2, dtype=dtype, device="cuda:0", ddp=False, channels_last=cl, graph=False)
    tr.set_epoch(2)
    x, y = tr.synthetic_batch()
    return float(tr.step(x, y))


def _warnings_of(fn):
    """Deterministic-mode alerts of fn(): Python warnings and what torch prints to stderr (alerts raised on the autograd thread)."""
    import tempfile
    with tempfile.TemporaryFile(mode="w+") as tmp, warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(tmp.fileno(), 2)
        try:
            fn()
            torch.cuda.synchronize()
        finally:
            sys.stderr.flush()
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        lines = [str(m.message) for m in w] + tmp.read().splitlines()
    return sorted({ln.strip()[:200] for ln in lines if "deterministic" in ln})


def flagged_ops():
    out = {}
    shipped = ops.resize_bilinear
    try:
        for dtype, cl in (("fp32", False), ("bf16", True)):
            key = f"{dtype}_{'channels_last' if cl else 'nchw'}"
            out[key] = {}
            for variant in ("interpolate", "shipped"):
                mm_net.ops.resize_bilinear = _plain_resize if variant == "interpolate" else shipped
                torch.use_deterministic_algorithms(True, warn_only=True)
                out[key][variant + "_warn_only"] = _warnings_of(lambda: one_step(dtype, cl))
                torch.use_deterministic_algorithms(True)
                try:
                    out[key][variant + "_strict"] = f"ok (loss {one_step(dtype, cl):.4f})"
                except RuntimeError as e:
                    out[key][variant + "_strict"] = "raised: " + str(e).strip().split("\n")[0][:300]
                torch.use_deterministic_algorithms(False)
    finally:
        mm_net.ops.resize_bilinear = shipped
        torch.use_deterministic_algorithms(False)
    return out


def step_cost(steps):
    trs = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        tr = Trainer(image_size=512, batch_per_rank=16, dtype="bf16", device="cuda:0", ddp=False, channels_last=True, graph=True)
        tr.set_epoch(2)
        batch = tr.synthetic_batch()
        for _ in range(tr.graph_warmup + 3):            # eager warm-up, capture, replays
            tr.step(*batch)
        torch.cuda.synchronize()
        trs[det] = (tr, batch)
    ms = {False: [], True: []}
    for _ in range(steps):
        for det in (False, True):
            torch.use_deterministic_algorithms(det)
            tr, batch = trs[det]
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(tr.stream)
            tr.step(*batch)
            b.record(tr.stream)
            b.synchronize()
            ms[det].append(a.elapsed_time(b))
    torch.use_deterministic_algorithms(False)
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    res = {"config": "MM_Net 512x512, batch 16, bf16 autocast, channels-last, whole-step CUDA graph, 1 GPU", "timed_steps": steps,
           "default_ms": round(med[False], 3), "deterministic_ms": round(med[True], 3), "ratio": round(med[True] / med[False], 3),
           "default_ms_all": [round(v, 3) for v in ms[False]], "deterministic_ms_all": [round(v, 3) for v in ms[True]],
           "graphed": [trs[d][0].graph is not None for d in (False, True)]}
    del trs
    torch.cuda.empty_cache()
    return res


# (C, H_in, W_in, H_out, W_out) of MM_Net at a 512x512 input
RESIZE_SHAPES = [(64, 16, 16, 32, 32), (64, 32, 32, 64, 64), (64, 64, 64, 128, 128), (64, 128, 128, 256, 256),
                 (64, 256, 256, 128, 128), (64, 256, 256, 64, 64), (64, 256, 256, 32, 32),
                 (1, 256, 256, 512, 512), (1, 128, 128, 512, 512), (1, 64, 64, 512, 512), (1, 32, 32, 512, 512)]


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def resize_cost(batch=16, reps=200):
    rows = []
    for dtype, cl in ((torch.bfloat16, True), (torch.float32, False)):
        fmt = torch.channels_last if cl else torch.contiguous_format
        for C, Hi, Wi, Ho, Wo in RESIZE_SHAPES:
            d = torch.randn(batch, C, Ho, Wo, device=DEV).to(dtype).contiguous(memory_format=fmt)
            ours = lambda: ops.resize_bilinear_bwd(d, (Hi, Wi), cl)
            aten = lambda: torch.ops.aten.upsample_bilinear2d_backward(d, [Ho, Wo], [batch, C, Hi, Wi], True, None, None)
            t = {}
            for _ in range(3):                           # alternate: three rounds, best of each
                for name, fn in (("ours", ours), ("aten", aten)):
                    t[name] = min(t.get(name, 1e9), time_ms(fn, reps))
            nbytes = (d.numel() + batch * C * Hi * Wi) * d.element_size()
            rows.append({"dtype": str(dtype).replace("torch.", ""), "layout": "NHWC" if cl else "NCHW", "shape": [batch, C, Hi, Wi, Ho, Wo],
                         "ours_us": round(t["ours"] * 1e3, 2), "aten_us": round(t["aten"] * 1e3, 2),
                         "ours_GBps": round(nbytes / (t["ours"] * 1e-3) / 1e9, 1), "aten_GBps": round(nbytes / (t["aten"] * 1e-3) / 1e9, 1),
                         "algorithmic_bytes": nbytes})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--skip", default="", help="comma-separated sections to skip: ops, step, resize")
    args = ap.parse_args()
    if os.environ.get("CUBLAS_WORKSPACE_CONFIG") not in (":4096:8", ":16:8"):
        sys.exit("set CUBLAS_WORKSPACE_CONFIG=:4096:8 before running (strict mode refuses cuBLAS otherwise)")
    assert torch.cuda.is_available(), "needs a CUDA device"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown", "torch": torch.__version__}
    skip = set(filter(None, args.skip.split(",")))
    if "ops" not in skip:
        res["flagged_ops"] = flagged_ops()
    if "resize" not in skip:
        res["resize_bwd"] = resize_cost()
    if "step" not in skip:
        res["train_step"] = step_cost(args.steps)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
