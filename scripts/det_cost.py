"""Cost of deterministic mode: the default (atomic) and the deterministic (_det) path of every accumulating op, timed alternately with
CUDA events at the sizes users run, plus the largest workspace the deterministic path allocated.
Usage: python scripts/det_cost.py [--out profiles/r3_deterministic.json] [--reps 20]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "mm-unet_b200")]
from mmunet_b200 import ops  # noqa: E402

DEV = "cuda"


def set_mode(det):
    torch.use_deterministic_algorithms(det, warn_only=True)


def time_pair(fn, reps):
    """Median ms of fn() with the mode off and on, the two alternating call by call (after a warm-up of each)."""
    ms = {False: [], True: []}
    for det in (False, True):
        set_mode(det)
        fn()
    torch.cuda.synchronize()
    for _ in range(reps):
        for det in (False, True):
            set_mode(det)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[det].append(a.elapsed_time(b))
    set_mode(False)
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    return {"default_ms": round(med[False], 4), "deterministic_ms": round(med[True], 4), "ratio": round(med[True] / med[False], 3)}


def scan_case(B, D, L, N, dtype):
    g = torch.Generator(device="cpu").manual_seed(0)
    u, z, dout = (torch.randn(B, D, L, generator=g).to(DEV, dtype) for _ in range(3))
    delta = (0.5 * torch.rand(B, D, L, generator=g)).to(DEV, dtype)
    A = (-0.5 * torch.rand(D, N, generator=g)).to(DEV)
    Bm, Cm = (torch.randn(B, 1, N, L, generator=g).to(DEV, dtype) for _ in range(2))
    Dp, bias = torch.randn(D, generator=g).to(DEV), (0.5 * torch.rand(D, generator=g)).to(DEV)
    _, x, _ = ops.selective_scan_fwd(u, delta, A, Bm, Cm, Dp, z, bias, True)
    return lambda: ops.selective_scan_bwd(u, delta, A, Bm, Cm, Dp, z, bias, dout, x, True)


def conv_case(B, D, L, dtype):
    x, dout = torch.randn(B, D, L, device=DEV).to(dtype), torch.randn(B, D, L, device=DEV).to(dtype)
    w, b = torch.randn(D, 4, device=DEV), torch.randn(D, device=DEV)
    return lambda: ops.causal_conv1d_bwd(x, w, b, dout, True)


def narrow_case(B, L, dtype):
    torch.manual_seed(0)
    dm, di, N = 3, 6, 16
    ws = [0.5 * torch.randn(2 * di, dm), 0.5 * torch.randn(di, 1, 4), 0.1 * torch.randn(di), 0.3 * torch.randn(1 + 2 * N, di),
          0.5 * torch.randn(di, 1), 0.4 * torch.randn(dm, di), -torch.rand(di, N) - 0.2, torch.randn(di), 0.3 * torch.rand(di)]
    ws = [w.to(DEV).requires_grad_() for w in ws]
    hidden = torch.randn(B, dm, L, device=DEV).to(dtype).requires_grad_()
    H = W = int(L ** 0.5)
    out = ops.mamba_narrow_fn(hidden, *ws, order=(3, H, W, 1))
    gy = torch.randn_like(out)
    return lambda: torch.autograd.grad(out, [hidden] + ws, gy, retain_graph=True)


def snake_case(B, C, H, W, K):
    feat = torch.randn(B, C, H, W, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_()
    y = (torch.arange(H, device=DEV).view(1, 1, H, 1) + 1.7 * torch.randn(B, K, H, W, device=DEV)).float().requires_grad_()
    out = ops.snake_sample(feat, y, torch.bfloat16)
    g = torch.randn_like(out)
    return lambda: torch.autograd.grad(out, (feat, y), g, retain_graph=True)


def gn_fwd_case(B, C, H, W):
    x = torch.randn(B, C, H, W, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    w, b = torch.randn(C, device=DEV), torch.randn(C, device=DEV)
    return lambda: ops.group_norm_nhwc(x, C // 4, w, b, 1e-5, torch.bfloat16)


def gn_bwd_case(B, C, H, W):
    x = torch.randn(B, C, H, W, device=DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_()
    w, b = torch.randn(C, device=DEV, requires_grad=True), torch.randn(C, device=DEV, requires_grad=True)
    y = ops.group_norm_nhwc(x, C // 4, w, b, 1e-5, torch.bfloat16)
    g = torch.randn_like(y)
    return lambda: torch.autograd.grad(y, (x, w, b), g, retain_graph=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_deterministic.json"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "det_cost.py needs a CUDA device"
    L_ = ops._lib.lib()
    cases = [
        ("scan_bwd config2 fp32 (B8 D384 L4096 N16)", lambda: scan_case(8, 384, 4096, 16, torch.float32),
         L_.mmu_selective_scan_bwd_det_workspace(8, 384, 4096, 16)),
        ("scan_bwd config2 bf16", lambda: scan_case(8, 384, 4096, 16, torch.bfloat16), L_.mmu_selective_scan_bwd_det_workspace(8, 384, 4096, 16)),
        ("scan_bwd RCG bf16 (B16 D128 L16384 N16)", lambda: scan_case(16, 128, 16384, 16, torch.bfloat16),
         L_.mmu_selective_scan_bwd_det_workspace(16, 128, 16384, 16)),
        ("conv_bwd config2 fp32 (B8 D384 L4096 W4)", lambda: conv_case(8, 384, 4096, torch.float32),
         L_.mmu_causal_conv1d_bwd_det_workspace(8, 384, 4096, 0)),
        ("conv_bwd config2 bf16", lambda: conv_case(8, 384, 4096, torch.bfloat16), L_.mmu_causal_conv1d_bwd_det_workspace(8, 384, 4096, 1)),
        ("narrow block bwd bf16 (B16 L65536, two-row order)", lambda: narrow_case(16, 65536, torch.bfloat16),
         max(L_.mmu_mamba_narrow_pre_bwd_det_workspace(16, 65536), L_.mmu_mamba_narrow_post_bwd_det_workspace(16, 65536))),
        ("snake sampler bwd NHWC bf16 (B16 C64 128x128 K3: 512^2 input, first stage)", lambda: snake_case(16, 64, 128, 128, 3), 0),
        ("group_norm NHWC fwd bf16 (B16 C64 128x128)", lambda: gn_fwd_case(16, 64, 128, 128),
         L_.mmu_group_norm_nhwc_fwd_det_workspace(16, 64, 128 * 128, 16)),
        ("group_norm NHWC bwd bf16 (B16 C64 128x128)", lambda: gn_bwd_case(16, 64, 128, 128),
         L_.mmu_group_norm_nhwc_bwd_det_workspace(16, 64, 128 * 128, 16)),
    ]
    rows = []
    for name, make, ws in cases:
        fn = make()
        r = time_pair(fn, args.reps)
        r.update(case=name, workspace_bytes=int(ws))
        rows.append(r)
        print(json.dumps(r), flush=True)
        del fn
        torch.cuda.empty_cache()
    res = {"gpu": gpu_info(), "timing": "CUDA events, median of %d alternating calls per mode, after one warm-up call each" % args.reps,
           "peak_workspace_bytes": max(r["workspace_bytes"] for r in rows), "cases": rows}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "peak_workspace_bytes": res["peak_workspace_bytes"]}))


if __name__ == "__main__":
    main()
