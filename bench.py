#!/usr/bin/env python
"""bench.py - headline benchmark of the B200-native Mamba-block hot path.

Workload (BASELINE.json configs[1]): the isolated Mamba block - causal_conv1d (width 4, SiLU) forward, selective scan
forward, selective scan backward, causal_conv1d backward - at B=8, D=384, L=4096 (a 64x64 map), d_state=16, with
z-gate, D-skip, delta-bias and softplus, on synthetic data in the reference tests' distributions.  One "step" is one
pass of those four kernels over one batch.  `value` is BASELINE.json's metric itself - selective-scan fwd+bwd algorithmic
HBM bytes ((11D+6N)BLs, BASELINE.md section 3) over the time the scan forward and backward took inside the step (CUDA
events around each kernel) - against the HBM roofline; the whole block including the conv kernels is the side key `block`.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype fp32|bf16] [--impl ours|reference] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as DIR/<name>.npy in float32: the results a caller of
the four ops receives (conv_out, scan_out, du, ddelta, dA, dB, dC, dD, dz, ddelta_bias, dx, dweight, dbias; not the saved-state
checkpoint, whose layout is private to the kernels).  The (batch, channel)-by-L tensors are cut to a fixed, seeded sample of
DUMP_ROWS rows so the dump stays near 30 MB; the inputs are seeded too, so two builds run with the same arguments can be
compared output for output.

N > 1 is launched by torchrun (one rank per GPU); every rank runs its own batch (weak scaling, no data-path collective:
every (batch, channel) scan lane is independent - SURVEY.md section 8e); time = max over ranks, value = sum of bytes / time.

`--impl reference` times the CPU path for the SAME step - same B, D, L, N, the same number of steps and warm-up steps - on
all host cores: the C/OpenMP restatement of the reference's selective_scan_ref / causal_conv1d_ref algorithm
(oracle/scan_oracle.c, kind "port"; the reference's pure-PyTorch loop needs ~17 s per full-config step).  The pure-PyTorch
form (oracle/torch_ref.py, the reference's own arithmetic op for op) is timed on a bounded sample and reported beside
it as `pytorch_ref_sample`, labelled as a sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "mm-unet_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

B, D, L, N, W = 8, 384, 4096, 16, 4
METRIC = "selective-scan fwd+bwd HBM GB/s vs peak (isolated Mamba block B8 D384 L4096 N16, algorithmic bytes); MM-UNet train img/s in `train`"


def algo_bytes(batch, s):
    scan_f = (4 * D + 2 * N) * batch * L * s
    scan_b = (7 * D + 4 * N) * batch * L * s
    conv_f = 2 * batch * D * L * s
    conv_b = 3 * batch * D * L * s
    return dict(scan_fwd=scan_f, scan_bwd=scan_b, conv_fwd=conv_f, conv_bwd=conv_b, step=scan_f + scan_b + conv_f + conv_b)


def make_inputs(batch, dtype, device, seed=0, pin=False):
    """Reference test distributions (tests/ops/test_selective_scan.py:58-88, tests/test_causal_conv1d.py:39-50)."""
    g = torch.Generator().manual_seed(seed)
    t = dict(
        x=torch.randn(batch, D, L, generator=g), delta=0.5 * torch.rand(batch, D, L, generator=g),
        z=torch.randn(batch, D, L, generator=g), Bm=torch.randn(batch, 1, N, L, generator=g),
        Cm=torch.randn(batch, 1, N, L, generator=g), dout=torch.randn(batch, D, L, generator=g))
    w = dict(A=-0.5 * torch.rand(D, N, generator=g), Dp=torch.randn(D, generator=g), dbias=0.5 * torch.rand(D, generator=g),
             cw=torch.randn(D, W, generator=g), cb=torch.randn(D, generator=g))
    t = {k: v.to(dtype) for k, v in t.items()}
    if pin:
        t = {k: v.pin_memory() for k, v in t.items()}
    else:
        t = {k: v.to(device) for k, v in t.items()}
    w = {k: v.to(device) for k, v in w.items()}
    return t, w


DUMP_ROWS = 256
GRAD_NAMES = ("du", "ddelta", "dA", "dB", "dC", "dD", "dz", "ddelta_bias")      # ops.selective_scan_bwd's results, in order


def dump_outputs(outdir, outs):
    """Writes outs (name -> tensor) as outdir/<name>.npy in float32.  A (B, D, L) tensor keeps only DUMP_ROWS of its B*D rows,
    the same seeded sample (in ascending row order) for every tensor and every run."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    rows = torch.randperm(B * D, generator=torch.Generator().manual_seed(1234))[:DUMP_ROWS].sort().values
    for name, v in outs.items():
        if v.shape[:2] == (B, D) and v.dim() == 3:
            v = v.reshape(B * D, -1)[rows.to(v.device)]
        np.save(os.path.join(outdir, name + ".npy"), v.detach().float().cpu().numpy())


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with nvidia-smi while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, threading.Event(), []

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bind_to_gpu_numa(index):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU BEFORE any pinned staging buffer is allocated:
    first-touch then places the staging pages on the GPU's NUMA node, so the per-step H2D copies of N ranks do not all cross one
    socket (VERDICT r1 weak item 5: e2e scaled 0.53 / 0.43 at 4 / 8 GPUs).  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, ((os.cpu_count() or 64) + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        numa = None
        try:
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
            numa = int(open(f"/sys/bus/pci/devices/{bus[-12:]}/numa_node").read())       # "00000000:1b:00.0" -> "0000:1b:00.0"
        except Exception:
            pass
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"cpus_bound": len(cpus), "first_cpu": cpus[0] if cpus else None, "gpu_numa_node": numa, "host_cpus": os.cpu_count()}
    except Exception as exc:
        return {"error": repr(exc)}


def reduce_max_ms(ms, dist, device=None):
    """Timing rule of the bench contract: a multi-rank number is the MAX over ranks (backend-agnostic: NCCL or gloo)."""
    if dist is None or not dist.is_initialized():
        return float(ms)
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_gbps(world, bytes_per_rank, ms):
    """Weak scaling: every rank processes its own batch; value = all ranks' algorithmic bytes / max-over-ranks time."""
    return world * bytes_per_rank / (ms * 1e-3) / 1e9


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu summary (profiles/), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def cpu_baseline_port(sample_batch=B, min_seconds=10.0, max_reps=8):
    """The oracle's C port (OpenMP over all host cores) on a bounded sample of the same step: the full batch, repeated
    until about 10 s of CPU work have been timed."""
    import oracle
    oracle.set_num_threads(len(os.sched_getaffinity(0)))
    t, w = make_inputs(sample_batch, torch.float32, "cpu")
    n = {k: v.numpy() for k, v in {**t, **w}.items()}
    reps, t0, scan_s = 0, time.perf_counter(), 0.0
    while reps < max_reps and (reps == 0 or time.perf_counter() - t0 < min_seconds):
        u = oracle.causal_conv1d_fwd(n["x"], n["cw"], n["cb"], True)
        t1 = time.perf_counter()
        oracle.selective_scan_fwd(u, n["delta"], n["A"], n["Bm"], n["Cm"], n["Dp"], n["z"], n["dbias"], True)
        g = oracle.selective_scan_bwd(u, n["delta"], n["A"], n["Bm"], n["Cm"], n["Dp"], n["z"], n["dbias"], n["dout"], True)
        scan_s += time.perf_counter() - t1
        oracle.causal_conv1d_bwd(n["x"], n["cw"], n["cb"], g["du"], True)
        reps += 1
    dt = (time.perf_counter() - t0) / reps
    nb = algo_bytes(sample_batch, 4)
    return {"value": (nb["scan_fwd"] + nb["scan_bwd"]) / (scan_s / reps) / 1e9, "unit": "GB/s", "cores": oracle.num_threads(),
            "kind": "port", "sample": f"{reps} x full step (batch {sample_batch}, D={D}, L={L}, N={N}), fp32, "
            f"oracle/scan_oracle.c (OpenMP), {dt:.2f} s per step; value = scan fwd+bwd bytes / scan seconds, as the GPU arm",
            "seconds_per_step": dt, "block_value": nb["step"] / dt / 1e9}


def run_reference(args):
    """Reference arm: the CPU path on the FULL config (B=8, D=384, L=4096, N=16), exactly `--steps` timed steps after `--warmup`
    warm-up steps, all host cores; the metric is the same one the GPU arm prints (scan fwd+bwd bytes / scan fwd+bwd time)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from oracle import torch_ref
    host_cores = len(os.sched_getaffinity(0))       # torchrun exports OMP_NUM_THREADS=1: use every core this process may run on
    torch.set_num_threads(host_cores)
    oracle.set_num_threads(host_cores)
    t, w = make_inputs(B, torch.float32, "cpu")
    n = {k: v.numpy() for k, v in {**t, **w}.items()}
    nb = algo_bytes(B, 4)

    def step():
        t0 = time.perf_counter()
        u = oracle.causal_conv1d_fwd(n["x"], n["cw"], n["cb"], True)
        t1 = time.perf_counter()
        oracle.selective_scan_fwd(u, n["delta"], n["A"], n["Bm"], n["Cm"], n["Dp"], n["z"], n["dbias"], True)
        g = oracle.selective_scan_bwd(u, n["delta"], n["A"], n["Bm"], n["Cm"], n["Dp"], n["z"], n["dbias"], n["dout"], True)
        t2 = time.perf_counter()
        oracle.causal_conv1d_bwd(n["x"], n["cw"], n["cb"], g["du"], True)
        return t2 - t1, time.perf_counter() - t0

    for _ in range(args.warmup):
        step()
    scan_s = step_s = 0.0
    for _ in range(args.steps):
        a, b_ = step()
        scan_s, step_s = scan_s + a, step_s + b_
    scan_s, step_s = scan_s / args.steps, step_s / args.steps
    val = (nb["scan_fwd"] + nb["scan_bwd"]) / scan_s / 1e9

    # the reference's own pure-PyTorch arithmetic on a bounded sample (batch 1 of 8, all 384 channels), 2 steps
    ts, ws = make_inputs(1, torch.float32, "cpu")
    pt = []
    for _ in range(2):
        leaves = {k: v.clone().requires_grad_() for k, v in {**ts, **ws}.items() if k != "dout"}
        t0 = time.perf_counter()
        u = torch_ref.causal_conv1d(leaves["x"], leaves["cw"], leaves["cb"], "silu")
        t1 = time.perf_counter()
        out = torch_ref.selective_scan(u, leaves["delta"], leaves["A"], leaves["Bm"], leaves["Cm"], leaves["Dp"], leaves["z"], leaves["dbias"], True)
        out.backward(ts["dout"])
        pt.append(time.perf_counter() - t1)
    nb1 = algo_bytes(1, 4)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config("fp32"),
            "value_basis": "scan fwd+bwd algorithmic bytes / scan fwd+bwd seconds inside the step (same definition as the GPU arm)",
            "block": {"value": nb["step"] / step_s / 1e9, "unit": "GB/s", "what": "whole step incl. causal_conv1d fwd/bwd"},
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": oracle.num_threads(), "kind": "port",
                             "sample": f"{args.steps} x the FULL step (batch {B}, D={D}, L={L}, N={N}), fp32, oracle/scan_oracle.c (C/OpenMP restatement of "
                                       f"selective_scan_ref / causal_conv1d_ref), {step_s:.2f} s per step"},
            "pytorch_ref_sample": {"value": (nb1["scan_fwd"] + nb1["scan_bwd"]) / min(pt) / 1e9, "unit": "GB/s", "cores": torch.get_num_threads(),
                                   "seconds_per_sample_step": min(pt),
                                   "sample": f"batch 1 of {B}, all {D} channels, L={L}: the reference's pure-PyTorch selective_scan_ref arithmetic "
                                             "(oracle/torch_ref.py, O(L) autograd form), scan fwd+bwd only; NOT the timed reference value"},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(io_dtype):
    """Identical for both arms, so the driver's same_config check compares like with like."""
    return {"workload": f"isolated Mamba block: causal_conv1d(w={W},silu) fwd -> selective_scan fwd -> bwd -> conv1d bwd; "
                        f"B={B} D={D} L={L} d_state={N}, z+D+delta_bias+softplus; per-GPU batch fixed (weak scaling)",
            "l2": "inputs (818 MB fp32 / 409 MB bf16 per step) larger than the 126 MB L2", "io_dtype": io_dtype}


def train_leg(args, rank, world, dev, dist, image_size, global_batch, steps):
    """MM-UNet (MM_Net) training img/s on synthetic DRIVE-shaped batches: forward, DiceFocal loss, backward, AdamW step;
    bf16 autocast; one rank per GPU with torch DDP (NCCL gradient all-reduce overlapped with backward).  STRONG scaling, as
    the reference's DDP run does (train.py:252-253, train.sh): the global batch is fixed and split over the ranks
    (BASELINE configs[2]: 16 -> 16/8/4/2 per rank; configs[3]: 8 -> 8/4/2/1).  Every step starts from PINNED HOST tensors
    (H2D inside the timed region) and ends with the loss copied back to the host."""
    from mmunet_b200.train import Trainer
    per_rank = max(1, global_batch // world)
    tr = Trainer(image_size=image_size, batch_per_rank=per_rank, dtype="bf16", device=dev, channels_last=True)
    tr.set_epoch(tr.warmup_epochs)        # full learning rate (epoch 0 of the reference's schedule trains with lr = 0)
    batches = [tr.synthetic_batch() for _ in range(2)]
    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    warm = tr.graph_warmup + 3 if tr.use_graph else 3     # eager warm-up, CUDA-graph capture, then replayed warm-up steps
    for i in range(warm):
        tr.step(*batches[i % 2])
    torch.cuda.synchronize()
    if dist: dist.barrier()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    s.record()
    for i in range(steps):
        loss = tr.step(*batches[i % 2])
        host_loss.copy_(loss.reshape(1), non_blocking=True)
    e.record()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = reduce_max_ms(s.elapsed_time(e), dist, dev) / steps
    xb, yb = batches[0]
    res = {"metric": "MM-UNet train img/s", "value": world * per_rank / (ms * 1e-3), "unit": "img/s",
           "ms_per_step": ms, "steps": steps, "warmup": warm, "n_gpus": world, "scaling": "strong",
           "cuda_graph": tr.graph is not None,
           "config": {"model": "MM_Net (mmunet_b200/mm_net.py, 50 Mamba blocks)", "image": f"{image_size}x{image_size} RGB",
                      "per_gpu_batch": per_rank, "global_batch": world * per_rank, "dtype": "bf16 autocast", "memory_format": "channels_last",
                      "optimizer": "AdamW lr 1e-3 wd 0.05 betas (0.9,0.95)", "loss": "DiceFocal",
                      "parallelism": f"dp{world}" + (" (DDP, NCCL all-reduce overlapped with backward)" if world > 1 else "")},
           "h2d_bytes_per_step": xb.numel() * xb.element_size() + yb.numel() * yb.element_size(), "d2h_bytes_per_step": 4,
           "hot_path_launches_per_step": int(tr.hot_path_launches),
           "loss": float(host_loss.item()), "wall_s": wall, "data": "synthetic", "peak_mem_gib": torch.cuda.max_memory_allocated() / 2**30}
    del tr, batches
    torch.cuda.empty_cache()
    return res


_REAL_STDOUT = None


def quiet_stdout():
    """Only the JSON line may reach stdout: libraries (NCCL prints its version banner there) get stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--dtype", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the MM_Net training leg (the `train` object)")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--train-batch", type=int, default=16, help="GLOBAL batch of the 512x512 training leg (BASELINE configs[2]); split over the ranks")
    ap.add_argument("--train-size", type=int, default=512)
    ap.add_argument("--no-hires", action="store_true", help="skip the 1024x1024 / global batch 8 training leg (BASELINE configs[3])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path: use it with --impl ours")
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)

    from mmunet_b200 import _lib, ops
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    host_binding = bind_to_gpu_numa(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float32 if args.dtype == "fp32" else torch.bfloat16
    s = 4 if dtype == torch.float32 else 2
    nbytes = algo_bytes(B, s)
    t, w = make_inputs(B, dtype, dev, seed=rank)
    warm = max(3, args.warmup)

    # ---------------- device-resident arm: raw kernels through the C-ABI, per-kernel CUDA events -------------------
    du = torch.empty_like(t["x"]); dd = torch.empty_like(t["x"]); dz = torch.empty_like(t["x"]); dx = torch.empty_like(t["x"])
    names = ("conv_fwd", "scan_fwd", "scan_bwd", "conv_bwd")
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(args.steps)]

    def step(e=None):
        if e: e[0].record()
        u = ops.causal_conv1d_fwd(t["x"], w["cw"], w["cb"], True)
        if e: e[1].record()
        out, xs, _ = ops.selective_scan_fwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], True)
        if e: e[2].record()
        g = ops.selective_scan_bwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], t["dout"], xs, True,
                                   du=du, ddelta=dd, dz=dz)
        if e: e[3].record()
        _, dw, db = ops.causal_conv1d_bwd(t["x"], w["cw"], w["cb"], du, True, dx=dx)
        if e: e[4].record()
        return {"conv_out": u, "scan_out": out, **dict(zip(GRAD_NAMES, g)), "dx": dx, "dweight": dw, "dbias": db}

    for _ in range(warm):
        step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    t0 = time.perf_counter()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(args.steps):
        outs = step(ev[i])
        if i + 1 < args.steps:
            # freed before the next step allocates, so every timed step gets the same buffer placement; outputs kept
            # alive across steps move the scan's buffers to other addresses, which slows the scan forward
            del outs
    stop.record()
    torch.cuda.synchronize()
    if dist: dist.barrier()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    launches = _lib.launch_count() - n0
    dev_ms = start.elapsed_time(stop)
    dev_ms = reduce_max_ms(dev_ms, dist, dev)
    per_kernel = {n: sum(ev[i][k].elapsed_time(ev[i][k + 1]) for i in range(args.steps)) / args.steps for k, n in enumerate(names)}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)
    del outs

    # ---------------- end-to-end arm: public autograd API, pinned host buffers, H2D + D2H inside the timed region ---
    # Every step copies ITS inputs from pinned host memory and reads its loss back.  The copies run on a second stream into
    # one of two device buffer sets, so the H2D of step i+1 overlaps the kernels of step i (PCIe is the e2e bound here:
    # 205 MB fp32 per step); events order copy -> compute -> buffer reuse.
    ht, _ = make_inputs(B, dtype, dev, seed=rank, pin=True)
    dbufs = [{k: torch.empty_like(v, device=dev) for k, v in ht.items()} for _ in range(2)]
    host_loss = torch.empty(1, dtype=torch.float32).pin_memory()
    params = {k: w[k].clone().requires_grad_() for k in ("A", "Dp", "dbias", "cw", "cb")}
    copy_stream = torch.cuda.Stream(dev)
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def e2e_copy(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])                 # the compute that last read this buffer set is done
            for k in ht:
                dbufs[i % 2][k].copy_(ht[k], non_blocking=True)
            copied[i % 2].record(copy_stream)

    def e2e_compute(i):
        dbuf = dbufs[i % 2]
        torch.cuda.current_stream().wait_event(copied[i % 2])
        x = dbuf["x"].requires_grad_()
        u = ops.causal_conv1d_fn(x, params["cw"], params["cb"], "silu")
        out = ops.selective_scan_fn(u, dbuf["delta"], params["A"], dbuf["Bm"], dbuf["Cm"], params["Dp"], dbuf["z"],
                                    params["dbias"], True)
        loss = (out.float() * dbuf["dout"].float()).sum()
        loss.backward()
        host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        consumed[i % 2].record()
        dbuf["x"] = dbuf["x"].detach()
        for p_ in params.values():
            p_.grad = None

    def e2e_run(n):
        e2e_copy(0)
        for i in range(n):
            if i + 1 < n:
                e2e_copy(i + 1)
            e2e_compute(i)

    e2e_steps = max(3, args.steps // 3)
    for ev_ in consumed:
        ev_.record()
    e2e_run(3)
    torch.cuda.synchronize()
    if dist: dist.barrier()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    copy_stream.wait_event(s2)                                      # no copy starts before the timed region does
    e2e_run(e2e_steps)
    e2.record()
    torch.cuda.synchronize()
    e2e_ms = reduce_max_ms(s2.elapsed_time(e2), dist, dev) / e2e_steps
    h2d = sum(v.numel() * v.element_size() for v in ht.values())

    # ---------------- MM-UNet training leg (BASELINE configs[2]): the caller of the path, img/s ---------------------
    train = None
    if not args.no_train:
        del ht, dbufs, t, du, dd, dz, dx
        torch.cuda.empty_cache()
        try:
            train = train_leg(args, rank, world, dev, dist, args.train_size, args.train_batch, args.train_steps)
        except Exception as exc:      # the training leg must not hide the hot-path numbers
            train = {"error": repr(exc)}
        if not args.no_hires:
            try:
                train["hires"] = train_leg(args, rank, world, dev, dist, 1024, 8, max(8, args.train_steps // 2))
            except Exception as exc:
                train["hires"] = {"error": repr(exc)}

    if rank == 0:          # the clock sampler runs through all three timed regions (device-resident, end-to-end, training)
        sampler.stop_flag.set()
        sampler.join(timeout=3)
    if rank != 0:
        if dist: dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    ms = dev_ms / args.steps
    scan_ms = per_kernel["scan_fwd"] + per_kernel["scan_bwd"]          # rank 0's CUDA events around the two scan passes
    scan_ms = scan_ms * (ms / sum(per_kernel.values())) if world > 1 else scan_ms      # scaled to the max-over-ranks step time
    value = whole_job_gbps(world, nbytes["scan_fwd"] + nbytes["scan_bwd"], scan_ms)
    dom = max(("scan_bwd", "scan_fwd"), key=lambda n: per_kernel[n])
    ach = nbytes[dom] / (per_kernel[dom] * 1e-3) / 1e9
    traffic = ncu_traffic().get(f"{dom}_{args.dtype}")
    line = {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if dtype == torch.float32 else "bf16 I/O, f32 state", "data": "synthetic",
        "config": workload_config(args.dtype),
        "value_basis": "scan fwd+bwd algorithmic bytes (11D+6N)BLs / (scan fwd + scan bwd time inside the step, CUDA events); "
                       "ms_per_step is the whole 4-kernel step",
        "block": {"value": whole_job_gbps(world, nbytes["step"], ms), "unit": "GB/s", "what": "whole step incl. causal_conv1d fwd/bwd (%d MB algorithmic per rank)" % round(nbytes["step"] / 1e6)},
        "e2e": {"value": whole_job_gbps(world, nbytes["scan_fwd"] + nbytes["scan_bwd"], e2e_ms), "unit": "GB/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms,
                "api": "causal_conv1d_fn + selective_scan_fn (autograd), pinned host inputs (H2D of step i+1 on a copy stream overlaps "
                       "step i), loss read back"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": nbytes[dom], "avg_launch_us": per_kernel[dom] * 1e3,
                     "frac_of_nominal_8000": ach / 8000.0},
        "kernels": {n: {"avg_us": per_kernel[n] * 1e3, "algorithmic_GBps": nbytes[n] / (per_kernel[n] * 1e-3) / 1e9,
                        "frac_of_peak": nbytes[n] / (per_kernel[n] * 1e-3) / 1e9 / peak} for n in names},
        "scan_fwd_bwd": {"us": (per_kernel["scan_fwd"] + per_kernel["scan_bwd"]) * 1e3,
                         "GBps": (nbytes["scan_fwd"] + nbytes["scan_bwd"]) / ((per_kernel["scan_fwd"] + per_kernel["scan_bwd"]) * 1e-3) / 1e9},
        "clocks": sampler.summary(), "wall_s": wall, "host_binding": host_binding,
    }
    if train is not None:
        line["train"] = train
    line["scan_fwd_bwd"]["frac_of_peak"] = line["scan_fwd_bwd"]["GBps"] / peak
    if world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_port()
        except Exception as exc:  # the oracle is a checker; its absence must not hide the GPU number
            line["cpu_baseline"] = {"error": repr(exc)}
    emit(line)
    if dist: dist.destroy_process_group()


if __name__ == "__main__":
    main()
