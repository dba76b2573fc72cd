"""Deterministic mode (torch.use_deterministic_algorithms(True), or MMU_DETERMINISTIC=1): every op that sums floats across CTAs
runs its _det entry point.  Each case runs three times - eagerly, on a side stream and as a CUDA-graph replay - and every output
must be bitwise equal across the three, within the oracle tolerances of test_gpu_kernels.py, and close to the default (atomic)
path.  Module cases hash the output and every gradient over two in-process runs and one run in a child process."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from conftest import ROOT
from test_gpu_kernels import check, make_scan_inputs, tol

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from mmunet_b200 import _lib, ops
DEV = "cuda"


@pytest.fixture
def det():
    """Deterministic mode on for the test (warn_only: the torch ops around ours that have no deterministic kernel only warn)."""
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    yield
    torch.use_deterministic_algorithms(was, warn_only=warn)


class _Off:
    def __enter__(self):
        self.was, self.warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
        torch.use_deterministic_algorithms(False)

    def __exit__(self, *a):
        torch.use_deterministic_algorithms(self.was, warn_only=self.warn)


def _flat(out):
    return [t.detach().clone() for t in (out if isinstance(out, (list, tuple)) else (out,)) if isinstance(t, torch.Tensor)]


def three_ways(fn):
    """fn() -> tensor or tuple of tensors (None entries dropped).  Eager, side stream, CUDA-graph replay; cloned results."""
    cur = torch.cuda.current_stream()
    a = _flat(fn())
    s = torch.cuda.Stream()
    s.wait_stream(cur)
    with torch.cuda.stream(s):
        b = _flat(fn())
    cur.wait_stream(s)
    s2 = torch.cuda.Stream()
    s2.wait_stream(cur)
    with torch.cuda.stream(s2):
        fn()                                    # warm-up on the capture stream's side
    cur.wait_stream(s2)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    g.replay()
    torch.cuda.synchronize()
    c = _flat(out)
    return a, b, c


def assert_bitwise(runs, names=None):
    a, b, c = runs
    assert len(a) == len(b) == len(c)
    for i, (x, y, z) in enumerate(zip(a, b, c)):
        n = names[i] if names else i
        assert torch.equal(x, y) or (x.isnan().any() and torch.equal(x.nan_to_num(), y.nan_to_num())), f"{n}: side stream differs"
        assert torch.equal(x, z) or (x.isnan().any() and torch.equal(x.nan_to_num(), z.nan_to_num())), f"{n}: graph replay differs"


def assert_close_to_default(got, want, rtol, atol_rel, names=None):
    for i, (x, y) in enumerate(zip(got, want)):
        n = names[i] if names else i
        y = y.float()
        torch.testing.assert_close(x.float(), y, rtol=rtol, atol=atol_rel * max(1.0, float(y.nan_to_num().abs().max())), equal_nan=True,
                                   msg=lambda m: f"{n}: {m}")


# ---------------------------------------------------------------------------------------------------------------------------------
# selective scan backward
# ---------------------------------------------------------------------------------------------------------------------------------
SCAN_NAMES = ["du", "ddelta", "dA", "dB", "dC", "dD", "dz", "ddelta_bias"]
SCAN_CASES = {
    "config2_chained": dict(B=8, D=384, L=4096, N=16),
    "reverse": dict(B=2, D=64, L=2048, N=16, reverse=True),
    "nslices": dict(B=2, D=12, L=2048, N=16, order=(2, 0, 0, 8)),          # (MMU_ORDER_NSLICES, H, W, nslices)
    "tworow": dict(B=2, D=12, L=2048, N=16, order=(3, 32, 64, 1)),         # MMU_ORDER_TWOROW over a 32 x 64 map
    "split_sequence": dict(B=16, D=6, L=65536, N=16),
    "ragged_v1": dict(B=2, D=6, L=999, N=16),                          # L % 8 != 0: the v1 kernels
    "grouped_n64": dict(B=2, D=20, L=264, N=64),
    "n_groups2": dict(B=2, D=8, L=512, N=16, G=2),
}


def _scan_setup(case, dtype):
    c = dict(SCAN_CASES[case])
    B, D, L, N, G = c.pop("B"), c.pop("D"), c.pop("L"), c.pop("N"), c.pop("G", 1)
    reverse, order = c.pop("reverse", False), c.pop("order", None)
    cpu, gpu = make_scan_inputs(B, D, L, N, G, dtype)
    _, x, _ = ops.selective_scan_fwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"], True,
                                     reverse=reverse, order=order)

    def fn():
        return ops.selective_scan_bwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"],
                                      gpu["dout"], x, True, reverse=reverse, order=order)
    return cpu, gpu, fn, (B, D, L, N, G, reverse, order)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", list(SCAN_CASES))
def test_scan_bwd_deterministic(det, case, dtype):
    cpu, gpu, fn, (B, D, L, N, G, reverse, order) = _scan_setup(case, dtype)
    n0 = _lib.launch_count()
    fn()
    n1 = _lib.launch_count()
    with _Off():
        fn()
    assert n1 - n0 > _lib.launch_count() - n1          # the _det entry point ran (its ordered reduces are extra launches)
    runs = three_ways(fn)
    names = [n for n, t in zip(SCAN_NAMES, fn()) if t is not None]
    assert_bitwise(runs, names)
    with _Off():
        ref = _flat(fn())
    rtol, atol = tol(dtype)
    assert_close_to_default(runs[0], ref, max(rtol, 1e-3), 5 * max(atol, 1e-3), names)
    if B * D * L <= 1 << 16 and order is None:      # the oracle at the small shapes (the large ones are covered through the default path)
        n = lambda t: None if t is None else t.numpy()
        c = cpu
        if reverse:
            c = {k: (v.flip(-1) if k in ("u", "delta", "B", "C", "z", "dout") and v is not None else v) for k, v in cpu.items()}
        rg = oracle.selective_scan_bwd(*(n(c[k]) for k in ("u", "delta", "A", "B", "C", "D", "z", "delta_bias", "dout")), True)
        got = dict(zip(SCAN_NAMES, fn()))
        check("dA", got["dA"], rg["dA"], max(rtol, 1e-3), 5 * max(atol, 1e-3))
        check("dD", got["dD"], rg["dD"], max(rtol, 1e-3), max(atol, 1e-3))


def test_scan_bwd_v1_fp16_deterministic(det):
    cpu, gpu = make_scan_inputs(2, 8, 512, 16, 1, torch.float16)
    _, x, _ = ops.selective_scan_fwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"], True)
    fn = lambda: ops.selective_scan_bwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"],
                                        gpu["dout"], x, True)
    runs = three_ways(fn)
    assert_bitwise(runs)
    n = lambda t: None if t is None else t.numpy()
    rg = oracle.selective_scan_bwd(*(n(cpu[k]) for k in ("u", "delta", "A", "B", "C", "D", "z", "delta_bias", "dout")), True)
    got = dict(zip(SCAN_NAMES, fn()))
    rtol, atol = tol(torch.float16)
    for k in ("dA", "dB", "dC", "dD"):
        ref = rg[k] if rg[k].ndim == got[k].ndim else rg[k][:, None]
        check(k, got[k], ref, max(rtol, 1e-3), 5 * max(atol, 1e-3))


@pytest.mark.parametrize("layout", ["batch_major", "row_major"])
def test_scan_bwd_dbc_views_deterministic(det, layout):
    """dB / dC accumulated into row slices of an x_proj gradient buffer, (B, R + 2N, L) or (R + 2N, B, L)."""
    B, D, L, N, R = 4, 64, 1024, 16, 4
    _, gpu = make_scan_inputs(B, D, L, N)
    _, x, _ = ops.selective_scan_fwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"], True)

    def fn():
        if layout == "batch_major":
            buf = torch.zeros(B, R + 2 * N, L, device=DEV)
            dB, dC = buf[:, R:R + N], buf[:, R + N:]
        else:
            buf = torch.zeros(R + 2 * N, B, L, device=DEV)
            dB, dC = buf[R:R + N].transpose(0, 1), buf[R + N:].transpose(0, 1)
        g = ops.selective_scan_bwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"],
                                   gpu["dout"], x, True, dBC=(dB, dC))
        return buf, g[2], g[5], g[7]
    runs = three_ways(fn)
    assert_bitwise(runs)
    with _Off():
        ref = _flat(fn())
    assert_close_to_default(runs[0], ref, 1e-3, 5e-3)


def test_scan_bwd_slot_workspace_is_capped(det):
    """A problem whose dB / dC slots exceed the cap runs over batch slices and stays deterministic."""
    L_ = _lib.lib()
    B, D, L, N = 4, 256, 65536, 16
    assert L_.mmu_selective_scan_bwd_det_workspace(B, D, L, N) > ops._DET_SCAN_WS_CAP
    _, gpu = make_scan_inputs(B, D, L, N, dtype=torch.bfloat16)
    _, x, _ = ops.selective_scan_fwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"], True)
    fn = lambda: ops.selective_scan_bwd(gpu["u"], gpu["delta"], gpu["A"], gpu["B"], gpu["C"], gpu["D"], gpu["z"], gpu["delta_bias"],
                                        gpu["dout"], x, True)
    a, b = _flat(fn()), _flat(fn())
    assert all(torch.equal(p, q) for p, q in zip(a, b))
    with _Off():
        ref = _flat(fn())
    assert_close_to_default(a, ref, 2e-2, 5e-2)


# ---------------------------------------------------------------------------------------------------------------------------------
# causal conv1d backward
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("width", [2, 4])
def test_conv_bwd_deterministic(det, dtype, width):
    torch.manual_seed(1)
    x = torch.randn(8, 384, 4096, device=DEV).to(dtype)
    w, b = torch.randn(384, width, device=DEV), torch.randn(384, device=DEV)
    dout = torch.randn_like(x)
    fn = lambda: ops.causal_conv1d_bwd(x, w, b, dout, True)
    runs = three_ways(fn)
    assert_bitwise(runs, ["dx", "dw", "db"])
    with _Off():
        ref = _flat(fn())
    assert_close_to_default(runs[0], ref, 1e-4 if dtype == torch.float32 else 1e-2, 1e-4, ["dx", "dw", "db"])


# ---------------------------------------------------------------------------------------------------------------------------------
# narrow Mamba block, GroupNorm NHWC, snake sampler: forward + backward through autograd (the backward runs on the forward's stream)
# ---------------------------------------------------------------------------------------------------------------------------------
def _narrow_inputs(dtype, coord, B=2, H=32, W=64):
    torch.manual_seed(2)
    dm, di, N = 3, 6, 16
    L = H * W
    p = dict(in_w=0.5 * torch.randn(2 * di, dm), conv_w=0.5 * torch.randn(di, 1, 4), conv_b=0.1 * torch.randn(di),
             x_w=0.3 * torch.randn(1 + 2 * N, di), dt_w=0.5 * torch.randn(di, 1), out_w=0.4 * torch.randn(dm, di),
             A=-torch.rand(di, N) - 0.2, D=torch.randn(di), dt_bias=0.3 * torch.rand(di), altho=torch.tensor(0.3))
    p = {k: v.to(DEV).requires_grad_() for k, v in p.items()}
    hidden = torch.randn(B, dm, L, device=DEV).to(dtype).requires_grad_()
    gy = torch.randn(B, dm, L, device=DEV)
    order = (_lib.ORDER_TWOROW, H, W, 1)
    c = (1.0, H, W) if coord else None

    def fn():
        out = ops.mamba_narrow_fn(hidden, p["in_w"], p["conv_w"], p["conv_b"], p["x_w"], p["dt_w"], p["out_w"], p["A"], p["D"],
                                  p["dt_bias"], order=order, altho=p["altho"] if coord else None, coord=c)
        leaves = [hidden] + [v for k, v in p.items() if coord or k != "altho"]
        return (out,) + torch.autograd.grad(out, leaves, gy.to(out.dtype))
    return fn


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("coord", [False, True])
def test_narrow_block_deterministic(det, dtype, coord):
    fn = _narrow_inputs(dtype, coord)
    runs = three_ways(fn)
    assert_bitwise(runs)
    with _Off():
        ref = _flat(fn())
    assert_close_to_default(runs[0], ref, 1e-3 if dtype == torch.float32 else 3e-2, 1e-3 if dtype == torch.float32 else 3e-2)


@pytest.mark.parametrize("dtypes", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16), (torch.float32, torch.bfloat16)])
@pytest.mark.parametrize("shape", [(2, 64, 128, 128), (1, 512, 8, 8)])
def test_group_norm_nhwc_deterministic(det, dtypes, shape):
    tin, tout = dtypes
    B, C, H, W = shape
    torch.manual_seed(5)
    x = (1.5 * torch.randn(B, C, H, W, device=DEV) + 0.7).to(tin).contiguous(memory_format=torch.channels_last).requires_grad_()
    w, b = torch.randn(C, device=DEV, requires_grad=True), torch.randn(C, device=DEV, requires_grad=True)
    gy = torch.randn(B, C, H, W, device=DEV).contiguous(memory_format=torch.channels_last)

    def fn():
        y = ops.group_norm_nhwc(x, C // 4, w, b, 1e-5, tout)
        return (y,) + torch.autograd.grad(y, (x, w, b), gy.to(tout))
    runs = three_ways(fn)
    assert_bitwise(runs, ["y", "dx", "dgamma", "dbeta"])
    with _Off():
        ref = _flat(fn())
    t = 1e-4 if tout == torch.float32 and tin == torch.float32 else 2e-2
    assert_close_to_default(runs[0], ref, t, t, ["y", "dx", "dgamma", "dbeta"])
    # the statistics are reduced in a fixed order: mean / rstd (hence y) do not depend on scheduling
    import torch.nn.functional as F
    torch.testing.assert_close(runs[0][0].float(), F.group_norm(x.detach().float(), C // 4, w.detach(), b.detach(), 1e-5), rtol=t, atol=t)


@pytest.mark.parametrize("dtypes", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16),
                                    (torch.bfloat16, torch.float32)])
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("shape", [(2, 16, 40, 36, 3), (1, 8, 64, 64, 9)])
def test_snake_sample_bwd_deterministic(det, dtypes, channels_last, shape):
    """Gather-side backward: y far outside [0, H-1] (clamp and gradient mask), one NaN coordinate (poisons its sample)."""
    tin, tout = dtypes
    B, C, H, W, K = shape
    torch.manual_seed(3)
    feat = torch.randn(B, C, H, W, device=DEV).to(tin)
    if channels_last:
        feat = feat.contiguous(memory_format=torch.channels_last)
    y = (torch.arange(H, device=DEV).view(1, 1, H, 1) + 1.7 * torch.randn(B, K, H, W, device=DEV)).float()
    y[0, K // 2, H // 3, W // 2] = float("nan")
    feat.requires_grad_()
    y.requires_grad_()
    g = torch.randn(B, C, H * K, W, device=DEV).to(tout)
    if channels_last:
        g = g.contiguous(memory_format=torch.channels_last)

    def fn():
        out = ops.snake_sample(feat, y, tout)
        return (out,) + torch.autograd.grad(out, (feat, y), g)
    runs = three_ways(fn)
    assert_bitwise(runs, ["out", "dfeat", "dy"])
    assert torch.isnan(runs[0][2][0, K // 2, H // 3, W // 2])
    with _Off():
        ref = _flat(fn())
    t = 1e-4 if tin == tout == torch.float32 else 2e-2
    assert_close_to_default(runs[0][:2], ref[:2], t, t, ["out", "dfeat"])
    # d/dy is piecewise constant in y: compare where both are finite
    dy, dy_ref = runs[0][2], ref[2]
    ok = dy.isfinite() & dy_ref.isfinite()
    assert torch.equal(dy.isnan(), dy_ref.isnan())
    bad = ((dy - dy_ref).abs() > t * (float(dy_ref[ok].abs().max()) + dy_ref.abs()))[ok].float().mean()
    assert bad <= 2e-3


# ---------------------------------------------------------------------------------------------------------------------------------
# modules: two runs in-process, one in a child process, SHA-256 of the output and every gradient
# ---------------------------------------------------------------------------------------------------------------------------------
def run_module(kind):
    """Forward + backward of one module on seeded inputs -> {name: SHA-256} of the output and every gradient."""
    from mmunet_b200 import Mamba, mm_net
    torch.manual_seed(0)
    if kind == "mamba":
        m = Mamba(d_model=64, d_state=16, bimamba_type="v3", nslices=4).cuda()
        x = torch.randn(2, 1024, 64, device=DEV, requires_grad=True)
        ctx = torch.autocast("cuda", enabled=False)
    else:                                  # mmconv<K>[_cl]: channels-last under bf16 autocast, or NCHW fp32
        K, cl = int(kind[6]), kind.endswith("_cl")
        m = mm_net.MMConv(16, 16, kernel_size=K).cuda()
        x = torch.randn(2, 16, 64, 64, device=DEV)
        if cl:
            m = m.to(memory_format=torch.channels_last)
            x = x.contiguous(memory_format=torch.channels_last)
        x.requires_grad_()
        ctx = torch.autocast("cuda", dtype=torch.bfloat16, enabled=cl)
    with ctx:
        y = m(x)
        y = y[0] if isinstance(y, tuple) else y
    y.backward(torch.randn(y.shape, generator=torch.Generator().manual_seed(1)).to(DEV, y.dtype))
    ts = [("out", y), ("dx", x.grad)] + [(n, p.grad) for n, p in m.named_parameters() if p.grad is not None]
    return {n: hashlib.sha256(t.detach().float().contiguous().cpu().numpy().tobytes()).hexdigest() for n, t in ts}


CHILD = ("import json, sys, torch; sys.path[:0] = sys.argv[1:4]; torch.use_deterministic_algorithms(True, warn_only=True); "
         "from test_gpu_deterministic import run_module; print(json.dumps(run_module(sys.argv[4])))")


@pytest.mark.parametrize("kind", ["mamba", "mmconv3", "mmconv1", "mmconv3_cl", "mmconv1_cl"])
def test_module_hashes_reproduce(det, kind, monkeypatch):
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    outs = [run_module(kind), run_module(kind)]
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, "-c", CHILD, os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "mm-unet_b200"), kind],
                       env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    outs.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert outs[0] == outs[1], [k for k in outs[0] if outs[0][k] != outs[1].get(k)]
    assert outs[0] == outs[2], [k for k in outs[0] if outs[0][k] != outs[2].get(k)]


# ---------------------------------------------------------------------------------------------------------------------------------
# bench.py under MMU_DETERMINISTIC=1: byte-identical dumps, equal to a direct deterministic run of the four ops
# ---------------------------------------------------------------------------------------------------------------------------------
def test_bench_dump_is_reproducible(tmp_path, det):
    env = dict(os.environ, MMU_DETERMINISTIC="1")
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-train", "--no-cpu-baseline",
                            "--dump-outputs", str(d)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
    names = sorted(f.name for f in dirs[0].iterdir())
    assert names and names == sorted(f.name for f in dirs[1].iterdir())
    for n in names:
        assert (dirs[0] / n).read_bytes() == (dirs[1] / n).read_bytes(), n

    import bench
    t, w = bench.make_inputs(bench.B, torch.float32, "cuda")
    u = ops.causal_conv1d_fwd(t["x"], w["cw"], w["cb"], True)
    out, xs, _ = ops.selective_scan_fwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], True)
    g = ops.selective_scan_bwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], t["dout"], xs, True)
    dx, dw, db = ops.causal_conv1d_bwd(t["x"], w["cw"], w["cb"], g[0], True)
    want = tmp_path / "direct"
    bench.dump_outputs(str(want), {"conv_out": u, "scan_out": out, **dict(zip(bench.GRAD_NAMES, g)), "dx": dx, "dweight": dw, "dbias": db})
    for n in names:
        assert np.array_equal(np.load(dirs[0] / n), np.load(want / n)), n
