"""Deterministic MM_Net training under torch.use_deterministic_algorithms(True).  The bilinear-resize backward (gather-side,
mmu_resize_bilinear_bwd_det) against a float64 CPU backward at MM_Net's own resize shapes, bitwise equal eagerly, on a side stream and
as a graph replay; the default path never calls it; and, in child processes under strict mode (not warn_only), MM_Net matches the
golden reference and two Trainer runs give byte-identical weights, AdamW state and losses."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from test_gpu_deterministic import _Off, assert_bitwise, det, three_ways  # noqa: F401  (det: fixture)

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from mmunet_b200 import ops
DEV = "cuda"
PATHS = [os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "mm-unet_b200")]

# (C, H_in, W_in, H_out, W_out)
RESIZE_CASES = {
    "decoder_up2": (64, 128, 128, 256, 256),         # DecoderBlock at 512x512 input: the last x2 upsample
    "rcg_256_128": (64, 256, 256, 128, 128),         # RCG: the contour map at H/2 resized to rcg2 / rcg3 / rcg4's maps
    "rcg_256_64": (64, 256, 256, 64, 64),
    "rcg_256_32": (64, 256, 256, 32, 32),
    "logits_256_512": (1, 256, 256, 512, 512),       # MM_Net: side outputs and the contour head to full size
    "ragged_19_38": (64, 19, 19, 38, 38),            # 608x608 input
    "ragged_38_19": (64, 38, 38, 19, 19),
    "ragged_76_19": (64, 76, 76, 19, 19),
    "ragged_tail": (6, 19, 21, 38, 11),              # C not a multiple of the 16-byte vector: scalar channels
    "deg_1_5": (3, 1, 1, 5, 5),
    "deg_5_1": (3, 5, 5, 1, 1),
    "deg_1_1": (3, 1, 1, 1, 1),
    "deg_mixed": (8, 1, 7, 5, 1),
}
B = 2


def _dout(case, dtype, cl):
    C, Hi, Wi, Ho, Wo = RESIZE_CASES[case]
    g = torch.Generator().manual_seed(list(RESIZE_CASES).index(case))
    d = torch.randn(B, C, Ho, Wo, generator=g).to(dtype)
    return d, (d.to(DEV).contiguous(memory_format=torch.channels_last) if cl else d.to(DEV))


def _adjoint64(d, hw):
    """F.interpolate's backward on CPU in float64 from the same dout."""
    x = torch.zeros(d.shape[0], d.shape[1], *hw, dtype=torch.float64, requires_grad=True)
    F.interpolate(x, size=d.shape[2:], mode="bilinear", align_corners=True).backward(d.double())
    return x.grad


def _axis(n_in, n_out):
    """-> (W, M, dr): the (n_out, n_in) weights of one axis as F.interpolate's CUDA forward computes them (fp32 scale, r, l0, l1), the
    0/1 mask of the taps, and how far those fp32 weights may be from the float64 ones (r = fl(fl(scale) * o): (in - 1) * 2^-23)."""
    s = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0)
    o = np.arange(n_out)
    r = s * o.astype(np.float32)
    i0 = r.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    l1 = r - i0.astype(np.float32)
    W, M = np.zeros((n_out, n_in)), np.zeros((n_out, n_in))
    np.add.at(W, (o, i0), (np.float32(1) - l1).astype(np.float64))
    np.add.at(W, (o, i1), l1.astype(np.float64))
    M[o, i0] = M[o, i1] = 1.0
    return torch.from_numpy(W), torch.from_numpy(M), (n_in - 1) * 2.0 ** -23 + 2.0 ** -24


def _bf16_ulp(v):
    _, e = torch.frexp(v)
    return torch.where(v == 0, torch.zeros_like(v), torch.ldexp(torch.ones_like(v), e - 8))


@pytest.mark.parametrize("cl", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", list(RESIZE_CASES))
def test_resize_bwd_matches_float64(case, dtype, cl):
    C, Hi, Wi, Ho, Wo = RESIZE_CASES[case]
    d_cpu, d = _dout(case, dtype, cl)
    got = ops.resize_bilinear_bwd(d, (Hi, Wi), cl)
    torch.cuda.synchronize()
    assert got.dtype == dtype and got.shape == (B, C, Hi, Wi)
    assert got.is_contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format)
    g = got.cpu().double()
    d64 = d_cpu.double()
    (Wh, Mh, dr_h), (Ww, Mw, dr_w) = _axis(Hi, Ho), _axis(Wi, Wo)
    # float64 sums over the forward's own fp32 weights: what the kernel computes up to its fp32 accumulation
    ref = Wh.T @ d64 @ Ww
    mag = Wh.T @ d64.abs() @ Ww                      # sum of |weight * dout|: bounds the fp32 accumulation error
    if dtype == torch.float32:
        err = (g - ref).abs() - 1e-5 * mag
    else:       # one rounding at the end: within one bf16 ulp of the float64 result rounded to bf16
        rb = ref.to(torch.bfloat16).double()
        err = (g - rb).abs() - (_bf16_ulp(rb) + 1e-5 * mag)
    assert float(err.max()) <= 0, f"{int((err > 0).sum())} elements out of tolerance, worst excess {float(err.max()):.3g}"
    # F.interpolate's backward on CPU in float64 (float64 weights): apart from the above, the fp32 rounding of the weights, at most
    # dr_h + dr_w per tap
    taps = Mh.T @ d64.abs() @ Mw
    cpu = _adjoint64(d_cpu, (Hi, Wi))
    lim = (1e-5 * mag + (dr_h + dr_w) * taps) if dtype == torch.float32 else (_bf16_ulp(g) + 1e-5 * mag + (dr_h + dr_w) * taps)
    assert float(((g - cpu).abs() - lim).max()) <= 0
    # close to torch's own CUDA backward (atomic scatter; for bf16 every add rounds to bf16)
    with _Off():
        x = torch.zeros(B, C, Hi, Wi, device=DEV, dtype=dtype, requires_grad=True)
        if cl:
            x = x.detach().contiguous(memory_format=torch.channels_last).requires_grad_()
        F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=True).backward(d)
    tol = 1e-5 if dtype == torch.float32 else 5e-2
    assert float(((g - x.grad.cpu().double()).abs() - tol * mag).max()) <= 0


@pytest.mark.parametrize("cl", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", ["decoder_up2", "rcg_256_64", "logits_256_512", "ragged_tail"])
def test_resize_bwd_bitwise(det, case, dtype, cl):
    """Through autograd (ops.resize_bilinear in deterministic mode): the same bits eagerly, on a side stream and as a graph replay;
    dx keeps the input's memory format."""
    C, Hi, Wi, Ho, Wo = RESIZE_CASES[case]
    _, d = _dout(case, dtype, cl)
    x = torch.randn(B, C, Hi, Wi, device=DEV).to(dtype)
    if cl:
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_()

    def fn():
        y = ops.resize_bilinear(x, size=(Ho, Wo))
        return (y,) + torch.autograd.grad(y, x, d)
    runs = three_ways(fn)
    assert_bitwise(runs, ["y", "dx"])
    y, dx = runs[0]
    assert torch.equal(y, F.interpolate(x.detach(), size=(Ho, Wo), mode="bilinear", align_corners=True))
    if C > 1 and Hi * Wi > 1:
        assert dx.is_contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format)
    assert torch.equal(dx, ops.resize_bilinear_bwd(d, (Hi, Wi), cl))


def _boom(*a, **k):
    raise AssertionError("the deterministic resize backward ran")


def test_default_path_never_calls_the_resize_kernel(monkeypatch):
    from mmunet_b200.mm_net import MM_Net
    monkeypatch.setattr(ops, "resize_bilinear_bwd", _boom)
    torch.manual_seed(0)
    net = MM_Net(num_classes=1).to(DEV).train()
    x = torch.randn(2, 3, 64, 64, device=DEV, requires_grad=True)
    with _Off():
        net(x).float().square().mean().backward()
    assert torch.isfinite(x.grad).all()
    # the same step in deterministic mode does reach it (so the monkeypatch is on the path it guards)
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        with pytest.raises(AssertionError, match="resize backward ran"):
            net(x).float().square().mean().backward()
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)


# ---------------------------------------------------------------------------------------------------------------------------------
# child processes under strict mode (torch.use_deterministic_algorithms(True), not warn_only)
# ---------------------------------------------------------------------------------------------------------------------------------
def _child(code, *args, cublas=":4096:8"):
    env = dict(os.environ)
    env.pop("CUBLAS_WORKSPACE_CONFIG", None)
    env.pop("MMU_DETERMINISTIC", None)
    if cublas:
        env["CUBLAS_WORKSPACE_CONFIG"] = cublas
    prologue = "import sys; sys.path[:0] = sys.argv[1:4]; import torch; torch.use_deterministic_algorithms(True); "
    r = subprocess.run([sys.executable, "-c", prologue + code, *PATHS, *map(str, args)], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stdout.strip().splitlines()[-1]


def test_mm_net_golden_under_strict_mode():
    code = ("torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False; "
            "import test_gpu_mm_net as t; t.test_mm_net_matches_reference_fp32(None); print('ok')")
    assert _child(code) == "ok"


def run_training(dtype, channels_last, graph, steps=6):
    """Strict-mode Trainer steps -> {"losses": [...], "sha256": digest of every parameter and every AdamW state tensor}."""
    import hashlib

    import numpy as np
    from mmunet_b200.train import Trainer
    tr = Trainer(image_size=64, batch_per_rank=2, dtype=dtype, device="cuda:0", ddp=False, channels_last=channels_last, graph=graph,
                 graph_warmup=3)
    tr.set_epoch(2)                                  # lr 1e-3 (epoch 0 of the warm-up has lr 0: the weights would not move)
    losses = []
    for _ in range(steps):
        x, y = tr.synthetic_batch()
        losses.append(float(tr.step(x, y)))
    assert (tr.graph is not None) == graph
    h = hashlib.sha256()
    for name, p in tr.net.named_parameters():
        h.update(name.encode())
        h.update(p.detach().float().contiguous().cpu().numpy().tobytes())
        for k, v in sorted(tr.opt.state.get(p, {}).items()):
            h.update(k.encode())
            h.update(v.detach().float().contiguous().cpu().numpy().tobytes() if torch.is_tensor(v) else repr(v).encode())
    return {"losses": losses, "finite": bool(np.isfinite(losses).all()), "sha256": h.hexdigest()}


@pytest.mark.parametrize("dtype,channels_last,graph", [("fp32", False, False), ("bf16", True, True)],
                         ids=["fp32_nchw_eager", "bf16_cl_graph"])
def test_training_is_reproducible_under_strict_mode(dtype, channels_last, graph):
    code = ("import json; from test_gpu_deterministic_training import run_training; "
            "print(json.dumps(run_training(sys.argv[4], sys.argv[5] == '1', sys.argv[6] == '1')))")
    runs = [json.loads(_child(code, dtype, int(channels_last), int(graph))) for _ in range(2)]
    assert runs[0]["finite"], runs[0]["losses"]
    assert runs[0]["losses"] == runs[1]["losses"]
    assert runs[0]["sha256"] == runs[1]["sha256"]
    assert len(set(runs[0]["losses"])) > 1                      # the weights moved


def test_trainer_refuses_strict_mode_without_cublas_config():
    code = ("from mmunet_b200.train import Trainer\n"
            "try:\n    Trainer(image_size=64, batch_per_rank=2, dtype='fp32', device='cuda:0', ddp=False, graph=False)\n"
            "except RuntimeError as e:\n    print('raised', 'CUBLAS_WORKSPACE_CONFIG=:4096:8' in str(e))\n"
            "else:\n    print('no error')")
    assert _child(code, cublas=None) == "raised True"
