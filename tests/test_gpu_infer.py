"""Sliding-window prediction on the GPU: the forward-only path of the Mamba Functions is bitwise the grad-saving forward and saves
memory; the stitch kernel (mmu_sw_stitch) against a torch restatement of monai's blending, its counts, and its reproducibility; the
predictor end to end on MM_Net; and a validation pass between training steps leaves the training bitwise unchanged."""
import hashlib
import json
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT

pytestmark = pytest.mark.gpu

DEV = "cuda"
PATHS = [os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "mm-unet_b200")]


@pytest.fixture()
def no_tf32():
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def _rand(*shape, scale=1.0, dtype=torch.float32, g=None):
    return (scale * torch.randn(*shape, generator=g)).to(DEV, dtype)


def _autocast(dtype):
    return torch.autocast("cuda", dtype=torch.bfloat16, enabled=dtype == torch.bfloat16)


def _forward_only_equal(fn):
    """fn(grad: bool) -> output tensor (or tuple).  The output with grad-requiring inputs (the grad-saving forward) must be bitwise the
    output of the same call under no_grad, launching the same kernels.  With grad mode on but no input requiring grad the call is
    forward-only too (no graph, the same launches); its values are not compared, since torch's own matmul picks its GEMM form from
    the operands' requires_grad (at::native::should_fold) in the fused out_proj."""
    from mmunet_b200 import _lib
    n0 = _lib.launch_count()
    want = fn(True)
    n1 = _lib.launch_count()
    want = want if isinstance(want, tuple) else (want,)
    assert want[0].grad_fn is not None
    with torch.no_grad():
        a = fn(True)
    n2 = _lib.launch_count()
    b = fn(False)
    n3 = _lib.launch_count()
    a = a if isinstance(a, tuple) else (a,)
    b = b if isinstance(b, tuple) else (b,)
    assert a[0].grad_fn is None and b[0].grad_fn is None
    for w, g in zip(want, a):
        assert torch.equal(w, g)
    assert n1 - n0 == n2 - n1 == n3 - n2               # the same kernels, none skipped or added


# (batch, dim, seqlen, dstate): which scan kernel the shape reaches (csrc/selective_scan_fwd.cu run_fwd)
SCAN_SHAPES = {
    "v5_wide": (4, 320, 512, 16),          # fp32: lane-ring kernel (>= 320 ring warps, L >= 512); bf16: v3
    "v3_chained": (1, 16, 4096, 16),       # few warps: v3 with the sequence split into chained segments
    "v1_ragged": (2, 6, 300, 16),          # L % 8 != 0: generic kernel
    "wide_state": (2, 8, 256, 32),         # d_state > 16: two 16-state passes
}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(SCAN_SHAPES))
def test_selective_scan_fn_forward_only(shape, dtype):
    from mmunet_b200 import ops
    B, D, L, N = SCAN_SHAPES[shape]
    g = torch.Generator().manual_seed(1)
    u, z = _rand(B, D, L, dtype=dtype, g=g), _rand(B, D, L, dtype=dtype, g=g)
    delta = (0.5 * torch.rand(B, D, L, generator=g)).to(DEV, dtype)
    A = (-0.5 * torch.rand(D, N, generator=g)).to(DEV)
    Bm, Cm = _rand(B, 1, N, L, dtype=dtype, g=g), _rand(B, 1, N, L, dtype=dtype, g=g)
    Dp, bias = _rand(D, g=g), (0.5 * torch.rand(D, generator=g)).to(DEV)

    def fn(grad):
        t = [v.detach().requires_grad_(grad) for v in (u, delta, A, Bm, Cm, Dp, z, bias)]
        return ops.selective_scan_fn(*t, delta_softplus=True, return_last_state=True)

    _forward_only_equal(fn)


def _inner_weights(di, N, R, dm, g):
    return dict(conv_w=_rand(di, 1, 4, scale=0.3, g=g), conv_b=_rand(di, scale=0.1, g=g), x_w=_rand(R + 2 * N, di, scale=di ** -0.5, g=g),
                dt_w=_rand(di, R, scale=R ** -0.5, g=g), out_w=_rand(dm, di, scale=di ** -0.5, g=g), out_b=_rand(dm, scale=0.1, g=g),
                A=-torch.rand(di, N, generator=g).add(0.5).to(DEV), A_b=-torch.rand(di, N, generator=g).add(0.5).to(DEV),
                D=_rand(di, g=g), dt_b=_rand(di, scale=0.5, g=g))


# (batch, d_inner, seqlen): v5 in fp32 (batch * d_inner / 4 >= 320 rows, L >= 512), chained v3, ragged L (generic kernel)
INNER_SHAPES = {"v5_wide": (4, 320, 512), "v3_chained": (1, 16, 4096), "v1_ragged": (2, 32, 300)}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", list(INNER_SHAPES))
@pytest.mark.parametrize("kind", ["no_out_proj", "no_out_proj_reversed", "no_out_proj_nslices", "inner", "inner_tworow", "bimamba"])
def test_inner_fns_forward_only(kind, shape, dtype):
    from mmunet_b200 import _lib, ops
    B, di, L = INNER_SHAPES[shape]
    N, R, dm = 16, 4, 8
    g = torch.Generator().manual_seed(2)
    w = _inner_weights(di, N, R, dm, g)
    xz0 = _rand(B, 2 * di, L, g=g)

    def fn(grad):
        t = {k: v.detach().requires_grad_(grad) for k, v in w.items()}
        xz = xz0.to(dtype).requires_grad_(grad)                                # in_proj's output: bf16 under autocast
        with _autocast(dtype):
            if kind == "no_out_proj":
                return ops.mamba_inner_fn_no_out_proj(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["A"], None, None, t["D"], t["dt_b"])
            if kind == "no_out_proj_reversed":
                return ops.mamba_inner_fn_no_out_proj_reversed(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["A"], t["D"], t["dt_b"])
            if kind == "no_out_proj_nslices":
                return ops.mamba_inner_fn_no_out_proj_ordered(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["A"], t["D"], t["dt_b"],
                                                              True, order=(_lib.ORDER_NSLICES, 1, L, 8 if L % 8 == 0 else 4))
            if kind == "inner":
                return ops.mamba_inner_fn(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["out_w"], t["out_b"], t["A"], None, None,
                                          t["D"], t["dt_b"])
            if kind == "inner_tworow":
                H = 4 if L % 4 == 0 else 2
                return ops.mamba_inner_fn_ordered(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["out_w"], t["out_b"], t["A"], t["D"],
                                                  t["dt_b"], True, order=(_lib.ORDER_TWOROW, H, L // H, 1))
            return ops.bimamba_inner_fn(xz, t["conv_w"], t["conv_b"], t["x_w"], t["dt_w"], t["out_w"], t["out_b"], t["A"], t["A_b"],
                                        None, None, t["D"], t["dt_b"])

    _forward_only_equal(fn)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("coord", [False, True], ids=["plain", "coord"])
@pytest.mark.parametrize("hw", [(16, 16), (24, 20), (64, 128)])
def test_narrow_block_forward_only(hw, coord, dtype):
    """MMConv's d_model = 3 Mamba (MambaNarrowFn), in its two-row scan order, with and without the coordinate epilogue."""
    from mmunet_b200 import Mamba, _lib
    torch.manual_seed(3)
    m = Mamba(d_model=3, d_state=16, d_conv=4, expand=2).to(DEV)
    H, W = hw
    x0 = torch.randn(2, 3, H * W, device=DEV)
    altho = torch.nn.Parameter(torch.tensor(0.3, device=DEV))
    assert m.narrow_block_available(x0.transpose(1, 2))

    def fn(grad):
        for p in m.parameters():
            p.requires_grad_(grad)
        altho.requires_grad_(grad)
        x = x0.detach().requires_grad_(grad).transpose(1, 2)
        with _autocast(dtype):
            return m(x, scan_order=(_lib.ORDER_TWOROW, H, W, 1), coord_epilogue=(altho, 1.0, H, W) if coord else None)[0]

    _forward_only_equal(fn)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("bimamba_type,L", [("none", 1024), ("none", 300), ("v3", 4096), ("v3", 1024)])
def test_mamba_modules_forward_only(bimamba_type, L, dtype):
    from mmunet_b200 import Mamba
    torch.manual_seed(4)
    m = Mamba(d_model=64, d_state=16, bimamba_type=bimamba_type, nslices=8).to(DEV)
    m.return_directional = False
    x0 = torch.randn(2, L, 64, device=DEV)

    def fn(grad):
        for p in m.parameters():
            p.requires_grad_(grad)
        with _autocast(dtype):
            return m(x0.detach().requires_grad_(grad))[0]

    _forward_only_equal(fn)


def test_forward_only_saves_state_memory():
    """RCG's Mamba (d_model 64, v3, 64 slices) on a 128 x 128 map: under no_grad the peak allocation is lower by at least the scan
    states x and pre-gate outputs y the grad-saving forward keeps for its three directions."""
    from mmunet_b200 import Mamba, _lib
    torch.manual_seed(5)
    m = Mamba(d_model=64, d_state=16, bimamba_type="v3", nslices=64).to(DEV)
    m.return_directional = False
    B, L, di, N = 2, 128 * 128, m.d_inner, 16
    x = torch.randn(B, 64, L, device=DEV).transpose(1, 2)
    stride = _lib.lib().mmu_scan_state_stride(B, di, L, N, _lib.F32)
    xy_bytes = 3 * (B * di * ((L + stride - 1) // stride) * N * 4 + B * di * L * 4)
    with torch.no_grad():
        m(x)                                                                  # one-time allocations (cuBLAS workspaces, grids)
    peaks = {}
    for mode in ("grad", "no_grad"):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        with torch.set_grad_enabled(mode == "grad"):
            out = m(x)[0]
        torch.cuda.synchronize()
        peaks[mode] = torch.cuda.max_memory_allocated() - base
        del out
    assert peaks["grad"] - peaks["no_grad"] >= xy_bytes, (peaks, xy_bytes)


# ---- stitch kernel ------------------------------------------------------------------------------------------------------------
def _head_sizes(roi):
    return [roi // 2, roi // 4, roi // 8, roi // 16, roi // 2]


def _random_heads(B, nwin, roi, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(B, nwin, s, s, generator=g).mul(3.0).to(DEV, dtype) for s in _head_sizes(roi)]


def _torch_stitch(heads, H, W, roi, overlap):
    """monai's SlidingWindowInferer blending (constant mode) restated in torch, with MM_Net's resize-and-sum per window."""
    from mmunet_b200.infer import pad_for_roi, window_starts
    B = heads[0].shape[0]
    (pt, pb), (pl, pr) = pad_for_roi(H, roi), pad_for_roi(W, roi)
    nh, nw = H + pt + pb, W + pl + pr
    acc = torch.zeros(B, 1, nh, nw, device=DEV)
    cnt = torch.zeros(1, 1, nh, nw, device=DEV)
    wins = [(a, b) for a in window_starts(nh, roi, overlap) for b in window_starts(nw, roi, overlap)]
    assert heads[0].shape[1] == len(wins)
    for w, (a, b) in enumerate(wins):
        v = None
        for h in heads:
            up = F.interpolate(h[:, w:w + 1].float(), size=(roi, roi), mode="bilinear", align_corners=True)
            v = up if v is None else v + up
        acc[:, :, a:a + roi, b:b + roi] += v
        cnt[:, :, a:a + roi, b:b + roi] += 1
    return (acc / cnt)[:, :, pt:pt + H, pl:pl + W]


def _nwin(H, W, roi, overlap):
    from mmunet_b200.infer import pad_for_roi, window_starts
    return (len(window_starts(H + sum(pad_for_roi(H, roi)), roi, overlap)) *
            len(window_starts(W + sum(pad_for_roi(W, roi)), roi, overlap)))


# (B, H, W, roi, overlap)
STITCH_CASES = {
    "image_eq_roi": (2, 512, 512, 512, 0.5),
    "drive_584x565": (1, 584, 565, 512, 0.5),
    "hrf_2336x3504": (1, 2336, 3504, 512, 0.5),
    "padded_300x200": (2, 300, 200, 512, 0.5),
    "roi64_overlap0": (3, 200, 150, 64, 0.0),
    "roi64_overlap50": (3, 200, 150, 64, 0.5),
    "roi64_overlap75": (3, 200, 150, 64, 0.75),
    "many_images": (7, 97, 130, 64, 0.5),
}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", list(STITCH_CASES))
def test_stitch_matches_torch(case, dtype):
    from mmunet_b200.infer import sw_stitch
    B, H, W, roi, ov = STITCH_CASES[case]
    heads = _random_heads(B, _nwin(H, W, roi, ov), roi, dtype, seed=list(STITCH_CASES).index(case))
    g = torch.Generator().manual_seed(6)
    target = (torch.rand(B, 1, H, W, generator=g) < 0.3).to(DEV, torch.uint8)
    fov = (torch.rand(H, W, generator=g) < 0.8).to(DEV)                       # one FOV shared by the images, bool
    logits, counts = sw_stitch(heads, (H, W), roi, ov, target=target, fov=fov)
    ref = _torch_stitch(heads, H, W, roi, ov)
    assert logits.shape == (B, 1, H, W) and logits.dtype == torch.float32
    torch.testing.assert_close(logits, ref, rtol=0, atol=1e-5 * float(ref.abs().max()))
    pos, t, inside = logits[:, 0] > 0, target[:, 0] != 0, fov.expand(B, H, W)
    want = torch.stack([(pos & t & inside).sum((1, 2)), (pos & ~t & inside).sum((1, 2)), (~pos & t & inside).sum((1, 2)),
                        (~pos & ~t & inside).sum((1, 2))], dim=1)
    assert counts.dtype == torch.int64 and torch.equal(counts, want)
    _, counts_all = sw_stitch(heads, (H, W), roi, ov, target=target)          # no FOV: every pixel
    assert int(counts_all.sum()) == B * H * W


@pytest.mark.parametrize("case", ["drive_584x565", "roi64_overlap75"])
def test_stitch_is_reproducible(case):
    """Two launches, a launch on a side stream and a CUDA-graph replay give the same bits (logits and counts)."""
    from mmunet_b200.infer import sw_stitch
    B, H, W, roi, ov = STITCH_CASES[case]
    heads = _random_heads(B, _nwin(H, W, roi, ov), roi, torch.bfloat16, seed=7)
    target = (torch.rand(B, 1, H, W, device=DEV) < 0.3).to(torch.uint8)
    a = sw_stitch(heads, (H, W), roi, ov, target=target)
    b = sw_stitch(heads, (H, W), roi, ov, target=target)
    cur, side = torch.cuda.current_stream(), torch.cuda.Stream()
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        c = sw_stitch(heads, (H, W), roi, ov, target=target)
    cur.wait_stream(side)
    out = torch.empty(B, 1, H, W, device=DEV)
    cnt = torch.zeros(B, 4, device=DEV, dtype=torch.int64)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        sw_stitch(heads, (H, W), roi, ov, target=target, counts=cnt, out=out)
    graph.replay()
    torch.cuda.synchronize()
    for lg, ct in (b, c, (out, cnt)):
        assert torch.equal(lg, a[0]) and torch.equal(ct, a[1])


def test_stitch_argument_errors():
    from mmunet_b200.infer import sw_stitch
    heads = _random_heads(1, 4, 64, torch.float32, seed=8)
    with pytest.raises(RuntimeError, match=r"\(1, 9, h, w\)"):
        sw_stitch(heads, (100, 100), 64, 0.5)                                # 9 windows, not 4
    with pytest.raises(RuntimeError, match="one dtype"):
        sw_stitch(heads[:4] + [heads[4].bfloat16()], (90, 90), 64, 0.5)
    with pytest.raises(RuntimeError, match="need a target"):
        sw_stitch(heads, (90, 90), 64, 0.5, fov=torch.ones(90, 90, device=DEV))


# ---- predictor end to end -------------------------------------------------------------------------------------------------------
def _net(channels_last=False):
    from mmunet_b200.mm_net import MM_Net
    torch.manual_seed(50)
    net = MM_Net(num_classes=1).to(DEV)
    return net.to(memory_format=torch.channels_last) if channels_last else net


def _monai_loop(net, x, roi, overlap):
    """Plain monai-style sliding window over model(window), fp32, one window at a time."""
    from mmunet_b200.infer import pad_for_roi, window_starts
    B, _, H, W = x.shape
    (pt, pb), (pl, pr) = pad_for_roi(H, roi), pad_for_roi(W, roi)
    xp = F.pad(x, (pl, pr, pt, pb))
    nh, nw = xp.shape[2:]
    acc = torch.zeros(B, 1, nh, nw, device=DEV)
    cnt = torch.zeros(1, 1, nh, nw, device=DEV)
    with torch.no_grad():
        for i in range(B):
            for a in window_starts(nh, roi, overlap):
                for b in window_starts(nw, roi, overlap):
                    acc[i:i + 1, :, a:a + roi, b:b + roi] += net(xp[i:i + 1, :, a:a + roi, b:b + roi]).float()
                    if i == 0:
                        cnt[:, :, a:a + roi, b:b + roi] += 1
    return (acc / cnt)[:, :, pt:pt + H, pl:pl + W]


def test_predict_equals_model_on_roi_sized_images(no_tf32):
    from mmunet_b200.infer import SlidingWindowPredictor
    net = _net().train()
    x = torch.randn(2, 3, 64, 64, device=DEV)
    pred = SlidingWindowPredictor(net, roi_size=64, sw_batch_size=2, dtype="fp32", graph=False)
    got = pred.predict(x)
    assert net.training and all(m.training for m in net.modules())          # the caller's mode is restored
    net.eval()
    with torch.no_grad():
        want = net(x)
    assert got.dtype == torch.float32 and got.shape == (2, 1, 64, 64)
    torch.testing.assert_close(got, want, rtol=0, atol=1e-5 * float(want.abs().max()))


def test_predict_equals_monai_loop_on_other_sizes(no_tf32):
    from mmunet_b200.infer import SlidingWindowPredictor
    net = _net().eval()
    imgs = [torch.randn(2, 3, 100, 90, device=DEV), torch.randn(1, 3, 40, 50, device=DEV)]
    pred = SlidingWindowPredictor(net, roi_size=64, overlap=0.5, sw_batch_size=1, dtype="fp32", graph=False)
    got = pred.predict(imgs)
    assert not net.training
    for x, lg in zip(imgs, got):
        want = _monai_loop(net, x, 64, 0.5)
        assert lg.shape == want.shape
        torch.testing.assert_close(lg, want, rtol=0, atol=1e-4 * float(want.abs().max()))
    one = pred.predict(imgs[0])                                               # a tensor in, a tensor out; same numbers
    torch.testing.assert_close(one, got[0], rtol=0, atol=1e-4 * float(got[0].abs().max()))


def _rel_l2(a, b):
    return float((a - b).norm() / b.norm())


def test_predict_bf16_channels_last_graph_and_batching(monkeypatch):
    """bf16 channels-last, graph on / off, one or three windows per batch.  The library's deterministic mode is on so that two replays
    can be compared bit for bit: by default the channels-last GroupNorm's statistics are summed with float atomics."""
    from mmunet_b200.infer import SlidingWindowPredictor
    monkeypatch.setenv("MMU_DETERMINISTIC", "1")
    net = _net(channels_last=True).eval()
    x = torch.randn(3, 3, 100, 90, device=DEV)
    target = torch.rand(3, 1, 100, 90, device=DEV) < 0.3
    runs = {}
    for graph in (False, True):
        for sw in (1, 3):
            pred = SlidingWindowPredictor(net, roi_size=64, overlap=0.5, sw_batch_size=sw, dtype="bf16", graph=graph)
            assert pred.channels_last
            lg = pred.predict(x)
            assert lg.dtype == torch.float32 and torch.isfinite(lg).all()
            counts = pred.evaluate(x, target)
            assert int(counts.sum()) == 3 * 100 * 90
            if graph:
                assert torch.equal(pred.predict(x), lg)                      # replay of the captured graph
                assert len(pred._graphs) == 1
                pred.reset()
                assert not pred._graphs
            runs[(graph, sw)] = lg
    ref = runs[(False, 1)]
    errs = {k: _rel_l2(lg, ref) for k, lg in runs.items()}
    print("relative L2 difference to eager, one window per batch:", errs)
    assert all(e < 5e-2 for e in errs.values()), errs              # bf16 activations; cuDNN picks per batch size


# ---- strict deterministic mode, in child processes ------------------------------------------------------------------------------
def _child(code, *args):
    env = dict(os.environ)
    env.pop("MMU_DETERMINISTIC", None)
    env["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
    prologue = "import sys; sys.path[:0] = sys.argv[1:4]; import torch; torch.use_deterministic_algorithms(True); "
    r = subprocess.run([sys.executable, "-c", prologue + code, *PATHS, *map(str, args)], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stdout.strip().splitlines()[-1]


def predictor_runs_bitwise():
    from mmunet_b200.infer import SlidingWindowPredictor
    net = _net(channels_last=True).eval()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 3, 100, 90, generator=g).to(DEV)
    t = (torch.rand(2, 1, 100, 90, generator=g) < 0.3).to(DEV)
    pred = SlidingWindowPredictor(net, roi_size=64, sw_batch_size=3, dtype="bf16")
    a, ca = pred.predict(x), pred.evaluate(x, t)
    b, cb = pred.predict(x), pred.evaluate(x, t)
    return bool(torch.equal(a, b) and torch.equal(ca, cb) and torch.isfinite(a).all())


def test_predictor_is_bitwise_reproducible_under_strict_mode():
    assert _child("from test_gpu_infer import predictor_runs_bitwise; print(predictor_runs_bitwise())") == "True"


def run_training_with_validation(validate):
    """6 strict-mode graphed bf16 channels-last Trainer steps, with (validate=1) or without a predictor evaluate() after step 3
    -> digest of the losses, every parameter, BatchNorm buffer and AdamW state tensor, and whether the net is in training mode."""
    from mmunet_b200.infer import SlidingWindowPredictor
    from mmunet_b200.train import Trainer
    tr = Trainer(image_size=64, batch_per_rank=2, dtype="bf16", device="cuda:0", ddp=False, channels_last=True, graph=True,
                 graph_warmup=3)
    tr.set_epoch(2)
    losses = []
    for i in range(6):
        if i == 3 and validate:
            g = torch.Generator().manual_seed(10)
            x = torch.randn(2, 3, 100, 90, generator=g)
            t = torch.rand(2, 1, 100, 90, generator=g) < 0.3
            counts = SlidingWindowPredictor(tr.net, roi_size=64, sw_batch_size=2, dtype="bf16").evaluate(x, t)
            assert int(counts.sum()) == 2 * 100 * 90
        xb, yb = tr.synthetic_batch()
        losses.append(float(tr.step(xb, yb)))
    assert tr.graph is not None
    h = hashlib.sha256(repr(losses).encode())
    for name, t in list(tr.net.named_parameters()) + list(tr.net.named_buffers()):
        h.update(name.encode())
        h.update(t.detach().cpu().contiguous().numpy().tobytes() if t.dtype != torch.bfloat16 else t.detach().float().cpu().numpy().tobytes())
        for k, v in sorted(tr.opt.state.get(t, {}).items()):
            h.update(k.encode())
            h.update(v.detach().float().cpu().contiguous().numpy().tobytes() if torch.is_tensor(v) else repr(v).encode())
    return {"digest": h.hexdigest(), "losses": losses, "training": tr.net.training}


def test_validation_does_not_perturb_training():
    code = ("import json; from test_gpu_infer import run_training_with_validation as r; "
            "print(json.dumps(r(int(sys.argv[4]))))")
    plain, validated = (json.loads(_child(code, v)) for v in (0, 1))
    assert validated["training"] is True
    assert plain["losses"] == validated["losses"]
    assert plain["digest"] == validated["digest"]
