"""bench.py --dump-outputs: the arrays it writes are what the four timed ops return on the benchmark's seeded inputs.
This checks the dump path only (names, row sample, dtype, size); the parity and golden tests check the kernels' results."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def run_bench(*args):
    return subprocess.run([sys.executable, BENCH, *args], cwd=ROOT, capture_output=True, text=True, timeout=900)


def test_bench_rejects_bad_arguments(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = run_bench(*args)
        assert r.returncode == 2 and "error" in r.stderr, (args, r.stderr[-2000:])
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_bench_dump_outputs_match_the_ops(tmp_path):
    got_dir, want_dir = tmp_path / "bench", tmp_path / "direct"
    r = run_bench("--steps", "2", "--warmup", "1", "--no-train", "--no-cpu-baseline", "--dump-outputs", str(got_dir))
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    files = sorted(got_dir.iterdir())
    assert sum(f.stat().st_size for f in files) <= 64 << 20

    # one step of the same four ops on the same inputs, written through the same sampling
    import bench
    from mmunet_b200 import ops
    t, w = bench.make_inputs(bench.B, torch.float32, "cuda")
    u = ops.causal_conv1d_fwd(t["x"], w["cw"], w["cb"], True)
    out, xs, _ = ops.selective_scan_fwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], True)
    g = ops.selective_scan_bwd(u, t["delta"], w["A"], t["Bm"], t["Cm"], w["Dp"], t["z"], w["dbias"], t["dout"], xs, True)
    dx, dw, db = ops.causal_conv1d_bwd(t["x"], w["cw"], w["cb"], g[0], True)
    bench.dump_outputs(str(want_dir), {"conv_out": u, "scan_out": out, **dict(zip(bench.GRAD_NAMES, g)),
                                       "dx": dx, "dweight": dw, "dbias": db})

    assert [f.name for f in files] == sorted(f.name for f in want_dir.iterdir())
    for f in files:
        a, b = np.load(f), np.load(want_dir / f.name)
        assert a.dtype == np.float32 and a.shape == b.shape, (f.name, a.dtype, a.shape, b.shape)
        assert a.shape[0] == bench.DUMP_ROWS or a.size <= 1 << 20, (f.name, a.shape)
        # dA / dB / dC / dD / ddelta_bias / dweight / dbias are accumulated with atomics: summation order may differ
        np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-5 * float(np.abs(b).max()), err_msg=f.name)
