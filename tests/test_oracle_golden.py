"""Pins oracle/ (C restatement + torch restatement) against golden vectors produced by the
unmodified reference (oracle/gen_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

import oracle
from oracle import torch_ref
from conftest import load_golden

SCAN = load_golden("selective_scan.npz")
CONV = load_golden("causal_conv1d.npz")
ORD = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "scan_orders.npz"))


def close(a, b, rtol=2e-4, atol=2e-4):
    np.testing.assert_allclose(np.asarray(a, np.float64), np.asarray(b, np.float64), rtol=rtol, atol=atol)


@pytest.mark.parametrize("name", sorted(SCAN))
def test_c_scan_matches_reference(name):
    c = SCAN[name]
    sp = bool(c["softplus"])
    out, last = oracle.selective_scan_fwd(c["u"], c["delta"], c["A"], c["B"], c["C"], c.get("D"), c.get("z"),
                                          c.get("delta_bias"), sp)
    close(out, c["out"])
    close(last, c["last_state"])
    g = oracle.selective_scan_bwd(c["u"], c["delta"], c["A"], c["B"], c["C"], c.get("D"), c.get("z"),
                                  c.get("delta_bias"), c["dout"], sp)
    for k in ("du", "ddelta", "dA", "dB", "dC", "dD", "dz", "ddelta_bias"):
        if k in c:
            scale = max(1.0, float(np.abs(c[k]).max()))
            close(g[k], c[k], rtol=5e-4, atol=5e-4 * scale)


@pytest.mark.parametrize("name", sorted(SCAN))
def test_torch_scan_matches_reference(name):
    c = SCAN[name]
    t = {k: torch.tensor(v, requires_grad=v.dtype == np.float32 and v.ndim > 0) for k, v in c.items()}
    out, last = torch_ref.selective_scan(t["u"], t["delta"], t["A"], t["B"], t["C"], t.get("D"), t.get("z"),
                                         t.get("delta_bias"), bool(c["softplus"]), True)
    close(out.detach(), c["out"])
    close(last.detach(), c["last_state"])
    out.backward(t["dout"].detach())
    for k, src in (("du", "u"), ("ddelta", "delta"), ("dA", "A"), ("dB", "B"), ("dC", "C"), ("dD", "D"),
                   ("dz", "z"), ("ddelta_bias", "delta_bias")):
        if k in c:
            scale = max(1.0, float(np.abs(c[k]).max()))
            close(t[src].grad, c[k], rtol=5e-4, atol=5e-4 * scale)


@pytest.mark.parametrize("name", sorted(CONV))
def test_conv_matches_reference(name):
    c = CONV[name]
    silu = bool(c["silu"])
    out = oracle.causal_conv1d_fwd(c["x"], c["w"], c.get("bias"), silu)
    close(out, c["out"], 1e-5, 1e-5)
    dx, dw, db = oracle.causal_conv1d_bwd(c["x"], c["w"], c.get("bias"), c["dout"], silu)
    close(dx, c["dx"], 1e-4, 1e-4)
    close(dw, c["dw"], 1e-4, 1e-4)
    if "dbias" in c:
        close(db, c["dbias"], 1e-4, 1e-4)
    o2 = torch_ref.causal_conv1d(torch.tensor(c["x"]), torch.tensor(c["w"]),
                                 torch.tensor(c["bias"]) if "bias" in c else None, "silu" if silu else None)
    close(o2, c["out"], 1e-5, 1e-5)


def test_scan_orders_bit_exact():
    for key in ORD.files:
        kind, _, spec = key.partition(".")
        if kind == "tworow":
            H, W = map(int, spec.split("x"))
            idx = oracle.scan_order_index(oracle.ORDER_TWOROW, H, W)
            src = torch.arange(H * W, dtype=torch.float32).reshape(1, 1, H, W)
            flat = torch_ref.two_row_flatten(src)
            assert np.array_equal(flat.reshape(-1).long().numpy(), ORD[key])
            assert torch.equal(torch_ref.two_row_unflatten(flat, H, W), src)
        elif kind == "nslices":
            L, ns = map(int, spec.split("_"))
            idx = oracle.scan_order_index(oracle.ORDER_NSLICES, 1, L, ns)
            src = torch.arange(L, dtype=torch.float32).reshape(1, 1, L)
            g = torch_ref.nslices_gather(src, ns)
            assert np.array_equal(g.reshape(-1).long().numpy(), ORD[key])
            assert torch.equal(torch_ref.nslices_scatter(g, ns), src)
        else:
            L = int(spec)
            idx = oracle.scan_order_index(oracle.ORDER_FLIP, 1, L)
        assert idx.dtype == np.int64 and np.array_equal(idx, ORD[key]), key
    with pytest.raises(ValueError):
        oracle.scan_order_index(oracle.ORDER_NSLICES, 1, 10, 4)     # L % ns != 0 (torch.stack raises in the reference)


def test_torch_inner_matches_reference():
    c = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "mamba_inner.npz"))
    t = {k: torch.tensor(c[k], requires_grad=True) for k in
         ("xz", "conv_w", "conv_b", "x_proj_w", "dt_proj_w", "out_proj_w", "A", "D", "dt_bias")}
    out = torch_ref.mamba_inner(t["xz"], t["conv_w"], t["conv_b"], t["x_proj_w"], t["dt_proj_w"], t["A"], t["D"],
                                t["dt_bias"], t["out_proj_w"], None)
    close(out.detach(), c["out"])
    out.backward(torch.tensor(c["dout"]))
    for k in t:
        scale = max(1.0, float(np.abs(c["d" + k]).max()))
        close(t[k].grad, c["d" + k], rtol=1e-3, atol=1e-3 * scale)


# SHA-256 of the reference's requirements/mamba_simple.py and src/UM_Net/MMUNet.py: the digests of the copies in
# tests/golden/_ref/ as they were added, after a byte-for-byte comparison with the reference's own files
REF_SHA256 = {"mamba_simple.py": "d8025f989f505225278f91576fd64a40acdecee8267ac865046d9b7740a9b626",
              "MMUNet.py": "c514237964c3dfeea7af9cd01cce8cf17537dc9d2f1a0d4f7698a533421b5818"}


def test_ref_fixtures_are_verbatim():
    """tests/golden/_ref/ holds unmodified copies of two reference files (the "runs unchanged" GPU test loads them by path)."""
    import hashlib
    import os
    from conftest import GOLDEN
    for name, digest in REF_SHA256.items():
        with open(os.path.join(GOLDEN, "_ref", name), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, f"tests/golden/_ref/{name} differs from the reference's file"
