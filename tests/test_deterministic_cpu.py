"""CPU-side checks of the deterministic-mode C-ABI: the workspace queries are pure host functions, a missing or too-small workspace
is refused before any CUDA call, and the MMU_DETERMINISTIC knob and torch's flag both select the mode."""
import ctypes
import os
import subprocess
import sys

import torch

from conftest import PKG, ROOT
from mmunet_b200 import _lib, ops

MMU_ERR_INVALID, MMU_ERR_WORKSPACE = -1, -3
FAKE_WS = 1 << 20          # a 256-byte aligned non-NULL address: never dereferenced when the size check refuses it


def _queries(lib):
    return {
        "scan": lambda: lib.mmu_selective_scan_bwd_det_workspace(8, 384, 4096, 16),
        "scan_rcg": lambda: lib.mmu_selective_scan_bwd_det_workspace(16, 128, 65536, 16),
        "scan_wide_state": lambda: lib.mmu_selective_scan_bwd_det_workspace(2, 20, 264, 64),
        "conv_f32": lambda: lib.mmu_causal_conv1d_bwd_det_workspace(8, 384, 4096, _lib.F32),
        "conv_bf16": lambda: lib.mmu_causal_conv1d_bwd_det_workspace(8, 384, 4096, _lib.BF16),
        "narrow_post": lambda: lib.mmu_mamba_narrow_post_bwd_det_workspace(16, 65536),
        "narrow_pre": lambda: lib.mmu_mamba_narrow_pre_bwd_det_workspace(16, 65536),
        "gn_fwd": lambda: lib.mmu_group_norm_nhwc_fwd_det_workspace(2, 64, 512 * 512, 16),
        "gn_bwd": lambda: lib.mmu_group_norm_nhwc_bwd_det_workspace(2, 64, 512 * 512, 16),
    }


def test_det_workspace_queries_are_pure():
    lib = _lib.lib()
    err = lib.mmu_last_error()
    for name, q in _queries(lib).items():
        a = q()
        assert a > 0 and a % 256 == 0 and a == q(), name
    assert lib.mmu_last_error() == err                        # a query sets no error state
    # dB / dC slots dominate the scan's: ceil(D / rows per CTA) * B * N * L * 8 bytes at most
    assert lib.mmu_selective_scan_bwd_det_workspace(8, 384, 4096, 16) >= (384 // 8) * 8 * 16 * 4096 * 8
    assert lib.mmu_selective_scan_bwd_det_workspace(0, 384, 4096, 16) == 0
    assert lib.mmu_snake_sample_bwd_det_workspace(2, 16, 512, 512, 9, 1) == 0      # gather-side: no slots


def test_det_entry_points_refuse_missing_or_small_workspace_without_gpu():
    lib = _lib.lib()
    p = _lib.ScanBwdParams()
    p.f.batch, p.f.dim, p.f.seqlen, p.f.dstate = 2, 6, 256, 16
    need = lib.mmu_selective_scan_bwd_det_workspace(2, 6, 256, 16)
    assert lib.mmu_selective_scan_bwd_det(ctypes.byref(p), None, need, None) == MMU_ERR_WORKSPACE
    assert lib.mmu_selective_scan_bwd_det(ctypes.byref(p), FAKE_WS, need - 1, None) == MMU_ERR_WORKSPACE
    assert b"workspace" in lib.mmu_last_error()
    assert lib.mmu_selective_scan_bwd_det(None, FAKE_WS, need, None) == MMU_ERR_INVALID
    p.f.batch = 0
    assert lib.mmu_selective_scan_bwd_det(ctypes.byref(p), FAKE_WS, need, None) == MMU_ERR_INVALID

    c = _lib.ConvParams()
    c.batch, c.dim, c.seqlen, c.width, c.dtype = 2, 8, 4096, 4, _lib.BF16
    need = lib.mmu_causal_conv1d_bwd_det_workspace(2, 8, 4096, _lib.BF16)
    assert lib.mmu_causal_conv1d_bwd_det(ctypes.byref(c), None, need, None) == MMU_ERR_WORKSPACE
    assert lib.mmu_causal_conv1d_bwd_det(ctypes.byref(c), FAKE_WS, need - 4, None) == MMU_ERR_WORKSPACE

    n = _lib.NarrowParams()
    n.d_model, n.d_inner, n.d_state, n.dt_rank, n.d_conv, n.batch, n.seqlen = 3, 6, 16, 1, 4, 2, 1024
    for fn, q in ((lib.mmu_mamba_narrow_post_bwd_det, lib.mmu_mamba_narrow_post_bwd_det_workspace),
                  (lib.mmu_mamba_narrow_pre_bwd_det, lib.mmu_mamba_narrow_pre_bwd_det_workspace)):
        need = q(2, 1024)
        assert fn(ctypes.byref(n), None, need, None) == MMU_ERR_WORKSPACE
        assert fn(ctypes.byref(n), FAKE_WS, need - 1, None) == MMU_ERR_WORKSPACE

    need = lib.mmu_group_norm_nhwc_fwd_det_workspace(2, 64, 1024, 16)
    gn = [FAKE_WS] * 7 + [_lib.F32, _lib.F32, 2, 64, 1024, 16, 1e-5]
    assert lib.mmu_group_norm_nhwc_fwd_det(*gn, None, need, None) == MMU_ERR_WORKSPACE
    assert lib.mmu_group_norm_nhwc_fwd_det(*gn, FAKE_WS, need - 1, None) == MMU_ERR_WORKSPACE
    need = lib.mmu_group_norm_nhwc_bwd_det_workspace(2, 64, 1024, 16)
    gb = [FAKE_WS] * 8 + [_lib.F32, _lib.F32, 2, 64, 1024, 16]
    assert lib.mmu_group_norm_nhwc_bwd_det(*gb, None, need, None) == MMU_ERR_WORKSPACE
    assert lib.mmu_group_norm_nhwc_bwd_det(*gb, FAKE_WS, need - 1, None) == MMU_ERR_WORKSPACE
    # null tensor pointers are refused as by the plain entry points
    assert lib.mmu_snake_sample_bwd_det(None, None, None, None, None, _lib.F32, _lib.F32, 1, 4, 8, 8, 3, 0, None, 0, None) == MMU_ERR_INVALID


def test_deterministic_mode_switches():
    was = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True, warn_only=True)
        assert ops._deterministic()
    finally:
        torch.use_deterministic_algorithms(was)
    code = ("import sys; sys.path[:0] = sys.argv[1:3]; from mmunet_b200 import _lib, ops; "
            "print(_lib.lib().mmu_deterministic_default(), int(ops._deterministic()))")
    for value, want in (("1", "1 1"), ("0", "0 0"), ("", "0 0")):
        env = dict(os.environ, MMU_DETERMINISTIC=value)
        out = subprocess.run([sys.executable, "-c", code, ROOT, PKG], env=env, capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr[-2000:]
        assert out.stdout.split() == want.split(), (value, out.stdout)
