"""CPU-side checks of the bilinear-resize backward (mmu_resize_bilinear_bwd_det): the header, the export table and the ctypes binding
agree; every bad argument is refused with MMU_ERR_INVALID before any CUDA call; ops.resize_bilinear is plain F.interpolate off the GPU;
and the trainer's check of CUBLAS_WORKSPACE_CONFIG under strict deterministic mode."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from mmunet_b200 import _lib, ops, train

MMU_ERR_INVALID = -1
FAKE = 1 << 20                     # a non-NULL, 16-byte aligned address: never dereferenced when the arguments are refused
NAME = "mmu_resize_bilinear_bwd_det"


def test_header_and_export_agree():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "mmunet_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+" + NAME + r"\s*\(([^)]*)\)\s*;", src)
    assert m, f"{NAME} is not declared in include/mmunet_b200.h"
    params = [p.strip() for p in m.group(1).split(",")]
    assert [p.split()[-1].lstrip("*") for p in params] == ["dout", "dx", "dtype", "B", "C", "H_in", "W_in", "H_out", "W_out",
                                                            "channels_last", "stream"]
    assert NAME in _lib.EXPORTS
    fn = getattr(_lib.lib(), NAME)
    assert len(fn.argtypes) == len(params)
    assert _lib.lib().mmu_version() == 100


def _call(dout=FAKE, dx=FAKE, dtype=_lib.F32, B=2, C=64, Hi=16, Wi=16, Ho=32, Wo=32, cl=0):
    return getattr(_lib.lib(), NAME)(dout, dx, dtype, B, C, Hi, Wi, Ho, Wo, cl, None)


@pytest.mark.parametrize("args,what", [
    (dict(dout=None), b"null"), (dict(dx=None), b"null"),
    (dict(dtype=_lib.F16), b"dtype"), (dict(dtype=7), b"dtype"), (dict(dtype=-1), b"dtype"),
    (dict(B=0), b"bad shape"), (dict(C=-3), b"bad shape"), (dict(Hi=0), b"bad shape"), (dict(Wi=-1), b"bad shape"),
    (dict(Ho=0), b"bad shape"), (dict(Wo=0, cl=1), b"bad shape"),
    (dict(Hi=65536, Wi=65536, C=1, B=1), b"index"),                         # one plane of 2^32 input pixels
    (dict(Ho=65536, Wo=32768, C=1, B=1), b"index"),                          # one plane of 2^31 output pixels
    (dict(Hi=16384, Wi=16384, C=64, B=1, cl=1), b"index"),                   # 2^28 pixels x 16 fp32 vectors
    (dict(B=2**31 - 1, C=2**31 - 1, Hi=2**15, Wi=2**15), b"index"),         # element count overflows int64
])
def test_bad_arguments_are_refused_without_gpu(args, what):
    assert _call(**args) == MMU_ERR_INVALID
    assert what in _lib.lib().mmu_last_error()


@pytest.mark.parametrize("det", [False, True])
def test_resize_bilinear_is_interpolate_off_the_gpu(det):
    """On CPU tensors (and for dtypes or layouts the kernel does not take) the op is F.interpolate itself, in either mode."""
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(det, warn_only=True)
    try:
        x = torch.randn(2, 3, 7, 9, dtype=torch.float64, requires_grad=True)
        for kw in (dict(size=(14, 5)), dict(scale_factor=2)):
            got = ops.resize_bilinear(x, **kw)
            want = F.interpolate(x, mode="bilinear", align_corners=True, **kw)
            assert got.grad_fn is not None and type(got.grad_fn).__name__ == type(want.grad_fn).__name__
            assert torch.equal(got, want)
    finally:
        torch.use_deterministic_algorithms(was)


def test_trainer_cublas_check(monkeypatch):
    was, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        monkeypatch.delenv("CUBLAS_WORKSPACE_CONFIG", raising=False)
        torch.use_deterministic_algorithms(False)
        train.check_deterministic_cublas()                       # mode off: nothing to check
        torch.use_deterministic_algorithms(True, warn_only=True)
        train.check_deterministic_cublas()                       # warn_only: torch itself only warns
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="CUBLAS_WORKSPACE_CONFIG=:4096:8"):
            train.check_deterministic_cublas()
        monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":0:0")
        with pytest.raises(RuntimeError, match="':0:0'"):
            train.check_deterministic_cublas()
        for ok in (":4096:8", ":16:8"):
            monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ok)
            train.check_deterministic_cublas()
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn)
