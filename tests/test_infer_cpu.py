"""CPU-side checks of sliding-window prediction: the window placement rule (monai's dense_patch_slices / _get_scan_interval and its
padding), the C-ABI of mmu_sw_stitch (header, export table and ctypes binding agree; every bad argument is refused with
MMU_ERR_INVALID before any CUDA call), segmentation_metrics, and the predictor's argument checks."""
import ctypes as ct
import math
import os
import re

import pytest
import torch

from conftest import ROOT
from mmunet_b200 import _lib
from mmunet_b200.infer import SlidingWindowPredictor, pad_for_roi, scan_interval, segmentation_metrics, window_starts

MMU_ERR_INVALID = -1
FAKE = 1 << 20                     # a non-NULL, 16-byte aligned address: never dereferenced when the arguments are refused


@pytest.mark.parametrize("n,roi,overlap,want", [
    (584, 512, .5, [0, 72]), (565, 512, .5, [0, 53]), (512, 512, .5, [0]), (960, 512, .5, [0, 256, 448]),
    (999, 512, .5, [0, 256, 487]), (512, 512, 0.0, [0]), (64, 64, .75, [0]),
])
def test_window_starts(n, roi, overlap, want):
    assert window_starts(n, roi, overlap) == want


def test_window_starts_long_axis_and_strides():
    s = window_starts(3504, 512, .5)
    assert len(s) == 13 and s[-1] == 2992 and s[:-1] == [256 * d for d in range(12)]
    assert scan_interval(100, 64, 0.0) == 64 and scan_interval(100, 64, 0.75) == 16 and scan_interval(64, 64, 0.75) == 64
    assert window_starts(200, 64, 0.0) == [0, 64, 128, 136]
    assert window_starts(100, 64, 0.75) == [0, 16, 32, 36]
    for n, roi, ov in ((584, 512, .5), (3504, 512, .5), (200, 64, 0.0), (100, 64, .75), (97, 32, .9)):
        s, iv = window_starts(n, roi, ov), scan_interval(n, roi, ov)
        assert s[-1] == n - roi and all(b > a for a, b in zip(s, s[1:]))
        assert all((d - 1) * iv + roi < n for d in range(1, len(s)))      # every window but the last one is needed
        covered = set()
        for a in s:
            covered.update(range(a, a + roi))
        assert covered == set(range(n))
    with pytest.raises(ValueError):
        window_starts(300, 512, .5)


def test_pad_for_roi():
    assert pad_for_roi(300, 512) == (106, 106)
    assert pad_for_roi(301, 512) == (105, 106)
    assert pad_for_roi(512, 512) == (0, 0) and pad_for_roi(2336, 512) == (0, 0)
    assert pad_for_roi(1, 64) == (31, 32)


# ---- C-ABI ---------------------------------------------------------------------------------------------------------------
def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "mmunet_b200.h")).read(), flags=re.S)


def test_header_export_and_binding_agree():
    src = _header()
    assert re.search(r"\bint\s+mmu_sw_stitch\s*\(\s*const\s+mmu_sw_stitch_params\s*\*\s*p\s*,\s*void\s*\*\s*stream\s*\)\s*;", src)
    assert re.search(r"#define\s+MMU_SW_HEADS\s+5\b", src) and _lib.SW_HEADS == 5
    body = re.search(r"typedef\s+struct\s+mmu_sw_stitch_params\s*\{(.*?)\}\s*mmu_sw_stitch_params\s*;", src, flags=re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            names.append(re.sub(r"\[.*?\]", "", part.strip().split()[-1]).lstrip("*"))
    assert names == [f[0] for f in _lib.SwStitchParams._fields_]
    # field sizes: arrays of 5, 4-byte ints up to the head sizes, then pointers and int64s
    assert ct.sizeof(_lib.SwStitchParams) == 11 * 4 + 10 * 4 + 4 + 5 * 8 + 15 * 8 + 3 * 8 * 3 + 8
    assert "mmu_sw_stitch" in _lib.EXPORTS
    fn = _lib.lib().mmu_sw_stitch
    assert len(fn.argtypes) == 2
    assert _lib.lib().mmu_version() == 100


def _params(**kw):
    p = _lib.SwStitchParams()
    p.dtype, p.batch, p.H, p.W, p.roi = _lib.F32, 2, 584, 565, 512
    p.n_h, p.n_w, p.pad_top, p.pad_left, p.interval_h, p.interval_w = 584, 565, 0, 0, 256, 256
    for k, s in enumerate((256, 128, 64, 32, 256)):
        p.head_h[k] = p.head_w[k] = s
        p.heads[k] = FAKE
        p.head_rs[k], p.head_ws[k], p.head_bs[k] = s, s * s, 4 * s * s
    p.logits, p.logits_bs, p.logits_rs = FAKE, 584 * 565, 565
    for name, v in kw.items():
        if isinstance(v, tuple):         # (field, index, value) for the per-head arrays
            getattr(p, v[0])[v[1]] = v[2]
        else:
            setattr(p, name, v)
    return p


def _call(p):
    return _lib.lib().mmu_sw_stitch(ct.byref(p), None)


@pytest.mark.parametrize("kw,what", [
    (dict(dtype=_lib.F16), b"dtype"), (dict(dtype=7), b"dtype"), (dict(dtype=-1), b"dtype"),
    (dict(batch=0), b"bad shape"), (dict(H=0), b"bad shape"), (dict(W=-1), b"bad shape"), (dict(roi=0), b"bad shape"),
    (dict(n_h=511, H=511), b"geometry"),                                    # n < roi
    (dict(n_w=500, W=500), b"geometry"),
    (dict(pad_top=-1), b"geometry"), (dict(pad_left=1), b"geometry"),      # pad + W > n
    (dict(interval_h=0), b"geometry"), (dict(interval_w=513), b"geometry"),
    (dict(logits=None), b"null logits"),
    (dict(counts=FAKE), b"target"),                                         # counts without a target
    (dict(counts=FAKE + 4, target=FAKE), b"aligned"),
    (dict(h=("heads", 3, None)), b"null head 3"),
    (dict(h=("head_h", 0, 0)), b"head 0"), (dict(h=("head_w", 4, -2)), b"head 4"),
    (dict(h=("head_rs", 1, -1)), b"negative stride"),
    (dict(h=("head_bs", 2, 2**63 - 1)), b"overflows"),                      # (batch - 1) * stride + ... > int64
    (dict(h=("head_ws", 0, 2**62)), b"overflows"),                          # (4 - 1) windows * 2^62
    (dict(logits_rs=-565), b"negative stride"),
    (dict(logits_bs=2**63 - 1), b"overflows"),
    (dict(batch=65536, h=("head_bs", 0, 0)), b"index range"),
])
def test_bad_arguments_are_refused_without_gpu(kw, what):
    h = kw.pop("h", None)
    p = _params(**kw)
    if h is not None:
        getattr(p, h[0])[h[1]] = h[2]
    if kw.get("batch") == 65536:                                             # keep every stride in range: only the grid is too big
        for k in range(5):
            p.head_bs[k] = 0
        p.logits_bs = 0
    assert _call(p) == MMU_ERR_INVALID
    assert what in _lib.lib().mmu_last_error()


def test_null_params_refused():
    assert _lib.lib().mmu_sw_stitch(None, None) == MMU_ERR_INVALID


def test_rows_past_the_grid_limit_refused():
    p = _params(H=8 * 65535 + 1, n_h=8 * 65535 + 1, logits_bs=0)
    assert _call(p) == MMU_ERR_INVALID
    assert b"index range" in _lib.lib().mmu_last_error()


# ---- metrics and arguments -----------------------------------------------------------------------------------------------
def test_segmentation_metrics():
    counts = torch.tensor([[30, 10, 20, 940], [0, 0, 0, 7], [0, 5, 0, 0], [4, 0, 0, 0]], dtype=torch.int64)
    m = segmentation_metrics(counts)
    assert all(v.dtype == torch.float64 and v.shape == (4,) for v in m.values())
    tp, fp, fn, tn = 30, 10, 20, 940
    assert m["dice"][0] == 2 * tp / (2 * tp + fp + fn)
    assert m["iou"][0] == tp / (tp + fp + fn)
    assert m["accuracy"][0] == (tp + tn) / 1000
    assert m["sensitivity"][0] == tp / (tp + fn)
    assert m["specificity"][0] == tn / (tn + fp)
    # image 1: no positives at all -> Dice, IoU, sensitivity undefined; image 2: no negatives predicted right, no positives
    assert math.isnan(m["dice"][1]) and math.isnan(m["iou"][1]) and math.isnan(m["sensitivity"][1])
    assert m["accuracy"][1] == 1.0 and m["specificity"][1] == 1.0
    assert m["dice"][2] == 0.0 and math.isnan(m["sensitivity"][2]) and m["specificity"][2] == 0.0
    assert m["dice"][3] == 1.0 and m["iou"][3] == 1.0 and math.isnan(m["specificity"][3])
    assert segmentation_metrics([1, 1, 1, 1])["accuracy"].item() == 0.5


class _Heads(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.conv = torch.nn.Conv2d(3, 1, 1)

    def forward_heads(self, x):
        return (self.conv(x),) * 5


@pytest.mark.parametrize("kw", [dict(roi_size=100), dict(roi_size=0), dict(roi_size=-32), dict(roi_size=64.0), dict(roi_size=True),
                                dict(overlap=1.0), dict(overlap=-0.1), dict(overlap=1.5),
                                dict(sw_batch_size=0), dict(sw_batch_size=-1), dict(sw_batch_size=2.0),
                                dict(dtype="int8")])
def test_predictor_refuses_bad_arguments(kw):
    with pytest.raises(ValueError):
        SlidingWindowPredictor(_Heads(), **kw)


def test_predictor_refuses_cpu_model_and_models_without_heads():
    with pytest.raises(RuntimeError, match="CUDA"):
        SlidingWindowPredictor(_Heads(), roi_size=64)
    with pytest.raises(TypeError, match="forward_heads"):
        SlidingWindowPredictor(torch.nn.Conv2d(3, 1, 1), roi_size=64)
