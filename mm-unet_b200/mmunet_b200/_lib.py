"""ctypes binding of libmmunet_b200.so (the C-ABI declared in include/mmunet_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails, a RuntimeError is
raised.  The product path never routes through PyTorch reference code or the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("MMU_LIB") or os.path.join(_HERE, "libmmunet_b200.so")   # MMU_LIB: an experiment build (csrc/build.sh MMU_VARIANT)

F32, BF16, F16 = 0, 1, 2
ORDER_ROWMAJOR, ORDER_FLIP, ORDER_NSLICES, ORDER_TWOROW = 0, 1, 2, 3
STATE_STRIDE = 64

_vp, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t


class ScanFwdParams(C.Structure):
    _fields_ = (
        [(n, _i32) for n in ("batch", "dim", "seqlen", "dstate", "dtype", "delta_softplus", "reverse", "x_stride")]
        + [(n, _vp) for n in ("u", "delta", "z", "B", "C", "A", "D", "delta_bias", "out", "x", "last_state")]
        + [(n, _i64) for n in ("u_bs", "u_ds", "delta_bs", "delta_ds", "z_bs", "z_ds", "out_bs", "out_ds",
                               "B_bs", "B_ns", "C_bs", "C_ns")]
        + [("workspace", _vp), ("workspace_bytes", _sz), ("y", _vp), ("y_bs", _i64), ("y_ds", _i64)]
        + [(n, _i32) for n in ("order", "order_h", "order_w", "order_ns")]
    )


class ScanBwdParams(C.Structure):
    _fields_ = (
        [("f", ScanFwdParams), ("dout", _vp), ("dout_bs", _i64), ("dout_ds", _i64)]
        + [(n, _vp) for n in ("du", "ddelta", "dz")]
        + [(n, _i64) for n in ("du_bs", "du_ds", "ddelta_bs", "ddelta_ds", "dz_bs", "dz_ds")]
        + [(n, _vp) for n in ("dA", "dB", "dC", "dD", "ddelta_bias")]
        + [("dB_bs", _i64), ("dC_bs", _i64), ("dB_ns", _i64), ("dC_ns", _i64)]
    )


class ConvParams(C.Structure):
    _fields_ = (
        [(n, _i32) for n in ("batch", "dim", "seqlen", "width", "dtype", "silu", "reverse", "reserved")]
        + [(n, _vp) for n in ("x", "weight", "bias", "out")]
        + [(n, _i64) for n in ("x_bs", "x_ds", "out_bs", "out_ds", "w_ds", "w_ws")]
        + [(n, _vp) for n in ("dout", "dx", "dweight", "dbias")]
        + [(n, _i64) for n in ("dout_bs", "dout_ds", "dx_bs", "dx_ds")]
        + [(n, _i32) for n in ("order", "order_h", "order_w", "order_ns")]
    )


class NarrowParams(C.Structure):
    """mmu_narrow_params (include/mmunet_b200.h)."""
    _fields_ = (
        [(n, _i32) for n in ("dtype", "batch", "seqlen", "d_model", "d_inner", "d_state", "dt_rank", "d_conv",
                             "order", "order_h", "order_w", "order_ns")]
        + [(n, _vp) for n in ("in_proj_w", "conv_w", "conv_b", "x_proj_w", "dt_proj_w", "out_proj_w", "hidden")]
        + [(n, _i64) for n in ("hidden_bs", "hidden_cs")]
        + [(n, _vp) for n in ("pre", "out_z", "out")]
        + [(n, _i64) for n in ("out_bs", "out_cs")]
        + [("dout", _vp)]
        + [(n, _i64) for n in ("dout_bs", "dout_cs")]
        + [(n, _vp) for n in ("dout_y", "gpre", "dBC", "dhidden")]
        + [(n, _i64) for n in ("dhidden_bs", "dhidden_cs")]
        + [("dweights", _vp)]
        + [(n, _i32) for n in ("hidden_dtype", "coord_mode", "map_h", "map_w")]
        + [("extend_scope", C.c_float)]
        + [(n, _vp) for n in ("altho", "coords", "dcoords")]
    )


EXPORTS = (
    "mmu_version", "mmu_last_error", "mmu_launch_count", "mmu_reload_knobs",
    "mmu_selective_scan_fwd_workspace", "mmu_selective_scan_fwd",
    "mmu_selective_scan_bwd_workspace", "mmu_selective_scan_bwd", "mmu_scan_state_stride",
    "mmu_causal_conv1d_fwd", "mmu_causal_conv1d_bwd",
    "mmu_scan_order_gather", "mmu_scan_order_scatter", "mmu_scan_order_index", "mmu_scan_order_fusable",
    "mmu_snake_sample_fwd", "mmu_snake_sample_bwd",
    "mmu_group_norm_nhwc_fwd", "mmu_group_norm_nhwc_bwd",
    "mmu_mamba_narrow_supported", "mmu_mamba_narrow_rows", "mmu_mamba_narrow_weight_floats",
    "mmu_mamba_narrow_pre_fwd", "mmu_mamba_narrow_post_fwd", "mmu_mamba_narrow_post_bwd", "mmu_mamba_narrow_pre_bwd",
    "mmu_deterministic_default",
    "mmu_selective_scan_bwd_det_workspace", "mmu_selective_scan_bwd_det",
    "mmu_causal_conv1d_bwd_det_workspace", "mmu_causal_conv1d_bwd_det",
    "mmu_mamba_narrow_post_bwd_det_workspace", "mmu_mamba_narrow_pre_bwd_det_workspace",
    "mmu_mamba_narrow_post_bwd_det", "mmu_mamba_narrow_pre_bwd_det",
    "mmu_group_norm_nhwc_fwd_det_workspace", "mmu_group_norm_nhwc_bwd_det_workspace",
    "mmu_group_norm_nhwc_fwd_det", "mmu_group_norm_nhwc_bwd_det",
    "mmu_snake_sample_bwd_det_workspace", "mmu_snake_sample_bwd_det",
)

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"mmunet_b200: CUDA extension {SO_PATH} is missing - build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or mm-unet_b200/csrc/build.sh. "
            "There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    L.mmu_version.restype = C.c_int
    L.mmu_last_error.restype = C.c_char_p
    L.mmu_launch_count.restype = C.c_uint64
    for n in ("mmu_selective_scan_fwd_workspace", "mmu_selective_scan_bwd_workspace"):
        getattr(L, n).restype = _sz
        getattr(L, n).argtypes = [_i32, _i32, _i32, _i32]
    L.mmu_scan_state_stride.restype = _i32
    L.mmu_scan_state_stride.argtypes = [_i32] * 5
    L.mmu_selective_scan_fwd.argtypes = [C.POINTER(ScanFwdParams), _vp]
    L.mmu_selective_scan_bwd.argtypes = [C.POINTER(ScanBwdParams), _vp]
    L.mmu_causal_conv1d_fwd.argtypes = [C.POINTER(ConvParams), _vp]
    L.mmu_causal_conv1d_bwd.argtypes = [C.POINTER(ConvParams), _vp]
    for n in ("mmu_scan_order_gather", "mmu_scan_order_scatter"):
        getattr(L, n).argtypes = [_vp, _vp, _i32, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp]
    L.mmu_scan_order_index.argtypes = [_vp, _i32, _i32, _i32, _i32, _vp]
    L.mmu_scan_order_fusable.restype = _i32
    L.mmu_scan_order_fusable.argtypes = [_i32] * 6
    L.mmu_snake_sample_fwd.argtypes = [_vp, _vp, _vp] + [_i32] * 8 + [_vp]
    L.mmu_snake_sample_bwd.argtypes = [_vp, _vp, _vp, _vp, _vp] + [_i32] * 8 + [_vp]
    L.mmu_group_norm_nhwc_fwd.argtypes = [_vp] * 7 + [_i32] * 6 + [C.c_float, _vp]
    L.mmu_group_norm_nhwc_bwd.argtypes = [_vp] * 8 + [_i32] * 6 + [_vp]
    L.mmu_mamba_narrow_supported.restype = _i32
    L.mmu_mamba_narrow_supported.argtypes = [_i32] * 6
    L.mmu_mamba_narrow_rows.restype = _i32
    L.mmu_mamba_narrow_rows.argtypes = [_i32] * 2
    L.mmu_mamba_narrow_weight_floats.restype = _i32
    L.mmu_mamba_narrow_weight_floats.argtypes = [_i32] * 5
    for n in ("mmu_mamba_narrow_pre_fwd", "mmu_mamba_narrow_post_fwd", "mmu_mamba_narrow_post_bwd", "mmu_mamba_narrow_pre_bwd"):
        getattr(L, n).argtypes = [C.POINTER(NarrowParams), _vp]
    # deterministic mode: the plain entry point's arguments + (workspace, workspace bytes) before the stream
    L.mmu_deterministic_default.restype = _i32
    L.mmu_deterministic_default.argtypes = []
    for n, args in (("mmu_selective_scan_bwd_det_workspace", [_i32] * 4), ("mmu_causal_conv1d_bwd_det_workspace", [_i32] * 4),
                    ("mmu_mamba_narrow_post_bwd_det_workspace", [_i32] * 2), ("mmu_mamba_narrow_pre_bwd_det_workspace", [_i32] * 2),
                    ("mmu_group_norm_nhwc_fwd_det_workspace", [_i32] * 4), ("mmu_group_norm_nhwc_bwd_det_workspace", [_i32] * 4)):
        getattr(L, n).restype = _sz
        getattr(L, n).argtypes = args
    L.mmu_selective_scan_bwd_det.argtypes = [C.POINTER(ScanBwdParams), _vp, _sz, _vp]
    L.mmu_causal_conv1d_bwd_det.argtypes = [C.POINTER(ConvParams), _vp, _sz, _vp]
    for n in ("mmu_mamba_narrow_post_bwd_det", "mmu_mamba_narrow_pre_bwd_det"):
        getattr(L, n).argtypes = [C.POINTER(NarrowParams), _vp, _sz, _vp]
    L.mmu_group_norm_nhwc_fwd_det.argtypes = [_vp] * 7 + [_i32] * 6 + [C.c_float, _vp, _sz, _vp]
    L.mmu_group_norm_nhwc_bwd_det.argtypes = [_vp] * 8 + [_i32] * 6 + [_vp, _sz, _vp]
    L.mmu_snake_sample_bwd_det_workspace.restype = _sz
    L.mmu_snake_sample_bwd_det_workspace.argtypes = [_i32] * 6
    L.mmu_snake_sample_bwd_det.argtypes = [_vp, _vp, _vp, _vp, _vp] + [_i32] * 8 + [_vp, _sz, _vp]
    for n in EXPORTS:      # fail loudly on a stale library
        getattr(L, n)
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().mmu_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def reload_knobs() -> None:
    """Re-read the MMU_* environment knobs (they are read once by the library)."""
    lib().mmu_reload_knobs()


def launch_count() -> int:
    return int(lib().mmu_launch_count())
