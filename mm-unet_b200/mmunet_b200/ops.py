"""Host-side mirror of the reference's fused-op interface, on top of the C-ABI CUDA library.

Same names, argument meaning and error behaviour as
  requirements/Mamba/mamba/mamba_ssm/ops/selective_scan_interface.py   (SelectiveScanFn :14-83,
      MambaInnerFnNoOutProj :155-289, MambaInnerFn :292-434, BiMambaInnerFn :437-603, wrappers :606-633)
  requirements/Mamba/causal-conv1d/causal_conv1d/causal_conv1d_interface.py  (CausalConv1dFn :10-46)

PyTorch is used for device memory, streams, autograd bookkeeping and the skinny projection GEMMs
(cuBLAS through F.linear / matmul, exactly where the reference uses them).  Every scan / conv / permutation
is a call into libmmunet_b200.so; there is no CPU or eager fallback - a missing library or a non-CUDA tensor
raises RuntimeError.
"""
from __future__ import annotations

import ctypes as ct

import torch
import torch.nn.functional as F

from . import _lib

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16, torch.float16: _lib.F16}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("mmunet_b200: expected CUDA tensors (there is no CPU path)")


# Deterministic mode (include/mmunet_b200.h, "Deterministic mode"): every op below that sums floats across CTAs then calls its _det
# entry point, which needs a workspace of partial-sum slots and gives bitwise reproducible results.
_DET_SCAN_WS_CAP = 512 << 20      # bytes of scan-backward slots per call; larger problems run over batch slices


def _deterministic() -> bool:
    """True when torch.use_deterministic_algorithms(True) is on or the environment knob MMU_DETERMINISTIC is set (for callers that
    cannot set torch's flag).  Checked when each kernel runs: backward functions at backward time."""
    return torch.are_deterministic_algorithms_enabled() or bool(_lib.lib().mmu_deterministic_default())


def _det_workspace(nbytes, device):
    """-> (tensor, pointer, bytes): a fresh workspace for a _det entry point from the caching allocator of the current stream (its
    contents do not matter: the kernels overwrite every slot they read)."""
    ws = torch.empty(max(int(nbytes), 1), device=device, dtype=torch.uint8)
    return ws, ws.data_ptr(), int(nbytes)


# ----------------------------------------------------------------------------------------------------------
# raw kernels
# ----------------------------------------------------------------------------------------------------------

def _scan_checks(u, delta, A, B, C, D, z, delta_bias):
    """Argument validation with the reference's rules (selective_scan.cpp:233-303)."""
    _require_cuda(u, delta, A, B, C, D, z, delta_bias)
    if u.dtype not in _DT:
        raise RuntimeError("selective_scan: input type must be float32, float16 or bfloat16")
    if A.is_complex():
        raise RuntimeError("selective_scan: complex A is not supported by mmunet_b200 (MM-UNet uses real A)")
    if A.dtype != torch.float32:
        raise RuntimeError("selective_scan: weight_type (A) must be float32")
    if B.dim() < 3 or C.dim() < 3:
        raise RuntimeError("selective_scan: constant (non input-dependent) B/C are not supported by mmunet_b200")
    if delta.dtype != u.dtype or B.dtype != u.dtype or C.dtype != u.dtype:
        raise RuntimeError("selective_scan: delta, B and C must have the same dtype as u")
    batch, dim, L = u.shape
    N = A.shape[1]
    if N > 256:
        raise RuntimeError("selective_scan only supports state dimension <= 256")
    if delta.shape != u.shape:
        raise RuntimeError(f"selective_scan: delta shape {tuple(delta.shape)} != u shape {tuple(u.shape)}")
    if A.shape[0] != dim:
        raise RuntimeError("selective_scan: A must be (dim, dstate)")
    for name, t in (("B", B), ("C", C)):
        if t.shape[0] != batch or t.shape[-2] != N or t.shape[-1] != L:
            raise RuntimeError(f"selective_scan: {name} must be (batch, n_groups, dstate, seqlen)")
        if dim % t.shape[1] != 0:
            raise RuntimeError("selective_scan: dim must be divisible by n_groups")
    for name, t in (("u", u), ("delta", delta), ("B", B), ("C", C), ("z", z)):
        if t is not None and t.stride(-1) != 1 and t.shape[-1] > 1:
            raise RuntimeError(f"selective_scan: {name}.stride(-1) must be 1")
    if D is not None and (D.dtype != torch.float32 or D.shape != (dim,)):
        raise RuntimeError("selective_scan: D must be float32 of shape (dim,)")
    if delta_bias is not None and (delta_bias.dtype != torch.float32 or delta_bias.shape != (dim,)):
        raise RuntimeError("selective_scan: delta_bias must be float32 of shape (dim,)")
    if z is not None and (z.dtype != u.dtype or z.shape != u.shape):
        raise RuntimeError("selective_scan: z must match u in dtype and shape")
    if B.shape[1] != C.shape[1]:
        raise RuntimeError("selective_scan: B and C must have the same n_groups")


def _fill_fwd(p, u, delta, A, B, C, D, z, delta_bias, softplus, reverse, g, G):
    """Fill a ScanFwdParams for group g of G (rows [g*H, (g+1)*H))."""
    batch, dim, L = u.shape
    H = dim // G
    es = u.element_size()
    p.batch, p.dim, p.seqlen, p.dstate = batch, H, L, A.shape[1]
    p.dtype, p.delta_softplus, p.reverse = _DT[u.dtype], int(bool(softplus)), int(bool(reverse))
    p.u = u.data_ptr() + g * H * u.stride(1) * es
    p.delta = delta.data_ptr() + g * H * delta.stride(1) * es
    p.z = None if z is None else z.data_ptr() + g * H * z.stride(1) * es
    p.B = B.data_ptr() + g * B.stride(1) * es
    p.C = C.data_ptr() + g * C.stride(1) * es
    p.A = A.data_ptr() + g * H * A.stride(0) * 4
    p.D = None if D is None else D.data_ptr() + g * H * 4
    p.delta_bias = None if delta_bias is None else delta_bias.data_ptr() + g * H * 4
    p.u_bs, p.u_ds = u.stride(0), u.stride(1)
    p.delta_bs, p.delta_ds = delta.stride(0), delta.stride(1)
    if z is not None:
        p.z_bs, p.z_ds = z.stride(0), z.stride(1)
    p.B_bs, p.B_ns, p.C_bs, p.C_ns = B.stride(0), B.stride(2), C.stride(0), C.stride(2)


def order_fusable(order, dstate, dtype):
    """order = (kind, H, W, nslices) or None.  True when the conv / scan kernels can apply the scan order themselves
    (mmu_scan_order_fusable): the gate / output tensors then stay in natural token order and no gather / scatter copy runs."""
    if order is None or order[0] == _lib.ORDER_ROWMAJOR:
        return True
    if dtype not in _DT:
        return False
    kind, H, W, ns = order
    return bool(_lib.lib().mmu_scan_order_fusable(kind, H, W, max(1, ns), dstate, _DT[dtype]))


def _set_order(p, order):
    if order is not None:
        p.order, p.order_h, p.order_w, p.order_ns = order[0], order[1], order[2], max(1, order[3])


class ScanStates(tuple):
    """What the forward saves for the backward: x = fp32 states after every 64th token (batch, dim, ceil(L/64), dstate),
    y = pre-gate output C.h + D*u (input dtype; None without a gate) - the role of the reference's `scan_intermediates`
    and `out` (selective_scan_interface.py:213-219)."""
    __slots__ = ()

    def __new__(cls, x, y=None):
        return super().__new__(cls, (x, y))

    x = property(lambda self: self[0])
    y = property(lambda self: self[1])


def _wide_state_groups(u, A, B):
    """d_state > 16 on the fast kernels: the register-resident kernels walk at most 16 states, and the recurrences of different
    states are independent - y = sum_n C_n h_n is a sum over state groups, every gradient either a sum over groups (du, ddelta,
    ddelta_bias) or group-local (dA, dB, dC).  So a wide state dimension runs as ceil(dstate/16) passes of the dstate <= 16 kernels
    over 16-state slices of A / B / C, with the D skip in the first pass and the gate applied once to the summed y (the
    reference walks `for state_idx < dstate` inside one kernel, selective_scan_fwd_kernel.cuh:163).  Needs what those kernels
    need (seqlen % 8 == 0, fp32 / bf16, n_groups == 1); anything else stays on the generic kernels."""
    N = A.shape[1]
    if N <= 16 or B.shape[1] != 1 or u.shape[-1] % 8 != 0 or u.dtype not in (torch.float32, torch.bfloat16):
        return None
    return [(n0, min(n0 + 16, N)) for n0 in range(0, N, 16)]


def _silu_parts(z):
    zf = z.float()
    sg = torch.sigmoid(zf)
    return zf * sg, sg * (1.0 + zf * (1.0 - sg))          # silu(z), d silu / dz


def selective_scan_fwd(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False, reverse=False,
                       save_states=True, return_last_state=False, order=None):
    """-> (out, states, last_state).  out is y*silu(z) when z is given; states is a ScanStates (or None).
    order = (kind, H, W, nslices): fused scan order - z and out are in natural token order and permuted by the kernel, u, delta,
    B, C in scan order (only where order_fusable() holds)."""
    _scan_checks(u, delta, A, B, C, D, z, delta_bias)
    if order is not None and order[0] == _lib.ORDER_ROWMAJOR:
        order = None
    groups = _wide_state_groups(u, A, B) if order is None else None
    if groups is None:
        return _selective_scan_fwd_single(u, delta, A, B, C, D, z, delta_bias, delta_softplus, reverse, save_states, return_last_state,
                                          order)
    io_dtype = u.dtype
    if io_dtype != torch.float32:
        # the per-group partial sums of y cancel against each other: rounding each of them to bf16 first would cost ~3 digits of
        # the total, so 2-byte inputs run the group passes in fp32 on the same (rounded) values and round the result once
        u, delta, B, C = u.float(), delta.float(), B.float(), C.float()
    y32, xs, lasts = None, [], []
    for gi, (n0, n1) in enumerate(groups):
        yg, st, last = _selective_scan_fwd_single(u, delta, A[:, n0:n1].contiguous(), B[:, :, n0:n1], C[:, :, n0:n1], D if gi == 0 else None,
                                                   None, delta_bias, delta_softplus, reverse, save_states, return_last_state)
        y32 = yg.float() if y32 is None else y32.add_(yg)
        if save_states:
            xs.append(st.x)
        if return_last_state:
            lasts.append(last)
    y = y32.to(io_dtype)
    out = y if z is None else (y32 * _silu_parts(z)[0]).to(io_dtype)
    states = ScanStates(xs, y if z is not None else None) if save_states else None     # x: one saved-state tensor per state group
    return out, states, (torch.cat(lasts, dim=-1) if return_last_state else None)


def _selective_scan_fwd_single(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False, reverse=False,
                               save_states=True, return_last_state=False, order=None):
    batch, dim, L = u.shape
    N = A.shape[1]
    G = B.shape[1]
    A = A.contiguous()
    out = torch.empty_like(u, memory_format=torch.contiguous_format)
    H = dim // G
    L_ = _lib.lib()
    xs = L_.mmu_scan_state_stride(batch, H, L, N, _DT[u.dtype]) if (save_states and order is None) else _lib.STATE_STRIDE
    nx = (L + xs - 1) // xs
    x = torch.empty((batch, dim, nx, N), device=u.device, dtype=torch.float32) if save_states else None
    y = torch.empty_like(out) if (save_states and z is not None) else None
    last = torch.empty((batch, dim, N), device=u.device, dtype=torch.float32) if return_last_state else None
    ws_bytes = L_.mmu_selective_scan_fwd_workspace(batch, H, L, N)
    ws = torch.empty(ws_bytes, device=u.device, dtype=torch.uint8) if ws_bytes else None
    with torch.cuda.device(u.device):
        for g in range(G):
            p = _lib.ScanFwdParams()
            _fill_fwd(p, u, delta, A, B, C, D, z, delta_bias, delta_softplus, reverse, g, G)
            p.x_stride = xs
            _set_order(p, order)
            p.out = out.data_ptr() + g * H * out.stride(1) * out.element_size()
            p.out_bs, p.out_ds = out.stride(0), out.stride(1)
            p.x = None if x is None else x.data_ptr() + g * H * x.stride(1) * 4
            if y is not None:
                p.y = y.data_ptr() + g * H * y.stride(1) * y.element_size()
                p.y_bs, p.y_ds = y.stride(0), y.stride(1)
            p.last_state = None if last is None else last.data_ptr() + g * H * N * 4
            if G > 1:   # per-group x / last_state slices are not batch-contiguous: run into temporaries
                xg = torch.empty((batch, H, nx, N), device=u.device, dtype=torch.float32) if save_states else None
                lg = torch.empty((batch, H, N), device=u.device, dtype=torch.float32) if return_last_state else None
                p.x, p.last_state = _ptr(xg), _ptr(lg)
            p.workspace, p.workspace_bytes = _ptr(ws), ws_bytes
            _lib.check(L_.mmu_selective_scan_fwd(ct.byref(p), _stream()), "selective_scan_fwd")
            if G > 1:
                if x is not None:
                    x[:, g * H:(g + 1) * H] = xg
                if last is not None:
                    last[:, g * H:(g + 1) * H] = lg
    return out, (ScanStates(x, y) if save_states else None), last


def _x_stride(x, L):
    """Token stride of the saved states, from the shape the forward allocated (see mmu_scan_state_stride)."""
    n8, n64 = (L + 7) // 8, (L + _lib.STATE_STRIDE - 1) // _lib.STATE_STRIDE
    return 8 if (x.shape[2] == n8 and n8 != n64) else _lib.STATE_STRIDE


def selective_scan_bwd(u, delta, A, B, C, D, z, delta_bias, dout, x, delta_softplus=False, reverse=False,
                       du=None, ddelta=None, dz=None, dBC=None, order=None):
    """-> (du, ddelta, dA, dB, dC, dD, dz, ddelta_bias); see _selective_scan_bwd_single.  A saved-state LIST (one tensor per group
    of 16 states, from the grouped forward) selects the grouped backward.  order: as the forward (z, dout, dz in natural order)."""
    xs = x.x if isinstance(x, ScanStates) else x
    if order is not None and order[0] == _lib.ORDER_ROWMAJOR:
        order = None
    if not isinstance(xs, (list, tuple)):
        return _selective_scan_bwd_single(u, delta, A, B, C, D, z, delta_bias, dout, x, delta_softplus, reverse, du, ddelta, dz, dBC, order)
    _scan_checks(u, delta, A, B, C, D, z, delta_bias)
    groups = _wide_state_groups(u, A, B)
    batch, dim, L = u.shape
    N = A.shape[1]
    io_dtype = u.dtype
    if dout.stride(-1) != 1 and L > 1:
        dout = dout.contiguous()
    dy = dout.float()
    if z is not None:
        y = x.y
        silu, dsilu = _silu_parts(z)
        dz_val = (dy * y.float() * dsilu).to(io_dtype)
        dz = dz_val if dz is None else dz.copy_(dz_val)
        dy = dy * silu
    if io_dtype != torch.float32:       # as the forward: the group passes run in fp32 on the rounded inputs
        u, delta, B, C = u.float(), delta.float(), B.float(), C.float()
    else:
        dy = dy.contiguous()
    if dBC is None:
        dB = torch.zeros((batch, 1, N, L), device=u.device, dtype=torch.float32)
        dC = torch.zeros_like(dB)
        dB3, dC3 = dB[:, 0], dC[:, 0]
    else:
        dB3, dC3 = dBC
        dB, dC = dB3.unsqueeze(1), dC3.unsqueeze(1)
    dA = torch.empty((dim, N), device=u.device, dtype=torch.float32)
    du32 = dd32 = dD = dbias = None
    for gi, (n0, n1) in enumerate(groups):
        g = _selective_scan_bwd_single(u, delta, A[:, n0:n1].contiguous(), B[:, :, n0:n1], C[:, :, n0:n1], D if gi == 0 else None, None,
                                       delta_bias, dy, ScanStates(xs[gi], None), delta_softplus, reverse, dBC=(dB3[:, n0:n1], dC3[:, n0:n1]))
        du32 = g[0].float() if du32 is None else du32.add_(g[0])
        dd32 = g[1].float() if dd32 is None else dd32.add_(g[1])
        dA[:, n0:n1] = g[2]
        if gi == 0:
            dD = g[5]
        if g[7] is not None:
            dbias = g[7] if dbias is None else dbias + g[7]
    du = du32.to(io_dtype) if du is None else du.copy_(du32)
    ddelta = dd32.to(io_dtype) if ddelta is None else ddelta.copy_(dd32)
    return du, ddelta, dA, dB, dC, dD, dz, dbias


def _selective_scan_bwd_single(u, delta, A, B, C, D, z, delta_bias, dout, x, delta_softplus=False, reverse=False,
                               du=None, ddelta=None, dz=None, dBC=None, order=None):
    """-> (du, ddelta, dA, dB, dC, dD, dz, ddelta_bias); dA/dB/dC/dD/ddelta_bias fp32.
    du / ddelta / dz may be pre-allocated views (e.g. halves of dxz, as selective_scan_interface.py:244-248).
    dBC: optional pair (dB, dC) of ZERO-FILLED fp32 (batch, dstate, L) views with unit sequence stride and free batch / state
    strides that receive the gradients in place (n_groups == 1 only), e.g. row slices of the x_proj gradient buffer."""
    _scan_checks(u, delta, A, B, C, D, z, delta_bias)
    y = None
    if isinstance(x, ScanStates):
        x, y = x.x, x.y
    _require_cuda(dout, x, y)
    batch, dim, L = u.shape
    N = A.shape[1]
    G = B.shape[1]
    H = dim // G
    A = A.contiguous()
    if dout.dtype != u.dtype or dout.shape != u.shape:
        raise RuntimeError("selective_scan_bwd: dout must match u in dtype and shape")
    if dout.stride(-1) != 1 and L > 1:
        dout = dout.contiguous()
    du = torch.empty_like(u, memory_format=torch.contiguous_format) if du is None else du
    ddelta = torch.empty_like(delta, memory_format=torch.contiguous_format) if ddelta is None else ddelta
    if z is not None and dz is None:
        dz = torch.empty_like(z, memory_format=torch.contiguous_format)
    # one zero fill for every accumulated-into output (they are atomically added to, selective_scan.cpp:458-466)
    nBC = batch * G * N * L if dBC is None else 0
    nA = (dim * N + 3) // 4 * 4           # keeps dB / dC 16-byte aligned
    acc = torch.zeros(2 * nBC + nA + 2 * dim, device=u.device, dtype=torch.float32)
    if dBC is None:
        dB = acc[:nBC].view(batch, G, N, L)
        dC = acc[nBC:2 * nBC].view(batch, G, N, L)
    else:
        dB, dC = dBC
        for t in (dB, dC):
            if G != 1 or t.dtype != torch.float32 or t.shape != (batch, N, L) or (t.stride(2) != 1 and L > 1):
                raise RuntimeError("selective_scan_bwd: dBC must be two fp32 (batch, dstate, L) views with stride(-1) == 1, n_groups == 1")
        dB, dC = dB.unsqueeze(1), dC.unsqueeze(1)
    dA = acc[2 * nBC:2 * nBC + dim * N].view(dim, N)
    dD = acc[2 * nBC + nA:2 * nBC + nA + dim] if D is not None else None
    dbias = acc[2 * nBC + nA + dim:] if delta_bias is not None else None
    L_ = _lib.lib()
    det = _deterministic()
    # deterministic mode: batch slices whose partial slots fit _DET_SCAN_WS_CAP (a function of the shape, so still reproducible);
    # dA / dD / ddelta_bias then sum over the slices in slice order
    nb = batch
    if det:
        while nb > 1 and L_.mmu_selective_scan_bwd_det_workspace(nb, H, L, N) > _DET_SCAN_WS_CAP:
            nb = (nb + 1) // 2
    for b0 in range(0, batch, nb):
        sl = slice(b0, min(batch, b0 + nb))
        _scan_bwd_launch(u[sl], delta[sl], A, B[sl], C[sl], D, z if z is None else z[sl], delta_bias, dout[sl], x[sl],
                         None if y is None else y[sl], delta_softplus, reverse, du[sl], ddelta[sl], dz if dz is None else dz[sl],
                         dB[sl], dC[sl], dA, dD, dbias, order, det)
    return du, ddelta, dA, dB, dC, dD, dz, dbias


def _scan_bwd_launch(u, delta, A, B, C, D, z, delta_bias, dout, x, y, delta_softplus, reverse, du, ddelta, dz, dB, dC, dA, dD, dbias,
                     order, det):
    """One mmu_selective_scan_bwd(_det) call per B/C group on prepared tensors (dB / dC: (batch, G, N, L) views)."""
    batch, dim, L = u.shape
    N = A.shape[1]
    G = B.shape[1]
    H = dim // G
    L_ = _lib.lib()
    ws_bytes = L_.mmu_selective_scan_bwd_workspace(batch, H, L, N)
    ws = torch.empty(ws_bytes, device=u.device, dtype=torch.uint8) if ws_bytes else None
    if det:
        dws, dws_ptr, dws_bytes = _det_workspace(L_.mmu_selective_scan_bwd_det_workspace(batch, H, L, N), u.device)
    es = u.element_size()
    with torch.cuda.device(u.device):
        for g in range(G):
            p = _lib.ScanBwdParams()
            _fill_fwd(p.f, u, delta, A, B, C, D, z, delta_bias, delta_softplus, reverse, g, G)
            xg = x if G == 1 else x[:, g * H:(g + 1) * H].contiguous()
            p.f.x = xg.data_ptr()
            p.f.x_stride = _x_stride(x, L)
            _set_order(p.f, order)
            if y is not None and z is not None:
                p.f.y = y.data_ptr() + g * H * y.stride(1) * es
                p.f.y_bs, p.f.y_ds = y.stride(0), y.stride(1)
            p.f.workspace, p.f.workspace_bytes = _ptr(ws), ws_bytes
            p.dout = dout.data_ptr() + g * H * dout.stride(1) * es
            p.dout_bs, p.dout_ds = dout.stride(0), dout.stride(1)
            p.du = du.data_ptr() + g * H * du.stride(1) * es
            p.du_bs, p.du_ds = du.stride(0), du.stride(1)
            p.ddelta = ddelta.data_ptr() + g * H * ddelta.stride(1) * es
            p.ddelta_bs, p.ddelta_ds = ddelta.stride(0), ddelta.stride(1)
            if dz is not None:
                p.dz = dz.data_ptr() + g * H * dz.stride(1) * es
                p.dz_bs, p.dz_ds = dz.stride(0), dz.stride(1)
            p.dA = dA.data_ptr() + g * H * N * 4
            if G == 1:
                p.dB, p.dC = dB.data_ptr(), dC.data_ptr()
                p.dB_bs, p.dC_bs, p.dB_ns, p.dC_ns = dB.stride(0), dC.stride(0), dB.stride(2), dC.stride(2)
            else:
                dBg = torch.zeros((batch, 1, N, L), device=u.device, dtype=torch.float32)
                dCg = torch.zeros_like(dBg)
                p.dB, p.dC = dBg.data_ptr(), dCg.data_ptr()
            p.dD = None if dD is None else dD.data_ptr() + g * H * 4
            p.ddelta_bias = None if dbias is None else dbias.data_ptr() + g * H * 4
            if det:
                _lib.check(L_.mmu_selective_scan_bwd_det(ct.byref(p), dws_ptr, dws_bytes, _stream()), "selective_scan_bwd_det")
            else:
                _lib.check(L_.mmu_selective_scan_bwd(ct.byref(p), _stream()), "selective_scan_bwd")
            if G > 1:
                dB[:, g:g + 1] = dBg
                dC[:, g:g + 1] = dCg


def _conv_params(x, weight, bias, silu, reverse=False, order=None):
    _require_cuda(x, weight, bias)
    if x.dtype not in _DT:
        raise RuntimeError("causal_conv1d: input type must be float32, float16 or bfloat16")
    if x.dim() != 3 or weight.dim() != 2 or weight.shape[0] != x.shape[1]:
        raise RuntimeError("causal_conv1d: x must be (batch, dim, seqlen) and weight (dim, width)")
    if not 2 <= weight.shape[1] <= 4:
        raise RuntimeError("causal_conv1d only supports width between 2 and 4")
    if bias is not None and bias.shape != (x.shape[1],):
        raise RuntimeError("causal_conv1d: bias must be (dim,)")
    p = _lib.ConvParams()
    p.batch, p.dim, p.seqlen = x.shape
    p.width, p.dtype, p.silu, p.reverse = weight.shape[1], _DT[x.dtype], int(bool(silu)), int(bool(reverse))
    p.x, p.weight, p.bias = x.data_ptr(), weight.data_ptr(), _ptr(bias)
    p.x_bs, p.x_ds, p.w_ds, p.w_ws = x.stride(0), x.stride(1), weight.stride(0), weight.stride(1)
    _set_order(p, order)
    return p


def causal_conv1d_fwd(x, weight, bias=None, silu=False, reverse=False, out=None, order=None):
    """x (B,D,L) with stride(-1)==1; weight (D,W) / bias (D) are used in fp32.  `out`: optional pre-allocated (B,D,L) result
    with unit sequence stride and free batch / channel strides.  order = (kind, H, W, nslices): x is read through the scan-order
    index map (it stays in natural token order), out is written in scan order."""
    if x.stride(-1) != 1 and x.shape[-1] > 1:
        x = x.contiguous()
    weight = weight.float()
    bias = None if bias is None else bias.float().contiguous()
    p = _conv_params(x, weight, bias, silu, reverse, order)
    if out is None:
        out = torch.empty_like(x, memory_format=torch.contiguous_format)
    elif out.shape != x.shape or out.dtype != x.dtype or (out.stride(-1) != 1 and out.shape[-1] > 1):
        raise RuntimeError("causal_conv1d_fwd: out must match x in shape / dtype with stride(-1) == 1")
    p.out, p.out_bs, p.out_ds = out.data_ptr(), out.stride(0), out.stride(1)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().mmu_causal_conv1d_fwd(ct.byref(p), _stream()), "causal_conv1d_fwd")
    return out


def causal_conv1d_bwd(x, weight, bias, dout, silu=False, dx=None, reverse=False, order=None):
    """-> (dx, dweight fp32 (D,W), dbias fp32 or None).  order: x / dx in natural token order, dout in scan order."""
    if x.stride(-1) != 1 and x.shape[-1] > 1:
        x = x.contiguous()
    if dout.stride(-1) != 1 and dout.shape[-1] > 1:
        dout = dout.contiguous()
    _require_cuda(dout)
    if dout.dtype != x.dtype or dout.shape != x.shape:
        raise RuntimeError("causal_conv1d_bwd: dout must match x in dtype and shape")
    weight = weight.float()
    bias = None if bias is None else bias.float().contiguous()
    p = _conv_params(x, weight, bias, silu, reverse, order)
    dx = torch.empty_like(x, memory_format=torch.contiguous_format) if dx is None else dx
    dw = torch.zeros(weight.shape, device=x.device, dtype=torch.float32)
    db = torch.zeros(x.shape[1], device=x.device, dtype=torch.float32) if bias is not None else None
    p.dout, p.dout_bs, p.dout_ds = dout.data_ptr(), dout.stride(0), dout.stride(1)
    p.dx, p.dx_bs, p.dx_ds = dx.data_ptr(), dx.stride(0), dx.stride(1)
    p.dweight, p.dbias = dw.data_ptr(), _ptr(db)
    L_ = _lib.lib()
    with torch.cuda.device(x.device):
        if _deterministic():
            ws, wp, wb = _det_workspace(L_.mmu_causal_conv1d_bwd_det_workspace(p.batch, p.dim, p.seqlen, p.dtype), x.device)
            _lib.check(L_.mmu_causal_conv1d_bwd_det(ct.byref(p), wp, wb, _stream()), "causal_conv1d_bwd_det")
        else:
            _lib.check(L_.mmu_causal_conv1d_bwd(ct.byref(p), _stream()), "causal_conv1d_bwd")
    return dx, dw, db


# ----------------------------------------------------------------------------------------------------------
# autograd functions with the reference's signatures
# ----------------------------------------------------------------------------------------------------------

def _save(ctx, saved):
    """ctx.save_for_backward for a tuple whose entries are None, tensors or lists of tensors (grouped saved states)."""
    flat, spec = [], []
    for t in saved:
        if t is None:
            spec.append(None)
        elif isinstance(t, (list, tuple)):
            spec.append(len(t))
            flat.extend(t)
        else:
            spec.append(-1)
            flat.append(t)
    ctx.save_for_backward(*flat)
    ctx.saved_spec = spec


def _load(ctx):
    it = iter(ctx.saved_tensors)
    return tuple(None if k is None else (next(it) if k == -1 else [next(it) for _ in range(k)]) for k in ctx.saved_spec)


class SelectiveScanFn(torch.autograd.Function):
    """selective_scan_interface.py:14-74."""

    @staticmethod
    def forward(ctx, u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                return_last_state=False):
        if u.stride(-1) != 1:
            u = u.contiguous()
        if delta.stride(-1) != 1:
            delta = delta.contiguous()
        if D is not None:
            D = D.contiguous()
        if B.stride(-1) != 1:
            B = B.contiguous()
        if C.stride(-1) != 1:
            C = C.contiguous()
        if z is not None and z.stride(-1) != 1:
            z = z.contiguous()
        ctx.squeeze_B = B.dim() == 3
        ctx.squeeze_C = C.dim() == 3
        if ctx.squeeze_B:
            B = B.unsqueeze(1)
        if ctx.squeeze_C:
            C = C.unsqueeze(1)
        out, x, last = selective_scan_fwd(u, delta, A, B, C, D, z, delta_bias, delta_softplus,
                                          save_states=True, return_last_state=return_last_state)
        ctx.delta_softplus = delta_softplus
        ctx.has_z = z is not None
        _save(ctx, (u, delta, A, B, C, D, z, delta_bias, x.x, x.y))
        return out if not return_last_state else (out, last)

    @staticmethod
    def backward(ctx, dout, *args):
        u, delta, A, B, C, D, z, delta_bias, x, y = _load(ctx)
        du, ddelta, dA, dB, dC, dD, dz, ddelta_bias = selective_scan_bwd(
            u, delta, A, B, C, D, z, delta_bias, dout, ScanStates(x, y), ctx.delta_softplus)
        dB = (dB.squeeze(1) if ctx.squeeze_B else dB).to(B.dtype)
        dC = (dC.squeeze(1) if ctx.squeeze_C else dC).to(C.dtype)
        return du, ddelta, dA, dB, dC, dD, dz, ddelta_bias, None, None


def selective_scan_fn(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                      return_last_state=False):
    """selective_scan_interface.py:77-83.  With return_last_state=True returns (out, last_state (B,D,N));
    the gradient of last_state is ignored, as in the reference."""
    return SelectiveScanFn.apply(u, delta, A, B, C, D, z, delta_bias, delta_softplus, return_last_state)


class CausalConv1dFn(torch.autograd.Function):
    """causal_conv1d_interface.py:10-34."""

    @staticmethod
    def forward(ctx, x, weight, bias=None, activation=None):
        if activation not in [None, "silu", "swish"]:
            raise NotImplementedError("activation must be None, silu, or swish")
        if x.stride(2) != 1:
            x = x.contiguous()
        bias = bias.contiguous() if bias is not None else None
        ctx.save_for_backward(x, weight, bias)
        ctx.activation = activation in ["silu", "swish"]
        return causal_conv1d_fwd(x, weight, bias, ctx.activation)

    @staticmethod
    def backward(ctx, dout):
        x, weight, bias = ctx.saved_tensors
        dx, dweight, dbias = causal_conv1d_bwd(x, weight, bias, dout, ctx.activation)
        return dx, dweight.to(weight.dtype), (dbias.to(bias.dtype) if bias is not None else None), None


def causal_conv1d_fn(x, weight, bias=None, activation=None):
    """x: (batch, dim, seqlen); weight: (dim, width); bias: (dim,); activation None | "silu" | "swish"."""
    return CausalConv1dFn.apply(x, weight, bias, activation)


def _autocast_dtype():
    return torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None


class _InnerCore:
    """Shared forward/backward of the fused inner functions (conv -> x_proj -> dt_proj -> scan).

    Layout: the tensors the skinny projections touch live channel-major ACROSS the batch, storage (channels, batch, L), so
    that every projection and every weight gradient is ONE 2-D GEMM on a (channels, batch*L) matrix (K = batch*L for the
    weight gradients: cuBLAS split-K instead of `batch` small K = L products), while the scan / conv kernels see the same
    storage as (batch, channels, L) views with strides (L, batch*L, 1).  x_dbl is (R + 2N, batch, L): B, C and the dt rows are
    row slices of it that the kernels read - and, in the backward, accumulate into - in place.  None of the reference's
    "(b l) d" flattening (selective_scan_interface.py:181-207), i.e. no transpose copies of conv_out, B, C or their gradients."""

    @staticmethod
    def _cbl(channels, batch, L, like, dtype=None, zero=False):
        """(channels, batch, L) storage and its (batch, channels, L) view."""
        mk = torch.zeros if zero else torch.empty
        st = mk((channels, batch, L), device=like.device, dtype=like.dtype if dtype is None else dtype)
        return st, st.permute(1, 0, 2)

    @staticmethod
    def forward(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B, C, D, delta_bias,
                B_proj_bias, C_proj_bias, delta_softplus, reverse=False, order=None):
        """order = (kind, H, W, nslices): the scan runs over xz in that token order WITHOUT permuted copies - the conv reads x
        through the index map and writes conv_out in scan order, the projections work on scan-order tensors (they are per-token),
        the scan reads the gate z and writes its output through the map: out_z comes back in natural token order
        (== scatter(inner(gather(xz))), requirements/mamba_simple.py:245-263, src/UM_Net/MMUNet.py:178-183)."""
        if B is not None or C is not None or B_proj_bias is not None or C_proj_bias is not None:
            raise NotImplementedError("mmunet_b200: only input-dependent B/C without projection bias are supported "
                                      "(the only form MM-UNet's Mamba uses)")
        if A.is_complex():
            raise NotImplementedError("mmunet_b200: complex A is not supported")
        R = delta_proj_weight.shape[1]
        N = A.shape[-1]
        if xz.stride(-1) != 1:
            xz = xz.contiguous()
        batch, L = xz.shape[0], xz.shape[-1]
        conv_w = conv1d_weight.reshape(conv1d_weight.shape[0], -1)
        d = conv_w.shape[0]
        x, z = xz.chunk(2, dim=1)
        conv_b = conv1d_bias.contiguous() if conv1d_bias is not None else None
        conv_st, conv_out = _InnerCore._cbl(d, batch, L, xz)
        causal_conv1d_fwd(x, conv_w, conv_b, True, reverse=reverse, out=conv_out, order=order)
        x_dbl = torch.mm(x_proj_weight, conv_st.view(d, batch * L))                 # (R+2N, b*l)     (:181)
        delta = torch.mm(delta_proj_weight, x_dbl[:R]).view(d, batch, L).permute(1, 0, 2)      # (b, d, l) view    (:182)
        x3 = x_dbl.view(-1, batch, L)
        Bm = x3[R:R + N].permute(1, 0, 2).unsqueeze(1)                              # (b, 1, n, l) views of x_dbl
        Cm = x3[R + N:].permute(1, 0, 2).unsqueeze(1)
        D = D.contiguous() if D is not None else None
        out_z, xs, _ = selective_scan_fwd(conv_out, delta, A, Bm, Cm, D, z, delta_bias, delta_softplus, reverse=reverse, order=order)
        saved = (xz, conv_w, conv_b, x_dbl, x_proj_weight, delta_proj_weight, conv_st, delta, A, None, None, D, delta_bias,
                 xs.x, xs.y)
        return out_z, saved

    @staticmethod
    def project_grads(x_dbl, x_proj_weight, delta_proj_weight, conv_st, ddelta_st, dBC_st, dconv_st):
        """Backward of the two skinny projections (selective_scan_interface.py:256-277) on (channels, batch*L) matrices.
        ddelta_st (d,b,l), dBC_st fp32 (2N,b,l), dconv_st (d,b,l) = the scan's du.  -> (dconv_out (b,d,l) view, dx_proj_w, ddt_proj_w)."""
        R = delta_proj_weight.shape[1]
        d, batch, L = conv_st.shape
        ddelta2 = ddelta_st.view(d, batch * L)
        dx_dbl = torch.empty_like(x_dbl)
        dx_dbl[R:] = dBC_st.view(-1, batch * L)                                      # one cast copy for dB and dC
        torch.mm(delta_proj_weight.t(), ddelta2, out=dx_dbl[:R])                     # (R, b*l)
        ddt_proj_w = torch.mm(ddelta2, x_dbl[:R].t())                                # (d, R), K = b*l
        dx_proj_w = torch.mm(dx_dbl, conv_st.view(d, batch * L).t())                 # (R+2N, d), K = b*l
        dconv = torch.addmm(dconv_st.view(d, batch * L), x_proj_weight.t(), dx_dbl)  # (d, b*l)
        return dconv.view(d, batch, L).permute(1, 0, 2), dx_proj_w, ddt_proj_w

    @staticmethod
    def backward(saved, dout_y, delta_softplus, reverse=False, order=None):
        """dout_y: (b, d, l).  Returns (dxz, dconv_w (d,1,w), dconv_b, dx_proj_w, ddt_proj_w, dA, dD, ddelta_bias)."""
        (xz, conv_w, conv_b, x_dbl, x_proj_weight, delta_proj_weight, conv_st, delta, A, _, _, D, delta_bias, xs_x, xs_y) = saved
        xs = ScanStates(xs_x, xs_y)
        R = delta_proj_weight.shape[1]
        N = A.shape[-1]
        d, batch, L = conv_st.shape
        x, z = xz.chunk(2, dim=1)
        conv_out = conv_st.permute(1, 0, 2)
        x3 = x_dbl.view(-1, batch, L)
        Bm, Cm = x3[R:R + N].permute(1, 0, 2).unsqueeze(1), x3[R + N:].permute(1, 0, 2).unsqueeze(1)
        dxz = torch.empty_like(xz)
        dx, dz = dxz.chunk(2, dim=1)
        du_st, du = _InnerCore._cbl(d, batch, L, xz)
        ddl_st, ddl = _InnerCore._cbl(d, batch, L, xz)
        dBC_st, _ = _InnerCore._cbl(2 * N, batch, L, xz, dtype=torch.float32, zero=True)
        dBC = (dBC_st[:N].permute(1, 0, 2), dBC_st[N:].permute(1, 0, 2))
        _, _, dA, _, _, dD, dz, ddelta_bias = selective_scan_bwd(
            conv_out, delta, A, Bm, Cm, D, z, delta_bias, dout_y, xs, delta_softplus, reverse=reverse, dz=dz, dBC=dBC,
            du=du, ddelta=ddl, order=order)
        dconv_out, dx_proj_w, ddt_proj_w = _InnerCore.project_grads(x_dbl, x_proj_weight, delta_proj_weight, conv_st, ddl_st,
                                                                    dBC_st, du_st)
        _, dconv_w, dconv_b = causal_conv1d_bwd(x, conv_w, conv_b, dconv_out, True, dx=dx, reverse=reverse, order=order)
        return dxz, dconv_w.unsqueeze(1), dconv_b, dx_proj_w, ddt_proj_w, dA, dD, ddelta_bias


def _out_proj(out_z, weight, bias):
    """(b, d, l) -> (b, l, e) = F.linear(out_z^T, W, bias) (selective_scan_interface.py:365) computed channel-major:
    the result is a transposed VIEW of a contiguous (b, e, l) tensor, which is what MM-UNet's callers transpose back to."""
    out = torch.matmul(weight, out_z)
    if bias is not None:
        out = out + bias.to(out.dtype)[:, None]
    return out.transpose(1, 2)


class _OutProjTokenMajorFn(torch.autograd.Function):
    """out_proj of the v2/v3 branch (requirements/mamba_simple.py:270): (b, d, l) -> (b, l, e) token-major.  Plain autograd would hand
    `total` a gradient that is a transposed VIEW of (b, l, d); each of the three directions' backward then makes it contiguous
    (three transpose copies of (b, d, l), 1.45 ms each at L = 65 536).  Here the gradient comes out of the GEMM as (b, d, l)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, total, weight, bias):
        weight, bias = _cast_proj(weight, bias)
        if weight.dtype != total.dtype:
            weight = weight.to(total.dtype)
        ctx.save_for_backward(total, weight)
        ctx.has_bias = bias is not None
        out = torch.matmul(total.transpose(1, 2), weight.t())
        if bias is not None:
            out = out + bias.to(out.dtype)
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        total, weight = ctx.saved_tensors
        dout_t = dout.to(weight.dtype).transpose(1, 2)                               # (b, e, l) view of the token-major gradient
        dtotal = torch.matmul(weight.t(), dout_t)                                    # (b, d, l) contiguous
        dweight = torch.bmm(dout_t, total.transpose(1, 2)).sum(0)                    # (e, d)
        return dtotal, dweight, (dout_t.sum((0, 2)) if ctx.has_bias else None)


def _out_proj_autograd(total, weight, bias):
    """(b, d, l) -> (b, l, e), token-major contiguous (the transposed operand goes into the GEMM as it is): reshaped to
    (b, e, H, W) by the caller it is a channels-last map."""
    return _OutProjTokenMajorFn.apply(total, weight, bias)


def _out_proj_bwd(dout, out_z, weight, has_bias):
    """dout (b, l, e) -> (dout_y (b, d, l) contiguous, dweight (e, d), dbias)."""
    dout_t = dout.transpose(1, 2)                                                    # (b, e, l)
    if dout_t.stride(-1) != 1:
        dout_t = dout_t.contiguous()
    dout_t = dout_t.to(weight.dtype)
    dout_y = torch.matmul(weight.t(), dout_t)                                        # (b, d, l)
    dweight = torch.bmm(dout_t, out_z.transpose(1, 2)).sum(0)                        # (e, d)
    return dout_y, dweight, (dout_t.sum((0, 2)) if has_bias else None)


def _cast_proj(*ws):
    dt = _autocast_dtype()
    return tuple(w.to(dt) if (dt is not None and w is not None) else w for w in ws)


class MambaInnerFnNoOutProj(torch.autograd.Function):
    """selective_scan_interface.py:155-289 (returns out_z (b, d, l))."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B=None, C=None, D=None,
                delta_bias=None, B_proj_bias=None, C_proj_bias=None, delta_softplus=True, checkpoint_lvl=1,
                reverse=False, order=None):
        x_proj_weight, delta_proj_weight = _cast_proj(x_proj_weight, delta_proj_weight)
        out_z, saved = _InnerCore.forward(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B, C, D,
                                          delta_bias, B_proj_bias, C_proj_bias, delta_softplus, reverse=reverse, order=order)
        ctx.delta_softplus = delta_softplus
        ctx.reverse = reverse
        ctx.order = order
        _save(ctx, saved)
        return out_z

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        saved = _load(ctx)
        dxz, dcw, dcb, dxw, ddw, dA, dD, ddb = _InnerCore.backward(saved, dout, ctx.delta_softplus, reverse=ctx.reverse, order=ctx.order)
        return (dxz, dcw, dcb, dxw, ddw, dA, None, None, dD, ddb, None, None, None, None, None, None)


class MambaInnerFn(torch.autograd.Function):
    """selective_scan_interface.py:292-434 (fused out_proj; returns (b, l, d_model))."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias,
                A, B=None, C=None, D=None, delta_bias=None, B_proj_bias=None, C_proj_bias=None, delta_softplus=True,
                checkpoint_lvl=1, order=None):
        x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias = _cast_proj(
            x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias)
        out_z, saved = _InnerCore.forward(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B, C, D,
                                          delta_bias, B_proj_bias, C_proj_bias, delta_softplus, order=order)
        ctx.delta_softplus = delta_softplus
        ctx.order = order
        ctx.out_proj_bias_is_None = out_proj_bias is None
        saved = saved + (out_proj_weight, out_z)
        _save(ctx, saved)
        return _out_proj(out_z, out_proj_weight, out_proj_bias)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        saved = _load(ctx)
        out_proj_weight, out_z = saved[-2], saved[-1]
        dout_y, dout_proj_w, dout_proj_b = _out_proj_bwd(dout, out_z, out_proj_weight, not ctx.out_proj_bias_is_None)
        dxz, dcw, dcb, dxw, ddw, dA, dD, ddb = _InnerCore.backward(saved[:-2], dout_y, ctx.delta_softplus, order=ctx.order)
        return (dxz, dcw, dcb, dxw, ddw, dout_proj_w, dout_proj_b, dA, None, None, dD, ddb, None, None, None, None, None)


class BiMambaInnerFn(torch.autograd.Function):
    """selective_scan_interface.py:437-603: one conv/projection feeding a forward scan (A) and a scan over the
    flipped sequence (A_b); the flip is fused into the kernels (`reverse`) instead of materialised."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias,
                A, A_b, B=None, C=None, D=None, delta_bias=None, B_proj_bias=None, C_proj_bias=None,
                delta_softplus=True, checkpoint_lvl=1):
        x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias = _cast_proj(
            x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias)
        out_f, saved = _InnerCore.forward(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B, C, D,
                                          delta_bias, B_proj_bias, C_proj_bias, delta_softplus)
        (xz_, conv_w, conv_b, x_dbl, xw, dw, conv_st, delta, A_, _, _, D_, db_, _xs_fx, _xs_fy) = saved
        R, N = dw.shape[1], A.shape[-1]
        d, batch, L = conv_st.shape
        x3 = x_dbl.view(-1, batch, L)
        Bm, Cm = x3[R:R + N].permute(1, 0, 2).unsqueeze(1), x3[R + N:].permute(1, 0, 2).unsqueeze(1)
        z = xz_.chunk(2, dim=1)[1]
        out_b, xs_b, _ = selective_scan_fwd(conv_st.permute(1, 0, 2), delta, A_b, Bm, Cm, D_, z, db_, delta_softplus, reverse=True)
        out_z = out_f + out_b            # out_b is already stored in un-flipped positions
        ctx.delta_softplus = delta_softplus
        ctx.out_proj_bias_is_None = out_proj_bias is None
        saved = saved + (out_proj_weight, out_z, A_b, xs_b.x, xs_b.y)
        _save(ctx, saved)
        return _out_proj(out_z, out_proj_weight, out_proj_bias)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        saved = _load(ctx)
        out_proj_weight, out_z, A_b, xs_bx, xs_by = saved[-5:]
        core = saved[:-5]
        (xz, conv_w, conv_b, x_dbl, xw, dw, conv_st, delta, A, _, _, D, dbias, xs_fx, xs_fy) = core
        xs_b, xs_f = ScanStates(xs_bx, xs_by), ScanStates(xs_fx, xs_fy)
        R, N = dw.shape[1], A.shape[-1]
        d, batch, L = conv_st.shape
        conv_out = conv_st.permute(1, 0, 2)
        x3 = x_dbl.view(-1, batch, L)
        Bm, Cm = x3[R:R + N].permute(1, 0, 2).unsqueeze(1), x3[R + N:].permute(1, 0, 2).unsqueeze(1)
        dout_y, dout_proj_w, dout_proj_b = _out_proj_bwd(dout, out_z, out_proj_weight, not ctx.out_proj_bias_is_None)
        x, z = xz.chunk(2, dim=1)
        # both directions accumulate dB / dC into the same buffer; the other gradients are summed afterwards
        dBC_st, _ = _InnerCore._cbl(2 * N, batch, L, xz, dtype=torch.float32, zero=True)
        dBC = (dBC_st[:N].permute(1, 0, 2), dBC_st[N:].permute(1, 0, 2))
        dub_st, dub = _InnerCore._cbl(d, batch, L, xz)
        ddb_st, ddb_ = _InnerCore._cbl(d, batch, L, xz)
        _, _, dA_b, _, _, dD_b, dz_b, ddb_b = selective_scan_bwd(
            conv_out, delta, A_b, Bm, Cm, D, z, dbias, dout_y, xs_b, ctx.delta_softplus, reverse=True, dBC=dBC, du=dub, ddelta=ddb_)
        dxz = torch.empty_like(xz)
        dx, dz = dxz.chunk(2, dim=1)
        duf_st, duf = _InnerCore._cbl(d, batch, L, xz)
        ddf_st, ddf = _InnerCore._cbl(d, batch, L, xz)
        _, _, dA, _, _, dD_f, dz, ddb_f = selective_scan_bwd(
            conv_out, delta, A, Bm, Cm, D, z, dbias, dout_y, xs_f, ctx.delta_softplus, dz=dz, dBC=dBC, du=duf, ddelta=ddf)
        dz += dz_b
        dD = None if D is None else dD_f + dD_b
        ddb = None if dbias is None else ddb_f + ddb_b
        dconv_out, dxw, ddw = _InnerCore.project_grads(x_dbl, xw, dw, conv_st, ddf_st + ddb_st, dBC_st, duf_st + dub_st)
        _, dcw, dcb = causal_conv1d_bwd(x, conv_w, conv_b, dconv_out, True, dx=dx)
        return (dxz, dcw.unsqueeze(1), dcb, dxw, ddw, dout_proj_w, dout_proj_b, dA, dA_b, None, None, dD, ddb,
                None, None, None, None)


def mamba_inner_fn(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias,
                   A, B=None, C=None, D=None, delta_bias=None, B_proj_bias=None, C_proj_bias=None,
                   delta_softplus=True):
    return MambaInnerFn.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight,
                              out_proj_bias, A, B, C, D, delta_bias, B_proj_bias, C_proj_bias, delta_softplus)


def bimamba_inner_fn(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias,
                     A, A_b, B=None, C=None, D=None, delta_bias=None, B_proj_bias=None, C_proj_bias=None,
                     delta_softplus=True):
    return BiMambaInnerFn.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight,
                                out_proj_bias, A, A_b, B, C, D, delta_bias, B_proj_bias, C_proj_bias, delta_softplus)


def mamba_inner_fn_no_out_proj(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B=None, C=None,
                               D=None, delta_bias=None, B_proj_bias=None, C_proj_bias=None, delta_softplus=True):
    return MambaInnerFnNoOutProj.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, B, C, D,
                                       delta_bias, B_proj_bias, C_proj_bias, delta_softplus)


def mamba_inner_fn_ordered(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias, A, D=None,
                           delta_bias=None, delta_softplus=True, order=None):
    """mamba_inner_fn over the tokens of xz taken in `order` = (kind, H, W, nslices), result in natural token order:
    == scatter(mamba_inner_fn(gather(xz), ...)) of MMConv (src/UM_Net/MMUNet.py:178-183) without the two permuted copies.
    Falls back to explicit gather / scatter kernels where the order cannot be fused."""
    N = A.shape[-1]
    if order is None or order_fusable(order, N, xz.dtype):
        return MambaInnerFn.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, out_proj_bias, A,
                                  None, None, D, delta_bias, None, None, delta_softplus, 1, order)
    kind, H, W, ns = order
    out = MambaInnerFn.apply(scan_order_gather(xz, kind, H, W, ns), conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight,
                             out_proj_weight, out_proj_bias, A, None, None, D, delta_bias, None, None, delta_softplus)
    return scan_order_scatter(out.transpose(1, 2), kind, H, W, ns).transpose(1, 2)


def mamba_inner_fn_no_out_proj_ordered(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, D=None, delta_bias=None,
                                       delta_softplus=True, order=None):
    """== scatter(mamba_inner_fn_no_out_proj(gather(xz), ...)) (requirements/mamba_simple.py:245-263) with the scan order fused into
    the conv / scan kernels' addressing; explicit gather / scatter where it cannot be fused."""
    N = A.shape[-1]
    if order is None or order_fusable(order, N, xz.dtype):
        return MambaInnerFnNoOutProj.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, None, None, D, delta_bias,
                                           None, None, delta_softplus, 1, False, order)
    kind, H, W, ns = order
    out = MambaInnerFnNoOutProj.apply(scan_order_gather(xz, kind, H, W, ns), conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight,
                                      A, None, None, D, delta_bias, None, None, delta_softplus)
    return scan_order_scatter(out, kind, H, W, ns)


def mamba_inner_fn_no_out_proj_reversed(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, D=None,
                                        delta_bias=None, delta_softplus=True):
    """== mamba_inner_fn_no_out_proj(xz.flip(-1), ...).flip(-1) (requirements/mamba_simple.py:229-241,270) without
    materialising either flip: the conv runs anti-causally and the scan walks l = L-1..0."""
    return MambaInnerFnNoOutProj.apply(xz, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, A, None, None,
                                       D, delta_bias, None, None, delta_softplus, 1, True)


# ----------------------------------------------------------------------------------------------------------
# scan-order permutations (bit-exact index maps)
# ----------------------------------------------------------------------------------------------------------

# ---- narrow Mamba block: fused prologue / epilogue around the scan (SURVEY.md section 8 row f3) ----------------------------------
def mamba_narrow_supported(d_model, d_inner, d_state, dt_rank, d_conv, dtype) -> bool:
    """True for the block shape the fused narrow kernels are built for (MMConv's Mamba: d_model 3, expand 2, d_state 16, dt_rank 1,
    d_conv 4; fp32 / bf16).  MMU_NARROW=0 in the environment disables them (the generic inner functions run instead)."""
    import os
    if os.environ.get("MMU_NARROW", "1") == "0" or dtype not in (torch.float32, torch.bfloat16):
        return False
    return bool(_lib.lib().mmu_mamba_narrow_supported(d_model, d_inner, d_state, dt_rank, d_conv, _DT[dtype]))


def _narrow_params(io, hid_dtype, batch, L, dims, order, weights, coord):
    p = _lib.NarrowParams()
    p.dtype, p.hidden_dtype, p.batch, p.seqlen = _DT[io], _DT[hid_dtype], batch, L
    p.d_model, p.d_inner, p.d_state, p.dt_rank, p.d_conv = dims
    _set_order(p, order)
    p.in_proj_w, p.conv_w, p.conv_b, p.x_proj_w, p.dt_proj_w, p.out_proj_w = [_ptr(w) for w in weights]
    if coord is not None:
        altho, scope, H, W = coord
        p.coord_mode, p.map_h, p.map_w, p.extend_scope, p.altho = 1, H, W, float(scope), altho.data_ptr()
    return p


class MambaNarrowFn(torch.autograd.Function):
    """The whole narrow Mamba block, requirements/mamba_simple.py:201-270 with bimamba_type "v1" (in_proj -> mamba_inner_fn ->
    out_proj, selective_scan_interface.py:292-434), on channel-major tokens: hidden (b, d_model, l) in NATURAL token order ->
    (b, d_model, l) in natural order, scanned in `order` = (kind, H, W, nslices) or None.  Three launches forward (prologue, scan,
    epilogue) and four backward instead of the separate projection / conv / cast ops; no in_proj / out_proj bias.
    coord = (altho, extend_scope, H, W): MMConv's coordinate epilogue (src/UM_Net/MMUNet.py:156-188) - the result is the fp32 map
    gain * block(hidden) + row index + snake_offsets(hidden) * extend_scope with gain = clamp(softplus(altho), 0.01)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, hidden, in_w, conv_w, conv_b, x_w, dt_w, out_w, A, D, dt_bias, order, altho, coord):
        io = _autocast_dtype() or hidden.dtype
        _require_cuda(hidden, in_w, conv_w, conv_b, x_w, dt_w, out_w, A, D, dt_bias, altho)
        batch, dm, L = hidden.shape
        di, N, R, kw = conv_w.shape[0], A.shape[1], dt_w.shape[1], conv_w.shape[-1]
        dims = (dm, di, N, R, kw)
        if not mamba_narrow_supported(*dims, io):
            raise RuntimeError(f"mamba_narrow_fn: unsupported block shape {dims} / dtype {io}")
        if order is not None and order[0] == _lib.ORDER_ROWMAJOR:
            order = None
        if not (hidden.dtype == io or (hidden.dtype == torch.float32 and io == torch.bfloat16)):
            hidden = hidden.to(io)
        if hidden.stride(-1) != 1:
            hidden = hidden.contiguous()
        weights = [w if w is None else w.detach().float().contiguous() for w in (in_w, conv_w.reshape(di, kw), conv_b, x_w, dt_w, out_w)]
        A, D, dt_bias = A.float().contiguous(), D.float().contiguous(), dt_bias.float().contiguous()
        if coord is not None:
            coord = (altho.detach().float().contiguous(),) + tuple(coord)
            if coord[2] * coord[3] != L:
                raise RuntimeError("mamba_narrow_fn: coord = (extend_scope, H, W) needs H * W == seqlen")
        L_ = _lib.lib()
        rows = L_.mmu_mamba_narrow_rows(di, N)
        pre = torch.empty((batch, rows, L), device=hidden.device, dtype=io)
        out = torch.empty((batch, dm, L), device=hidden.device, dtype=torch.float32 if coord is not None else io)
        with torch.cuda.device(hidden.device):
            p = _narrow_params(io, hidden.dtype, batch, L, dims, order, weights, coord)
            p.hidden, p.hidden_bs, p.hidden_cs, p.pre = hidden.data_ptr(), hidden.stride(0), hidden.stride(1), pre.data_ptr()
            _lib.check(L_.mmu_mamba_narrow_pre_fwd(ct.byref(p), _stream()), "mamba_narrow_pre_fwd")
            u, delta, z = pre[:, :di], pre[:, di:2 * di], pre[:, 2 * di:3 * di]
            Bm, Cm = pre[:, 3 * di:3 * di + N].unsqueeze(1), pre[:, 3 * di + N:].unsqueeze(1)
            out_z, xs, _ = selective_scan_fwd(u, delta, A, Bm, Cm, D, z, dt_bias, True)
            p.out_z = out_z.data_ptr()
            if coord is not None:
                p.coords = out.data_ptr()
            else:
                p.out, p.out_bs, p.out_cs = out.data_ptr(), out.stride(0), out.stride(1)
            _lib.check(L_.mmu_mamba_narrow_post_fwd(ct.byref(p), _stream()), "mamba_narrow_post_fwd")
        ctx.dims, ctx.order, ctx.io, ctx.has_conv_b = dims, order, io, conv_b is not None
        ctx.wdtypes = [None if w is None else w.dtype for w in (in_w, conv_w, conv_b, x_w, dt_w, out_w)]
        ctx.conv_w_shape = conv_w.shape
        ctx.coord = None if coord is None else coord[1:]
        ctx.altho_dtype = None if altho is None else altho.dtype
        ctx.save_for_backward(hidden, pre, out_z, xs.x, xs.y, A, D, dt_bias, coord[0] if coord is not None else None,
                              *[w for w in weights if w is not None])
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        hidden, pre, out_z, xs_x, xs_y, A, D, dt_bias, altho, *ws = ctx.saved_tensors
        if not ctx.has_conv_b:
            ws.insert(2, None)
        dm, di, N, R, kw = ctx.dims
        io = ctx.io
        coord = None if ctx.coord is None else (altho,) + tuple(ctx.coord)
        batch, _, L = hidden.shape
        dout = dout.to(torch.float32 if coord is not None else io)
        if coord is not None:
            dout = dout.contiguous()
        elif dout.stride(-1) != 1:
            dout = dout.contiguous()
        L_ = _lib.lib()
        nW = L_.mmu_mamba_narrow_weight_floats(dm, di, N, R, kw)
        nBC = batch * 2 * N * L
        acc = torch.zeros(nBC + nW, device=hidden.device, dtype=torch.float32)      # one fill: dB | dC (16-byte aligned rows) | weight grads
        dBC, dW = acc[:nBC].view(batch, 2 * N, L), acc[nBC:]
        dout_y = torch.empty((batch, di, L), device=hidden.device, dtype=io)
        gpre = torch.empty((batch, 3 * di, L), device=hidden.device, dtype=io)
        dhidden = torch.empty_like(hidden)
        det = _deterministic()
        if det:
            dws, dws_ptr, dws_bytes = _det_workspace(max(L_.mmu_mamba_narrow_post_bwd_det_workspace(batch, L),
                                                             L_.mmu_mamba_narrow_pre_bwd_det_workspace(batch, L)), hidden.device)
        with torch.cuda.device(hidden.device):
            p = _narrow_params(io, hidden.dtype, batch, L, ctx.dims, ctx.order, ws, coord)
            p.out_z, p.dout_y, p.dweights = out_z.data_ptr(), dout_y.data_ptr(), dW.data_ptr()
            if coord is not None:
                p.dcoords = dout.data_ptr()
            else:
                p.dout, p.dout_bs, p.dout_cs = dout.data_ptr(), dout.stride(0), dout.stride(1)
            if det:
                _lib.check(L_.mmu_mamba_narrow_post_bwd_det(ct.byref(p), dws_ptr, dws_bytes, _stream()), "mamba_narrow_post_bwd_det")
            else:
                _lib.check(L_.mmu_mamba_narrow_post_bwd(ct.byref(p), _stream()), "mamba_narrow_post_bwd")
            u, delta, z = pre[:, :di], pre[:, di:2 * di], pre[:, 2 * di:3 * di]
            Bm, Cm = pre[:, 3 * di:3 * di + N].unsqueeze(1), pre[:, 3 * di + N:].unsqueeze(1)
            _, _, dA, _, _, dD, _, ddt_bias = selective_scan_bwd(
                u, delta, A, Bm, Cm, D, z, dt_bias, dout_y, ScanStates(xs_x, xs_y), True, du=gpre[:, :di], ddelta=gpre[:, di:2 * di],
                dz=gpre[:, 2 * di:], dBC=(dBC[:, :N], dBC[:, N:]))
            p.hidden, p.hidden_bs, p.hidden_cs, p.pre = hidden.data_ptr(), hidden.stride(0), hidden.stride(1), pre.data_ptr()
            p.gpre, p.dBC = gpre.data_ptr(), dBC.data_ptr()
            p.dhidden, p.dhidden_bs, p.dhidden_cs = dhidden.data_ptr(), dhidden.stride(0), dhidden.stride(1)
            if det:
                _lib.check(L_.mmu_mamba_narrow_pre_bwd_det(ct.byref(p), dws_ptr, dws_bytes, _stream()), "mamba_narrow_pre_bwd_det")
            else:
                _lib.check(L_.mmu_mamba_narrow_pre_bwd(ct.byref(p), _stream()), "mamba_narrow_pre_bwd")
        sizes = (2 * di * dm, di * kw, di, (R + 2 * N) * di, di * R, dm * di, 1)
        g_in, g_cw, g_cb, g_x, g_dt, g_out, g_al = torch.split(dW, sizes)
        wd = ctx.wdtypes
        d_altho = g_al.reshape(()).to(ctx.altho_dtype) if coord is not None else None
        return (dhidden, g_in.view(2 * di, dm).to(wd[0]), g_cw.view(ctx.conv_w_shape).to(wd[1]), g_cb.to(wd[2]) if ctx.has_conv_b else None,
                g_x.view(R + 2 * N, di).to(wd[3]), g_dt.view(di, R).to(wd[4]), g_out.view(dm, di).to(wd[5]), dA, dD, ddt_bias, None,
                d_altho, None)


def mamba_narrow_fn(hidden, in_proj_weight, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight, A, D,
                    delta_bias, order=None, altho=None, coord=None):
    """hidden (b, d_model, l), natural token order -> (b, d_model, l); see MambaNarrowFn.  coord = (extend_scope, H, W) with the
    parameter altho selects MMConv's coordinate epilogue (fp32 result)."""
    return MambaNarrowFn.apply(hidden, in_proj_weight, conv1d_weight, conv1d_bias, x_proj_weight, delta_proj_weight, out_proj_weight,
                               A, D, delta_bias, order, altho, coord)


def _order_call(fn_name, src, order, H, W, nslices):
    _require_cuda(src)
    if src.dtype not in _DT:
        raise RuntimeError("scan_order: dtype must be float32, float16 or bfloat16")
    L = H * W
    if src.shape[-1] != L:
        raise RuntimeError(f"scan_order: last dim {src.shape[-1]} != H*W = {L}")
    if order == _lib.ORDER_NSLICES and (nslices <= 0 or L % nslices):
        raise RuntimeError(f"scan_order: sequence length {L} is not divisible by nslices {nslices}")
    # the (b, 2d, l) view produced by in_proj is (2d, b, l)-contiguous: permute instead of copying
    swap = src.dim() == 3 and not src.is_contiguous() and src.transpose(0, 1).is_contiguous()
    base = src.transpose(0, 1) if swap else src
    src2 = base.reshape(-1, L)
    if src2.stride(-1) != 1:
        src2 = src2.contiguous()
    dst = torch.empty((src2.shape[0], L), device=src.device, dtype=src.dtype)
    with torch.cuda.device(src.device):
        rc = getattr(_lib.lib(), fn_name)(src2.data_ptr(), dst.data_ptr(), _DT[src.dtype], src2.shape[0],
                                          src2.stride(0), dst.stride(0), order, H, W, max(1, nslices), _stream())
    _lib.check(rc, fn_name)
    dst = dst.view(*base.shape[:-1], L)
    return dst.transpose(0, 1) if swap else dst


class _ScanOrderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, order, H, W, nslices, scatter):
        ctx.args = (order, H, W, nslices, scatter)
        return _order_call("mmu_scan_order_scatter" if scatter else "mmu_scan_order_gather", x, order, H, W, nslices)

    @staticmethod
    def backward(ctx, g):
        order, H, W, nslices, scatter = ctx.args
        # the adjoint of a permutation gather is the scatter with the same index map, and vice versa
        return (_order_call("mmu_scan_order_gather" if scatter else "mmu_scan_order_scatter", g, order, H, W, nslices),
                None, None, None, None, None)


def scan_order_gather(x, order, H, W, nslices=1):
    """y[..., l] = x[..., idx(l)]  (x: (..., H*W))."""
    return _ScanOrderFn.apply(x, order, H, W, nslices, False)


def scan_order_scatter(y, order, H, W, nslices=1):
    """x[..., idx(l)] = y[..., l]."""
    return _ScanOrderFn.apply(y, order, H, W, nslices, True)


def scan_order_index(order, H, W, nslices=1, device="cuda"):
    idx = torch.empty(H * W, device=device, dtype=torch.int64)
    with torch.cuda.device(idx.device):
        _lib.check(_lib.lib().mmu_scan_order_index(idx.data_ptr(), order, H, W, max(1, nslices), _stream()),
                   "mmu_scan_order_index")
    return idx


def two_row_flatten(x):
    """(B,C,H,W) -> (B,C,H*W) in MMConv's morph order (MMUNet.py:68-93)."""
    B, C_, H, W = x.shape
    return scan_order_gather(x.reshape(B, C_, H * W), _lib.ORDER_TWOROW, H, W)


def two_row_unflatten(x_flat, H, W):
    """inverse (MMUNet.py:95-121): (B,C,L) -> (B,C,H,W)."""
    B, C_, L = x_flat.shape
    return scan_order_scatter(x_flat, _lib.ORDER_TWOROW, H, W).view(B, C_, H, W)


# ----------------------------------------------------------------------------------------------------------
# MMConv's snake row sampler (the caller of the Mamba block; replaces coordinate rescale + F.grid_sample, MMUNet.py:190-224)
# ----------------------------------------------------------------------------------------------------------

def _nhwc_ok(t):
    C_ = t.shape[1]
    return (t.dim() == 4 and C_ % 4 == 0 and ((C_ // 4) & (C_ // 4 - 1)) == 0 and not t.is_contiguous()
            and t.is_contiguous(memory_format=torch.channels_last))


class _SnakeSampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, y, out_dtype):
        _require_cuda(feat, y)
        if feat.dtype not in (torch.float32, torch.bfloat16) or out_dtype not in (torch.float32, torch.bfloat16):
            raise RuntimeError("snake_sample: feature / output dtype must be float32 or bfloat16")
        if feat.dim() != 4 or y.dim() != 4 or y.shape[0] != feat.shape[0] or y.shape[2:] != feat.shape[2:]:
            raise RuntimeError(f"snake_sample: feat (B,C,H,W) / y (B,K,H,W) mismatch: {tuple(feat.shape)} vs {tuple(y.shape)}")
        cl = _nhwc_ok(feat)                       # channels-last feature maps are consumed and produced in place (NHWC kernels)
        fmt = torch.channels_last if cl else torch.contiguous_format
        feat = feat.contiguous(memory_format=fmt)
        y = y.float().contiguous()
        B, C_, H, W = feat.shape
        K = y.shape[1]
        out = torch.empty((B, C_, H * K, W), device=feat.device, dtype=out_dtype, memory_format=fmt)
        with torch.cuda.device(feat.device):
            _lib.check(_lib.lib().mmu_snake_sample_fwd(feat.data_ptr(), y.data_ptr(), out.data_ptr(), _DT[feat.dtype], _DT[out_dtype],
                                                       B, C_, H, W, K, int(cl), _stream()), "snake_sample_fwd")
        ctx.save_for_backward(feat, y)
        ctx.out_dtype, ctx.cl = out_dtype, cl
        return out

    @staticmethod
    def backward(ctx, dout):
        feat, y = ctx.saved_tensors
        B, C_, H, W = feat.shape
        K = y.shape[1]
        fmt = torch.channels_last if ctx.cl else torch.contiguous_format
        dout = dout.to(ctx.out_dtype).contiguous(memory_format=fmt)
        nf = feat.numel()
        acc = torch.zeros(nf + y.numel(), device=feat.device, dtype=torch.float32)     # one zero fill for both accumulators
        dfeat = acc[:nf].view(B, H, W, C_).permute(0, 3, 1, 2) if ctx.cl else acc[:nf].view(B, C_, H, W)
        dy = acc[nf:].view_as(y)
        L_ = _lib.lib()
        args = (feat.data_ptr(), y.data_ptr(), dout.data_ptr(), dfeat.data_ptr(), dy.data_ptr(), _DT[feat.dtype], _DT[ctx.out_dtype],
                B, C_, H, W, K, int(ctx.cl))
        with torch.cuda.device(feat.device):
            if _deterministic():
                ws, wp, wb = _det_workspace(L_.mmu_snake_sample_bwd_det_workspace(B, C_, H, W, K, int(ctx.cl)), feat.device)
                _lib.check(L_.mmu_snake_sample_bwd_det(*args, wp, wb, _stream()), "snake_sample_bwd_det")
            else:
                _lib.check(L_.mmu_snake_sample_bwd(*args, _stream()), "snake_sample_bwd")
        return dfeat.to(feat.dtype), dy, None


def snake_sample(feat, y, out_dtype=None):
    """feat (B,C,H,W), y (B,K,H,W) fp32 row coordinates in pixels -> (B,C,H*K,W): row-interpolated samples at
    (clamp(y,0,H-1), clamp(w+k-K//2,0,W-1)) - MMConv's deformed feature map (MMUNet.py:190-224)."""
    return _SnakeSampleFn.apply(feat, y, feat.dtype if out_dtype is None else out_dtype)


# ----------------------------------------------------------------------------------------------------------
# channels-last GroupNorm with 4 channels per group (MMConv's closing norm, MMUNet.py:46, 271)
# ----------------------------------------------------------------------------------------------------------

def group_norm_nhwc_supported(x, num_groups):
    C_ = x.shape[1] if x.dim() == 4 else 0
    G = num_groups
    return (x.is_cuda and x.dim() == 4 and C_ == 4 * G and (G >= 256 or 256 % G == 0) and x.dtype in (torch.float32, torch.bfloat16)
            and x.is_contiguous(memory_format=torch.channels_last) and not (x.is_contiguous() and C_ > 1 and x.shape[2] * x.shape[3] > 1))


class _GroupNormNhwcFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, num_groups, eps, out_dtype):
        B, C_, H, W = x.shape
        G = num_groups
        w32, b32 = weight.float().contiguous(), bias.float().contiguous()
        y = torch.empty((B, C_, H, W), device=x.device, dtype=out_dtype, memory_format=torch.channels_last)
        stats = torch.zeros(4 * B * G, device=x.device, dtype=torch.float32)          # sums (2BG) | mean (BG) | rstd (BG)
        sums, mean, rstd = stats[:2 * B * G], stats[2 * B * G:3 * B * G], stats[3 * B * G:]
        L_ = _lib.lib()
        args = (x.data_ptr(), w32.data_ptr(), b32.data_ptr(), y.data_ptr(), sums.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _DT[x.dtype],
                _DT[out_dtype], B, C_, H * W, G, float(eps))
        with torch.cuda.device(x.device):
            if _deterministic():
                ws, wp, wb = _det_workspace(L_.mmu_group_norm_nhwc_fwd_det_workspace(B, C_, H * W, G), x.device)
                _lib.check(L_.mmu_group_norm_nhwc_fwd_det(*args, wp, wb, _stream()), "group_norm_nhwc_fwd_det")
            else:
                _lib.check(L_.mmu_group_norm_nhwc_fwd(*args, _stream()), "group_norm_nhwc_fwd")
        ctx.save_for_backward(x, w32, mean, rstd)
        ctx.G, ctx.out_dtype, ctx.wdtype = G, out_dtype, weight.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w32, mean, rstd = ctx.saved_tensors
        B, C_, H, W = x.shape
        G = ctx.G
        dy = dy.to(ctx.out_dtype).contiguous(memory_format=torch.channels_last)
        dx = torch.empty_like(x, memory_format=torch.channels_last)
        acc = torch.zeros(2 * B * G + 2 * C_, device=x.device, dtype=torch.float32)    # S1,S2 per (b, group) | dgamma | dbeta
        L_ = _lib.lib()
        args = (x.data_ptr(), w32.data_ptr(), dy.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(), acc.data_ptr(),
                acc[2 * B * G:].data_ptr(), _DT[x.dtype], _DT[ctx.out_dtype], B, C_, H * W, G)
        with torch.cuda.device(x.device):
            if _deterministic():
                ws, wp, wb = _det_workspace(L_.mmu_group_norm_nhwc_bwd_det_workspace(B, C_, H * W, G), x.device)
                _lib.check(L_.mmu_group_norm_nhwc_bwd_det(*args, wp, wb, _stream()), "group_norm_nhwc_bwd_det")
            else:
                _lib.check(L_.mmu_group_norm_nhwc_bwd(*args, _stream()), "group_norm_nhwc_bwd")
        dgamma, dbeta = acc[2 * B * G:2 * B * G + C_], acc[2 * B * G + C_:]
        return dx, dgamma.to(ctx.wdtype), dbeta.to(ctx.wdtype), None, None, None


def group_norm_nhwc(x, num_groups, weight, bias, eps=1e-5, out_dtype=None):
    """F.group_norm for a channels-last (B, C, H, W) tensor with C == 4 * num_groups; statistics in fp32, output channels-last in
    `out_dtype` (default: x.dtype).  Raises if the layout / shape is not supported - check group_norm_nhwc_supported first."""
    if not group_norm_nhwc_supported(x, num_groups):
        raise RuntimeError("group_norm_nhwc: needs a CUDA channels-last (B, 4*G, H, W) fp32/bf16 tensor with G | 256 or G >= 256")
    return _GroupNormNhwcFn.apply(x, weight, bias, num_groups, eps, x.dtype if out_dtype is None else out_dtype)
