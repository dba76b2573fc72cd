"""MM-UNet (`MM_Net`) on top of the B200 Mamba hot path - the caller of the path (SURVEY.md section 8 rows f1/f2).

Restates src/UM_Net/MMUNet.py so that the model can run where the reference tree is not mounted (the GPU box):
  MMConv          MMUNet.py:10-274    snake (dynamic) conv whose row offsets are refined by a v1 Mamba over the morph
                                      (two-row, column-interleaved) scan order
  CBAM            MMUNet.py:313-338
  SideoutBlock    MMUNet.py:341-352
  RCG             MMUNet.py:354-418   reverse-attention gate with a v3 Mamba over the 2x up-sampled map
  DecoderBlock    MMUNet.py:420-431
  ResidualBlock   MMUNet.py:433-467
  MM_Net          MMUNet.py:474-585
Module / parameter names, shapes, initialisers and creation ORDER are the reference's, so a reference
`state_dict()` loads as is and a given torch seed yields the same initial weights (tests/test_mm_net_cpu.py,
tests/golden/mm_net.npz).

What differs from the reference (performance only, same arithmetic):
  * the morph flatten / inverse (MMUNet.py:68-121) are the closed-form gather / scatter kernels (`ops.two_row_*`)
    instead of view/permute/reshape/cat chains;
  * the cumulative snake offsets (MMUNet.py:156-174: K//2 Python iterations of in-place row sums over a cloned
    buffer) are two cumsums away from the centre tap;
  * coordinate grids are built once per (H, W, K, device) and cached; no `device="cuda"` constructor default
    (SURVEY.md section 0.5) - tensors follow the input's device;
  * `Mamba` is `mmunet_b200.mamba.Mamba` (hosts bimamba_type="v1", which the reference constructor rejects,
    SURVEY.md section 0.4).
  * the bilinear resizes (F.interpolate, align_corners=True) go through `ops.resize_bilinear`: the same call, except that in
    deterministic mode their backward is the library's gather-side kernel instead of ATen's atomic scatter.
`MM_Net` is the only model of the reference's zoo built here: it is the one that calls the hot path.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .mamba import Mamba

# Tests swap these three for CPU oracle stand-ins (the product path has no CPU implementation).
_flatten_two_row = ops.two_row_flatten
_unflatten_two_row = ops.two_row_unflatten
_snake_sample = ops.snake_sample          # None -> the reference's torch formulation (grid rescale + F.grid_sample)
_group_norm_nhwc = ops.group_norm_nhwc    # None -> always nn.GroupNorm
_fuse_scan_order = True                   # False -> always materialise the two-row flatten / inverse around the Mamba block


class MMConv(nn.Module):
    """Snake convolution along rows with Mamba-refined offsets (morph 0) - MMUNet.py:10-274."""

    def __init__(self, in_channels=1, out_channels=1, kernel_size=9, extend_scope=1.0, morph=0, if_offset=True,
                 device=None, num_slices=4):
        super().__init__()
        if morph not in (0, 1):
            raise ValueError("morph should be 0 or 1.")
        if kernel_size % 2 == 0:
            raise ValueError("MMConv: kernel_size must be odd (the reference's offset recursion indexes past the "
                             "last tap otherwise, MMUNet.py:164-170)")
        K = kernel_size
        self.mamba = Mamba(d_model=K, d_state=16, d_conv=4, expand=2, bimamba_type="v1", nslices=num_slices)
        self.kernel_size, self.extend_scope, self.morph, self.if_offset = K, extend_scope, morph, if_offset
        self.gn_offset = nn.GroupNorm(K, 2 * K)
        self.gn = nn.GroupNorm(out_channels // 4, out_channels)
        self.gn_fp32_out = False     # channels-last path only: True = fp32 result under autocast, as torch's GroupNorm returns
        self.relu = nn.ReLU(inplace=False)
        self.tanh = nn.Tanh()
        self.offset_conv = nn.Conv2d(in_channels, 2 * K, 3, padding=1)
        self.dsc_conv_x = nn.Conv2d(in_channels, out_channels, kernel_size=(K, 1), stride=(K, 1), padding=0)
        self.dsc_conv_y = nn.Conv2d(in_channels, out_channels, kernel_size=(1, K), stride=(1, K), padding=0)
        self.altho = nn.Parameter(torch.log(torch.exp(torch.tensor(1.0)) - 1.0))
        self._grid_cache = {}

    # ---- static coordinate grids ---------------------------------------------------------------------------------
    def _base_grids(self, H, W, device):
        """rows (1,1,H,1) = h; cols (K*H... ) see below.  x map (MMUNet.py:141-151,191): x[(h k), w] = w + (k - K//2),
        already clamped to [0, W-1] and scaled to [-1, 1] (MMUNet.py:229-242) since it carries no learned offset."""
        key = (H, W, str(device))
        hit = self._grid_cache.get(key)
        if hit is None:
            K, c = self.kernel_size, self.kernel_size // 2
            rows = torch.arange(H, dtype=torch.float32, device=device).view(1, 1, H, 1)
            taps = torch.linspace(-c, c, K, device=device)                            # (K)
            cols = torch.arange(W, dtype=torch.float32, device=device)                # (W)
            xk = (cols.view(1, W) + taps.view(K, 1)).clamp(0, W - 1)                  # (K, W)
            xk = -1.0 + (2.0 / (W - 1)) * xk
            xmap = xk.view(1, 1, K, W).expand(1, H, K, W).reshape(1, H * K, W)
            hit = (rows, xmap)
            self._grid_cache = {key: hit}
        return hit

    def _snake_offsets(self, dy):
        """dy (B,K,H,W) -> cumulative offsets away from the centre tap (MMUNet.py:156-174): tap c stays 0,
        tap c+i = sum_{j<=i} dy[c+j], tap c-i = sum_{j<=i} dy[c-j]."""
        c = self.kernel_size // 2
        if c == 0:
            return torch.zeros_like(dy)
        right = torch.cumsum(dy[:, c + 1:], dim=1)
        left = torch.cumsum(dy[:, :c].flip(1), dim=1).flip(1)
        return torch.cat([left, torch.zeros_like(dy[:, :1]), right], dim=1)

    def row_coordinates(self, offset):
        """offset (B,2K,H,W) in [-1,1] -> y coordinates (B,K,H,W) of the K taps (MMUNet.py:122-188)."""
        B, _, H, W = offset.shape
        K = self.kernel_size
        dy = offset[:, :K]                                    # the second K channels (x offsets) are unused (:136)
        rows, _ = self._base_grids(H, W, offset.device)
        if (_fuse_scan_order and dy.is_cuda and isinstance(self.mamba, Mamba) and self.morph == 0 and dy.dtype in (torch.float32, torch.bfloat16)
                and self.mamba.narrow_block_available(dy)):
            # narrow fused block with the coordinate arithmetic below as its epilogue: offset map in, y coordinates out
            from . import _lib
            y = self.mamba(dy.reshape(B, K, H * W).transpose(-1, -2), scan_order=(_lib.ORDER_TWOROW, H, W, 1),
                           coord_epilogue=(self.altho, self.extend_scope, H, W))[0]
            return y.transpose(-1, -2).reshape(B, K, H, W)
        if _fuse_scan_order and dy.is_cuda and isinstance(self.mamba, Mamba) and self.mamba.bimamba_type not in ("v2", "v3"):
            # the morph (two-row) order is applied inside the conv / scan kernels' addressing: the tokens stay in natural order,
            # no flatten / inverse-flatten copies (:178-183); explicit gather / scatter kernels where the map cannot be fused
            from . import _lib
            refined = self.mamba(dy.reshape(B, K, H * W).transpose(-1, -2), scan_order=(_lib.ORDER_TWOROW, H, W, 1))[0]
            refined = refined.transpose(-1, -2).reshape(B, K, H, W)
        else:
            tokens = _flatten_two_row(dy.contiguous())            # (B, K, L) in morph scan order        (:178)
            refined = self.mamba(tokens.transpose(-1, -2))[0]     # (B, L, K)                             (:180-181)
            refined = _unflatten_two_row(refined.transpose(-1, -2), H, W)      # (B, K, H, W)         (:182-183)
        gain = torch.clamp(F.softplus(self.altho), min=0.01)                   #                      (:186-187)
        return gain * refined.float() + (rows + self._snake_offsets(dy).float() * self.extend_scope)

    def _grid_sample(self, input, y):
        """The reference formulation: rescale both coordinate maps to [-1, 1] and bilinear grid_sample."""
        B, K, H, W = y.shape
        _, xmap = self._base_grids(H, W, y.device)
        ymap = y.permute(0, 2, 1, 3).reshape(B, H * K, W)                      # "b k h w -> b (h k) w"   (:190)
        ymap = -1.0 + (2.0 / (H - 1)) * ymap.clamp(0, H - 1)                   # (:205-209, 229-242)
        grid = torch.stack([xmap.expand(B, -1, -1), ymap], dim=-1)             # (B, H*K, W, 2) = (x, y)  (:211-216)
        src = input if input.dtype == grid.dtype or torch.is_autocast_enabled(input.device.type) else input.to(grid.dtype)
        return F.grid_sample(src, grid, mode="bilinear", padding_mode="zeros", align_corners=True)

    def forward(self, input):
        offset = self.tanh(self.gn_offset(self.offset_conv(input)))            # (:247-250)
        B, _, H, W = offset.shape
        K = self.kernel_size
        y = self.row_coordinates(offset)                                       # (B, K, H, W)
        if _snake_sample is not None and self.morph == 0 and input.is_cuda and input.dtype in (torch.float32, torch.bfloat16):
            # fused clamp + row interpolation, written in the dtype the strided conv consumes (MMUNet.py:190-224)
            dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else input.dtype
            feat = _snake_sample(input, y, dt if dt in (torch.float32, torch.bfloat16) else torch.float32)
        else:
            feat = self._grid_sample(input, y)
        out = self.dsc_conv_x(feat) if self.morph == 0 else self.dsc_conv_y(feat)
        if _group_norm_nhwc is not None and out.is_cuda and ops.group_norm_nhwc_supported(out, self.gn.num_groups):
            # channels-last model: normalise in place of layout (ATen's GroupNorm would copy to NCHW, return NCHW and, under
            # autocast, fp32); the output keeps the conv's dtype, statistics are fp32
            # (MMConv.gn_fp32_out = True restores torch's autocast behaviour: an fp32 result)
            return _group_norm_nhwc(out, self.gn.num_groups, self.gn.weight, self.gn.bias, self.gn.eps,
                                    torch.float32 if self.gn_fp32_out else None)
        return self.gn(out)


class CBAM(nn.Module):
    """Channel then spatial attention - MMUNet.py:313-338."""

    def __init__(self, channel, reduction=16):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.max_pool = nn.AdaptiveMaxPool2d(1)
        self.mlp = nn.Sequential(nn.Conv2d(channel, channel // reduction, kernel_size=1, bias=False), nn.ReLU(inplace=True),
                                 nn.Conv2d(channel // reduction, channel, kernel_size=1, bias=False))
        self.conv = nn.Conv2d(2, 1, kernel_size=7, stride=1, padding=3, bias=False)
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        # amax == AdaptiveMaxPool2d(1) (one reduction kernel instead of the 3.4 ms adaptive-pool kernel at 256x256)
        y = self.sigmoid(self.mlp(self.avg_pool(x)) + self.mlp(x.amax(dim=(2, 3), keepdim=True))) * x
        s = torch.cat((y.amax(dim=1, keepdim=True), y.mean(dim=1, keepdim=True)), 1)
        return self.sigmoid(self.conv(s)) * y


def _mm_bn_relu(cin, cout, ns, k=3):
    return nn.Sequential(MMConv(cin, cout, num_slices=ns, kernel_size=k), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))


class SideoutBlock(nn.Module):
    """MMUNet.py:341-352."""

    def __init__(self, in_channels, out_channels, num_slices=4):
        super().__init__()
        self.conv1 = _mm_bn_relu(in_channels, in_channels // 4, num_slices)
        self.dropout = nn.Dropout2d(0.1)
        self.conv2 = nn.Conv2d(in_channels // 4, out_channels, kernel_size=1)

    def forward(self, x):
        return self.conv2(self.dropout(self.conv1(x)))


class RCG(nn.Module):
    """Reverse-attention gate; a v3 (forward + flipped + slice-interleaved) Mamba runs over the 2x up-sampled,
    row-major flattened map - MMUNet.py:354-418."""

    def __init__(self, d_state=16, d_conv=4, expand=2, head=4, num_slices=4, step=1):
        super().__init__()
        self.conv1 = _mm_bn_relu(128, 64, num_slices)
        self.upsample = nn.ConvTranspose2d(64, 64, kernel_size=4, stride=2, padding=1, output_padding=0)
        self.downsample = nn.Conv2d(64, 64, kernel_size=4, stride=2, padding=1)
        self.mamba = Mamba(d_model=64, d_state=d_state, d_conv=d_conv, expand=expand, bimamba_type="v3", nslices=num_slices)
        self.mamba.return_directional = False          # o_1..o_3 are discarded here (:407)
        self.mlp = nn.Sequential(nn.Conv2d(64, 1, kernel_size=1), nn.Sigmoid())

    def forward(self, pre, edge, f):
        r = (1.0 - torch.sigmoid(pre)) * f                                               # (:390-392)
        edge1 = ops.resize_bilinear(edge, size=f.shape[2:])
        x2 = self.conv1(torch.cat((edge1, r), 1))
        x0 = self.upsample(x2)
        B, C, H, W = x0.shape
        tokens = x0.reshape(B, C, H * W).transpose(-1, -2)                               # row-major scan order (:405)
        out = self.mamba(tokens)[0]
        x0 = self.downsample(out.transpose(-1, -2).reshape(B, C, H, W))
        return x0 * self.mlp(x2) * x2 + f                                                # (:414-416)


class DecoderBlock(nn.Module):
    """MMUNet.py:420-431."""

    def __init__(self, in_channels, out_channels, num_slices=4):
        super().__init__()
        self.conv1 = _mm_bn_relu(in_channels, in_channels // 4, num_slices)
        self.conv2 = _mm_bn_relu(in_channels // 4, out_channels, num_slices)

    def forward(self, x):
        return ops.resize_bilinear(self.conv2(self.conv1(x)), scale_factor=2)


class ResidualBlock(nn.Module):
    """ResNet-34-shaped block whose 3x3 convs are MMConvs - MMUNet.py:433-467."""

    def __init__(self, in_channels, out_channels, num_slices, downsample=False):
        super().__init__()
        self.downsample = downsample
        if downsample:
            self.block1 = nn.Sequential(
                nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=2, padding=1, bias=False),
                nn.BatchNorm2d(out_channels), nn.ReLU(inplace=True),
                MMConv(out_channels, out_channels, num_slices=num_slices, kernel_size=3), nn.BatchNorm2d(out_channels))
            self.block2 = nn.Sequential(nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=2, bias=False),
                                        nn.BatchNorm2d(out_channels))
        else:
            self.block1 = nn.Sequential(
                MMConv(in_channels, out_channels, num_slices=num_slices, kernel_size=3), nn.BatchNorm2d(out_channels),
                nn.ReLU(inplace=True),
                MMConv(out_channels, out_channels, num_slices=num_slices, kernel_size=3), nn.BatchNorm2d(out_channels))
        self.relu = nn.ReLU(inplace=True)

    def forward(self, x):
        y = self.block1(x)
        return self.relu((self.block2(x) if self.downsample else x) + y)


def _stage(cin, cout, n, ns, down):
    return nn.Sequential(*[ResidualBlock(cin if i == 0 else cout, cout, num_slices=ns, downsample=down and i == 0)
                           for i in range(n)])


class MM_Net(nn.Module):
    """MMUNet.py:474-585.  forward: (B,3,H,W) -> logits (B,1,H,W) = sum of 4 side outputs + the contour head."""

    def __init__(self, num_classes=1, num_slices_list=(64, 32, 16, 8), out_indices=(0, 1, 2, 3), heads=(1, 2, 4, 4)):
        super().__init__()
        ns = list(num_slices_list)
        self.encoder1 = nn.Sequential(nn.Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False), nn.BatchNorm2d(64),
                                      nn.ReLU(inplace=True))
        self.maxpool = nn.MaxPool2d(kernel_size=3, stride=2, padding=1, dilation=1, ceil_mode=False)
        self.encoder2 = _stage(64, 64, 3, ns[0], False)
        self.encoder3 = _stage(64, 128, 4, ns[1], True)
        self.encoder4 = _stage(128, 256, 6, ns[2], True)
        self.encoder5 = _stage(256, 512, 3, ns[3], True)
        self.down3 = _mm_bn_relu(128, 64, ns[-1], k=1)
        self.down4 = _mm_bn_relu(256, 64, ns[-1], k=1)
        self.down5 = _mm_bn_relu(512, 64, ns[-1], k=1)
        self.cbam = nn.Sequential(nn.Conv2d(64, 64, 3, 1, 1), nn.BatchNorm2d(64), nn.ReLU(inplace=True), CBAM(64),
                                  nn.Conv2d(64, 64, 3, 1, 1), nn.BatchNorm2d(64), nn.ReLU(inplace=True))
        self.line_predict = nn.Conv2d(64, 1, 3, 1, 1)
        self.side2 = SideoutBlock(64, 1, num_slices=ns[0])
        self.side3 = SideoutBlock(64, 1, num_slices=ns[1])
        self.side4 = SideoutBlock(64, 1, num_slices=ns[2])
        self.side5 = SideoutBlock(64, 1, num_slices=ns[3])
        self.rcg2 = RCG(num_slices=ns[0], head=heads[0])
        self.rcg3 = RCG(num_slices=ns[1], head=heads[1])
        self.rcg4 = RCG(num_slices=ns[2], head=heads[2])
        self.decoder5 = DecoderBlock(in_channels=64, out_channels=64, num_slices=ns[3])
        self.decoder4 = DecoderBlock(in_channels=128, out_channels=64, num_slices=ns[2])
        self.decoder3 = DecoderBlock(in_channels=128, out_channels=64, num_slices=ns[1])
        self.decoder2 = DecoderBlock(in_channels=128, out_channels=64, num_slices=ns[0])

    def forward(self, x):
        total = None
        for t in self.forward_heads(x):                      # (:577)
            up = ops.resize_bilinear(t, size=x.shape[2:])
            total = up if total is None else total + up
        return total

    def forward_heads(self, x):
        """The five (B, 1, h, w) logit maps (out2, out3, out4, out5, p_c) of a (B, 3, H, W) input, at 1/2, 1/4, 1/8, 1/16 and 1/2 of
        its size, before forward's bilinear resize to (H, W) and sum (what the sliding-window predictor stitches)."""
        e1 = self.encoder1(x)
        e2 = self.encoder2(self.maxpool(e1))
        e3 = self.encoder3(e2)
        e4 = self.encoder4(e3)
        e5 = self.down5(self.encoder5(e4))
        e3, e4 = self.down3(e3), self.down4(e4)

        d5 = self.decoder5(e5)
        out5 = self.side5(d5)
        c1 = self.cbam(e1)                                   # contour branch
        p_c = self.line_predict(c1)
        d4 = self.decoder4(torch.cat((d5, self.rcg4(out5, c1, e4)), dim=1))
        out4 = self.side4(d4)
        d3 = self.decoder3(torch.cat((d4, self.rcg3(out4, c1, e3)), dim=1))
        out3 = self.side3(d3)
        d2 = self.decoder2(torch.cat((d3, self.rcg2(out3, c1, e2)), dim=1))
        out2 = self.side2(d2)
        return out2, out3, out4, out5, p_c

    def unused_parameters(self):
        """Parameters that never receive a gradient in MM_Net: the `_b`/`_s` sets of the v1 Mambas and `dsc_conv_y`
        (morph is always 0) - what a data-parallel wrapper must not wait for (SURVEY.md section 8b 'v1 shim')."""
        names = []
        for mod_name, m in self.named_modules():
            if isinstance(m, MMConv):
                pre = mod_name + "." if mod_name else ""
                names += [pre + "dsc_conv_y.weight", pre + "dsc_conv_y.bias"]
                for pn, _ in m.mamba.named_parameters():
                    if "_b" in pn.split(".")[0] or "_s" in pn.split(".")[0]:
                        names.append(pre + "mamba." + pn)
        return names
