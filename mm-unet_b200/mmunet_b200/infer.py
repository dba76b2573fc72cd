"""Sliding-window MM_Net prediction: what the reference's validation (train.py:180, monai SlidingWindowInferer(roi_size=image_size,
overlap=0.5), constant blending) does with a trained model, on images of any size.

  window_starts / pad_for_roi   the window placement rule (monai's _get_scan_interval / dense_patch_slices and its padding)
  sw_stitch                     one mmu_sw_stitch launch: the windows' five head maps -> full-size fp32 logits (+ confusion counts)
  SlidingWindowPredictor        pad, cut windows, run MM_Net.forward_heads in batches (optionally a captured CUDA graph), stitch
  segmentation_metrics          Dice, IoU, accuracy, sensitivity, specificity from the counts

The model's own final resize-and-sum (MMUNet.py:577) is fused into the stitch: each window's logit map is never formed at full size.
There is no CPU path: the predictor needs a CUDA model and the stitch is a CUDA kernel.
"""
from __future__ import annotations

import contextlib
import ctypes as ct

import torch
import torch.nn.functional as F

from . import _lib

_HEAD_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}
_AUTOCAST = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": None, "f32": None}


def scan_interval(n: int, roi: int, overlap: float) -> int:
    """Window stride along a padded axis of size n: roi when n == roi, else max(int(roi * (1 - overlap)), 1)."""
    return roi if n == roi else max(int(roi * (1 - overlap)), 1)


def window_starts(n: int, roi: int, overlap: float) -> list:
    """Starts of the windows along a padded axis of size n >= roi: window d starts at min(d * interval, n - roi), for d up to the first
    with d * interval + roi >= n (monai's dense_patch_slices)."""
    if n < roi:
        raise ValueError(f"window_starts: axis {n} is shorter than the roi {roi} (pad it first, see pad_for_roi)")
    iv = scan_interval(n, roi, overlap)
    d = 0
    while d * iv + roi < n:
        d += 1
    return [min(k * iv, n - roi) for k in range(d + 1)]


def pad_for_roi(h: int, roi: int) -> tuple:
    """(before, after) zero padding of an image side h < roi up to roi: (roi - h) // 2 before, the rest after; (0, 0) when h >= roi."""
    diff = max(roi - h, 0)
    return diff // 2, diff - diff // 2


def _check_head(t, k):
    if not t.is_cuda or t.dtype not in _HEAD_DT or t.dim() != 4 or (t.stride(-1) != 1 and t.shape[-1] > 1):
        raise RuntimeError(f"sw_stitch: head {k} must be a CUDA fp32 / bf16 (images, windows, h, w) tensor with column stride 1")


def _mask(m, B, H, W, device):
    """uint8 (B, H, W) view (batch stride 0 for one shared map) of a target / FOV map given as (B, 1, H, W), (B, H, W) or (H, W)."""
    m = torch.as_tensor(m, device=device)
    if m.dim() == 4:
        m = m[:, 0]
    if m.dim() == 2:
        m = m.unsqueeze(0).expand(B, H, W)
    if m.shape != (B, H, W):
        raise RuntimeError(f"sw_stitch: mask of shape {tuple(m.shape)} does not match the images ({B}, {H}, {W})")
    if m.dtype != torch.uint8:
        m = (m != 0).to(torch.uint8)
    return m if (m.stride(-1) == 1 or W == 1) else m.contiguous()


def sw_stitch(heads, image_size, roi: int, overlap: float, target=None, fov=None, counts=None, out=None):
    """heads: the five head maps (out2, out3, out4, out5, p_c) of every window of B images of size image_size = (H, W), each a
    (B, windows, h_k, w_k) tensor (fp32 or bf16, one dtype, column stride 1), windows in row-major order of the padded image.
    -> (logits (B, 1, H, W) fp32, counts (B, 4) int64 or None): the window-blended sum of the heads' bilinear upsamplings to roi x roi
    (include/mmunet_b200.h, mmu_sw_stitch).  With a target, counts gets TP, FP, FN, TN of logit > 0 inside the FOV added to it (a
    zero-filled tensor is made when counts is None).  out: optional fp32 (B, 1, H, W) result with column stride 1."""
    heads = list(heads)
    if len(heads) != _lib.SW_HEADS:
        raise RuntimeError(f"sw_stitch: expected {_lib.SW_HEADS} head maps, got {len(heads)}")
    for k, t in enumerate(heads):
        _check_head(t, k)
    dt = heads[0].dtype
    if any(t.dtype != dt for t in heads):
        raise RuntimeError("sw_stitch: the head maps must share one dtype")
    H, W = (int(v) for v in image_size)
    (pt, pb), (pl, pr) = pad_for_roi(H, roi), pad_for_roi(W, roi)
    n_h, n_w = H + pt + pb, W + pl + pr
    nwin = len(window_starts(n_h, roi, overlap)) * len(window_starts(n_w, roi, overlap))
    B, dev = heads[0].shape[0], heads[0].device
    if any(t.shape[0] != B or t.shape[1] != nwin for t in heads):
        raise RuntimeError(f"sw_stitch: every head map must be ({B}, {nwin}, h, w) for a {H}x{W} image at roi {roi}, overlap {overlap}")
    logits = torch.empty((B, 1, H, W), device=dev, dtype=torch.float32) if out is None else out
    if logits.shape != (B, 1, H, W) or logits.dtype != torch.float32 or logits.device != dev or (logits.stride(-1) != 1 and W > 1):
        raise RuntimeError(f"sw_stitch: out must be an fp32 ({B}, 1, {H}, {W}) tensor on the heads' device with column stride 1")
    p = _lib.SwStitchParams()
    p.dtype, p.batch, p.H, p.W, p.roi = _HEAD_DT[dt], B, H, W, roi
    p.n_h, p.n_w, p.pad_top, p.pad_left = n_h, n_w, pt, pl
    p.interval_h, p.interval_w = scan_interval(n_h, roi, overlap), scan_interval(n_w, roi, overlap)
    for k, t in enumerate(heads):
        p.head_h[k], p.head_w[k] = t.shape[2], t.shape[3]
        p.heads[k] = t.data_ptr()
        p.head_bs[k], p.head_ws[k], p.head_rs[k] = t.stride(0), t.stride(1), t.stride(2)
    p.logits, p.logits_bs, p.logits_rs = logits.data_ptr(), logits.stride(0), logits.stride(2)
    if target is not None:
        tg = _mask(target, B, H, W, dev)
        p.target, p.target_bs, p.target_rs = tg.data_ptr(), tg.stride(0), tg.stride(1)
        if fov is not None:
            fv = _mask(fov, B, H, W, dev)
            p.fov, p.fov_bs, p.fov_rs = fv.data_ptr(), fv.stride(0), fv.stride(1)
        if counts is None:
            counts = torch.zeros((B, 4), device=dev, dtype=torch.int64)
        elif counts.shape != (B, 4) or counts.dtype != torch.int64 or not counts.is_contiguous() or counts.device != dev:
            raise RuntimeError("sw_stitch: counts must be a contiguous int64 (B, 4) tensor on the heads' device")
        p.counts = counts.data_ptr()
    elif counts is not None or fov is not None:
        raise RuntimeError("sw_stitch: counts and fov need a target")
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().mmu_sw_stitch(ct.byref(p), torch.cuda.current_stream().cuda_stream), "sw_stitch")
    return logits, counts


def segmentation_metrics(counts) -> dict:
    """counts (..., 4) = TP, FP, FN, TN -> float64 tensors (...): dice (= F1), iou, accuracy, sensitivity, specificity.  A zero
    denominator gives NaN."""
    c = torch.as_tensor(counts).to(torch.float64)
    tp, fp, fn, tn = c.unbind(-1)
    return {"dice": 2 * tp / (2 * tp + fp + fn), "iou": tp / (tp + fp + fn), "accuracy": (tp + tn) / (tp + fp + fn + tn),
            "sensitivity": tp / (tp + fn), "specificity": tn / (tn + fp)}


class SlidingWindowPredictor:
    """Segment images of any size with a (trained) MM_Net, as monai's SlidingWindowInferer(roi_size, overlap, mode="constant") around
    the model does in the reference's validation.

    Every image is zero-padded up to roi where it is smaller, cut into roi x roi windows (window_starts), and the windows of all
    images are run through model.forward_heads in batches of sw_batch_size (the last batch filled with zero windows whose outputs are
    ignored), under autocast(dtype) as in Trainer.  The heads are copied into per-image slabs and one mmu_sw_stitch launch per group
    of same-size images blends them.  Runs under torch.no_grad() (not inference_mode: MMConv caches coordinate grids that a later
    training step reuses), with the model in eval() for the call and every module's previous mode restored afterwards.  The work runs
    on a side stream ordered with the caller's stream like Trainer.step.

    predict returns fp32 logits also under bf16 autocast, where eager model(x) returns bf16: the heads are upsampled and summed in
    fp32 by the stitch.  The stitch itself gives the same bits on every run; the model's forward does too only in deterministic
    mode (torch.use_deterministic_algorithms(True) or MMU_DETERMINISTIC=1), since by default the channels-last GroupNorm sums its
    statistics with float atomics.

    graph=True: the first call for a (roi, sw_batch_size, dtype, layout) captures forward_heads on one static (sw_batch_size, 3, roi,
    roi) input into a CUDA graph (after an eager warm-up); later batches replay it.  The graph reads the parameters and BatchNorm
    buffers in place, so it sees the weights a trainer has just updated; after model.to(...), load_state_dict(assign=True) or anything
    else that reallocates them, call reset()."""

    def __init__(self, model, roi_size=512, overlap=0.5, sw_batch_size=4, dtype="bf16", channels_last=None, graph=True):
        if isinstance(roi_size, bool) or not isinstance(roi_size, int) or roi_size <= 0 or roi_size % 32:
            raise ValueError(f"SlidingWindowPredictor: roi_size must be a positive multiple of 32 (MM_Net's stride), got {roi_size!r}")
        if not 0 <= overlap < 1:
            raise ValueError(f"SlidingWindowPredictor: overlap must be in [0, 1), got {overlap!r}")
        if isinstance(sw_batch_size, bool) or not isinstance(sw_batch_size, int) or sw_batch_size < 1:
            raise ValueError(f"SlidingWindowPredictor: sw_batch_size must be an integer >= 1, got {sw_batch_size!r}")
        if dtype not in _AUTOCAST:
            raise ValueError(f"SlidingWindowPredictor: dtype must be one of {sorted(_AUTOCAST)}, got {dtype!r}")
        if not hasattr(model, "forward_heads"):
            raise TypeError("SlidingWindowPredictor: the model must provide forward_heads (MM_Net)")
        param = next(model.parameters(), None)
        if param is None or not param.is_cuda:
            raise RuntimeError("SlidingWindowPredictor: the model must be on a CUDA device (there is no CPU path)")
        if channels_last is None:          # follow the model's layout
            channels_last = any(p.dim() == 4 and not p.is_contiguous() and p.is_contiguous(memory_format=torch.channels_last)
                                for p in model.parameters())
        self.model, self.roi, self.overlap, self.sw_batch = model, roi_size, float(overlap), sw_batch_size
        self.dtype, self.autocast_dtype, self.channels_last, self.use_graph = dtype, _AUTOCAST[dtype], bool(channels_last), bool(graph)
        self.device = param.device
        self.stream = None
        self._graphs = {}

    def reset(self):
        """Drop the captured CUDA graphs (needed after the model's parameters or buffers were reallocated)."""
        self._graphs.clear()

    def predict(self, images):
        """images: (B, 3, H, W) with any H, W >= 1, or a list of such tensors (one per image size) -> fp32 logits (B, 1, H, W) (a list
        for a list)."""
        logits, _ = self._run(images, None, None)
        return logits

    def evaluate(self, images, targets, fov=None):
        """-> int64 (B, 4) counts TP, FP, FN, TN of logit > 0 against targets != 0 over the pixels with fov != 0 (all without a fov),
        computed in the stitch kernel (a list for a list of image tensors).  targets / fov: (B, 1, H, W), (B, H, W) or (H, W)."""
        _, counts = self._run(images, targets, fov)
        return counts

    # ---- internals -----------------------------------------------------------------------------------------------------------
    def _heads(self, x):
        ctx = torch.autocast("cuda", dtype=self.autocast_dtype) if self.autocast_dtype is not None else contextlib.nullcontext()
        with ctx:
            return tuple(self.model.forward_heads(x))

    def _new_input(self):
        x = torch.zeros((self.sw_batch, 3, self.roi, self.roi), device=self.device)
        return x.contiguous(memory_format=torch.channels_last) if self.channels_last else x

    def _graph(self):
        key = (self.roi, self.sw_batch, self.dtype, self.channels_last)
        ent = self._graphs.get(key)
        if ent is None:
            static_in = self._new_input()
            for _ in range(2):                                   # eager warm-up: cuDNN / cuBLAS choices, MMConv grid caches
                self._heads(static_in)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.stream):
                outs = self._heads(static_in)
            # the graph reads the grid tensors the MMConvs cached during the warm-up: keep them alive while the graph lives
            caches = [m._grid_cache for m in self.model.modules() if hasattr(m, "_grid_cache")]
            ent = self._graphs[key] = (g, static_in, outs, caches)
        return ent

    def _run(self, images, targets, fov):
        single = torch.is_tensor(images)
        groups = [images] if single else list(images)
        tgs = [targets] if single else (list(targets) if targets is not None else [None] * len(groups))
        fvs = [fov] if single else (list(fov) if fov is not None else [None] * len(groups))
        for x in groups:
            if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] < 1 or x.shape[3] < 1:
                raise RuntimeError(f"SlidingWindowPredictor: images must be (B, 3, H, W), got {tuple(x.shape)}")
        if len(tgs) != len(groups) or len(fvs) != len(groups):
            raise RuntimeError("SlidingWindowPredictor: one targets / fov entry per image group")
        dev, S, nb = self.device, self.roi, self.sw_batch
        cur = torch.cuda.current_stream(dev)
        if self.stream is None:
            self.stream = torch.cuda.Stream(dev)
        logits = [torch.empty((x.shape[0], 1, x.shape[2], x.shape[3]), device=dev, dtype=torch.float32) for x in groups]
        counts = [torch.zeros((x.shape[0], 4), device=dev, dtype=torch.int64) for x in groups] if targets is not None else None
        modes = [(m, m.training) for m in self.model.modules()]
        grid_caches = [(m, m._grid_cache) for m in self.model.modules() if hasattr(m, "_grid_cache")]
        self.stream.wait_stream(cur)
        try:
            with torch.cuda.device(dev), torch.cuda.stream(self.stream), torch.no_grad():
                self.model.eval()
                # pad every group, list its windows (image-major, then row-major) and their flat slab positions
                padded, geo, wins = [], [], []
                for g, x in enumerate(groups):
                    B, _, H, W = x.shape
                    (pt, pb), (pl, pr) = pad_for_roi(H, S), pad_for_roi(W, S)
                    xp = F.pad(x.to(device=dev, dtype=torch.float32), (pl, pr, pt, pb))
                    sh = window_starts(H + pt + pb, S, self.overlap)
                    sw = window_starts(W + pl + pr, S, self.overlap)
                    padded.append(xp)
                    geo.append(len(sh) * len(sw))
                    wins += [(g, i, a, b) for i in range(B) for a in sh for b in sw]
                if self.use_graph:
                    graph, buf, outs, _ = self._graph()
                else:
                    graph, buf = None, self._new_input()
                slabs = None
                pos = [0] * len(groups)                            # next flat slab position of each group
                for j0 in range(0, len(wins), nb):
                    chunk = wins[j0:j0 + nb]
                    for j, (g, i, a, b) in enumerate(chunk):
                        buf[j].copy_(padded[g][i, :, a:a + S, b:b + S])
                    if len(chunk) < nb:
                        buf[len(chunk):].zero_()
                    if graph is not None:
                        graph.replay()
                    else:
                        outs = self._heads(buf)
                    if slabs is None:
                        dt = outs[0].dtype if all(o.dtype == outs[0].dtype for o in outs) and outs[0].dtype in _HEAD_DT else torch.float32
                        slabs = [[torch.empty((x.shape[0] * geo[g], o.shape[2], o.shape[3]), device=dev, dtype=dt) for o in outs]
                                 for g, x in enumerate(groups)]
                    j = 0
                    while j < len(chunk):                          # one copy per head for each run of windows of one group
                        g = chunk[j][0]
                        m = 1
                        while j + m < len(chunk) and chunk[j + m][0] == g:
                            m += 1
                        for k, o in enumerate(outs):
                            slabs[g][k][pos[g]:pos[g] + m].copy_(o[j:j + m, 0])
                        pos[g] += m
                        j += m
                for g, x in enumerate(groups):
                    heads = [s.view(x.shape[0], geo[g], s.shape[1], s.shape[2]) for s in slabs[g]]
                    sw_stitch(heads, x.shape[2:], S, self.overlap, tgs[g] if targets is not None else None, fvs[g],
                              counts[g] if counts is not None else None, out=logits[g])
        finally:
            for m, t in modes:
                m.training = t
            for m, c in grid_caches:
                m._grid_cache = c
            cur.wait_stream(self.stream)
        if single:
            return logits[0], (counts[0] if counts is not None else None)
        return logits, counts
