"""Torch-facing operators of the B200 hot path: thin wrappers that hand raw device pointers of torch
tensors (device memory + streams are the only thing torch provides here) to libsfod_b200.so.

Signatures follow the operators the reference reaches through detectron2/torchvision:
``nms`` / ``batched_nms`` / ``roi_align`` / ``roi_pool`` have torchvision's signatures
(torchvision/ops/boxes.py:20,51 and roi_align.py:204); the fused entry points (``rpn_select``,
``frcnn_postprocess``) replace whole per-image Python loops of detectron2 (SURVEY.md 8a).
Every function requires CUDA tensors and raises if the native library is unavailable.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor

from . import _lib
from ._lib import EmaTensor, EraseParams, FrcnnParams, JitterParams, ResizeImage, RpnParams, check

NCHW, NHWC = 0, 1
DT_F32, DT_I64, DT_U8 = 0, 1, 2   # enum sfod_dtype
SCALE_CLAMP = math.log(1000.0 / 16)
COORD_TRICK_MAX_N = 1000  # torchvision CPU switches batched_nms strategy at boxes.numel() > 4000
BN_FUSED_MAX_BYTES = 100 * 1024 * 1024   # activations up to this size take the single-launch L2-resident BatchNorm (0 disables it)

_ws_cache: Dict[Tuple[str, int, int], Tensor] = {}
_small_cache: Dict[Tuple, Tensor] = {}


# ---- optional per-call device timing (bench.py's roofline numbers): CUDA events recorded on the launching stream
# around the C-ABI call, so they measure exactly the kernels the call enqueues.  Off by default (zero overhead).
class KernelTimers:
    def __init__(self):
        self.enabled = False
        self.records: Dict[str, List[Tuple[torch.cuda.Event, torch.cuda.Event]]] = {}

    def start(self) -> None:
        self.records = {}
        self.enabled = True

    def stop(self) -> Dict[str, Tuple[int, float]]:
        """-> {tag: (number of calls, total milliseconds)}; synchronises."""
        self.enabled = False
        torch.cuda.synchronize()
        out = {t: (len(ev), sum(a.elapsed_time(b) for a, b in ev)) for t, ev in self.records.items()}
        self.records = {}
        return out


timers = KernelTimers()


class _timed:
    __slots__ = ("tag", "ev")

    def __init__(self, tag: str):
        self.tag = tag
        self.ev = None

    def __enter__(self):
        if timers.enabled:
            self.ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            self.ev[0].record()
        return self

    def __exit__(self, *exc):
        if self.ev is not None:
            self.ev[1].record()
            timers.records.setdefault(self.tag, []).append(self.ev)
        return False


def launch_count() -> int:
    """Kernel launches issued by libsfod_b200 in this process so far."""
    return int(_lib.lib().sfod_debug_launch_count())


def _stream(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _require_cuda(*ts: Tensor) -> torch.device:
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("sfod_b200 operators run on CUDA tensors only (no CPU fallback); got a "
                               f"{t.device} tensor")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must be on the same CUDA device")
    assert dev is not None
    return dev


def _workspace(dev: torch.device, tag: str, nbytes: int) -> Tensor:
    """Grow-only workspace per (tag, device, STREAM): reuse is stream-ordered, so a buffer is shared only by calls that are
    enqueued on the same stream (forward and backward of an op on one stream may share it; another stream -- or a CUDA-graph
    capture, which runs on its own stream and keeps replaying the addresses it recorded -- gets its own)."""
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    key = (tag, idx, torch.cuda.current_stream(dev).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
        _ws_cache[key] = buf
    return buf


def _small_i32(dev: torch.device, values: Sequence[int]) -> Tensor:
    key = (dev.index, tuple(int(v) for v in values))
    t = _small_cache.get(key)
    if t is None:
        if len(_small_cache) > 4096:
            _small_cache.clear()
        t = torch.tensor(list(key[1]), dtype=torch.int32, device=dev)
        _small_cache[key] = t
    return t


def _f32c(t: Tensor) -> Tensor:
    return t.detach().to(torch.float32).contiguous()


# ----------------------------------------------------------------------------------------------- NMS
def _nms_impl(boxes: Tensor, scores: Tensor, idxs: Optional[Tensor], iou_threshold: float) -> Tensor:
    dev = _require_cuda(boxes, scores, idxs)
    if boxes.dim() != 2 or boxes.shape[1] != 4:
        raise ValueError(f"boxes should be a 2d tensor of shape [N, 4], got {tuple(boxes.shape)}")
    if scores.dim() != 1 or scores.shape[0] != boxes.shape[0]:
        raise ValueError("boxes and scores should have same number of elements in dimension 0, got "
                         f"{boxes.shape[0]} and {scores.shape[0]}")
    n = boxes.shape[0]
    if n == 0:
        return torch.empty((0,), dtype=torch.int64, device=dev)
    b, s = _f32c(boxes), _f32c(scores)
    ix = None
    if idxs is not None:
        if idxs.shape[0] != n:
            raise ValueError("idxs must have one entry per box")
        ix = idxs.detach().to(torch.int64).contiguous()
    L = _lib.lib()
    with torch.cuda.device(dev):
        ws = _workspace(dev, "nms", L.sfod_nms_workspace_bytes(n))
        keep = torch.empty((n,), dtype=torch.int64, device=dev)
        cnt = torch.empty((1,), dtype=torch.int64, device=dev)
        check(L.sfod_nms(b.data_ptr(), s.data_ptr(), ix.data_ptr() if ix is not None else None, n, float(iou_threshold),
                         COORD_TRICK_MAX_N, keep.data_ptr(), cnt.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "sfod_nms")
        k = int(cnt.item())  # variable-length result: one D2H read, as in torchvision's own CUDA nms
    return keep[:k]


def nms(boxes: Tensor, scores: Tensor, iou_threshold: float) -> Tensor:
    """torchvision.ops.nms(boxes, scores, iou_threshold) -> int64 indices, score-descending."""
    return _nms_impl(boxes, scores, None, iou_threshold)


def batched_nms(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float) -> Tensor:
    """torchvision.ops.batched_nms / detectron2.layers.batched_nms (boxes are cast to fp32 as d2 does)."""
    return _nms_impl(boxes, scores, idxs, iou_threshold)


# ----------------------------------------------------------------------------------------------- ROI pooling
def _layout_of(x: Tensor) -> Tuple[Tensor, int]:
    """Returns (tensor whose storage is dense in the reported layout, layout)."""
    if x.dim() != 4:
        raise ValueError("input must be a 4-d (N, C, H, W) tensor")
    if x.is_contiguous():
        return x, NCHW
    if x.is_contiguous(memory_format=torch.channels_last):
        return x, NHWC
    return x.contiguous(), NCHW


def convert_boxes_to_roi_format(boxes: List[Tensor]) -> Tensor:
    """torchvision.ops._utils.convert_boxes_to_roi_format / d2 convert_boxes_to_pooler_format."""
    if len(boxes) == 0:
        raise ValueError("empty box list")
    parts = [torch.cat([torch.full((len(b), 1), i, dtype=b.dtype, device=b.device), b], dim=1) for i, b in enumerate(boxes)]
    return torch.cat(parts, dim=0)


def _check_rois(boxes: Union[Tensor, List[Tensor]]) -> Tensor:
    if isinstance(boxes, (list, tuple)):
        for b in boxes:
            if b.dim() != 2 or b.shape[1] != 4:
                raise ValueError("Expected Tensor[L, 4] in the box list")
        return convert_boxes_to_roi_format(list(boxes))
    if boxes.dim() != 2 or boxes.shape[1] != 5:
        raise ValueError("Expected Tensor[K, 5] rois: (batch_index, x1, y1, x2, y2)")
    return boxes


def _pair(v) -> Tuple[int, int]:
    return (int(v), int(v)) if isinstance(v, int) else (int(v[0]), int(v[1]))


class _RoIAlignFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, rois: Tensor, ph: int, pw: int, scale: float, sr: int, aligned: bool, exact: bool):
        dev = _require_cuda(x, rois)
        xin, layout = _layout_of(x.detach().to(torch.float32))
        r = _f32c(rois)
        N, Cc, H, W = xin.shape
        R = r.shape[0]
        out = torch.empty((R, Cc, ph, pw), dtype=torch.float32, device=dev)
        L = _lib.lib()
        if R > 0:
            with torch.cuda.device(dev):
                ws = _workspace(dev, "roi", L.sfod_roi_align_fwd_workspace_bytes(N, Cc, H, W, R, layout, int(exact)))
                with _timed("roi_align_fwd"):
                    check(L.sfod_roi_align_fwd(xin.data_ptr(), layout, r.data_ptr(), N, Cc, H, W, R, ph, pw, float(scale), int(sr),
                                               int(aligned), int(exact), out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)),
                          "sfod_roi_align_fwd")
        ctx.save_for_backward(r)
        ctx.meta = (N, Cc, H, W, ph, pw, float(scale), int(sr), int(aligned), layout, x.dtype)
        return out.to(x.dtype)

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        (r,) = ctx.saved_tensors
        N, Cc, H, W, ph, pw, scale, sr, aligned, layout, dtype = ctx.meta
        dev = grad_out.device
        g = _f32c(grad_out)
        fmt = torch.channels_last if layout == NHWC else torch.contiguous_format
        gin = torch.empty((N, Cc, H, W), dtype=torch.float32, device=dev, memory_format=fmt)
        L = _lib.lib()
        with torch.cuda.device(dev):
            ws = _workspace(dev, "roi", L.sfod_roi_align_bwd_workspace_bytes(N, Cc, H, W, layout))
            with _timed("roi_align_bwd"):
                check(L.sfod_roi_align_bwd(g.data_ptr(), r.data_ptr(), N, Cc, H, W, r.shape[0], ph, pw, scale, sr, aligned,
                                           gin.data_ptr(), layout, ws.data_ptr(), ws.numel(), _stream(dev)), "sfod_roi_align_bwd")
        return gin.to(dtype), None, None, None, None, None, None, None


def roi_align(input: Tensor, boxes: Union[Tensor, List[Tensor]], output_size, spatial_scale: float = 1.0,
              sampling_ratio: int = -1, aligned: bool = False, exact: bool = False) -> Tensor:
    """torchvision.ops.roi_align signature (roi_align.py:204-211).  ``exact=True`` reproduces torchvision's
    summation order bit for bit; the default separable kernel agrees to <= 1e-5 relative."""
    rois = _check_rois(boxes)
    ph, pw = _pair(output_size)
    return _RoIAlignFn.apply(input, rois, ph, pw, spatial_scale, sampling_ratio, aligned, exact)


class _RoIPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, rois: Tensor, ph: int, pw: int, scale: float):
        dev = _require_cuda(x, rois)
        xin = _f32c(x)
        r = _f32c(rois)
        N, Cc, H, W = xin.shape
        R = r.shape[0]
        out = torch.empty((R, Cc, ph, pw), dtype=torch.float32, device=dev)
        argmax = torch.empty((R, Cc, ph, pw), dtype=torch.int32, device=dev)
        if R > 0:
            with torch.cuda.device(dev):
                check(_lib.lib().sfod_roi_pool_fwd(xin.data_ptr(), r.data_ptr(), N, Cc, H, W, R, ph, pw, float(scale),
                                                   out.data_ptr(), argmax.data_ptr(), _stream(dev)), "sfod_roi_pool_fwd")
        ctx.save_for_backward(r, argmax)
        ctx.meta = (N, Cc, H, W, ph, pw, x.dtype)
        return out.to(x.dtype)

    @staticmethod
    def backward(ctx, grad_out: Tensor):
        r, argmax = ctx.saved_tensors
        N, Cc, H, W, ph, pw, dtype = ctx.meta
        dev = grad_out.device
        g = _f32c(grad_out)
        gin = torch.empty((N, Cc, H, W), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(_lib.lib().sfod_roi_pool_bwd(g.data_ptr(), r.data_ptr(), argmax.data_ptr(), N, Cc, H, W, r.shape[0], ph, pw,
                                               gin.data_ptr(), _stream(dev)), "sfod_roi_pool_bwd")
        return gin.to(dtype), None, None, None, None


def roi_pool(input: Tensor, boxes: Union[Tensor, List[Tensor]], output_size, spatial_scale: float = 1.0) -> Tensor:
    """torchvision.ops.roi_pool signature."""
    rois = _check_rois(boxes)
    ph, pw = _pair(output_size)
    return _RoIPoolFn.apply(input, rois, ph, pw, spatial_scale)


# ----------------------------------------------------------------------------------------------- box coder / softmax
def apply_deltas(deltas: Tensor, boxes: Tensor, weights: Sequence[float], scale_clamp: float = SCALE_CLAMP) -> Tensor:
    """detectron2 Box2BoxTransform.apply_deltas: deltas (R, 4k), boxes (R, 4) -> (R, 4k)."""
    dev = _require_cuda(deltas, boxes)
    d, b = _f32c(deltas), _f32c(boxes)
    if d.dim() != 2 or d.shape[1] % 4 != 0 or b.shape != (d.shape[0], 4):
        raise ValueError(f"apply_deltas: deltas {tuple(d.shape)} / boxes {tuple(b.shape)} mismatch")
    out = torch.empty_like(d)
    w = (C.c_float * 4)(*[float(v) for v in weights])
    with torch.cuda.device(dev):
        check(_lib.lib().sfod_apply_deltas(d.data_ptr(), b.data_ptr(), d.shape[0], d.shape[1] // 4, w, float(scale_clamp),
                                           out.data_ptr(), _stream(dev)), "sfod_apply_deltas")
    return out


def softmax_lastdim(x: Tensor) -> Tensor:
    dev = _require_cuda(x)
    xin = _f32c(x)
    x2 = xin.reshape(-1, xin.shape[-1])
    out = torch.empty_like(x2)
    with torch.cuda.device(dev):
        check(_lib.lib().sfod_softmax_lastdim(x2.data_ptr(), x2.shape[0], x2.shape[1], out.data_ptr(), _stream(dev)),
              "sfod_softmax_lastdim")
    return out.reshape(xin.shape)


def threshold_select(values: Tensor, counts: Tensor, thres: float) -> Tuple[Tensor, Tensor]:
    """Per-row stable selection of ``values > thres`` among the first counts[s] entries.
    values (S, stride) fp32, counts (S) int32 -> (index (S, stride) int64, count (S) int32)."""
    dev = _require_cuda(values, counts)
    v = _f32c(values)
    c = counts.to(torch.int32).contiguous()
    S, stride = v.shape
    idx = torch.empty((S, stride), dtype=torch.int64, device=dev)
    cnt = torch.empty((S,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().sfod_threshold_select(v.data_ptr(), c.data_ptr(), S, stride, float(thres), idx.data_ptr(),
                                               cnt.data_ptr(), _stream(dev)), "sfod_threshold_select")
    return idx, cnt


def class_threshold_select(values: Tensor, classes: Tensor, counts: Tensor, class_thresh: Tensor) -> Tuple[Tensor, Tensor]:
    """Per-row stable selection of ``values >= class_thresh[classes]`` among the first counts[s] entries.
    values (S, stride) fp32, classes (S, stride) int64, class_thresh (K) fp32 -> (index (S, stride) int64, count (S) int32)."""
    dev = _require_cuda(values, classes, counts, class_thresh)
    v = _f32c(values)
    cl = classes.detach().to(torch.int64).contiguous()
    c = counts.to(torch.int32).contiguous()
    th = _f32c(class_thresh)
    if v.dim() != 2 or cl.shape != v.shape or c.shape != (v.shape[0],):
        raise ValueError("values/classes must be (S, stride) and counts (S)")
    S, stride = v.shape
    idx = torch.empty((S, stride), dtype=torch.int64, device=dev)
    cnt = torch.empty((S,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().sfod_class_threshold_select(v.data_ptr(), cl.data_ptr(), c.data_ptr(), S, stride, th.numel(), th.data_ptr(),
                                                     idx.data_ptr(), cnt.data_ptr(), _stream(dev)), "sfod_class_threshold_select")
    return idx, cnt


def class_histogram(values: Tensor, classes: Tensor, counts: Tensor, num_classes: int, thres: float) -> Tensor:
    """Per-class count of entries with ``values > thres`` over all rows (count_label_prediction for a batch) -> (K) int64."""
    dev = _require_cuda(values, classes, counts)
    v = _f32c(values)
    cl = classes.detach().to(torch.int64).contiguous()
    c = counts.to(torch.int32).contiguous()
    S, stride = v.shape
    hist = torch.empty((int(num_classes),), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(_lib.lib().sfod_class_histogram(v.data_ptr(), cl.data_ptr(), c.data_ptr(), S, stride, int(num_classes), float(thres),
                                              hist.data_ptr(), _stream(dev)), "sfod_class_histogram")
    return hist


# ----------------------------------------------------------------------------------------------- image preprocessing
def normalize_pad(images: Union[Tensor, Sequence[Tensor]], pixel_mean: Sequence[float], pixel_std: Sequence[float],
                  size_divisibility: int = 0, channels_last: bool = False) -> Tuple[Tensor, List[Tuple[int, int]]]:
    """``ImageList.from_tensors([(x - mean) / std for x in images], size_divisibility)`` in one pass per image size:
    images is a (N, C, H, W) uint8/float32 tensor or a list of (C, H, W) tensors of any sizes; returns the padded fp32
    batch (zeros in the padding; channels-last storage on request) and the true (h, w) of every image."""
    if isinstance(images, Tensor):
        if images.dim() != 4:
            raise ValueError("a batched input must be (N, C, H, W)")
        groups = [(images, list(range(images.shape[0])))]
        sizes = [(int(images.shape[2]), int(images.shape[3]))] * images.shape[0]
        C_ = int(images.shape[1])
        dev = _require_cuda(images)
    else:
        if len(images) == 0:
            raise ValueError("empty image list")
        dev = _require_cuda(*images)
        C_ = int(images[0].shape[0])
        sizes = [(int(im.shape[-2]), int(im.shape[-1])) for im in images]
        groups = [(im.unsqueeze(0), [i]) for i, im in enumerate(images)]
    mean = [float(v) for v in pixel_mean]
    std = [float(v) for v in pixel_std]
    if len(mean) != C_ or len(std) != C_:
        raise ValueError("pixel_mean / pixel_std must have one value per channel")
    Hp, Wp = max(s[0] for s in sizes), max(s[1] for s in sizes)
    if size_divisibility > 1:
        Hp = (Hp + size_divisibility - 1) // size_divisibility * size_divisibility
        Wp = (Wp + size_divisibility - 1) // size_divisibility * size_divisibility
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    out = torch.empty((len(sizes), C_, Hp, Wp), dtype=torch.float32, device=dev, memory_format=fmt)
    cm, cs = (C.c_float * C_)(*mean), (C.c_float * C_)(*std)
    L = _lib.lib()
    slot = C_ * Hp * Wp
    with torch.cuda.device(dev):
        for t, idxs in groups:
            if t.dtype == torch.uint8:
                dt = DT_U8
            elif t.dtype == torch.float32:
                dt = DT_F32
            else:
                raise TypeError("images must be uint8 or float32")
            t = t.contiguous()
            n, _, H, W = t.shape
            check(L.sfod_normalize_pad(t.data_ptr(), dt, C_ * H * W, n, C_, H, W, cm, cs, Hp, Wp, NHWC if channels_last else NCHW,
                                       out.data_ptr() + idxs[0] * slot * 4, _stream(dev)), "sfod_normalize_pad")
    return out, sizes


# ----------------------------------------------------------------------------------------------- label sub-sampling
_MASK64 = (1 << 64) - 1


def sample_hash(seed: int, seg, idx):
    """The counter-based key of ``sfod_subsample_labels`` (csrc/sample.cuh ``sample_hash``) restated on the host (numpy uint64):
    splitmix64 finaliser of ``seed + golden * (seg << 32 | idx)``, upper 32 bits.  Pure arithmetic, used to derive the
    permutation the kernel realises (tests, RNG-parity callers)."""
    import numpy as np
    with np.errstate(over="ignore"):
        seg = np.asarray(seg, dtype=np.uint64); idx = np.asarray(idx, dtype=np.uint64)
        x = np.uint64(seed & _MASK64) + np.uint64(0x9E3779B97F4A7C15) * ((seg << np.uint64(32)) | idx)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return (x >> np.uint64(32)).astype(np.uint32)


def subsample_labels_batched(labels: Tensor, lengths: Sequence[int], num_samples: int, positive_fraction: float, bg_label: int,
                             seed: int) -> Tuple[Tensor, Tensor]:
    """detectron2 ``subsample_labels`` for all segments of ``labels`` (1-D int64, segment s = ``lengths[s]`` consecutive entries)
    in one launch and without host synchronisation: returns (sampled (S, num_samples) int64 segment-local indices padded with
    -1 -- positives first --, counts (S, 2) int32 (num_pos, num_neg)), both on the device."""
    dev = _require_cuda(labels)
    lab = labels.detach()
    if lab.dtype != torch.int64:
        lab = lab.to(torch.int64)
    lab = lab.contiguous()
    S = len(lengths)
    if sum(int(v) for v in lengths) != lab.numel():
        raise ValueError("lengths must sum to labels.numel()")
    offs = [0]
    for v in lengths:
        offs.append(offs[-1] + int(v))
    sampled = torch.empty((S, int(num_samples)), dtype=torch.int64, device=dev)
    counts = torch.empty((S, 2), dtype=torch.int32, device=dev)
    if S == 0:
        return sampled, counts
    max_pos = int(num_samples * positive_fraction)
    with torch.cuda.device(dev), _timed("subsample_labels"):
        offs_host = (C.c_int32 * len(offs))(*offs)      # host array: passed to the kernel by value (no H2D copy, no sync)
        check(_lib.lib().sfod_subsample_labels(lab.data_ptr(), offs_host, S, int(num_samples), max_pos, int(bg_label),
                                               int(seed) & _MASK64, sampled.data_ptr(), counts.data_ptr(), _stream(dev)),
              "sfod_subsample_labels")
    return sampled, counts


# ----------------------------------------------------------------------------------------------- box matching
def iou_match(gt_boxes: Tensor, boxes: Tensor, thresholds: Sequence[float], labels: Sequence[int],
              allow_low_quality_matches: bool = False) -> Tuple[Tensor, Tensor, Tensor]:
    """Fused ``pairwise_iou(gt_boxes, boxes)`` + detectron2 ``Matcher(thresholds, labels, allow_low_quality_matches)``:
    gt_boxes (M, 4), boxes (N, 4) -> (matches (N) int64, match_labels (N) int8, matched_vals (N) float32).
    ``thresholds`` are the Matcher's inner thresholds (ascending), ``labels`` has one more entry."""
    dev = _require_cuda(gt_boxes, boxes)
    g, b = _f32c(gt_boxes).reshape(-1, 4), _f32c(boxes).reshape(-1, 4)
    th = [float(t) for t in thresholds]
    lb = [int(v) for v in labels]
    if len(lb) != len(th) + 1 or any(v not in (-1, 0, 1) for v in lb):
        raise ValueError("labels must hold len(thresholds) + 1 values from {-1, 0, 1}")
    M, N = g.shape[0], b.shape[0]
    matches = torch.empty((N,), dtype=torch.int64, device=dev)
    mlabels = torch.empty((N,), dtype=torch.int8, device=dev)
    vals = torch.empty((N,), dtype=torch.float32, device=dev)
    if N == 0:
        return matches, mlabels, vals
    L = _lib.lib()
    cth = (C.c_float * max(len(th), 1))(*th)
    clb = (C.c_int * len(lb))(*lb)
    with torch.cuda.device(dev):
        ws = _workspace(dev, "match", L.sfod_iou_match_workspace_bytes(M))
        check(L.sfod_iou_match(g.data_ptr() if M else None, b.data_ptr(), M, N, cth, clb, len(th), int(bool(allow_low_quality_matches)),
                               matches.data_ptr(), mlabels.data_ptr(), vals.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)),
              "sfod_iou_match")
    return matches, mlabels, vals


# ----------------------------------------------------------------------------------------------- RPN selection
def rpn_select(logits: Tensor, deltas: Tensor, image_sizes: Sequence[Tuple[int, int]], *, anchors: Optional[Tensor] = None,
               cell_anchors: Optional[Tensor] = None, feat_hw: Optional[Tuple[int, int]] = None, stride: int = 0,
               anchor_offset: float = 0.0, weights: Sequence[float] = (1.0, 1.0, 1.0, 1.0), scale_clamp: float = SCALE_CLAMP,
               pre_nms_topk: int = 12000, post_nms_topk: int = 2000, nms_thresh: float = 0.7, min_box_size: float = 0.0):
    """Single-level RPN.predict_proposals for all images: logits (N, HWA), deltas (N, HWA, 4) -- or the RPN head's outputs as they
    lie, logits (N, A, Hf, Wf) and deltas (N, 4A, Hf, Wf): the flatten of reference rpn.py:28-41 is then folded into the kernels
    (no permute copy); indices keep the flattened (Hf, Wf, A) numbering either way.
    Either ``anchors`` (HWA, 4) or (``cell_anchors`` (A, 4), ``feat_hw``, ``stride``) must be given.
    Returns (boxes (N, P, 4), logits (N, P), src_index (N, P) int64, count (N) int32, invalid (N) int32)."""
    dev = _require_cuda(logits, deltas, anchors)
    if (logits.dim() == 4 and deltas.dim() == 4 and not logits.is_contiguous() and not deltas.is_contiguous()
            and logits.is_contiguous(memory_format=torch.channels_last) and deltas.is_contiguous(memory_format=torch.channels_last)
            and deltas.shape[1] == 4 * logits.shape[1]):
        # channels-last head outputs (NHWC backbone): the reference's flatten is a free VIEW of this memory, (N, H, W, A) and
        # (N, H, W, A, 4) -- take it instead of an NCHW copy
        if feat_hw is None:
            feat_hw = (int(logits.shape[2]), int(logits.shape[3]))
        n_img = logits.shape[0]
        logits = logits.permute(0, 2, 3, 1).reshape(n_img, -1)
        deltas = deltas.permute(0, 2, 3, 1).reshape(n_img, -1, 4)
    lg, dl = _f32c(logits), _f32c(deltas)
    native = lg.dim() == 4
    if native:
        N, A_head, Hh, Wh = lg.shape
        HWA = A_head * Hh * Wh
        if dl.shape != (N, 4 * A_head, Hh, Wh):
            raise ValueError(f"deltas must be (N, 4A, Hf, Wf) = {(N, 4 * A_head, Hh, Wh)}, got {tuple(dl.shape)}")
        if feat_hw is not None and (int(feat_hw[0]), int(feat_hw[1])) != (Hh, Wh):
            raise ValueError("feat_hw does not match the head outputs")
    else:
        N, HWA = lg.shape
        if dl.shape != (N, HWA, 4):
            raise ValueError(f"deltas must be (N, HWA, 4) = {(N, HWA, 4)}, got {tuple(dl.shape)}")
    if len(image_sizes) != N:
        raise ValueError("one image size per image is required")
    p = RpnParams()
    p.N, p.HWA = N, HWA
    p.stride, p.anchor_offset = int(stride), float(anchor_offset)
    for i in range(4):
        p.weights[i] = float(weights[i])
    p.scale_clamp = float(scale_clamp)
    p.pre_nms_topk, p.post_nms_topk = int(pre_nms_topk), int(post_nms_topk)
    p.min_box_size, p.nms_thresh = float(min_box_size), float(nms_thresh)
    anc = None
    if anchors is not None:
        anc = _f32c(anchors)
        if anc.shape != (HWA, 4):
            raise ValueError("anchors must be (HWA, 4)")
        p.A, p.Hf, p.Wf = (A_head, Hh, Wh) if native else (0, 0, 0)
    else:
        if cell_anchors is None or feat_hw is None or stride <= 0:
            raise ValueError("need anchors or (cell_anchors, feat_hw, stride)")
        ca = cell_anchors.detach().to("cpu", torch.float32).reshape(-1).tolist()
        A = len(ca) // 4
        if A > 64:
            raise ValueError("at most 64 cell anchors are supported in closed form; pass `anchors`")
        if native and A != A_head:
            raise ValueError(f"{A} cell anchors for head outputs with {A_head} anchors per cell")
        p.A, p.Hf, p.Wf = A, int(feat_hw[0]), int(feat_hw[1])
        for i, v in enumerate(ca):
            p.cell_anchors[i] = v
    p.head_layout = 1 if native else 0
    P = int(post_nms_topk)
    L = _lib.lib()
    with torch.cuda.device(dev):
        hw = _small_i32(dev, [v for s in image_sizes for v in (int(s[0]), int(s[1]))])
        out_boxes = torch.empty((N, P, 4), dtype=torch.float32, device=dev)
        out_logits = torch.empty((N, P), dtype=torch.float32, device=dev)
        out_src = torch.empty((N, P), dtype=torch.int64, device=dev)
        out_cnt = torch.empty((N,), dtype=torch.int32, device=dev)
        invalid = torch.empty((N,), dtype=torch.int32, device=dev)
        ws = _workspace(dev, "rpn", L.sfod_rpn_select_workspace_bytes(C.byref(p)))
        with _timed("rpn_select"):
            check(L.sfod_rpn_select(C.byref(p), lg.data_ptr(), dl.data_ptr(), anc.data_ptr() if anc is not None else None,
                                    hw.data_ptr(), out_boxes.data_ptr(), out_logits.data_ptr(), out_src.data_ptr(),
                                    out_cnt.data_ptr(), invalid.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "sfod_rpn_select")
    return out_boxes, out_logits, out_src, out_cnt, invalid


# ----------------------------------------------------------------------------------------------- Fast R-CNN post-process
def frcnn_postprocess(cls_logits: Tensor, deltas: Tensor, proposals: Tensor, rows_per_image, image_sizes: Sequence[Tuple[int, int]], *,
                      weights: Sequence[float] = (10.0, 10.0, 5.0, 5.0), scale_clamp: float = SCALE_CLAMP, score_thresh: float = 0.05,
                      nms_thresh: float = 0.5, topk: int = 100, pseudo_thresh: float = 0.8, want_probs: bool = False,
                      want_boxes: bool = False, rows_stride: int = 0):
    """FastRCNNOutputLayers.inference + threshold_bbox("roih") for all images in one call.
    cls_logits (R, K+1), deltas (R, 4K) or (R, 4), proposals (R, 4) concatenated over images.
    ``rows_per_image``: a list of ints (rows of image i follow those of image i-1), or -- packed layout, ``rows_stride > 0`` --
    an int32 DEVICE tensor of N row counts, image i owning rows [i*rows_stride, i*rows_stride + count[i]) (no host sync)."""
    dev = _require_cuda(cls_logits, deltas, proposals)
    cl, dl, pr = _f32c(cls_logits), _f32c(deltas), _f32c(proposals)
    R, K1 = cl.shape
    K = K1 - 1
    if K < 1:
        raise ValueError("cls_logits must have K+1 >= 2 columns")
    if dl.shape[0] != R or dl.shape[1] not in (4, 4 * K) or pr.shape != (R, 4):
        raise ValueError("deltas / proposals shapes do not match cls_logits")
    packed = rows_stride > 0
    if packed:
        if not isinstance(rows_per_image, Tensor) or rows_per_image.dtype != torch.int32 or not rows_per_image.is_cuda:
            raise ValueError("packed layout needs an int32 CUDA tensor of per-image row counts")
        if rows_per_image.numel() != len(image_sizes) or rows_stride * len(image_sizes) != R:
            raise ValueError("packed layout: R must equal N * rows_stride and counts must have N entries")
    elif sum(rows_per_image) != R or len(rows_per_image) != len(image_sizes):
        raise ValueError("rows_per_image must sum to R and match image_sizes")
    if topk < 0:
        raise ValueError("topk_per_image < 0 (return all) is not supported by the fused path")
    N = len(image_sizes)
    p = FrcnnParams()
    p.N, p.R, p.K = N, R, K
    p.class_agnostic = int(dl.shape[1] == 4 and K != 1)
    p.rows_stride = int(rows_stride) if packed else 0
    p.max_rows_per_image = int(rows_stride) if packed else (max(1, max(rows_per_image)) if N else 1)
    for i in range(4):
        p.weights[i] = float(weights[i])
    p.scale_clamp, p.score_thresh, p.nms_thresh = float(scale_clamp), float(score_thresh), float(nms_thresh)
    p.topk, p.pseudo_thresh, p.coord_trick_max_n = int(topk), float(pseudo_thresh), COORD_TRICK_MAX_N
    T = int(topk)
    L = _lib.lib()
    with torch.cuda.device(dev):
        if packed:
            row_off = rows_per_image.contiguous()
        else:
            offs = [0]
            for r in rows_per_image:
                offs.append(offs[-1] + int(r))
            row_off = _small_i32(dev, offs)
        hw = _small_i32(dev, [v for s in image_sizes for v in (int(s[0]), int(s[1]))])
        det_boxes = torch.empty((N, T, 4), dtype=torch.float32, device=dev)
        det_scores = torch.empty((N, T), dtype=torch.float32, device=dev)
        det_classes = torch.empty((N, T), dtype=torch.int64, device=dev)
        det_rows = torch.empty((N, T), dtype=torch.int64, device=dev)
        det_count = torch.empty((N,), dtype=torch.int32, device=dev)
        pseudo_count = torch.empty((N,), dtype=torch.int32, device=dev)
        probs = torch.empty((R, K1), dtype=torch.float32, device=dev) if want_probs else None
        boxes = torch.empty((R, dl.shape[1]), dtype=torch.float32, device=dev) if want_boxes else None
        ws = _workspace(dev, "frcnn", L.sfod_frcnn_postprocess_workspace_bytes(C.byref(p)))
        with _timed("frcnn_postprocess"):
            check(L.sfod_frcnn_postprocess(C.byref(p), cl.data_ptr(), dl.data_ptr(), pr.data_ptr(), row_off.data_ptr(), hw.data_ptr(),
                                           det_boxes.data_ptr(), det_scores.data_ptr(), det_classes.data_ptr(), det_rows.data_ptr(),
                                           det_count.data_ptr(), pseudo_count.data_ptr(),
                                           probs.data_ptr() if probs is not None else None,
                                           boxes.data_ptr() if boxes is not None else None, ws.data_ptr(), ws.numel(), _stream(dev)),
                  "sfod_frcnn_postprocess")
    return dict(boxes=det_boxes, scores=det_scores, classes=det_classes, rows=det_rows, count=det_count,
                pseudo_count=pseudo_count, probs=probs, decoded=boxes)


# ----------------------------------------------------------------------------------------------- box-head FC
def linear_3xtf32_supported(in_features: int, out_features: int) -> bool:
    """Shapes ``linear_3xtf32`` covers (TMA row strides are 16-byte multiples; the epilogue stores groups of 16 columns)."""
    return in_features % 4 == 0 and out_features % 16 == 0


def linear_3xtf32(x: Tensor, weight: Tensor, bias: Optional[Tensor] = None, relu: bool = False) -> Tensor:
    """``F.linear(x, weight, bias)`` (then ``torch.relu`` when ``relu``) in fp32 on the tensor cores with 3xTF32 arithmetic:
    fp32-level accuracy whatever ``torch.backends.cuda.matmul.allow_tf32`` says.  x (M, K), weight (N, K); no autograd."""
    dev = _require_cuda(x, weight, bias)
    x, w = _f32c(x), _f32c(weight)
    b = _f32c(bias) if bias is not None else None
    M, K = x.shape
    N = w.shape[0]
    if w.shape[1] != K or (b is not None and b.shape != (N,)):
        raise ValueError(f"linear_3xtf32: x {tuple(x.shape)}, weight {tuple(w.shape)}, bias {None if b is None else tuple(b.shape)}")
    y = torch.empty((M, N), dtype=torch.float32, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        ws = _workspace(dev, "linear_3xtf32", L.sfod_linear_3xtf32_workspace_bytes(M, N, K))
        with _timed("box_head_fc"):
            check(L.sfod_linear_3xtf32(x.data_ptr(), M, K, w.data_ptr(), N, b.data_ptr() if b is not None else None, int(bool(relu)),
                                       y.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "sfod_linear_3xtf32")
    return y


# ----------------------------------------------------------------------------------------------- EMA
class EmaPlan:
    """One-launch mean-teacher EMA over a fixed set of (student, teacher) tensor pairs.

    The chunk table is built once (tensor storages of a model are stable across steps) and kept on the
    device; ``step(keep_rate)`` is a single kernel launch at 12 B/element.
    """

    def __init__(self, pairs: Sequence[Tuple[Tensor, Tensor]]):
        if len(pairs) == 0:
            raise ValueError("EmaPlan needs at least one tensor pair")
        dev = _require_cuda(*[t for pr in pairs for t in pr])
        arr = (EmaTensor * len(pairs))()
        self._keepalive = []
        self.numel = 0
        for i, (s, t) in enumerate(pairs):
            if s.shape != t.shape:
                raise ValueError(f"EMA pair {i}: shape mismatch {tuple(s.shape)} vs {tuple(t.shape)}")
            if s.dtype != t.dtype:
                raise ValueError(f"EMA pair {i}: dtype mismatch {s.dtype} vs {t.dtype}")
            if s.dtype == torch.float32:
                code = 0
            elif s.dtype == torch.int64:
                code = 1
            else:
                raise TypeError(f"EMA supports float32 and int64 state tensors, got {s.dtype}")
            # elementwise over the storage: any dense layout works as long as both tensors share it (e.g. channels_last weights)
            if not (s.is_contiguous() and t.is_contiguous()):
                cl = s.dim() == 4 and s.is_contiguous(memory_format=torch.channels_last) and t.is_contiguous(memory_format=torch.channels_last)
                if not cl or s.stride() != t.stride():
                    raise ValueError(f"EMA pair {i}: tensors must be dense and share one memory layout")
            arr[i].student, arr[i].teacher = s.data_ptr(), t.data_ptr()
            arr[i].numel, arr[i].dtype = s.numel(), code
            self._keepalive.append((s, t))
            self.numel += s.numel()
        L = _lib.lib()
        self.n_chunks = int(L.sfod_ema_plan_chunks(arr, len(pairs)))
        nbytes = int(L.sfod_ema_plan_bytes(self.n_chunks))
        host = torch.empty(max(nbytes, 8), dtype=torch.uint8).pin_memory() if torch.cuda.is_available() else None
        check(L.sfod_ema_plan_build(arr, len(pairs), host.data_ptr(), nbytes), "sfod_ema_plan_build")
        self.device = dev
        self.plan = host.to(dev, non_blocking=False)

    def step(self, keep_rate: float) -> None:
        with torch.cuda.device(self.device), _timed("ema_multi_tensor"):
            check(_lib.lib().sfod_ema_multi_tensor(self.plan.data_ptr(), self.n_chunks, float(keep_rate), _stream(self.device)),
                  "sfod_ema_multi_tensor")


# ----------------------------------------------------------------------------------------------- BatchNorm (AdaBN)
# Multi-GPU statistics over peer memory: 0 = the payload is delivered by the finalize kernel itself (default), 1 = by the last CTA
# of the statistics kernel (overlapping the launch gap before the finalize kernel, at the price of a ticket atomic per CTA).  Both
# are correct and tested; bench.py measures both (no difference beyond noise in the AdaBN step at 2 GPUs: DESIGN.md section 7).
BN_P2P_TAIL_PUSH = int(os.environ.get("SFOD_P2P_TAIL_PUSH", "0"))


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return t.data_ptr() if t is not None else None


def _residual_like(residual: Tensor, xin: Tensor, layout: int) -> Tensor:
    """``residual`` in the memory layout of ``xin`` (the fused residual add reads both with the same indexing)."""
    res, rl = _layout_of(residual.detach())
    if res.shape != xin.shape or res.dtype != torch.float32:
        raise ValueError("residual must have the shape and dtype of x")
    if rl != layout:
        res = res.contiguous(memory_format=torch.channels_last if layout == NHWC else torch.contiguous_format)
    return res


def bn_train_forward(x: Tensor, weight: Optional[Tensor], bias: Optional[Tensor], running_mean: Optional[Tensor],
                     running_var: Optional[Tensor], num_batches_tracked: Optional[Tensor], momentum: float = 0.1,
                     eps: float = 1e-5, fuse_relu: bool = False, inplace: bool = False, group=None,
                     compute_output: bool = True, pre_bias: Optional[Tensor] = None, fuse_maxpool: bool = False,
                     residual: Optional[Tensor] = None) -> Optional[Tensor]:
    """Train-mode BatchNorm2d forward without autograd (the AdaBN / no_grad-teacher case): batch statistics,
    running-stat update, normalise(+residual)(+ReLU)(+2x2 max-pool).  ``pre_bias`` (C) is added to ``x`` first (the bias of the
    convolution feeding the BN, so the convolution itself can run bias-free); ``residual`` (same shape and layout as ``x``) is
    added to the normalised value before the ReLU (tail of a ResNet bottleneck).  With ``group`` (a torch.distributed process
    group, ``True`` = default group) the per-channel (sum, sum^2, count) payload is all-reduced on the device -- the count stays
    there, phase 2 reads it from the payload -- so that all ranks normalise with the statistics of the concatenated batch
    without a host read (SURVEY.md 8e)."""
    dev = _require_cuda(x, pre_bias, residual)
    xin, layout = _layout_of(x.detach())
    if xin.dtype != torch.float32:
        raise TypeError("bn_train_forward computes in float32")
    N, Cc, H, W = xin.shape
    pb = None
    if pre_bias is not None:
        pb = pre_bias.detach()
        if pb.dtype != torch.float32 or pb.numel() != Cc or not pb.is_contiguous():
            raise ValueError("pre_bias must be a contiguous float32 tensor with one entry per channel")
    if residual is not None and fuse_maxpool:
        raise ValueError("residual and fuse_maxpool are mutually exclusive")
    res = _residual_like(residual, xin, layout) if residual is not None else None
    L = _lib.lib()
    with torch.cuda.device(dev):
        stats = torch.empty((L.sfod_bn_stats_bytes(Cc) // 8,), dtype=torch.float64, device=dev)
        if (group is None and layout == NCHW and compute_output and not fuse_maxpool and xin.numel() * 4 <= BN_FUSED_MAX_BYTES
                and BN_FUSED_MAX_BYTES > 0):
            # activation fits L2: statistics -> grid barrier -> normalise in ONE cooperative launch (second read of x from L2)
            y = xin if inplace else torch.empty_like(xin)
            with _timed("bn_train_fused_res" if res is not None else "bn_train_fused"):
                rc = L.sfod_bn_train_fused(xin.data_ptr(), _ptr(pb), _ptr(res), y.data_ptr(), N, Cc, H, W, stats.data_ptr(),
                                           _ptr(weight), _ptr(bias), _ptr(running_mean), _ptr(running_var), _ptr(num_batches_tracked),
                                           float(momentum), float(eps), int(fuse_relu), _stream(dev))
            if rc == 0:
                return y
            if rc != 3:   # SFOD_ERR_UNSUPPORTED: no cooperative grid -> the two-phase path below
                check(rc, "sfod_bn_train_fused")
        comm = None
        if group is not None:
            from .engine.p2p import PeerStatExchange
            if isinstance(group, PeerStatExchange):
                # the all-reduce happens inside the finalize kernel (or the statistics kernel's last CTA), over NVLink peer memory
                if Cc > group.max_channels:
                    raise ValueError(f"PeerStatExchange carries at most {group.max_channels} channels per layer")
                comm = C.byref(group.comm)
        with _timed("bn_partial_stats"):
            check(L.sfod_bn_partial_stats(xin.data_ptr(), _ptr(pb), layout, N, Cc, H * W, stats.data_ptr(),
                                          comm if BN_P2P_TAIL_PUSH else None, _stream(dev)), "sfod_bn_partial_stats")
        if group is not None and comm is None:
            from .engine.adabn_dist import allreduce_bn_stats_device
            allreduce_bn_stats_device(stats, Cc, group=group if group is not True else None)   # payload [0, 2C] incl. the count
        y = None
        if compute_output:
            if fuse_maxpool:
                fmt = torch.channels_last if layout == NHWC else torch.contiguous_format
                y = torch.empty((N, Cc, H // 2, W // 2), dtype=torch.float32, device=dev, memory_format=fmt)
            else:
                y = xin if inplace else torch.empty_like(xin)
        if comm is not None:
            tag = "bn_exchange_finalize_apply"
        else:
            tag = "bn_finalize_apply_pool" if fuse_maxpool else ("bn_finalize_apply_res" if res is not None else "bn_finalize_apply")
        with _timed(tag):
            check(L.sfod_bn_finalize_apply(xin.data_ptr() if compute_output else None, _ptr(pb), _ptr(res) if compute_output else None,
                                           _ptr(y), layout, N, Cc, H, W, stats.data_ptr(), comm, _ptr(weight), _ptr(bias),
                                           _ptr(running_mean), _ptr(running_var), _ptr(num_batches_tracked), float(momentum), float(eps),
                                           int(fuse_relu), int(fuse_maxpool), _stream(dev)), "sfod_bn_finalize_apply")
    return y


def bn_frozen_forward(x: Tensor, weight: Optional[Tensor], bias: Optional[Tensor], running_mean: Tensor, running_var: Tensor,
                      eps: float = 1e-5, fuse_relu: bool = False, inplace: bool = False, residual: Optional[Tensor] = None) -> Tensor:
    """FrozenBatchNorm2d / eval-mode BatchNorm forward with the fused neighbours (ReLU, residual add); no autograd."""
    dev = _require_cuda(x, residual, running_mean, running_var)
    xin, layout = _layout_of(x.detach())
    if xin.dtype != torch.float32:
        raise TypeError("bn_frozen_forward computes in float32")
    N, Cc, H, W = xin.shape
    res = _residual_like(residual, xin, layout) if residual is not None else None
    L = _lib.lib()
    with torch.cuda.device(dev):
        scratch = torch.empty((L.sfod_bn_frozen_scratch_bytes(Cc),), dtype=torch.uint8, device=dev)
        y = xin if inplace else torch.empty_like(xin)
        with _timed("bn_frozen_apply"):
            check(L.sfod_bn_frozen_apply(xin.data_ptr(), _ptr(res), y.data_ptr(), layout, N, Cc, H, W, _ptr(weight), _ptr(bias),
                                         running_mean.data_ptr(), running_var.data_ptr(), float(eps), int(fuse_relu),
                                         scratch.data_ptr(), _stream(dev)), "sfod_bn_frozen_apply")
    return y


# ----------------------------------------------------------------------------------------------- strong augmentation (8f rank 3)
def _u8_batch(images: Tensor) -> Tuple[Tensor, torch.device]:
    dev = _require_cuda(images)
    if images.dim() != 4 or images.shape[1] != 3 or images.dtype != torch.uint8:
        raise ValueError("images must be a (N, 3, H, W) uint8 tensor")
    return images.contiguous(), dev


def _struct_array_to_device(arr, dev: torch.device) -> Tensor:
    raw = bytes(arr)
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)


def color_jitter(images: Tensor, params: Sequence[dict]) -> Tensor:
    """torchvision ColorJitter (+ RandomGrayscale) on a uint8 batch with per-image decisions ``params[n] = dict(order=[...],
    factors=[...], grayscale=bool)``: ``order`` lists op codes (0 brightness, 1 contrast, 2 saturation, 3 hue) in application
    order with their ``factors`` (Python floats); an empty order = jitter not applied.  Follows torchvision's PIL path
    (ImageEnhance / Image.convert: what the reference runs, since its mapper feeds PIL images) in Pillow's arithmetic, bit for bit."""
    x, dev = _u8_batch(images)
    N, _, H, W = x.shape
    if len(params) != N:
        raise ValueError("one parameter record per image")
    arr = (JitterParams * max(N, 1))()
    for n, p in enumerate(params):
        order, fac = list(p.get("order", [])), list(p.get("factors", []))
        if len(order) != len(fac) or len(order) > 4 or any(o not in (0, 1, 2, 3) for o in order):
            raise ValueError("order / factors: up to four ops from {0, 1, 2, 3} with one factor each")
        arr[n].n_ops = len(order)
        for k, (o, f) in enumerate(zip(order, fac)):
            arr[n].op[k], arr[n].factor[k] = int(o), float(f)
            if int(o) == 3:
                if not -0.5 <= float(f) <= 0.5:
                    raise ValueError("hue factor must lie in [-0.5, 0.5]")
                arr[n].hue_shift[k] = int(float(f) * 255) & 0xFF   # np.int32(hue * 255).astype(np.uint8) of torchvision's PIL path
        arr[n].grayscale = int(bool(p.get("grayscale", False)))
    out = torch.empty_like(x)
    if N == 0:
        return out
    with torch.cuda.device(dev), _timed("color_jitter"):
        rec = _struct_array_to_device(arr, dev)
        ws = _workspace(dev, "jitter", 8 * N)
        check(_lib.lib().sfod_color_jitter_pil(x.data_ptr(), N, H, W, rec.data_ptr(), ws.data_ptr(), ws.numel(), out.data_ptr(),
                                               _stream(dev)), "sfod_color_jitter_pil")
    return out


def pil_blur_params(sigma: float, passes: int = 3) -> Tuple[int, int, int]:
    """(box radius, ww, fw) of Pillow's GaussianBlur(radius=sigma): the float32 arithmetic of ``_gaussian_blur_radius`` and
    ``ImagingHorizontalBoxBlur`` (Pillow src/libImaging/BoxBlur.c), operation by operation."""
    import numpy as np
    f = np.float32
    rad = f(sigma)
    sigma2 = f(rad * rad / f(passes))
    L = f(np.sqrt(12.0 * float(sigma2) + 1.0))
    l = f(np.floor((float(L) - 1.0) / 2.0))
    a = f(f(f(2) * l + f(1)) * f(f(l * f(l + f(1))) - f(f(3) * sigma2)))
    a = f(a / f(f(6) * f(sigma2 - f(f(l + f(1)) * f(l + f(1))))))
    fr = f(l + a)
    r = int(fr)
    ww = int(f(16777216.0) / f(fr * f(2) + f(1)))
    fw = ((1 << 24) - (r * 2 + 1) * ww) // 2
    return r, ww, fw


def gaussian_blur_pil(images: Tensor, sigmas: Sequence[Optional[float]]) -> Tensor:
    """``PIL.ImageFilter.GaussianBlur(radius=sigma)`` on a uint8 batch, bit for bit -- the blur of the reference's strong augmentation
    (reference daod/data/transforms/augmentations.py:18-21).  ``sigmas[n] is None`` (or 0) leaves image n untouched."""
    x, dev = _u8_batch(images)
    N, _, H, W = x.shape
    if len(sigmas) != N:
        raise ValueError("one sigma (or None) per image")
    radius, wws, fws = [-1] * N, [0] * N, [0] * N
    for n, sg in enumerate(sigmas):
        if sg is None or float(sg) == 0.0:
            continue
        if float(sg) < 0:
            raise ValueError("sigma must be >= 0")
        radius[n], wws[n], fws[n] = pil_blur_params(float(sg))
        if radius[n] > 9:
            raise ValueError("sigma too large for the fused tile kernel (box radius <= 9, sigma <= ~10)")
    out = torch.empty_like(x)
    if N == 0:
        return out
    with torch.cuda.device(dev), _timed("gaussian_blur_pil"):
        r_dev = _small_i32(dev, radius)
        w_dev = _small_i32(dev, wws + fws)     # both weights are < 2^24: int32 and uint32 share the bit pattern
        check(_lib.lib().sfod_gaussian_blur_pil(x.data_ptr(), N, H, W, r_dev.data_ptr(), w_dev.data_ptr(), w_dev.data_ptr() + 4 * N,
                                                max(max(radius), 0), out.data_ptr(), _stream(dev)), "sfod_gaussian_blur_pil")
    return out


def random_erase_(images: Tensor, rects: Sequence[Sequence[Tuple[int, int, int, int]]], noise: Optional[Tensor] = None, seed: int = 0) -> Tensor:
    """In place RandomErasing(value="random") on a uint8 batch: ``rects[n]`` = up to four (top, left, height, width) rectangles
    applied in order; the fill is ``byte(255 * v)`` with v ~ N(0, 1) (device generator keyed by ``seed``), or
    ``v = noise[n, k, c, y, x]`` ((N, 4, 3, H, W) float32) when given."""
    dev = _require_cuda(images, noise)
    if images.dim() != 4 or images.shape[1] != 3 or images.dtype != torch.uint8 or not images.is_contiguous():
        raise ValueError("images must be a contiguous (N, 3, H, W) uint8 tensor (modified in place)")
    N, _, H, W = images.shape
    if len(rects) != N:
        raise ValueError("one rectangle list per image")
    arr = (EraseParams * max(N, 1))()
    for n, rl in enumerate(rects):
        if len(rl) > 4:
            raise ValueError("at most four rectangles per image")
        arr[n].n_rects = len(rl)
        for k, (i, j, h, w) in enumerate(rl):
            if i < 0 or j < 0 or h < 0 or w < 0 or i + h > H or j + w > W:
                raise ValueError(f"rectangle {(i, j, h, w)} outside the image")
            arr[n].rect[k][0], arr[n].rect[k][1], arr[n].rect[k][2], arr[n].rect[k][3] = int(i), int(j), int(h), int(w)
    if noise is not None and (noise.shape != (N, 4, 3, H, W) or noise.dtype != torch.float32 or not noise.is_contiguous()):
        raise ValueError("noise must be a contiguous (N, 4, 3, H, W) float32 tensor")
    if N == 0:
        return images
    with torch.cuda.device(dev), _timed("random_erase"):
        rec = _struct_array_to_device(arr, dev)
        check(_lib.lib().sfod_random_erase(images.data_ptr(), N, H, W, rec.data_ptr(), noise.data_ptr() if noise is not None else None,
                                           int(seed) & _MASK64, _stream(dev)), "sfod_random_erase")
    return images


# ----------------------------------------------------------------------------------------------- weak augmentation (8f rank 3)
RESIZE_MAX_KSIZE = 9          # ksize = 2 * ceil(max(in / out, 1)) + 1: down-scales up to 4 per axis


def pil_resize_coeffs(in_size: int, out_size: int) -> Tuple[Tensor, Tensor]:
    """Bounds ``(out, 2)`` int32 ``[xmin, xmax]`` and taps ``(out, ksize)`` int32 (zero past ``xmax``) of Pillow's 8-bit BILINEAR
    resampler along one axis (Pillow src/libImaging/Resample.c: ``precompute_coeffs`` + ``normalize_coeffs_8bpc``), in Python
    floats (C doubles) and in Pillow's order: the weights are summed sequentially before they are normalised."""
    in_size, out_size = int(in_size), int(out_size)
    if in_size <= 0 or out_size <= 0:
        raise ValueError("sizes must be positive")
    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = 1.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    ss = 1.0 / fs
    bounds = [[0, 0] for _ in range(out_size)]
    taps = [[0] * ksize for _ in range(out_size)]
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        w = []
        for x in range(xmax):
            t = abs((x + xmin - center + 0.5) * ss)
            w.append(1.0 - t if t < 1.0 else 0.0)
        ww = 0.0
        for v in w:
            ww += v
        for x, v in enumerate(w):
            if ww != 0.0:
                v = v / ww
            taps[xx][x] = int(-0.5 + v * (1 << 22)) if v < 0 else int(0.5 + v * (1 << 22))
        bounds[xx] = [xmin, xmax]
    return torch.tensor(bounds, dtype=torch.int32), torch.tensor(taps, dtype=torch.int32)


# device-resident coefficient tables: one growing int32 arena per device, every (in, out) pair uploaded once.  The kernel addresses
# the tables by int32 offsets into the arena; a grown arena copies the old tables to the same offsets, and the old one stays alive
# (a launch enqueued earlier may still read it).
_resize_arena: Dict[int, dict] = {}


def _resize_table(dev: torch.device, in_size: int, out_size: int) -> Tuple[int, int]:
    """-> (offset into the device arena, ksize) of the table of one axis."""
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    a = _resize_arena.setdefault(idx, {"buf": None, "used": 0, "index": {}, "old": []})
    hit = a["index"].get((in_size, out_size))
    if hit is not None:
        return hit
    bounds, taps = pil_resize_coeffs(in_size, out_size)
    table = torch.cat([bounds.reshape(-1), taps.reshape(-1)])
    off, n = a["used"], table.numel()
    if a["buf"] is None or off + n > a["buf"].numel():
        grown = torch.empty(max(2 * (off + n), 1 << 16), dtype=torch.int32, device=dev)
        if a["buf"] is not None:
            grown[:off].copy_(a["buf"][:off])
            a["old"].append(a["buf"])
        a["buf"] = grown
    a["buf"][off:off + n].copy_(table)
    a["used"] = off + n
    a["index"][(in_size, out_size)] = (off, int(taps.shape[1]))
    return off, int(taps.shape[1])


class ResizePlan:
    """Host-side part of one ``resize_pil`` call: the per-image records (uploaded to the device), the output layout and the launch
    geometry.  ``launch(out)`` enqueues the kernel; a plan can be launched again while its inputs and tables stay alive."""

    def __init__(self, images: Union[Tensor, Sequence[Tensor]], sizes: Sequence[Tuple[int, int]], hflip: Optional[Sequence[bool]] = None):
        imgs = list(images.unbind(0)) if isinstance(images, Tensor) else list(images)
        if isinstance(images, Tensor) and images.dim() != 4:
            raise ValueError("a batched input must be (N, H, W, 3)")
        if not imgs:
            raise ValueError("empty image batch")
        dev = _require_cuda(*imgs)
        N = len(imgs)
        sizes = [(int(h), int(w)) for h, w in sizes]
        flips = [False] * N if hflip is None else [bool(f) for f in hflip]
        if len(sizes) != N or len(flips) != N:
            raise ValueError("one output size and one flip flag per image")
        for im in imgs:
            if im.dim() != 3 or im.shape[2] != 3 or im.dtype != torch.uint8:
                raise ValueError("images must be (H, W, 3) uint8 (a CHW image as x.permute(1, 2, 0))")
        arr = (ResizeImage * N)()
        self.offsets, total, max_k = [], 0, 0
        with torch.cuda.device(dev):
            for n, (im, (h, w)) in enumerate(zip(imgs, sizes)):
                H, W = int(im.shape[0]), int(im.shape[1])
                if H <= 0 or W <= 0 or h <= 0 or w <= 0:
                    raise ValueError("image and output sizes must be positive")
                if H > 4 * h or W > 4 * w:
                    raise ValueError(f"resize {H}x{W} -> {h}x{w}: down-scales beyond 4 per axis are not supported")
                if h * w > 0x7FFFFFFF:
                    raise ValueError("output plane too large")
                kxo, kxs = _resize_table(dev, W, w)
                kyo, kys = _resize_table(dev, H, h)
                max_k = max(max_k, kxs, kys)
                r = arr[n]
                r.src = im.data_ptr()
                r.stride_row, r.stride_px, r.stride_ch = (int(v) for v in im.stride())
                r.in_h, r.in_w, r.out_h, r.out_w = H, W, h, w
                r.out_offset = total
                r.hflip = int(flips[n])
                r.kx_offset, r.kx_size, r.ky_offset, r.ky_size = kxo, kxs, kyo, kys
                self.offsets.append(total)
                total += 3 * h * w
            self.records = _struct_array_to_device(arr, dev)
            self.coeffs = _resize_arena[dev.index if dev.index is not None else torch.cuda.current_device()]["buf"]
        self.images, self.dev, self.n, self.sizes, self.nbytes, self.max_k = imgs, dev, N, sizes, total, max_k

    def launch(self, out: Tensor) -> None:
        if out.device != self.dev or out.dtype != torch.uint8 or out.numel() < self.nbytes or not out.is_contiguous():
            raise ValueError("out must be a contiguous uint8 tensor of at least nbytes on the images' device")
        with torch.cuda.device(self.dev):
            check(_lib.lib().sfod_resize_pil(self.records.data_ptr(), self.n, self.coeffs.data_ptr(), out.data_ptr(),
                                             max(h for h, _ in self.sizes), max(w for _, w in self.sizes), self.max_k,
                                             _stream(self.dev)), "sfod_resize_pil")


def resize_pil(images: Union[Tensor, Sequence[Tensor]], sizes: Sequence[Tuple[int, int]],
               hflip: Optional[Sequence[bool]] = None) -> Union[Tensor, List[Tensor]]:
    """``np.flip(np.asarray(Image.fromarray(img).resize((w, h), Image.BILINEAR)), 1)`` (flip optional) for every image of a batch,
    bit for bit, transposed to CHW -- detectron2's ResizeTransform (uint8 path) + HFlipTransform + the mapper's HWC -> CHW copy.

    ``images``: a (N, H, W, 3) tensor, or a list of (H, W, 3) CUDA uint8 tensors or views of any strides (a CHW image passes as
    ``x.permute(1, 2, 0)``); ``sizes[n]`` = output (h, w); ``hflip[n]`` = mirror the output horizontally.  Returns a (N, 3, h, w)
    tensor when all output sizes are equal, otherwise a list of (3, h, w) views into one allocation.  One launch."""
    with _timed("resize_pil"):
        plan = ResizePlan(images, sizes, hflip)
        out = torch.empty(plan.nbytes, dtype=torch.uint8, device=plan.dev)
        plan.launch(out)
    N, sz = plan.n, plan.sizes
    if all(s == sz[0] for s in sz):
        return out.view(N, 3, sz[0][0], sz[0][1])
    return [out[o:o + 3 * h * w].view(3, h, w) for o, (h, w) in zip(plan.offsets, sz)]


# ----------------------------------------------------------------------------------------------- COCO box AP
def coco_eval_out_numel(T: int, R: int, K: int, A: int, M: int) -> int:
    """Elements of the packed fp64 result of ``coco_box_eval``: precision and scores (T, R, K, A, M), then recall (T, K, A, M)."""
    return 2 * T * R * K * A * M + T * K * A * M


def coco_box_eval(gt_offsets: Sequence[int], gt_boxes: Tensor, gt_area: Tensor, gt_iscrowd: Tensor, gt_ids: Tensor, gt_categories: Tensor,
                  dt_boxes: Tensor, dt_scores: Tensor, dt_classes: Tensor, dt_counts: Tensor, num_categories: int,
                  iou_thrs: Sequence[float], rec_thrs: Sequence[float], area_rngs: Sequence[Sequence[float]], max_dets: Sequence[int],
                  out: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """pycocotools ``COCOeval(iouType="bbox")``: ``evaluate()`` + ``accumulate()`` on the device, bit-equal (include/sfod_b200.h,
    ``sfod_coco_eval``).  Images are the ground truth's images in ascending id order, categories its categories in ascending
    id order (index 0..K-1).

    ``gt_offsets`` (host, I + 1 ints): the gt of image i are rows [gt_offsets[i], gt_offsets[i+1]) of ``gt_boxes`` (n_gt, 4)
    fp64 XYWH, ``gt_area`` fp64 (the annotations' area), ``gt_iscrowd``, ``gt_ids`` and ``gt_categories`` int64, in annotation
    order.  Detections: one padded row per image, ``dt_boxes`` (I, P, 4) fp32 XYWH, ``dt_scores`` (I, P), ``dt_classes``
    (I, P) int64 and the device-side valid counts ``dt_counts`` (I).  ``out``: optional fp64 buffer of at least
    ``coco_eval_out_numel`` elements.  Returns (precision, recall, scores) as views into it, with COCOeval's -1 where a cell is
    undefined.  No host synchronisation."""
    dev = _require_cuda(gt_boxes, gt_area, gt_iscrowd, gt_ids, gt_categories, dt_boxes, dt_scores, dt_classes, dt_counts, out)
    offs = [int(v) for v in gt_offsets]
    I = len(offs) - 1
    if I < 0 or offs[0] != 0 or any(b < a for a, b in zip(offs, offs[1:])):
        raise ValueError("coco_box_eval: gt_offsets must start at 0 and be non-decreasing (ground truth sorted by image)")
    n_gt = offs[-1]
    if max((b - a for a, b in zip(offs, offs[1:])), default=0) > 1024:
        raise ValueError("coco_box_eval: more than 1024 ground-truth boxes in one image")
    if tuple(gt_boxes.shape) != (n_gt, 4) or any(t.shape != (n_gt,) for t in (gt_area, gt_iscrowd, gt_ids, gt_categories)):
        raise ValueError(f"coco_box_eval: ground truth of {n_gt} boxes expected, got boxes {tuple(gt_boxes.shape)}")
    if dt_boxes.dim() != 3 or dt_boxes.shape[0] != I or dt_boxes.shape[2] != 4:
        raise ValueError(f"coco_box_eval: dt_boxes must be ({I}, P, 4), got {tuple(dt_boxes.shape)}")
    P = dt_boxes.shape[1]
    if dt_scores.shape != (I, P) or dt_classes.shape != (I, P) or dt_counts.shape != (I,):
        raise ValueError("coco_box_eval: dt_scores / dt_classes must be (I, P) and dt_counts (I,)")
    if not 1 <= P <= 1024 or I * P >= 1 << 24:
        raise ValueError(f"coco_box_eval: {P} detection slots per image (1..1024, images x slots < 2^24)")
    K, T, R, A, M = int(num_categories), len(iou_thrs), len(rec_thrs), len(area_rngs), len(max_dets)
    if not (1 <= K <= _lib.COCO_MAX_CATEGORIES and 1 <= T <= _lib.COCO_MAX_IOU_THRS and 1 <= R <= _lib.COCO_MAX_REC_THRS
            and 1 <= A <= _lib.COCO_MAX_AREA_RNGS and 1 <= M <= _lib.COCO_MAX_MAX_DETS):
        raise ValueError(f"coco_box_eval: unsupported sizes K={K} T={T} R={R} A={A} M={M}")
    if any(not 1 <= int(m) <= 128 for m in max_dets):
        raise ValueError(f"coco_box_eval: maxDets must lie in 1..128, got {list(max_dets)}")
    if any(t.dtype != d for t, d in ((gt_boxes, torch.float64), (gt_area, torch.float64), (gt_ids, torch.int64), (gt_categories, torch.int64),
                                     (dt_boxes, torch.float32), (dt_scores, torch.float32), (dt_classes, torch.int64), (dt_counts, torch.int32))):
        raise ValueError("coco_box_eval: gt boxes / area fp64, ids / categories / dt classes int64, dt boxes / scores fp32, counts int32")
    need = coco_eval_out_numel(T, R, K, A, M)
    if out is None:
        out = torch.empty(need, dtype=torch.float64, device=dev)
    elif out.dtype != torch.float64 or not out.is_contiguous() or out.numel() < need:
        raise ValueError(f"coco_box_eval: out must be a contiguous fp64 tensor of >= {need} elements")
    p = _lib.CocoEvalParams()
    p.n_images, p.n_categories, p.dt_stride = I, K, P
    p.n_iou_thrs, p.n_rec_thrs, p.n_area_rngs, p.n_max_dets = T, R, A, M
    for i, v in enumerate(max_dets):
        p.max_dets[i] = int(v)
    for i, v in enumerate(iou_thrs):
        p.iou_thrs[i] = float(v)
    for i, v in enumerate(rec_thrs):
        p.rec_thrs[i] = float(v)
    for i, (lo, hi) in enumerate(area_rngs):
        p.area_rng[i][0], p.area_rng[i][1] = float(lo), float(hi)
    host_offs = (C.c_int64 * (I + 1))(*offs)
    gt = [t.contiguous() for t in (gt_boxes, gt_area, gt_iscrowd.to(torch.uint8), gt_ids, gt_categories)]
    dt = [t.contiguous() for t in (dt_boxes, dt_scores, dt_classes, dt_counts)]
    n1 = T * R * K * A * M
    precision, scores, recall = out[:n1], out[n1:2 * n1], out[2 * n1:need]
    L = _lib.lib()
    with torch.cuda.device(dev):
        ws = _workspace(dev, "coco_eval", L.sfod_coco_eval_workspace_bytes(C.byref(p)))
        with _timed("coco_eval"):
            check(L.sfod_coco_eval(C.byref(p), host_offs, *[_ptr(t) if t.numel() else None for t in gt], *[_ptr(t) if t.numel() else None for t in dt],
                                   precision.data_ptr(), scores.data_ptr(), recall.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)),
                  "sfod_coco_eval")
    return precision.view(T, R, K, A, M), recall.view(T, K, A, M), scores.view(T, R, K, A, M)
