"""Weak and strong augmentation of the input batch on the GPU (SURVEY.md 8f rank 3).

Weak: the reference's mapper first applies detectron2's ``build_augmentation(cfg, is_train)`` -- ResizeShortestEdge, then (training)
RandomFlip -- to every image; the teacher consumes this weak image and the strong chain below runs on it.  ``draw_weak_params``
draws the decisions with the same numpy calls in the same order as detectron2's ``get_transform``s, ``weak_augment`` does the
pixel work in one launch (``ops.resize_pil``: Pillow's BILINEAR resize + flip + HWC -> CHW, bit for bit) and
``apply_weak_to_boxes`` maps annotation boxes as ``transform_instance_annotations`` does.

Strong:

The reference builds, per image and on the CPU (PIL), reference daod/data/detection_utils.py:7-37:

    RandomApply([ColorJitter(0.4, 0.4, 0.4, 0.1)], p=0.8) -> RandomGrayscale(p=0.2) -> RandomApply([GaussianBlur((0.1, 2.0))], p=0.5)
    -> ToTensor -> RandomErasing(0.7, (0.05, 0.2), (0.3, 3.3), "random") -> RandomErasing(0.5, (0.02, 0.2), (0.1, 6), "random")
    -> RandomErasing(0.3, (0.02, 0.2), (0.05, 8), "random") -> ToPILImage

and applies it in the data mapper (daod/data/mappers/two_crop_augmentation_mapper.py:141-157).  Here the random DECISIONS are
drawn on the host with the same distributions and in the same order as torchvision draws them (``draw_params``), and the
pixel work runs on the batch in HBM (``ops.color_jitter`` / ``ops.gaussian_blur_pil`` / ``ops.random_erase_``: 4 launches per batch
instead of ~10 PIL passes per image on one CPU core).  Images are RGB uint8 (N, 3, H, W), as the mapper's PIL images are.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import Tensor

from .. import ops
from ..config import CfgNode, get_cfg

JITTER = dict(brightness=(0.6, 1.4), contrast=(0.6, 1.4), saturation=(0.6, 1.4), hue=(-0.1, 0.1), p=0.8)   # ColorJitter(0.4, 0.4, 0.4, 0.1)
GRAYSCALE_P = 0.2
BLUR = dict(sigma=(0.1, 2.0), p=0.5)
ERASERS = [dict(p=0.7, scale=(0.05, 0.2), ratio=(0.3, 3.3)), dict(p=0.5, scale=(0.02, 0.2), ratio=(0.1, 6.0)),
           dict(p=0.3, scale=(0.02, 0.2), ratio=(0.05, 8.0))]


def _uniform(g: torch.Generator, lo: float, hi: float) -> float:
    return float(torch.empty(1).uniform_(lo, hi, generator=g))


def draw_erase_rect(g: torch.Generator, H: int, W: int, scale, ratio):
    """torchvision RandomErasing.get_params (10 attempts; None if no rectangle fits)."""
    area = H * W
    log_ratio = (math.log(ratio[0]), math.log(ratio[1]))
    for _ in range(10):
        erase_area = area * _uniform(g, scale[0], scale[1])
        aspect_ratio = math.exp(_uniform(g, log_ratio[0], log_ratio[1]))
        h = int(round(math.sqrt(erase_area * aspect_ratio)))
        w = int(round(math.sqrt(erase_area / aspect_ratio)))
        if not (h < H and w < W):
            continue
        i = int(torch.randint(0, H - h + 1, size=(1,), generator=g))
        j = int(torch.randint(0, W - w + 1, size=(1,), generator=g))
        return (i, j, h, w)
    return None


def draw_params(N: int, H: int, W: int, generator: Optional[torch.Generator] = None) -> List[Dict]:
    """The per-image decisions of the reference's strong augmentation: same distributions, same order of draws."""
    g = generator if generator is not None else torch.default_generator
    out = []
    for _ in range(N):
        p: Dict = {"order": [], "factors": [], "grayscale": False, "sigma": None, "rects": []}
        if not (JITTER["p"] < float(torch.rand(1, generator=g))):           # RandomApply
            fn_idx = torch.randperm(4, generator=g).tolist()                # ColorJitter.get_params
            vals = [_uniform(g, *JITTER["brightness"]), _uniform(g, *JITTER["contrast"]), _uniform(g, *JITTER["saturation"]),
                    _uniform(g, *JITTER["hue"])]
            p["order"], p["factors"] = fn_idx, [vals[k] for k in fn_idx]
        p["grayscale"] = bool(float(torch.rand(1, generator=g)) < GRAYSCALE_P)
        if not (BLUR["p"] < float(torch.rand(1, generator=g))):
            p["sigma"] = _uniform(g, *BLUR["sigma"])
        for e in ERASERS:
            if float(torch.rand(1, generator=g)) < e["p"]:
                r = draw_erase_rect(g, H, W, e["scale"], e["ratio"])
                if r is not None:
                    p["rects"].append(r)
        out.append(p)
    return out


def strong_augment(images: Tensor, params: Optional[List[Dict]] = None, generator: Optional[torch.Generator] = None,
                   noise: Optional[Tensor] = None, seed: Optional[int] = None) -> Tensor:
    """(N, 3, H, W) uint8 RGB CUDA batch -> strongly augmented uint8 batch (a new tensor).

    ColorJitter / RandomGrayscale run in Pillow's arithmetic (torchvision's PIL path, which the reference's mapper takes:
    daod/data/mappers/two_crop_augmentation_mapper.py:141-157), bit for bit.  The blur is the reference's filter,
    ``PIL.ImageFilter.GaussianBlur(radius=sigma)`` (reference daod/data/transforms/augmentations.py:18-21) reproduced bit for bit
    (``ops.gaussian_blur_pil``: Pillow's three extended box-blur passes per axis)."""
    N, _, H, W = images.shape
    if params is None:
        params = draw_params(N, H, W, generator)
    x = ops.color_jitter(images, params)
    if any(p["sigma"] is not None for p in params):
        x = ops.gaussian_blur_pil(x, [p["sigma"] for p in params])
    if any(p["rects"] for p in params):
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,), generator=generator if generator is not None else torch.default_generator))
        ops.random_erase_(x, [p["rects"] for p in params], noise=noise, seed=seed)
    return x


# ------------------------------------------------------------------------------------------------------------- weak augmentation
def _resize_shortest_edge_shape(h: int, w: int, size: int, max_size: int) -> Tuple[int, int]:
    """detectron2 ResizeShortestEdge.get_output_shape."""
    size = size * 1.0
    scale = size / min(h, w)
    if h < w:
        newh, neww = size, scale * w
    else:
        newh, neww = scale * h, size
    if max(newh, neww) > max_size:
        scale = max_size * 1.0 / max(newh, neww)
        newh = newh * scale
        neww = neww * scale
    return int(newh + 0.5), int(neww + 0.5)


def draw_weak_params(image_sizes: Sequence[Tuple[int, int]], cfg: CfgNode, is_train: bool = True,
                     rng: Optional[np.random.RandomState] = None) -> List[Dict]:
    """Per image ``{"size": (h, w), "hflip": bool}``: the decisions of detectron2's ``build_augmentation(cfg, is_train)`` --
    ``ResizeShortestEdge(MIN_SIZE_*, MAX_SIZE_*, sampling)`` and, in training, ``RandomFlip`` -- drawn with the same numpy calls in
    the same order as their ``get_transform``s (per image: the short edge, then the flip on the resized image).  ``rng=None``
    draws from numpy's global state, as detectron2 does."""
    r = np.random if rng is None else rng
    if is_train:
        short, max_size, style = cfg.INPUT.MIN_SIZE_TRAIN, cfg.INPUT.MAX_SIZE_TRAIN, cfg.INPUT.get("MIN_SIZE_TRAIN_SAMPLING", "choice")
        flip = cfg.INPUT.get("RANDOM_FLIP", "horizontal")
    else:
        short, max_size, style, flip = cfg.INPUT.MIN_SIZE_TEST, cfg.INPUT.MAX_SIZE_TEST, "choice", "none"
    if style not in ("range", "choice"):
        raise ValueError(f"MIN_SIZE_TRAIN_SAMPLING {style!r}")
    if flip not in ("horizontal", "none"):
        raise NotImplementedError(f"RANDOM_FLIP {flip!r}: only 'horizontal' and 'none' are supported")
    if isinstance(short, int):
        short = (short, short)
    if style == "range" and len(short) != 2:
        raise ValueError("MIN_SIZE_TRAIN_SAMPLING 'range' needs two sizes")
    out = []
    for h, w in image_sizes:
        size = r.randint(short[0], short[1] + 1) if style == "range" else r.choice(short)
        if size == 0:                                                    # NoOpTransform
            newh, neww = int(h), int(w)
        else:
            newh, neww = _resize_shortest_edge_shape(int(h), int(w), size, max_size)
        do_flip = bool(r.uniform(0, 1.0, []) < 0.5) if flip == "horizontal" else False   # RandomFlip._rand_range() < prob
        out.append({"size": (newh, neww), "hflip": do_flip})
    return out


def weak_augment(images: Union[Tensor, Sequence[Tensor]], params: Optional[List[Dict]] = None, cfg: Optional[CfgNode] = None,
                 is_train: bool = True, rng: Optional[np.random.RandomState] = None) -> Tuple[Union[Tensor, List[Tensor]], List[Dict]]:
    """Resize (+ flip) a batch of decoded uint8 RGB images on the GPU: ``images`` is a (N, H, W, 3) tensor or a list of (H, W, 3)
    CUDA tensors or views (``x.permute(1, 2, 0)`` for a CHW image).  Without ``params`` the decisions are drawn by
    ``draw_weak_params`` from ``cfg`` (detectron2's defaults, ``config.get_cfg()``, when None).  Returns the CHW weak images -- a
    (N, 3, h, w) tensor when all sizes agree, otherwise a list -- and the parameters used."""
    imgs = list(images.unbind(0)) if isinstance(images, Tensor) else list(images)
    if params is None:
        params = draw_weak_params([(int(im.shape[0]), int(im.shape[1])) for im in imgs], cfg if cfg is not None else get_cfg(),
                                  is_train, rng)
    out = ops.resize_pil(images, [p["size"] for p in params], [p["hflip"] for p in params])
    return out, params


def apply_weak_to_boxes(boxes_xyxy, image_size: Tuple[int, int], param: Dict) -> np.ndarray:
    """detectron2 ``transform_instance_annotations`` for the weak transforms: each transform maps the four corners of every box
    (resize ``x * (new_w / w)``, ``y * (new_h / h)``; flip ``x -> new_w - x``) and takes their min / max; the result is clipped
    to ``[0, new size]``.  float64 arithmetic; float32 result (what ``Boxes`` stores).  ``image_size`` = the original (h, w)."""
    h, w = int(image_size[0]), int(image_size[1])
    newh, neww = (int(v) for v in param["size"])
    box = np.asarray(boxes_xyxy, dtype=np.float64).reshape(-1, 4)
    idxs = np.array([(0, 1), (2, 1), (0, 3), (2, 3)]).flatten()

    def apply_box(b, fn):
        coords = fn(b[:, idxs].reshape(-1, 2)).reshape((-1, 4, 2))
        return np.concatenate((coords.min(axis=1), coords.max(axis=1)), axis=1)

    def resize(c):
        c[:, 0] = c[:, 0] * (neww * 1.0 / w)
        c[:, 1] = c[:, 1] * (newh * 1.0 / h)
        return c

    def hflip(c):
        c[:, 0] = neww - c[:, 0]
        return c

    box = apply_box(box, resize)
    if param["hflip"]:
        box = apply_box(box, hflip)
    box = np.minimum(box.clip(min=0), [neww, newh, neww, newh])
    return box.astype(np.float32)
