"""CPU tests (no GPU) of the weak augmentation: detectron2's ResizeShortestEdge + RandomFlip as the reference's mapper applies them.

* resize_bilinear below (a numpy restatement of Pillow's 8-bit BILINEAR resampler, test infrastructure) against live Pillow;
* ops.pil_resize_coeffs against the restatement's tables;
* engine.draw_weak_params against a literal restatement of detectron2's two get_transform()s on an identically seeded RNG;
* engine.apply_weak_to_boxes against the float64 restatement of transform_instance_annotations;
* the C ABI surface of sfod_resize_pil: exported, mirrored, argument checks without a launch; no CPU fallback.
"""
import ctypes as C
import sys

import numpy as np
import pytest
import torch
from PIL import Image

import sfod_b200  # noqa: F401
from sfod_b200 import _lib, config, engine, ops

# --------------------------------------------------------------------------------------------------------------------------
# Image.resize((w, h), Image.BILINEAR) on an 8-bit image: Pillow's src/libImaging/Resample.c, restated in numpy.  detectron2's
# ResizeTransform.apply_image calls it for uint8 images (the weak augmentation of the reference's mapper).  Per axis, in C double:
#   scale = in / out, fs = max(scale, 1), support = fs, ksize = 2 ceil(support) + 1; per output xx: center = (xx + 0.5) scale,
#   xmin = max(int(center - support + 0.5), 0), xmax = min(int(center + support + 0.5), in) - xmin,
#   w[x] = bilinear((x + xmin - center + 0.5) / fs), normalised by their sequential sum, k[x] = int(w[x] 2^22 + 0.5).
# Horizontal pass first, over the input rows the vertical taps use, rounded to a uint8 temporary image; then the vertical pass.
# Each output is clip8(2^21 + sum in * k) with clip8(s) = 0 / 255 / s >> 22.  Pinned against live Pillow below.
PRECISION_BITS = 22


def resize_coeffs(in_size: int, out_size: int):
    """-> (bounds (out, 2) int64 [xmin, xmax], taps (out, ksize) int64, zero-padded past xmax)."""
    scale = float(in_size) / out_size
    fs = max(scale, 1.0)
    support = 1.0 * fs
    ksize = int(np.ceil(support)) * 2 + 1
    taps = np.zeros((out_size, ksize), np.int64)
    bounds = np.zeros((out_size, 2), np.int64)
    ss = 1.0 / fs
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
        if ww != 0.0:
            w = [v / ww for v in w]
        for x, v in enumerate(w):
            taps[xx, x] = int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
        bounds[xx] = (xmin, xmax)
    return bounds, taps


def _resample_rows(img: np.ndarray, bounds: np.ndarray, taps: np.ndarray) -> np.ndarray:
    """One pass along axis 1 of an (H, W, C) uint8 array."""
    H, _, C = img.shape
    src = img.astype(np.int64)
    out = np.empty((H, len(bounds), C), np.uint8)
    for xx, (xmin, xmax) in enumerate(bounds):
        acc = np.full((H, C), 1 << (PRECISION_BITS - 1), np.int64)
        for x in range(xmax):
            acc += src[:, xmin + x, :] * taps[xx, x]
        out[:, xx, :] = np.where(acc <= 0, 0, np.where(acc >= 255 << PRECISION_BITS, 255, acc >> PRECISION_BITS))
    return out


def resize_bilinear(img_hwc: np.ndarray, w: int, h: int) -> np.ndarray:
    """(H, W, C) uint8 -> what ``Image.fromarray(img_hwc).resize((w, h), Image.BILINEAR)`` returns, as an (h, w, C) array."""
    H, W, _ = img_hwc.shape
    out = img_hwc
    bv, kv = resize_coeffs(H, h)
    if w != W:
        bh, kh = resize_coeffs(W, w)
        y0, y1 = int(bv[0, 0]), int(bv[-1, 0] + bv[-1, 1])
        out = _resample_rows(out[y0:y1], bh, kh)
        bv = bv.copy()
        bv[:, 0] -= y0
    if h != H:
        out = _resample_rows(out.transpose(1, 0, 2), bv, kv).transpose(1, 0, 2)
    return np.ascontiguousarray(out)


# (H, W, h, w): the three dataset shapes, pure up / down, mixed, one axis unchanged, 1-pixel outputs, a scale of exactly 4, odd sizes
SHAPES = [
    (1024, 2048, 600, 1200),     # Cityscapes / Foggy Cityscapes at MIN_SIZE_TRAIN 600
    (375, 1242, 403, 1333),      # KITTI with MAX_SIZE 1333 (enlarges vertically)
    (1052, 1914, 600, 1092),     # Sim10k
    (37, 53, 80, 111),           # up
    (64, 128, 38, 75),           # down
    (20, 30, 7, 200),            # down vertically, up horizontally
    (100, 100, 100, 57),         # height unchanged
    (61, 90, 30, 90),            # width unchanged
    (3, 4, 1, 1),                # 1-pixel output
    (1, 40, 1, 13),              # 1-row image
    (40, 64, 10, 16),            # scale of exactly 4 (ksize 9)
    (31, 17, 9, 5),              # odd sizes
    (333, 517, 129, 701),
]


def _pil_resize(img, w, h):
    return np.asarray(Image.fromarray(img).resize((w, h), Image.BILINEAR))


@pytest.mark.parametrize("H,W,h,w", SHAPES)
def test_restated_resize_equals_pillow(H, W, h, w):
    rng = np.random.default_rng(H * 7919 + W)
    img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    img[:2, :5] = 255                                                   # saturated corner: the 255 clamp is reachable
    assert np.array_equal(resize_bilinear(img, w, h), _pil_resize(img, w, h))


def test_restated_resize_extreme_values_hit_both_clamps():
    img = np.zeros((16, 16, 3), np.uint8)
    img[::2, ::2] = 255
    for (h, w) in ((7, 5), (16, 40), (4, 4)):
        assert np.array_equal(resize_bilinear(img, w, h), _pil_resize(img, w, h))


@pytest.mark.parametrize("n_in,n_out", [(2048, 1200), (1024, 600), (1242, 1333), (375, 403), (1914, 1092), (1052, 600), (64, 16),
                                        (53, 111), (100, 100), (4, 1), (1, 1), (17, 5)])
def test_pil_resize_coeffs_equal_the_restated_tables(n_in, n_out):
    bounds, taps = ops.pil_resize_coeffs(n_in, n_out)
    ob, ot = resize_coeffs(n_in, n_out)
    assert bounds.dtype == torch.int32 and taps.dtype == torch.int32
    assert np.array_equal(bounds.numpy(), ob) and np.array_equal(taps.numpy(), ot)
    assert taps.shape[1] == 2 * int(np.ceil(max(n_in / n_out, 1.0))) + 1
    assert (ob[:, 0] + ob[:, 1] <= n_in).all() and (ot >= 0).all()


# ---------------------------------------------------------------------------------------------------------------- draws
class _D2ResizeShortestEdge:
    """detectron2 0.6 detectron2/data/transforms/augmentation_impl.py ResizeShortestEdge, restated (np.random -> rs)."""

    def __init__(self, short_edge_length, max_size=sys.maxsize, sample_style="range"):
        self.is_range = sample_style == "range"
        if isinstance(short_edge_length, int):
            short_edge_length = (short_edge_length, short_edge_length)
        self.short_edge_length, self.max_size = short_edge_length, max_size

    def get_transform(self, image, rs):
        h, w = image.shape[:2]
        if self.is_range:
            size = rs.randint(self.short_edge_length[0], self.short_edge_length[1] + 1)
        else:
            size = rs.choice(self.short_edge_length)
        if size == 0:
            return (h, w)
        return self.get_output_shape(h, w, size, self.max_size)

    @staticmethod
    def get_output_shape(oldh, oldw, short_edge_length, max_size):
        h, w = oldh, oldw
        size = short_edge_length * 1.0
        scale = size / min(h, w)
        if h < w:
            newh, neww = size, scale * w
        else:
            newh, neww = scale * h, size
        if max(newh, neww) > max_size:
            scale = max_size * 1.0 / max(newh, neww)
            newh = newh * scale
            neww = neww * scale
        neww = int(neww + 0.5)
        newh = int(newh + 0.5)
        return (newh, neww)


class _D2RandomFlip:
    """detectron2 RandomFlip(prob=0.5, horizontal=True).get_transform with Augmentation._rand_range, restated."""

    def get_transform(self, image, rs):
        low, high = 0, 1.0
        return rs.uniform(low, high, []) < 0.5


def _d2_draw(sizes, short, max_size, style, is_train, rs):
    augs = [_D2ResizeShortestEdge(short, max_size, style)] + ([_D2RandomFlip()] if is_train else [])
    out = []
    for h, w in sizes:
        image = np.empty((h, w, 0))                                       # AugmentationList: each transform sees the current image
        newh, neww = augs[0].get_transform(image, rs)
        flip = bool(augs[1].get_transform(np.empty((newh, neww, 0)), rs)) if is_train else False
        out.append({"size": (newh, neww), "hflip": flip})
    return out


def _same_state(a, b):
    sa, sb = a.get_state(), b.get_state()
    return sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


SIZES = [(1024, 2048), (1024, 2048), (375, 1242), (1052, 1914), (2048, 1024), (600, 600), (17, 999)]


@pytest.mark.parametrize("short,max_size,style", [((600,), 1333, "choice"), ((480, 512, 544, 576, 608), 1333, "choice"),
                                                  ((480, 800), 1333, "range"), ((600,), 1000, "choice"), (600, 1333, "choice")])
def test_draw_weak_params_is_detectron2s_random_stream(short, max_size, style):
    cfg = config.vgg_source_free_cfg()
    cfg.INPUT.MIN_SIZE_TRAIN, cfg.INPUT.MAX_SIZE_TRAIN, cfg.INPUT.MIN_SIZE_TRAIN_SAMPLING = short, max_size, style
    for seed in (0, 1, 2024):
        a, b = np.random.RandomState(seed), np.random.RandomState(seed)
        got = engine.draw_weak_params(SIZES * 3, cfg, True, a)
        assert got == _d2_draw(SIZES * 3, short, max_size, style, True, b)
        assert _same_state(a, b)
    assert any(p["hflip"] for p in got) and not all(p["hflip"] for p in got)


def test_draw_weak_params_dataset_shapes_and_test_mode():
    cfg = config.vgg_source_free_cfg()
    assert cfg.INPUT.MIN_SIZE_TRAIN == (600,) and cfg.INPUT.MIN_SIZE_TRAIN_SAMPLING == "choice" and cfg.INPUT.RANDOM_FLIP == "horizontal"
    got = engine.draw_weak_params([(1024, 2048), (375, 1242), (1052, 1914), (2048, 1024)], cfg, True, np.random.RandomState(5))
    # KITTI: max_size caps the long side, 375 * 1333 / 1242 = 402.48 -> 402
    assert [p["size"] for p in got] == [(600, 1200), (402, 1333), (600, 1092), (1200, 600)]
    # a one-element "choice" draws no number: only the flips consume the stream
    a, b = np.random.RandomState(9), np.random.RandomState(9)
    engine.draw_weak_params([(1024, 2048)] * 4, cfg, True, a)
    b.uniform(0, 1.0, [4])
    assert _same_state(a, b)
    # test mode: ResizeShortestEdge(MIN_SIZE_TEST, MAX_SIZE_TEST, "choice") only -- no flip draw
    for seed in (3, 4):
        a, b = np.random.RandomState(seed), np.random.RandomState(seed)
        got = engine.draw_weak_params(SIZES, cfg, False, a)
        assert got == _d2_draw(SIZES, cfg.INPUT.MIN_SIZE_TEST, cfg.INPUT.MAX_SIZE_TEST, "choice", False, b)
        assert not any(p["hflip"] for p in got) and _same_state(a, b)
    # the default is numpy's global state, as in detectron2
    np.random.seed(77)
    got = engine.draw_weak_params(SIZES, cfg)
    assert got == _d2_draw(SIZES, (600,), 1333, "choice", True, np.random.RandomState(77))


def test_draw_weak_params_rejects_unsupported_settings():
    cfg = config.get_cfg()
    cfg.INPUT.RANDOM_FLIP = "vertical"
    with pytest.raises(NotImplementedError):
        engine.draw_weak_params([(10, 10)], cfg, True, np.random.RandomState(0))
    cfg = config.get_cfg()
    cfg.INPUT.MIN_SIZE_TRAIN_SAMPLING = "range"
    with pytest.raises(ValueError):
        engine.draw_weak_params([(10, 10)], cfg, True, np.random.RandomState(0))     # (800,) is not a range


# ---------------------------------------------------------------------------------------------------------------- boxes
def _d2_transform_boxes(bbox, image_size, param):
    """detectron2 transform_instance_annotations for [ResizeTransform, HFlipTransform] (Transform.apply_box per transform), then
    Boxes(...) -> float32."""
    h, w = image_size
    newh, neww = param["size"]
    idxs = np.array([(0, 1), (2, 1), (0, 3), (2, 3)]).flatten()

    def apply_box(box, apply_coords):
        coords = np.asarray(box).reshape(-1, 4)[:, idxs].reshape(-1, 2)
        coords = apply_coords(coords).reshape((-1, 4, 2))
        return np.concatenate((coords.min(axis=1), coords.max(axis=1)), axis=1)

    def resize_coords(coords):
        coords[:, 0] = coords[:, 0] * (neww * 1.0 / w)
        coords[:, 1] = coords[:, 1] * (newh * 1.0 / h)
        return coords

    def hflip_coords(coords):
        coords[:, 0] = neww - coords[:, 0]
        return coords

    out = []
    for b in bbox:
        box = apply_box(np.array([b]), resize_coords)
        if param["hflip"]:
            box = apply_box(box, hflip_coords)
        box = box[0].clip(min=0)
        out.append(np.minimum(box, list((newh, neww) + (newh, neww))[::-1]))
    return torch.tensor(np.array(out), dtype=torch.float32).numpy()


def test_apply_weak_to_boxes_equals_detectron2():
    rng = np.random.default_rng(3)
    boxes = np.concatenate([rng.uniform(0, 2048, (40, 2)), rng.uniform(0, 1024, (40, 2))], 1)[:, [0, 2, 1, 3]]
    boxes[:, 2:] = boxes[:, :2] + rng.uniform(0.1, 400, (40, 2))              # some run past the image: clipped
    boxes[0] = (-5.0, -3.0, 10.0, 12.0)                                          # negative corner: clipped to 0
    boxes = boxes.tolist()
    for size, param in (((1024, 2048), {"size": (600, 1200), "hflip": False}), ((1024, 2048), {"size": (600, 1200), "hflip": True}),
                        ((375, 1242), {"size": (403, 1333), "hflip": True}), ((1052, 1914), {"size": (600, 1092), "hflip": False})):
        got = engine.apply_weak_to_boxes(boxes, size, param)
        want = _d2_transform_boxes(boxes, size, param)
        assert got.dtype == np.float32 and got.shape == (40, 4)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (size, param)
        assert (got >= 0).all() and (got[:, 0::2] <= param["size"][1]).all() and (got[:, 1::2] <= param["size"][0]).all()


# ---------------------------------------------------------------------------------------------------------------- C ABI
def test_resize_entry_point_is_exported_mirrored_and_checks_arguments():
    L = _lib.lib()
    launches = L.sfod_debug_launch_count()
    assert "sfod_resize_pil" in _lib.SIGNATURES and _lib.ABI_STRUCTS[6] is _lib.ResizeImage
    assert L.sfod_abi_sizeof(6) == C.sizeof(_lib.ResizeImage) == 80
    rec, cf, out = 0x1000, 0x2000, 0x3000                                         # never dereferenced: every call below is refused
    assert L.sfod_resize_pil(rec, -1, cf, out, 600, 1200, 5, None) == 1         # N < 0
    assert L.sfod_resize_pil(None, 1, cf, out, 600, 1200, 5, None) == 1         # null pointers
    assert L.sfod_resize_pil(rec, 1, None, out, 600, 1200, 5, None) == 1
    assert L.sfod_resize_pil(rec, 1, cf, None, 600, 1200, 5, None) == 1
    assert L.sfod_resize_pil(rec, 1, cf, out, 0, 1200, 5, None) == 1           # non-positive sizes
    assert L.sfod_resize_pil(rec, 1, cf, out, 600, -1, 5, None) == 1
    assert L.sfod_resize_pil(rec, 1, cf, out, 600, 1200, 0, None) == 1
    assert L.sfod_resize_pil(rec, 1, cf, out, 65536, 32768, 5, None) == 1      # 2^31 pixels: int32 plane index overflows
    assert L.sfod_resize_pil(rec, 1, cf, out, 600, 1200, 11, None) == 3        # down-scale beyond 4: unsupported
    assert L.sfod_resize_pil(rec, 0, cf, out, 600, 1200, 5, None) == 0         # empty batch: nothing to do
    assert L.sfod_debug_launch_count() == launches


def test_resize_pil_refuses_cpu_tensors():
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.resize_pil(torch.zeros(2, 8, 8, 3, dtype=torch.uint8), [(4, 4)] * 2, [False, True])
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        engine.weak_augment([torch.zeros(8, 8, 3, dtype=torch.uint8)], params=[{"size": (4, 4), "hflip": False}])
