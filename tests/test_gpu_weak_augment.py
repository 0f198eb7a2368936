"""GPU tests of the weak augmentation: ops.resize_pil / engine.weak_augment against live Pillow, bit for bit.

detectron2's ResizeTransform.apply_image for uint8 images is ``Image.fromarray(img).resize((w, h), Image.BILINEAR)``, RandomFlip's
HFlipTransform is ``np.flip(img, axis=1)`` after it, and the mapper then transposes HWC -> CHW; the kernel fuses the three.
"""
import numpy as np
import pytest
import torch
from PIL import Image

import sfod_b200  # noqa: F401
from sfod_b200 import config, engine, ops

pytestmark = pytest.mark.gpu

SHAPES = [
    (1024, 2048, 600, 1200),     # Cityscapes / Foggy Cityscapes at MIN_SIZE_TRAIN 600
    (375, 1242, 403, 1333),      # KITTI-like, enlarges vertically
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


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _image(H, W, seed):
    img = np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)
    img[:2, :5] = 255                                                      # saturated corner: the 255 clamp is reachable
    return img


def _want(img, h, w, flip):
    """The mapper's weak image as CHW: Pillow resize, np.flip, transpose."""
    out = np.asarray(Image.fromarray(img).resize((w, h), Image.BILINEAR))
    if flip:
        out = np.flip(out, axis=1)
    return torch.from_numpy(np.array(out.transpose(2, 0, 1), order="C", copy=True))    # a fresh array: no negative stride


@pytest.mark.parametrize("H,W,h,w", SHAPES)
def test_resize_pil_equals_pillow_hwc_and_chw_views(dev, H, W, h, w):
    img = _image(H, W, H * 31 + W)
    hwc = torch.from_numpy(img).to(dev)
    chw = torch.from_numpy(np.ascontiguousarray(img.transpose(2, 0, 1))).to(dev)     # what decode_jpeg(device="cuda") returns
    for flip in (False, True):
        want = _want(img, h, w, flip)
        for src in (hwc, chw.permute(1, 2, 0)):
            launches = ops.launch_count()
            got = ops.resize_pil([src], [(h, w)], [flip])
            assert ops.launch_count() == launches + 1
            assert got.shape == (1, 3, h, w) and got.dtype == torch.uint8
            assert torch.equal(got[0].cpu(), want), (flip, src.stride(), int((got[0].cpu() != want).sum()))


def test_resize_pil_mixed_batch_returns_a_list_and_equal_batch_a_tensor(dev):
    cases = SHAPES[3:]                                                     # small shapes, every kind of scale, one launch
    imgs = [_image(H, W, k) for k, (H, W, _, _) in enumerate(cases)]
    flips = [k % 2 == 1 for k in range(len(cases))]
    # alternate HWC tensors and permuted CHW views inside one batch
    srcs = [torch.from_numpy(im).to(dev) if k % 3 else torch.from_numpy(np.ascontiguousarray(im.transpose(2, 0, 1))).to(dev).permute(1, 2, 0)
            for k, im in enumerate(imgs)]
    launches = ops.launch_count()
    got = ops.resize_pil(srcs, [(h, w) for _, _, h, w in cases], flips)
    assert ops.launch_count() == launches + 1
    assert isinstance(got, list) and len(got) == len(cases)
    base = got[0].untyped_storage().data_ptr()
    for k, ((H, W, h, w), im) in enumerate(zip(cases, imgs)):
        assert got[k].shape == (3, h, w) and got[k].untyped_storage().data_ptr() == base       # views into one allocation
        assert torch.equal(got[k].cpu(), _want(im, h, w, flips[k])), (cases[k], flips[k])
    # equal output sizes -> one (N, 3, h, w) tensor; a (N, H, W, 3) batch input
    batch = np.stack([_image(75, 130, 100 + k) for k in range(5)])
    flips = [True, False, False, True, True]
    launches = ops.launch_count()
    got = ops.resize_pil(torch.from_numpy(batch).to(dev), [(48, 83)] * 5, flips)
    assert ops.launch_count() == launches + 1
    assert isinstance(got, torch.Tensor) and got.shape == (5, 3, 48, 83) and got.is_contiguous()
    for k in range(5):
        assert torch.equal(got[k].cpu(), _want(batch[k], 48, 83, flips[k]))
    # different input sizes to one output size still give a tensor
    got = ops.resize_pil([torch.from_numpy(imgs[0]).to(dev), torch.from_numpy(imgs[1]).to(dev)], [(30, 40)] * 2, [False, True])
    assert isinstance(got, torch.Tensor) and got.shape == (2, 3, 30, 40)
    assert torch.equal(got[1].cpu(), _want(imgs[1], 30, 40, True))


def test_resize_pil_cityscapes_batch_of_eight(dev):
    """The timed size: eight 1024x2048 images -> 600x1200, half of them flipped."""
    g = torch.Generator().manual_seed(8)
    x = torch.randint(0, 256, (8, 1024, 2048, 3), dtype=torch.uint8, generator=g)
    flips = [bool(k % 2) for k in range(8)]
    got = ops.resize_pil(x.to(dev), [(600, 1200)] * 8, flips).cpu()
    for k in range(8):
        assert torch.equal(got[k], _want(x[k].numpy(), 600, 1200, flips[k])), k


def test_resize_pil_rejects_unsupported_input(dev):
    x = torch.zeros(41, 64, 3, dtype=torch.uint8, device=dev)
    with pytest.raises(ValueError, match="beyond 4"):
        ops.resize_pil([x], [(10, 16)], [False])                          # 41 / 10 > 4
    with pytest.raises(ValueError):
        ops.resize_pil([x.float()], [(20, 32)], [False])
    with pytest.raises(ValueError):
        ops.resize_pil([x[..., :2]], [(20, 32)], [False])
    with pytest.raises(ValueError):
        ops.resize_pil([x], [(20, 32), (20, 32)], [False])


def _tv_jitter(img, p):
    import torchvision.transforms.functional as TF
    for o, f in zip(p["order"], p["factors"]):
        img = (TF.adjust_brightness, TF.adjust_contrast, TF.adjust_saturation, TF.adjust_hue)[o](img, f)
    if p.get("grayscale"):
        img = TF.rgb_to_grayscale(img, num_output_channels=3)
    return img


def test_weak_then_strong_equals_the_reference_mapper_on_pil_images(dev):
    """The reference mapper's image path: ResizeShortestEdge (Pillow BILINEAR) + RandomFlip (np.flip) with detectron2's draws, then the
    strong chain on the PIL weak image (ColorJitter + RandomGrayscale, GaussianBlur, ToTensor, RandomErasing with the drawn noise,
    ToPILImage), against engine.weak_augment -> engine.strong_augment with the same decisions and noise: bit-equal."""
    import torchvision.transforms.functional as TF
    from PIL import ImageFilter
    N, H, W = 10, 120, 200
    cfg = config.get_cfg()
    cfg.INPUT.MIN_SIZE_TRAIN, cfg.INPUT.MAX_SIZE_TRAIN = (72,), 1333
    imgs = [_image(H, W, 500 + k) for k in range(N)]
    weak, wp = engine.weak_augment(torch.from_numpy(np.stack(imgs)).to(dev), cfg=cfg, rng=np.random.RandomState(12))
    assert [p["size"] for p in wp] == [(72, 120)] * N
    assert any(p["hflip"] for p in wp) and not all(p["hflip"] for p in wp)
    h, w = wp[0]["size"]
    g = torch.Generator().manual_seed(2026)
    sp = engine.draw_strong_augmentation_params(N, h, w, g)
    assert any(p["order"] for p in sp) and any(p["sigma"] is not None for p in sp) and any(p["rects"] for p in sp)
    noise = torch.randn(N, 4, 3, h, w, generator=g)
    got = engine.strong_augment(weak, params=sp, noise=noise.to(dev)).cpu()
    for n in range(N):
        img = np.asarray(Image.fromarray(imgs[n]).resize((w, h), Image.BILINEAR))                  # ResizeTransform.apply_image
        if wp[n]["hflip"]:
            img = np.flip(img, axis=1)                                                             # HFlipTransform.apply_image
        pil = Image.fromarray(np.ascontiguousarray(img), "RGB")
        pil = _tv_jitter(pil, sp[n])
        if sp[n]["sigma"] is not None:
            pil = pil.filter(ImageFilter.GaussianBlur(radius=sp[n]["sigma"]))
        t = TF.to_tensor(pil)
        for k, (i, j, hh, ww) in enumerate(sp[n]["rects"]):
            t = TF.erase(t, i, j, hh, ww, noise[n, k, :, i:i + hh, j:j + ww])
        want = torch.from_numpy(np.array(TF.to_pil_image(t))).permute(2, 0, 1)
        assert torch.equal(got[n], want), (n, wp[n], sp[n], int((got[n] != want).sum()))
