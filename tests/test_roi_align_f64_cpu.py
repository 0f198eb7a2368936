"""CPU tests (no GPU): pin the float64 ROIAlign reference of oracle/roi_align_f64.py, which the GPU path tests compare
every kernel with.

1. Its fp32 geometry is the kernels' (and torchvision's): the fp32 terms it produces, summed in torchvision's order, equal
   torchvision.ops.roi_align in fp32 bit for bit, forward and backward, on the edge ROIs of the path tests and the
   adversarial ROIs of the forward parity test.
2. Its float64 accumulation is right: where the fp32 geometry is exact (dyadic coordinates, power-of-two scale, bin sizes
   that are dyadic multiples of 1 / 7 of the ROI and power-of-two grids) it equals torchvision run on float64 tensors to
   1e-12 of the error scale S . |X|; on general ROIs the difference is the fp32 rounding of the sample coordinates.
3. The workspace query of the default forward covers the exact-kernel fallback of a channels-last call.
"""
import numpy as np
import pytest
import torch
import torchvision

from oracle import roi_align_f64 as rf

ADVERSARIAL = np.array([[0, -500, -500, -100, -100], [1, 100, 100, 100, 100], [0, 300, 300, 200, 250],
                        [1, 0, 0, 1200, 600], [0, 10.3, 20.7, 12.1, 22.9], [1, 1100, 500, 1400, 800]], np.float32)


def _rois(N, H, W, scale, aligned, sr, seed, sweep=40):
    b = rf.roi_set(H, W, scale, aligned, sr, seed, sweep=sweep, wide=20)
    n = np.random.default_rng(seed).integers(0, N, (len(b), 1)).astype(np.float32)
    return np.vstack([np.hstack([n, b]), ADVERSARIAL])


def _bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
def test_fp32_terms_in_torchvision_order_equal_torchvision_forward(aligned, sr):
    N, C, H, W, scale = 2, 5, 18, 37, 1 / 32
    rois = _rois(N, H, W, scale, aligned, sr, 3)
    x = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(4)) * 3 + 1
    ref = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr)
    tv = torchvision.ops.roi_align(x, torch.from_numpy(rois), (7, 7), scale, sr, aligned)
    assert _bits(ref.fp32_forward(x), tv.numpy())


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
def test_fp32_terms_in_torchvision_order_equal_torchvision_backward(aligned, sr):
    N, C, H, W, scale = 2, 3, 9, 13, 1 / 16
    rois = _rois(N, H, W, scale, aligned, sr, 5, sweep=12)
    rois[-6:, 1:] *= 0.5                                    # the adversarial ROIs of the 600 x 1200 image on this map
    g = torch.randn(len(rois), C, 7, 7, generator=torch.Generator().manual_seed(6))
    x = torch.zeros(N, C, H, W, requires_grad=True)
    torchvision.ops.roi_align(x, torch.from_numpy(rois), (7, 7), scale, sr, aligned).backward(g)
    ref = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr)
    assert _bits(ref.fp32_backward(g), x.grad.numpy())


def _dyadic_rois(N, H, W, scale, rng, n=120):
    """Starts on a 1/8 feature-pixel grid, bins of k/4 feature pixels with a power-of-two adaptive grid (k/4 <= 1, 2 or 4),
    so that every fp32 operation of the geometry is exact -- for aligned on and off, with sampling ratio 0 or 2."""
    bins = np.array([0.25, 0.5, 0.75, 1.0, 1.25, 1.5, 2.0, 3.25, 3.5, 4.0])
    sw = rng.integers(-24, 8 * W, n) / 8.0; sh = rng.integers(-24, 8 * H, n) / 8.0
    bw = rng.choice(bins, n); bh = rng.choice(bins, n)
    feat = np.stack([sw, sh, sw + 7 * bw, sh + 7 * bh], 1)
    return np.hstack([rng.integers(0, N, (n, 1)), feat / scale]).astype(np.float32)


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 2])
def test_float64_accumulation_equals_torchvision_float64_where_the_geometry_is_exact(aligned, sr):
    N, C, H, W, scale = 2, 6, 18, 37, 1 / 32
    rng = np.random.default_rng(7)
    rois = _dyadic_rois(N, H, W, scale, rng)
    x = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(8), dtype=torch.float64) * 10
    g = torch.randn(len(rois), C, 7, 7, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    r64 = torch.from_numpy(rois).double()
    xr = x.clone().requires_grad_(True)
    tv = torchvision.ops.roi_align(xr, r64, (7, 7), scale, sr, aligned)
    tv.backward(g)
    ref = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr)
    for rows, out, sc, _, _ in ref.forward(x):
        assert np.all(np.abs(out - tv.detach().numpy()[rows]) <= 1e-12 * sc)
    grad, sc, _, _ = ref.backward(g)
    assert np.all(np.abs(grad - xr.grad.numpy()) <= 1e-12 * sc)


def test_float64_reference_on_general_rois_is_limited_by_the_fp32_geometry():
    """Random ROIs (no sample within reach of a discontinuity): each fp32 sample coordinate is at most 4 roundings from the
    real one, |dv| <= 4 * 2^-24 * 2^ceil(log2(max(H, W) + 1)), and moves each bilinear weight by at most |dv|, so the bin
    average moves by at most 2 * |dv| * max|X| (two weights per axis, a convex combination)."""
    N, C, H, W, scale = 2, 4, 38, 75, 1 / 16
    rng = np.random.default_rng(10)
    b = rf.roi_set(H, W, scale, True, 0, 11, sweep=150, wide=40)[:190]
    rois = np.hstack([rng.integers(0, N, (len(b), 1)), b]).astype(np.float32)
    x = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(12), dtype=torch.float64)
    tv = torchvision.ops.roi_align(x, torch.from_numpy(rois).double(), (7, 7), scale, 0, True).numpy()
    dv = 4 * 2.0 ** -24 * 2.0 ** np.ceil(np.log2(max(H, W) + 1))
    bound = 2 * 2 * dv * float(x.abs().max())
    worst = 0.0
    for rows, out, _, _, _ in rf.RoiAlignF64(rois, N, H, W, scale, True, 0).forward(x):
        worst = max(worst, float(np.abs(out - tv[rows]).max()))
    assert worst <= bound, (worst, bound)


def test_window_classes_follow_the_table_kernel_rule():
    """Hand-checked windows: a bin of 0.5 pixel (one sample, two columns), of 2 pixels (two samples 1 apart: three columns),
    a 5-pixel bin with five samples (six columns), and a bin wider than the map (dense tables)."""
    rois = np.array([[0, 8.25, 1, 11.75, 3], [0, 2.0, 1, 16.0, 3], [0, 0.5, 1, 35.5, 3], [0, -40, 1, 60, 3]], np.float32)
    ref = rf.RoiAlignF64(rois, 1, 6, 37, 1.0, False, 0)
    assert ref.nx.tolist() == [2, 3, 6, rf.DENSE]


def test_roi_align_workspace_covers_the_exact_fallback_of_a_channels_last_call():
    """A channels-last call whose shape the separable path does not take (C % 4 != 0, a map too large for its tables, or an
    output other than 7 x 7) runs the exact kernel on an NCHW copy made in the workspace: the size the default call asks for
    must hold that copy even for a handful of ROIs."""
    from sfod_b200 import _lib
    L = _lib.lib()
    NHWC = 1
    for N, C, H, W in ((2, 6, 18, 37), (1, 32, 400, 1300), (2, 512, 18, 37)):
        for R in (1, 5, 300):
            assert L.sfod_roi_align_fwd_workspace_bytes(N, C, H, W, R, NHWC, 0) >= N * C * H * W * 4, (N, C, H, W, R)
