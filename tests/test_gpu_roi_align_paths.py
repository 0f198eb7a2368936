"""Every ROIAlign forward and backward kernel of csrc/roi.cu against the float64 reference of oracle/roi_align_f64.py.

Each case declares the kernel instantiation it targets and asserts with torch.profiler that it ran, so a change to the
dispatch cannot move a case to another path unnoticed.  The ROI sets (oracle.roi_align_f64.roi_set) put samples exactly on
the discontinuities of the operator and one fp32 step either side of them, and cover every compact column window.

Criterion.  For every output element, with u = 2^-24, ``|got - ref| <= (m + c) * u * scale``: ref and scale = S . |X|
(forward) or S^T . |G| (backward) from the reference, m its term count.  The bound is a standard error analysis of the
kernels' summation structure; every term is non-negative-weighted, so relative perturbations of terms add up to an error
bounded by (their number of roundings) * u * scale, and gamma_n = n u / (1 - n u) <= (n + 1) u for n < 2^11.

* Weight tables (separable kernels).  Ad[y, ph] = sum over the samples of h * inv and l * inv with inv = fl(1 / g): every
  entry sums k <= K non-zero sample terms (each sample puts one non-zero weight on an entry: lo == hi only with l = 0), with
  a product and an addition (or one FMA) per term, so it carries a relative error <= gamma_{K + 1}; Bc / Bd likewise.
  K = sampling_ratio for a fixed grid.  For the adaptive grid (g = ceil(bin)) the samples are more than 1/2 pixel apart
  (bin / g > (g - 1) / g >= 1/2 for g >= 2), and an entry collects the samples within one pixel of its row, or the clamped
  ones in [-1, 0] / [size - 1, size] together with those within one pixel: K = 4.
* Forward (slab and L2 kernels, compact or dense columns).  out[ph, pw] = sum_y Ad[y, ph] * T[y, pw] with T[y, pw] =
  sum_x Bc[pw, x] * X[y, x], both FMA chains; zero weights add exact zeros.  A term passes n_x roundings in T and n_y in the
  row chain, where n_x, n_y are the non-zero columns / rows of the bin, and m = n_x * n_y >= n_x + n_y - 1.  Per term:
  (m + 1) + 2 (K + 1) roundings, plus one for gamma:  c_fwd = 2 K + 4.
* Backward (separable).  Per ROI and row, U[pw] = sum over the bins of the row's pass of Ad * gOut (FMA chain), then
  v = sum_pw Bd[x, pw] * U[pw] (product + FMA chain), and one float atomic per (ROI, pass, pixel) in any order: a sum of p
  values in any order is within gamma_{p - 1} of their sum.  A pixel's m = sum over ROIs of n_a * n_b, and the two register
  passes give a ROI at most two atomics per pixel, so n_a + n_b + p - 1 <= m + 2; with the tables and gamma:  c_bwd = 2 K + 5.
* Generic backward.  Per sample corner: fl(hy * hx), fl(go * w), fl(/ count), then one atomic: m counts the sample corners
  (``terms``) and a term sees 3 + (m - 1) roundings: c = 3 (plus one for gamma).
* Exact forward.  Per sample: four products of fl(hy * hx) and the pixel, three additions, one addition to val, then / count:
  m counts sample corners and a term sees at most 2 + 3 + n_s + 1 <= m + 6 roundings: c = 7.  The exact kernel is also
  bit-equal to torchvision.

The sensitivity tests run the same criterion on outputs computed with ROIs shifted by 2^-6 feature pixel, with ``aligned``
flipped and with the sampling ratio increased by one, and require it to reject each of them, for every kernel family.
"""
import time

import numpy as np
import pytest
import torch
import torchvision
from torch.profiler import ProfilerActivity, profile

from oracle import roi_align_f64 as rf
import sfod_b200  # noqa: F401

pytestmark = pytest.mark.gpu

U = 2.0 ** -24


def _K(sr):
    return 4 if sr <= 0 else sr


C_EXACT, C_GENERIC = 7, 4


def c_fwd(sr):
    return 2 * _K(sr) + 4


def c_bwd(sr):
    return 2 * _K(sr) + 5


@pytest.fixture(scope="module")
def ops(cuda_device):
    return sfod_b200.ops


@pytest.fixture(scope="module")
def sms(cuda_device):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _profiled(fn):
    """Runs fn under torch.profiler (CUDA activity) and returns (result, names of the CUDA kernels that ran).  The call is
    made once before the profiler starts (lazy module loading) and twice under it: a call that launches a single kernel
    cold can go unrecorded."""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        out = fn()
        torch.cuda.synchronize()
    return out, {e.name for e in prof.events()}


def _assert_ran(names, target, what):
    hits = sorted(n for n in names if target in n)
    assert hits, f"{what}: no kernel named {target!r} ran; ROI kernels seen: {sorted(n for n in names if 'roi' in n)}"
    return hits[0]


class _Check:
    """The criterion, accumulated over chunks: ok, and the largest err / (u * scale)."""

    def __init__(self):
        self.ok, self.worst = True, 0.0

    def add(self, got, ref, scale, m, c):
        err = np.abs(np.asarray(got, np.float64) - ref)
        self.ok &= bool(np.all(err <= (m + c) * U * scale))
        pos = scale > 0
        if pos.any():
            self.worst = max(self.worst, float((err[pos] / (U * scale[pos])).max()))
        return self


def _rois(N, H, W, scale, aligned, sr, seed, empty=(), extra=0):
    """The ROI set of the map (oracle.roi_align_f64.roi_set) over the images not in ``empty``, followed by ``extra`` random
    filler ROIs (they only make the launch bigger).  Returns (rois (R, 5) float32, number of designed rows)."""
    rng = np.random.default_rng(seed)
    imgs = np.setdiff1d(np.arange(N), np.asarray(empty, np.int64))
    # the 400 x 1300 map: fewer ROIs, since a map-sized one there has bins of 69 x 223 samples
    b = rf.roi_set(H, W, scale, aligned, sr, seed, **(dict(sweep=60, wide=40) if H * W > 100_000 else {}))
    parts = [np.hstack([rng.choice(imgs, (len(b), 1)).astype(np.float32), b])]
    if extra:
        wh = rng.uniform(0.3, 0.9, (extra, 2)) ** 2 * np.array([W, H]) + 0.2
        c0 = rng.uniform(0, 1, (extra, 2)) * np.array([W, H])
        fb = np.hstack([c0 - wh / 2, c0 + wh / 2]) / scale
        parts.append(np.hstack([rng.choice(imgs, (extra, 1)), fb]).astype(np.float32))
    return np.vstack(parts), len(b)


def _features(N, C, H, W, seed):
    """Normal values with magnitudes spread over four decades, so that small and large bins sit side by side."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, C, H, W, generator=g) * torch.exp(torch.rand(N, 1, H, W, generator=g) * 9.2 - 4.6)


# ------------------------------------------------------------------------------------------------ forward
FWD_CASES = {
    # id: (N, C, H, W, stride, kernel for NCHW, kernel for channels-last, extra ROIs, images without ROIs)
    "slab16": (2, 512, 18, 37, 32, "roi_align_fwd_slab_kernel<16, 33>", "roi_align_fwd_slab_kernel<16, 32>", 0, ()),
    "slab8": (4, 512, 25, 42, 32, "roi_align_fwd_slab_kernel<8, 33>", "roi_align_fwd_slab_kernel<8, 32>", 0, ()),
    "many_images": (70, 32, 8, 12, 32, "roi_align_fwd_slab_kernel<16, 33>", "roi_align_fwd_slab_kernel<16, 32>", 0, (5, 33, 40, 69)),
    "too_many_images": (1025, 32, 8, 12, 32, "roi_align_fwd_sep_kernel<0>", "roi_align_fwd_sep_kernel<0>", 0, ()),
    "l2_256": (2, 256, 38, 75, 16, "roi_align_fwd_sep_kernel<256>", "roi_align_fwd_sep_kernel<256>", 0, ()),
    "l2_512": (2, 512, 38, 75, 16, "roi_align_fwd_sep_kernel<512>", "roi_align_fwd_sep_kernel<512>", 0, ()),
    "l2_2048": (1, 2048, 38, 75, 16, "roi_align_fwd_sep_kernel<2048>", "roi_align_fwd_sep_kernel<2048>", 0, ()),
    "partial_slab": (2, 260, 38, 75, 16, "roi_align_fwd_sep_kernel<0>", "roi_align_fwd_sep_kernel<0>", 0, ()),
    "r101_lpt": (2, 1024, 38, 75, 16, "roi_align_fwd_sep_kernel<1024>", "roi_align_fwd_sep_kernel<1024>", 0.5, ()),
    "r101_arrival": (8, 1024, 38, 75, 16, "roi_align_fwd_sep_kernel<1024>", "roi_align_fwd_sep_kernel<1024>", 2.0, ()),
    "exact_c6": (2, 6, 18, 37, 32, "roi_align_fwd_exact_kernel", "roi_align_fwd_exact_kernel", 0, ()),
    "exact_big_map": (1, 32, 400, 1300, 4, "roi_align_fwd_exact_kernel", "roi_align_fwd_exact_kernel", 0, ()),
}
WINDOW_CLASSES = (2, 3, 4, 6, 8, rf.DENSE)


def _run_forward_case(ops, dev, name, sms, configs, report):
    N, C, H, W, stride, k_nchw, k_cl, extra, empty = FWD_CASES[name]
    scale = 1.0 / stride
    exact = "exact" in k_nchw
    nslab = -(-C // 256)
    x = _features(N, C, H, W, sum(map(ord, name)))
    xd = x.to(dev)
    xcl = xd.contiguous(memory_format=torch.channels_last)
    for ci, (aligned, sr) in enumerate(configs):
        n_extra = 0
        if isinstance(extra, float):      # R * ceil(C / 256) at the given multiple of the cost-order threshold 64 * 3 * SMs
            n_extra = int(extra * 64 * 3 * sms / nslab) + 1
        rois, n_design = _rois(N, H, W, scale, aligned, sr, 100 + ci, empty=empty)
        if n_extra:
            rois, n_design = _rois(N, H, W, scale, aligned, sr, 100 + ci, empty=empty, extra=max(n_extra - n_design, 0))
            items = len(rois) * nslab
            assert (items < 64 * 3 * sms) == (extra < 1), "the case must sit on its side of the cost-order threshold"
        rd = torch.from_numpy(rois).to(dev)
        call = lambda inp, r=rd, a=aligned, s=sr: ops.roi_align(inp, r, (7, 7), scale, s, a)
        if ci == 0:
            out, names = _profiled(lambda: call(xd))
            kn = _assert_ran(names, k_nchw, f"{name} NCHW")
            out_cl, names = _profiled(lambda: call(xcl))
            kc = _assert_ran(names, k_cl, f"{name} channels-last")
            report.append(f"{name}: NCHW ran {kn.split('(')[0]}; channels-last ran {kc.split('(')[0]}")
        else:
            out, out_cl = call(xd), call(xcl)
        assert torch.equal(out_cl, out), f"{name}: channels-last and NCHW inputs differ"
        assert torch.equal(call(xd), out), f"{name}: two calls differ (the forward has no atomics)"
        perm = torch.from_numpy(np.random.default_rng(ci).permutation(len(rois))).to(dev)
        assert torch.equal(call(xd, rd[perm]), out[perm]), f"{name}: shuffled ROI / image order changes results"
        bad = rd.clone(); bad[::7, 0] = float(N + 2); bad[3::11, 0] = -1.0
        inval = (bad[:, 0] < 0) | (bad[:, 0] >= N)
        ob = call(xd, bad)
        assert torch.count_nonzero(ob[inval]) == 0 and torch.equal(ob[~inval], out[~inval]), f"{name}: invalid image index"
        # the reference: every row, or the designed ROIs and a seeded sample of the filler (each row depends on its ROI only)
        idx = np.arange(len(rois))
        if len(rois) > 1200:
            rng = np.random.default_rng(ci)
            idx = np.concatenate([np.arange(n_design), n_design + rng.choice(len(rois) - n_design, 100, replace=False)])
        ref = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr)
        if not exact:
            nxs = ref.nx[idx]
            few = {k: int((nxs == k).sum()) for k in WINDOW_CLASSES if (nxs == k).sum() < 20}
            assert not few, f"{name}: fewer than 20 ROIs of window classes {few}"
        got = out[torch.from_numpy(idx).to(dev)].cpu().numpy()
        pos = {r: i for i, r in enumerate(idx)}
        chk = _Check()
        for rows, rv, sc, nnz, terms in ref.forward(x, idx):
            g = got[[pos[r] for r in rows]]
            if exact:
                chk.add(g, rv, sc, terms, C_EXACT)
            else:
                chk.add(g, rv, sc, nnz, c_fwd(sr))
        report.append(f"  {name} aligned={aligned} sr={sr} R={len(rois)}: max err/(u*scale) {chk.worst:.2f}")
        assert chk.ok, f"{name} aligned={aligned} sr={sr}: error above (m + c) u scale (max ratio {chk.worst:.2f})"
        if exact:
            tv = torchvision.ops.roi_align(x, torch.from_numpy(rois), (7, 7), scale, sr, aligned)
            assert torch.equal(out.cpu(), tv), f"{name}: exact fallback must be bit-equal to torchvision"
    return xd, x


ALL_CONFIGS = [(True, 0), (True, 2), (False, 0), (False, 2)]


@pytest.mark.parametrize("name", list(FWD_CASES))
def test_roi_align_forward_path(ops, cuda_device, sms, name):
    t0 = time.time()
    report = []
    _run_forward_case(ops, cuda_device, name, sms, ALL_CONFIGS, report)
    print("\n" + "\n".join(report) + f"\n  {name}: {time.time() - t0:.1f} s")


# ------------------------------------------------------------------------------------------------ backward
BWD_CASES = {
    # id: (N, C, H, W, stride, (PH, PW), kernel, layouts, configs); one more image without any ROI is appended
    "bwd_sep512": (2, 512, 18, 37, 32, (7, 7), "roi_align_bwd_sep_kernel<512>", ("nchw", "nhwc"), ALL_CONFIGS[:1] + ALL_CONFIGS[3:]),
    "bwd_r101": (2, 1024, 38, 75, 16, (7, 7), "roi_align_bwd_sep_kernel<1024>", ("nhwc",), ALL_CONFIGS[:1]),
    "bwd_sep256": (2, 256, 38, 75, 16, (7, 7), "roi_align_bwd_sep_kernel<256>", ("nhwc",), ALL_CONFIGS[:1]),
    "bwd_sep2048": (1, 2048, 38, 75, 16, (7, 7), "roi_align_bwd_sep_kernel<2048>", ("nhwc",), ALL_CONFIGS[:1]),
    "bwd_sep260": (2, 260, 38, 75, 16, (7, 7), "roi_align_bwd_sep_kernel<0>", ("nchw",), ALL_CONFIGS[:1]),
    "bwd_generic_big_map": (1, 32, 400, 1300, 4, (7, 7), "roi_align_bwd_generic_kernel", ("nchw",), ALL_CONFIGS[:1]),
    "bwd_generic_5x3": (2, 16, 18, 37, 32, (5, 3), "roi_align_bwd_generic_kernel", ("nchw", "nhwc"), ALL_CONFIGS[3:]),
}


def _stacked(H, W, scale, n, rng):
    """n ROIs over the same few pixels of image 0 (atomic contention on every pixel of the region)."""
    c = np.array([W * 0.4, H * 0.45]); half = rng.uniform(0.5, 3.0, (n, 2)) + rng.uniform(0, 0.01, (n, 1))
    return np.hstack([np.zeros((n, 1)), np.hstack([c - half, c + half]) / scale]).astype(np.float32)


def _backward(ops, xd, rd, g, ph_pw, scale, sr, aligned):
    xd = xd.detach().clone().requires_grad_(True)
    ops.roi_align(xd, rd, ph_pw, scale, sr, aligned).backward(g)
    return xd.grad


@pytest.mark.parametrize("name", list(BWD_CASES))
def test_roi_align_backward_path(ops, cuda_device, name):
    t0 = time.time()
    N, C, H, W, stride, ph_pw, kern, layouts, configs = BWD_CASES[name]
    generic = "generic" in kern
    scale = 1.0 / stride
    Nt = N + 1                                                      # image N gets no ROI
    x = torch.zeros(Nt, C, H, W, device=cuda_device)
    report = []
    for ci, (aligned, sr) in enumerate(configs):
        rng = np.random.default_rng(200 + ci)
        rois, _ = _rois(N, H, W, scale, aligned, sr, 200 + ci, extra=1300 if name == "bwd_r101" else 0)
        rois = np.vstack([rois, _stacked(H, W, scale, 300, rng)])
        rd = torch.from_numpy(rois).to(cuda_device)
        g = torch.randn(len(rois), C, *ph_pw, generator=torch.Generator().manual_seed(ci))
        gd = g.to(cuda_device)
        ref = rf.RoiAlignF64(rois, Nt, H, W, scale, aligned, sr, *ph_pw)
        grad, sc, nnz, terms = ref.backward(g)
        grads = []
        for layout in layouts:
            xl = x if layout == "nchw" else x.contiguous(memory_format=torch.channels_last)
            if ci == 0:
                gr, names = _profiled(lambda: _backward(ops, xl, rd, gd, ph_pw, scale, sr, aligned))
                report.append(f"{name} {layout}: ran {_assert_ran(names, kern, f'{name} {layout}').split('(')[0]}")
            else:
                gr = _backward(ops, xl, rd, gd, ph_pw, scale, sr, aligned)
            got = gr.cpu().numpy()
            assert not np.any(got[N]), f"{name}: an image without ROIs must get a zero gradient"
            chk = _Check().add(got, grad, sc, terms if generic else nnz, C_GENERIC if generic else c_bwd(sr))
            report.append(f"  {name} {layout} aligned={aligned} sr={sr} R={len(rois)}: max err/(u*scale) {chk.worst:.2f}")
            assert chk.ok, f"{name} {layout} aligned={aligned} sr={sr}: error above (m + c) u scale (max ratio {chk.worst:.2f})"
            grads.append(got)
    # no ROI at all: a zero gradient
    xr = x.detach().clone().requires_grad_(True)
    y = ops.roi_align(xr, torch.zeros(0, 5, device=cuda_device), ph_pw, scale, 0, True)
    y.backward(torch.zeros_like(y))
    assert xr.grad is not None and torch.count_nonzero(xr.grad) == 0
    print("\n" + "\n".join(report) + f"\n  {name}: {time.time() - t0:.1f} s")


# ------------------------------------------------------------------------------------------------ sensitivity
def _perturbed(rois, scale):
    shifted = rois.copy()
    shifted[:, 1:] = (shifted[:, 1:].astype(np.float64) + 2.0 ** -6 / scale).astype(np.float32)
    return shifted


@pytest.mark.parametrize("name", ["slab16", "l2_512", "exact_c6"])
def test_forward_criterion_rejects_wrong_answers(ops, cuda_device, name):
    """Shifted ROIs, flipped ``aligned`` and a sampling ratio one higher each fail the forward criterion, per kernel family."""
    N, C, H, W, stride, _, _, _, _ = FWD_CASES[name]
    scale, aligned, sr = 1.0 / stride, True, 0
    x = _features(N, C, H, W, 5)
    xd = x.to(cuda_device)
    rois, _ = _rois(N, H, W, scale, aligned, sr, 300)
    ref = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr)
    c = C_EXACT if "exact" in name else c_fwd(sr)
    wrong = {"shifted 2^-6 pixel": (_perturbed(rois, scale), aligned, sr), "aligned flipped": (rois, not aligned, sr),
             "sampling ratio + 1": (rois, aligned, sr + 1)}
    right = ops.roi_align(xd, torch.from_numpy(rois).to(cuda_device), (7, 7), scale, sr, aligned).cpu().numpy()
    for what, (r, a, s) in [("unperturbed", (rois, aligned, sr))] + list(wrong.items()):
        got = right if what == "unperturbed" else \
            ops.roi_align(xd, torch.from_numpy(r).to(cuda_device), (7, 7), scale, s, a).cpu().numpy()
        chk = _Check()
        for rows, rv, sc, nnz, terms in ref.forward(x):
            chk.add(got[rows], rv, sc, terms if "exact" in name else nnz, c)
        print(f"{name} {what}: max err/(u*scale) {chk.worst:.3g}")
        assert chk.ok == (what == "unperturbed"), f"{name}: the criterion {'rejects' if not chk.ok else 'accepts'} {what}"


@pytest.mark.parametrize("name", ["bwd_sep512", "bwd_generic_5x3"])
def test_backward_criterion_rejects_wrong_answers(ops, cuda_device, name):
    N, C, H, W, stride, ph_pw, kern, _, _ = BWD_CASES[name]
    scale, aligned, sr = 1.0 / stride, True, 0
    rois, _ = _rois(N, H, W, scale, aligned, sr, 400)
    g = torch.randn(len(rois), C, *ph_pw, generator=torch.Generator().manual_seed(4))
    gd, rd = g.to(cuda_device), torch.from_numpy(rois).to(cuda_device)
    x = torch.zeros(N, C, H, W, device=cuda_device)
    grad, sc, nnz, terms = rf.RoiAlignF64(rois, N, H, W, scale, aligned, sr, *ph_pw).backward(g)
    m, c = (terms, C_GENERIC) if "generic" in kern else (nnz, c_bwd(sr))
    cases = [("unperturbed", rd, aligned, sr), ("shifted 2^-6 pixel", torch.from_numpy(_perturbed(rois, scale)).to(cuda_device), aligned, sr),
             ("aligned flipped", rd, not aligned, sr), ("sampling ratio + 1", rd, aligned, sr + 1)]
    for what, r, a, s in cases:
        got = _backward(ops, x, r, gd, ph_pw, scale, s, a).cpu().numpy()
        chk = _Check().add(got, grad, sc, m, c)
        print(f"{name} {what}: max err/(u*scale) {chk.worst:.3g}")
        assert chk.ok == (what == "unperturbed"), f"{name}: the criterion {'rejects' if not chk.ok else 'accepts'} {what}"
