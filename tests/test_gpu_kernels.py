"""GPU parity tests: every CUDA entry point (through the C ABI via sfod_b200.ops) against the CPU oracle
on the same seeded inputs.  Integer results (keep indices, top-k indices, classes, rows, counts) must be
bit-exact; floating-point results match within the tolerance stated in each test (BASELINE.json: 1e-5
relative fp32; where the CUDA arithmetic is *defined* identically to the oracle's we assert equality)."""
import numpy as np
import pytest
import torch
import torchvision

from oracle import d2_cpu as o
import sfod_b200  # noqa: F401
from sfod_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops(cuda_device):
    import sfod_b200
    return sfod_b200.ops


def _bits_equal(got: torch.Tensor, ref: torch.Tensor) -> bool:
    """Bit-exact fp32 equality; NaNs match NaNs regardless of payload (-0.0 != +0.0 is enforced)."""
    g, r = got.detach().cpu().contiguous().numpy(), ref.detach().cpu().contiguous().numpy()
    nan = np.isnan(r)
    return bool(np.array_equal(np.isnan(g), nan) and np.array_equal(g.view(np.uint32)[~nan], r.view(np.uint32)[~nan]))


def _close(a, b, rtol=1e-5, atol_scale=1e-5):
    a = a.detach().cpu().double(); b = b.detach().cpu().double()
    scale = max(float(b.abs().max()), 1e-30) if b.numel() else 1.0
    assert a.shape == b.shape, (a.shape, b.shape)
    err = (a - b).abs()
    tol = atol_scale * scale + rtol * b.abs()
    assert bool((err <= tol).all()), f"max err {float(err.max()):.3e} (scale {scale:.3e})"


# ------------------------------------------------------------------------------------------------ EMA
@pytest.mark.parametrize("keep_rate", [0.9996, 0.999696, 0.0])
def test_ema_multi_tensor_bit_exact(ops, cuda_device, keep_rate):
    g = torch.Generator().manual_seed(7)
    shapes = [(64,), (64, 3, 3, 3), (1,), (7,), (1000003,), (512, 512, 3, 3), (33, 5), (4099,)]
    student = {f"p{i}": torch.randn(s, generator=g) for i, s in enumerate(shapes)}
    teacher = {f"p{i}": torch.randn(s, generator=g) for i, s in enumerate(shapes)}
    student["nbt"] = torch.tensor(1000, dtype=torch.int64); teacher["nbt"] = torch.tensor(1000, dtype=torch.int64)
    student["nbt2"] = torch.tensor([5, 0, 123456789], dtype=torch.int64); teacher["nbt2"] = torch.tensor([7, 3, 123456000], dtype=torch.int64)
    student["p0"][3] = float("nan"); teacher["p1"].view(-1)[5] = -0.0; student["p1"].view(-1)[5] = 0.0
    ref_t = {k: v.clone() for k, v in teacher.items()}
    o.load_state_dict_like(ref_t, o.update_teacher_model(student, ref_t, keep_rate))
    sd = {k: v.to(cuda_device) for k, v in student.items()}
    td = {k: v.to(cuda_device) for k, v in teacher.items()}
    plan = ops.EmaPlan([(sd[k], td[k]) for k in td])
    plan.step(keep_rate)
    torch.cuda.synchronize()
    for k in td:
        got, ref = td[k].cpu(), ref_t[k]
        if got.dtype == torch.float32:
            assert _bits_equal(got, ref), k
        else:
            assert torch.equal(got, ref), k
    # second step keeps matching (state carried on the device)
    o.load_state_dict_like(ref_t, o.update_teacher_model(student, ref_t, keep_rate))
    plan.step(keep_rate)
    assert _bits_equal(td["p4"], ref_t["p4"])


# ------------------------------------------------------------------------------------------------ NMS
@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 500, 2000, 4000, 9990])
@pytest.mark.parametrize("kind", ["low", "high"])
def test_nms_bit_exact(ops, cuda_device, n, kind):
    if kind == "low":
        b, s = synth.boxes_low_suppression(synth.V, n, 1234)
    else:
        b, s = synth.boxes_high_suppression(n, 1234)
    n = b.shape[0]
    for thr in (0.7, 0.5):
        ref = torchvision.ops.nms(b, s, thr)
        got = ops.nms(b.to(cuda_device), s.to(cuda_device), thr).cpu()
        assert torch.equal(got, ref), f"n={n} thr={thr}: {got.numel()} vs {ref.numel()} kept"


def test_nms_large_multi_tile_sort(ops, cuda_device):
    b, s = synth.boxes_high_suppression(20000, 99, clusters=600)
    ref = torchvision.ops.nms(b, s, 0.7)
    got = ops.nms(b.to(cuda_device), s.to(cuda_device), 0.7).cpu()
    assert torch.equal(got, ref)


def test_nms_semantics_kats(ops, cuda_device):
    """SURVEY.md B-1: ties keep the lowest index; degenerate boxes (IoU NaN) are never suppressed; strict >."""
    d = cuda_device
    b = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 10], [20, 20, 30, 30], [20, 20, 30, 30]], dtype=torch.float32)
    s = torch.ones(4)
    assert ops.nms(b.to(d), s.to(d), 0.5).cpu().tolist() == [0, 2]
    b = torch.tensor([[5, 5, 5, 5], [5, 5, 5, 5], [0, 0, 10, 10]], dtype=torch.float32)
    assert ops.nms(b.to(d), torch.tensor([0.9, 0.8, 0.7]).to(d), 0.5).cpu().tolist() == [0, 1, 2]
    b = torch.tensor([[0, 0, 10, 10], [0, 0, 10, 5]], dtype=torch.float32)  # IoU exactly 0.5
    assert ops.nms(b.to(d), torch.tensor([0.9, 0.8]).to(d), 0.5).cpu().tolist() == [0, 1]
    assert ops.nms(torch.zeros(0, 4, device=d), torch.zeros(0, device=d), 0.5).numel() == 0
    with pytest.raises(ValueError):
        ops.nms(torch.zeros(3, 5, device=d), torch.zeros(3, device=d), 0.5)
    with pytest.raises(RuntimeError):
        ops.nms(torch.zeros(3, 4), torch.zeros(3), 0.5)  # CPU tensors: no fallback


@pytest.mark.parametrize("thr,num,den", [(0.5, 1.0, 3.0), (0.7, 3.0, 17.0)])
def test_nms_decisions_at_the_threshold(ops, cuda_device, thr, num, den):
    """Pairs of equal boxes shifted by w * num / den have IoU = (w - dx) / (w + dx) = thr in exact arithmetic; in fp32 they
    land a few ulps on either side of it.  The kernels decide `fl(inter / union) > thr` without dividing when inter is
    far from thr * union and with the exact division otherwise: the keep set must still be torchvision's, pair by pair."""
    g = torch.Generator().manual_seed(77)
    P = 3000
    w = torch.rand(P, generator=g) * 200 + 10
    h = torch.rand(P, generator=g) * 200 + 10
    x0 = torch.rand(P, generator=g) * 50
    y0 = torch.rand(P, generator=g) * 50
    dx = w * num / den
    # second half: just OUTSIDE the band in which the exact division runs (relative distance 2e-6 .. 3e-5, both sides)
    eps = 10.0 ** (torch.rand(P, generator=g) * 1.2 - 5.7) * (torch.randint(0, 2, (P,), generator=g) * 2 - 1)
    eps[: P // 2] = 0.0
    dx = dx * (1.0 + eps)
    a = torch.stack([x0, y0, x0 + w, y0 + h], 1)
    b = torch.stack([x0 + dx, y0, x0 + dx + w, y0 + h], 1)
    boxes = torch.cat([a, b]).contiguous()
    scores = torch.cat([torch.full((P,), 0.9), torch.full((P,), 0.8)]) + torch.arange(2 * P) * 1e-6
    idx = torch.cat([torch.arange(P), torch.arange(P)])
    ref = o.batched_nms(boxes, scores, idx, thr)
    suppressed = 2 * P - ref.numel()
    assert 0.05 * P < suppressed < 0.95 * P, f"the construction must straddle the threshold ({suppressed} of {P} pairs suppressed)"
    got = ops.batched_nms(boxes.to(cuda_device), scores.to(cuda_device), idx.to(cuda_device), thr).cpu()
    assert torch.equal(got, ref)
    # the same pairs as one segment each of the plain operator (class-unaware kernels): shift pairs apart instead
    sub = slice(0, 400)
    off = (torch.arange(400, dtype=torch.float32) * 512.0)[:, None] * torch.tensor([1.0, 0.0, 1.0, 0.0])
    bb = torch.cat([a[sub] + off, b[sub] + off]).contiguous()
    ss = torch.cat([scores[:P][sub], scores[P:][sub]])
    assert torch.equal(ops.nms(bb.to(cuda_device), ss.to(cuda_device), thr).cpu(), torchvision.ops.nms(bb, ss, thr))


@pytest.mark.parametrize("n", [900, 1000, 1001, 6000])
def test_batched_nms_matches_torchvision_cpu_strategy(ops, cuda_device, n):
    """n <= 1000 -> coordinate trick arithmetic, above -> per-class (SURVEY.md B-2)."""
    b, s = synth.boxes_high_suppression(n, 5, clusters=60)
    g = torch.Generator().manual_seed(3)
    idx = torch.randint(0, 8, (n,), generator=g)
    ref = o.batched_nms(b, s, idx, 0.5)
    got = ops.batched_nms(b.to(cuda_device), s.to(cuda_device), idx.to(cuda_device), 0.5).cpu()
    assert torch.equal(got, ref)


# ------------------------------------------------------------------------------------------------ ROIAlign / ROIPool
@pytest.mark.parametrize("cfg", [synth.V, synth.R101], ids=["V", "R"])
@pytest.mark.parametrize("aligned", [True, False])
def test_roi_align_forward(ops, cuda_device, cfg, aligned):
    N, R = 2, 300
    x = synth.features(cfg, N, 11)
    rois = synth.random_rois(N, R, 12)
    # a few adversarial rois: outside the image, zero / negative size, whole image, tiny
    extra = torch.tensor([[0, -500, -500, -100, -100], [1, 100, 100, 100, 100], [0, 300, 300, 200, 250],
                          [1, 0, 0, 1200, 600], [0, 10.3, 20.7, 12.1, 22.9], [1, 1100, 500, 1400, 800]], dtype=torch.float32)
    rois = torch.cat([rois, extra])
    scale = 1.0 / cfg["stride"]
    for sr in (0, 2):
        ref = torchvision.ops.roi_align(x, rois, (7, 7), scale, sr, aligned)
        xe = x.to(cuda_device); re_ = rois.to(cuda_device)
        exact = ops.roi_align(xe, re_, (7, 7), scale, sr, aligned, exact=True).cpu()
        assert _bits_equal(exact, ref), "exact kernel must be bit-exact"
        fast = ops.roi_align(xe, re_, (7, 7), scale, sr, aligned).cpu()
        _close(fast, ref)
        fast_cl = ops.roi_align(xe.contiguous(memory_format=torch.channels_last), re_, (7, 7), scale, sr, aligned).cpu()
        assert torch.equal(fast_cl, fast), "NHWC input must give the same result as the internally transposed NCHW input"


def test_roi_align_kat_and_api(ops, cuda_device):
    """SURVEY.md B-3 known answers + torchvision API forms (list of boxes, other output sizes)."""
    d = cuda_device
    x = torch.arange(25, dtype=torch.float32).reshape(1, 1, 5, 5).to(d)
    rois = torch.tensor([[0, 1, 1, 3, 3]], dtype=torch.float32).to(d)
    a = ops.roi_align(x, rois, (4, 4), 1.0, 0, False).cpu().reshape(4, 4)
    assert a.tolist() == [[7.5, 8, 8.5, 9], [10, 10.5, 11, 11.5], [12.5, 13, 13.5, 14], [15, 15.5, 16, 16.5]]
    a = ops.roi_align(x, rois, (4, 4), 1.0, 0, True).cpu().reshape(4, 4)
    assert a.tolist() == [[4.5, 5, 5.5, 6], [7, 7.5, 8, 8.5], [9.5, 10, 10.5, 11], [12, 12.5, 13, 13.5]]
    p = ops.roi_pool(x, rois, (2, 2), 1.0).cpu().reshape(2, 2)
    assert p.tolist() == [[12, 13], [17, 18]]
    xs = torch.randn(2, 8, 20, 30)
    bl = [torch.tensor([[1.0, 2.0, 15.0, 12.0]]), torch.tensor([[0.0, 0.0, 29.0, 19.0], [3.0, 3.0, 9.0, 9.0]])]
    ref = torchvision.ops.roi_align(xs, bl, 7, 1.0, 0, True)
    got = ops.roi_align(xs.to(d), [b.to(d) for b in bl], 7, 1.0, 0, True).cpu()
    _close(got, ref)
    assert ops.roi_align(xs.to(d), torch.zeros(0, 5, device=d), 7).shape == (0, 8, 7, 7)
    # maps narrower than the compact column window (dense-table fallback) and a partial 256-channel slab
    for shape in ((1, 4, 6, 3), (2, 260, 9, 2), (1, 12, 3, 40)):
        xn = torch.randn(*shape, generator=torch.Generator().manual_seed(sum(shape)))
        rn = torch.tensor([[0, 0.2, 0.4, shape[3] - 0.5, shape[2] - 0.7], [shape[0] - 1, 0.0, 0.0, 1.0, 1.0],
                           [0, -3.0, -2.0, shape[3] + 4.0, shape[2] + 1.0], [0, 1.2, 1.1, 1.3, 1.15]], dtype=torch.float32)
        for sr in (0, 3):
            _close(ops.roi_align(xn.to(d), rn.to(d), 7, 1.0, sr, True).cpu(), torchvision.ops.roi_align(xn, rn, 7, 1.0, sr, True))
    with pytest.raises(ValueError):
        ops.roi_align(xs.to(d), torch.zeros(3, 4, device=d), 7)


@pytest.mark.parametrize("cfg", [synth.V, synth.R101, dict(name="mid-even-W", C=48, H=40, W=50, stride=16)], ids=["V", "R", "mid"])
def test_roi_align_forward_any_image_order_and_invalid_index(ops, cuda_device, cfg):
    """The slab-resident forward (32-channel slab: V) serves the ROIs of one image at a time from shared memory; R101-C4 and
    the 40 x 50 map, whose slabs do not fit, run the persistent L2 forward.  ROIs must be accepted in any image order
    (detectron2 passes them grouped by image, torchvision's API does not require it), images without ROIs are skipped, and an
    out-of-range batch index yields zeros (library contract; torchvision reads out of bounds)."""
    N, R = (5, 700) if cfg["C"] <= 512 else (3, 260)
    x = synth.features(cfg, N, 51)
    rois = synth.random_rois(N, R, 52)
    rois[:, 0] = torch.randint(0, N, (R,), generator=torch.Generator().manual_seed(53)).float()
    rois[rois[:, 0] == 3, 0] = 1.0                      # image 3 has no ROI at all
    sc = 1.0 / cfg["stride"]
    if cfg["stride"] == 16 and cfg["W"] == 50:
        rois[:, 1::2] *= 50 * 16 / 1200.0; rois[:, 2::2] *= 40 * 16 / 600.0     # keep the boxes on the smaller map
    ref = torchvision.ops.roi_align(x, rois, (7, 7), sc, 0, True)
    got = ops.roi_align(x.to(cuda_device), rois.to(cuda_device), (7, 7), sc, 0, True).cpu()
    _close(got, ref)
    got_cl = ops.roi_align(x.to(cuda_device).contiguous(memory_format=torch.channels_last), rois.to(cuda_device), (7, 7), sc, 0, True).cpu()
    assert torch.equal(got_cl, got)
    bad = rois.clone(); bad[::7, 0] = float(N + 2); bad[3::11, 0] = -1.0
    got = ops.roi_align(x.to(cuda_device), bad.to(cuda_device), (7, 7), sc, 0, True).cpu()
    invalid = (bad[:, 0] < 0) | (bad[:, 0] >= N)
    assert torch.count_nonzero(got[invalid]) == 0
    _close(got[~invalid], ref[~invalid])


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_roi_align_backward(ops, cuda_device, layout):
    cfg = synth.V
    N, R = 2, 512
    x = synth.features(cfg, N, 21)
    rois = synth.random_rois(N, R, 22)
    g = torch.randn(R, cfg["C"], 7, 7, generator=torch.Generator().manual_seed(23))
    xr = x.clone().requires_grad_(True)
    torchvision.ops.roi_align(xr, rois, (7, 7), 1 / 32, 0, True).backward(g)
    xd = x.to(cuda_device)
    if layout == "nhwc":
        xd = xd.contiguous(memory_format=torch.channels_last)
    xd.requires_grad_(True)
    y = ops.roi_align(xd, rois.to(cuda_device), (7, 7), 1 / 32, 0, True)
    y.backward(g.to(cuda_device))
    _close(xd.grad, xr.grad, rtol=1e-5, atol_scale=1e-5)
    # generic (non 7x7) path
    xr2 = x[:, :16].clone().requires_grad_(True)
    g2 = torch.randn(R, 16, 5, 3, generator=torch.Generator().manual_seed(24))
    torchvision.ops.roi_align(xr2, rois, (5, 3), 1 / 32, 2, False).backward(g2)
    xd2 = x[:, :16].to(cuda_device).requires_grad_(True)
    ops.roi_align(xd2, rois.to(cuda_device), (5, 3), 1 / 32, 2, False).backward(g2.to(cuda_device))
    _close(xd2.grad, xr2.grad)


@pytest.mark.parametrize("sr", [0, 2])
def test_roi_align_backward_many_images(ops, cuda_device, sr):
    """ROIs in any image order, an image without ROIs (its gradient must be all zeros), wide bins with a fixed sampling
    ratio; NCHW and channels-last gradients agree."""
    cfg = synth.V
    N, R = 6, 600
    x = synth.features(cfg, N, 61)
    rois = synth.random_rois(N, R, 62)
    rois[rois[:, 0] == 4, 0] = 2.0
    g = torch.randn(R, cfg["C"], 7, 7, generator=torch.Generator().manual_seed(63))
    xr = x.clone().requires_grad_(True)
    torchvision.ops.roi_align(xr, rois, (7, 7), 1 / 32, sr, True).backward(g)
    xd = x.to(cuda_device).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    ops.roi_align(xd, rois.to(cuda_device), (7, 7), 1 / 32, sr, True).backward(g.to(cuda_device))
    _close(xd.grad.cpu(), xr.grad, rtol=1e-5, atol_scale=1e-5)
    assert torch.count_nonzero(xd.grad[4]) == 0
    xn = x.to(cuda_device).requires_grad_(True)                      # NCHW gradient: accumulated channels-last, transposed
    ops.roi_align(xn, rois.to(cuda_device), (7, 7), 1 / 32, sr, True).backward(g.to(cuda_device))
    _close(xn.grad.cpu(), xr.grad, rtol=1e-5, atol_scale=1e-5)


def test_roi_pool_forward_backward(ops, cuda_device):
    cfg = synth.V
    N, R = 2, 256
    x = synth.features(cfg, N, 31)[:, :64].contiguous()
    rois = synth.random_rois(N, R, 32)
    xr = x.clone().requires_grad_(True)
    ref = torchvision.ops.roi_pool(xr, rois, (7, 7), 1 / 32)
    g = torch.randn_like(ref)
    ref.backward(g)
    xd = x.to(cuda_device).requires_grad_(True)
    got = ops.roi_pool(xd, rois.to(cuda_device), (7, 7), 1 / 32)
    assert torch.equal(got.detach().cpu(), ref.detach()), "max pooling must be bit-exact"
    got.backward(g.to(cuda_device))
    _close(xd.grad, xr.grad)


# ------------------------------------------------------------------------------------------------ box decode / softmax
def test_apply_deltas_and_softmax_defined_arithmetic(ops, cuda_device):
    g = torch.Generator().manual_seed(41)
    R = 5000
    ctr = torch.rand(R, 2, generator=g) * 1000; wh = torch.rand(R, 2, generator=g) * 300 + 1
    boxes = torch.cat([ctr - wh / 2, ctr + wh / 2], 1)
    d = torch.randn(R, 32, generator=g) * 2
    d[0, 3] = 100.0  # clamp path
    got = ops.apply_deltas(d.to(cuda_device), boxes.to(cuda_device), (10, 10, 5, 5)).cpu()
    spec = o.apply_deltas(d, boxes, (10, 10, 5, 5), exp=o.exp_correctly_rounded)
    assert torch.equal(got, spec), "decode must equal the defined (correctly-rounded-exp) arithmetic bit for bit"
    _close(got, o.apply_deltas(d, boxes, (10, 10, 5, 5)), rtol=1e-5, atol_scale=0)  # vs ATen exp: <= 1 ulp on the exp term
    kat = ops.apply_deltas(torch.tensor([[0.1, -0.2, 0.3, 10.0]]).to(cuda_device), torch.tensor([[10.0, 20, 50, 100]]).to(cuda_device),
                           (1, 1, 1, 1)).cpu()[0].tolist()
    assert kat == [7.0028228759765625, -2456.000244140625, 60.99717712402344, 2544.000244140625]
    x = torch.randn(4000, 9, generator=g) * 4
    sm = ops.softmax_lastdim(x.to(cuda_device)).cpu()
    assert torch.equal(sm, o.softmax_defined(x))
    _close(sm, torch.softmax(x, -1), rtol=1e-5, atol_scale=0)


# ------------------------------------------------------------------------------------------------ RPN selection
def _head_layout(cfg, logits, deltas):
    """Undo the flatten of reference rpn.py:28-41: (N, HWA) -> (N, A, H, W), (N, HWA, 4) -> (N, 4A, H, W) as the head writes them."""
    N, H, W = logits.shape[0], cfg["H"], cfg["W"]
    A = logits.shape[1] // (H * W)
    return (logits.view(N, H, W, A).permute(0, 3, 1, 2).contiguous(),
            deltas.view(N, H, W, A, 4).permute(0, 3, 4, 1, 2).reshape(N, 4 * A, H, W).contiguous())


def _rpn_case(ops, dev, cfg, N, seed, pre, post, image_sizes, use_anchor_tensor=False, delta_std=0.5, native=False):
    logits, deltas, cell, anchors = synth.rpn_head_outputs(cfg, N, seed, delta_std)
    ref = o.rpn_predict_proposals([anchors], [logits], [deltas], image_sizes, 0.7, pre, post, 0.0, False,
                                  exp=o.exp_correctly_rounded)
    kw = dict(anchors=anchors.to(dev)) if use_anchor_tensor else dict(cell_anchors=cell, feat_hw=(cfg["H"], cfg["W"]), stride=cfg["stride"])
    lg_in, dl_in = _head_layout(cfg, logits, deltas) if native else (logits, deltas)
    boxes, lg, src, cnt, invalid = ops.rpn_select(lg_in.to(dev), dl_in.to(dev), image_sizes, pre_nms_topk=pre,
                                                  post_nms_topk=post, nms_thresh=0.7, **kw)
    cnt = cnt.cpu().tolist()
    assert invalid.cpu().tolist() == [0] * N
    for i in range(N):
        k = cnt[i]
        assert k == len(ref[i]["src_index"]), (i, k, len(ref[i]["src_index"]))
        assert torch.equal(src[i, :k].cpu(), ref[i]["src_index"]), f"image {i}: proposal index mismatch"
        assert torch.equal(boxes[i, :k].cpu(), ref[i]["proposal_boxes"])
        assert torch.equal(lg[i, :k].cpu(), ref[i]["objectness_logits"])
    return ref, (boxes, lg, src, cnt)


def test_rpn_select_vgg_teacher_train_mode(ops, cuda_device):
    _rpn_case(ops, cuda_device, synth.V, 2, 1234, 12000, 2000, [(600, 1200), (600, 1200)])


def test_rpn_select_vgg_eval_and_ragged_image_sizes(ops, cuda_device):
    _rpn_case(ops, cuda_device, synth.V, 3, 1235, 6000, 1000, [(600, 1200), (576, 1100), (300, 400)])


def test_rpn_select_explicit_anchor_tensor(ops, cuda_device):
    _rpn_case(ops, cuda_device, synth.V, 1, 1236, 12000, 2000, [(600, 1200)], use_anchor_tensor=True)


def test_rpn_select_r101_topk_12000_of_34200(ops, cuda_device):
    _rpn_case(ops, cuda_device, synth.R101, 1, 1237, 12000, 2000, [(600, 1200)])


@pytest.mark.parametrize("cfg_name,use_anchor_tensor", [("V", False), ("V", True), ("R101", False)])
def test_rpn_select_reads_the_head_outputs_as_they_lie(ops, cuda_device, cfg_name, use_anchor_tensor):
    """head_layout 1: (N, A, H, W) logits / (N, 4A, H, W) deltas straight from the RPN head's convolutions -- the permute
    copies of reference rpn.py:28-41 are folded into the key build and the top-k gather.  Same oracle, same bits; ragged
    image sizes; non-finite entries are counted at the same flattened positions."""
    cfg = getattr(synth, cfg_name)
    _rpn_case(ops, cuda_device, cfg, 3, 1241, 12000, 2000, [(600, 1200), (576, 1100), (300, 400)],
              use_anchor_tensor=use_anchor_tensor, native=True)
    logits, deltas, cell, anchors = synth.rpn_head_outputs(cfg, 1, 78)
    deltas[0, 5, 0] = float("inf"); logits[0, 9] = float("nan")
    kw = dict(cell_anchors=cell, feat_hw=(cfg["H"], cfg["W"]), stride=cfg["stride"], pre_nms_topk=12000, post_nms_topk=2000)
    flat = ops.rpn_select(logits.to(cuda_device), deltas.to(cuda_device), [(600, 1200)], **kw)
    lg4, dl4 = _head_layout(cfg, logits, deltas)
    nat = ops.rpn_select(lg4.to(cuda_device), dl4.to(cuda_device), [(600, 1200)], **kw)
    for a, b in zip(flat, nat):
        assert torch.equal(a, b)
    with pytest.raises(ValueError):
        ops.rpn_select(lg4.to(cuda_device), dl4[:, :-4].contiguous().to(cuda_device), [(600, 1200)], **kw)
    # channels-last head outputs (NHWC backbone): the flatten is a free view of that memory; same results, no copy of the inputs
    lg_cl = lg4.to(cuda_device).contiguous(memory_format=torch.channels_last)
    dl_cl = dl4.to(cuda_device).contiguous(memory_format=torch.channels_last)
    cl = ops.rpn_select(lg_cl, dl_cl, [(600, 1200)], **kw)
    for a, b in zip(flat, cl):
        assert torch.equal(a, b)


@pytest.mark.parametrize("H,W,sizes,ratios", [(1, 1, (64,), (1.0,)), (2, 3, (32, 64), (0.5, 1.0, 2.0)), (1, 40, (32,), (0.5, 2.0))])
@pytest.mark.parametrize("native", [False, True])
def test_rpn_select_tiny_maps_both_head_layouts(ops, cuda_device, H, W, sizes, ratios, native):
    """Degenerate feature maps (a single cell with a single anchor, fewer anchors than post_nms_topk, one row): the sort tile is
    mostly padding and every count is below the caps -- both head layouts equal the oracle bit for bit."""
    cfg = dict(name="tiny", C=8, H=H, W=W, stride=32, sizes=sizes, ratios=ratios, image=(32 * H, 32 * W))
    _rpn_case(ops, cuda_device, cfg, 2, 1300 + H * W, 12000, 2000, [(32 * H, 32 * W), (max(16, 32 * H - 7), max(16, 32 * W - 5))],
              native=native)


def test_rpn_select_high_suppression_and_reference_exp(ops, cuda_device):
    """Tiny deltas -> anchors at the same cell overlap heavily -> few survivors (count < post_nms_topk).
    Also compares with the reference-faithful oracle (ATen exp): boxes within 1e-5, keep sets reported."""
    cfg = synth.V
    ref_cr, (boxes, lg, src, cnt) = _rpn_case(ops, cuda_device, cfg, 1, 1238, 12000, 2000, [(600, 1200)], delta_std=0.05)
    logits, deltas, cell, anchors = synth.rpn_head_outputs(cfg, 1, 1238, 0.05)
    ref_aten = o.rpn_predict_proposals([anchors], [logits], [deltas], [(600, 1200)], 0.7, 12000, 2000, 0.0, False)
    a, b = set(ref_aten[0]["src_index"].tolist()), set(src[0, :cnt[0]].cpu().tolist())
    # the 1-ulp exp difference may flip an IoU decision in rare cases; sets must agree to >= 99.9 %
    assert len(a ^ b) <= max(2, len(a) // 1000), f"{len(a ^ b)} proposals differ between ATen-exp and defined-exp"


def test_rpn_select_invalid_counts_nonfinite(ops, cuda_device):
    logits, deltas, cell, anchors = synth.rpn_head_outputs(synth.V, 1, 77)
    deltas[0, 5, 0] = float("inf"); logits[0, 9] = float("nan")
    _, _, _, cnt, invalid = ops.rpn_select(logits.to(cuda_device), deltas.to(cuda_device), [(600, 1200)], cell_anchors=cell,
                                           feat_hw=(18, 37), stride=32)
    assert invalid.cpu().tolist() == [2]
    ref = o.rpn_predict_proposals([anchors], [logits], [deltas], [(600, 1200)], training=False, exp=o.exp_correctly_rounded)
    assert cnt.cpu().tolist()[0] == len(ref[0]["src_index"])


# ------------------------------------------------------------------------------------------------ Fast R-CNN post-process
def _frcnn_case(ops, dev, rows, K, seed, logit_std, image_sizes, delta_std=1.0, pseudo=0.8):
    R = sum(rows)
    cls, dl = synth.box_head_outputs(R, K, seed, logit_std, delta_std)
    props = synth.random_rois(1, R, seed + 1)[:, 1:].contiguous()
    plist = list(props.split(rows))
    ref = o.box_predictor_inference(cls, dl, plist, image_sizes, 0.05, 0.5, 100, exp=o.exp_correctly_rounded,
                                    softmax=o.softmax_defined)
    out = ops.frcnn_postprocess(cls.to(dev), dl.to(dev), props.to(dev), rows, image_sizes, pseudo_thresh=pseudo,
                                want_probs=True, want_boxes=True)
    cnt = out["count"].cpu().tolist(); pc = out["pseudo_count"].cpu().tolist()
    for i, r in enumerate(ref):
        k = cnt[i]
        assert k == len(r["scores"]), (i, k, len(r["scores"]))
        assert torch.equal(out["classes"][i, :k].cpu(), r["pred_classes"])
        assert torch.equal(out["rows"][i, :k].cpu(), r["kept_rows"])
        assert torch.equal(out["scores"][i, :k].cpu(), r["scores"])
        assert torch.equal(out["boxes"][i, :k].cpu(), r["pred_boxes"])
        pl = o.threshold_bbox(r, pseudo, "roih")
        assert pc[i] == len(pl["scores"]), "pseudo-label set size"
        assert torch.equal(out["boxes"][i, :pc[i]].cpu(), pl["gt_boxes"]) and torch.equal(out["classes"][i, :pc[i]].cpu(), pl["gt_classes"])
    assert torch.equal(out["probs"].cpu(), o.softmax_defined(cls))
    assert torch.equal(out["decoded"].cpu(), o.apply_deltas(dl, props, (10, 10, 5, 5), exp=o.exp_correctly_rounded))
    return ref, out, (cls, dl, plist)


def test_frcnn_postprocess_confident_logits(ops, cuda_device):
    """logits N(0,4): ~25 % of the 16 000 (row, class) pairs pass 0.05, some scores exceed 0.8."""
    ref, out, _ = _frcnn_case(ops, cuda_device, [2000, 2000], 8, 51, 4.0, [(600, 1200), (600, 1200)])
    assert sum(out["pseudo_count"].cpu().tolist()) > 0


def test_frcnn_postprocess_random_init_like(ops, cuda_device):
    """near-uniform softmax (random-init heads): all 16 000 candidates pass 0.05, empty pseudo-label set."""
    ref, out, _ = _frcnn_case(ops, cuda_device, [2000], 8, 52, 0.05, [(600, 1200)], delta_std=0.1)
    assert out["pseudo_count"].cpu().tolist() == [0]


def test_frcnn_postprocess_small_uses_coordinate_trick_and_ragged(ops, cuda_device):
    """<= 1000 candidates per image -> torchvision-CPU's coordinate-trick arithmetic; ragged rows incl. an empty image."""
    _frcnn_case(ops, cuda_device, [150, 0, 37, 1000], 8, 53, 4.0, [(600, 1200), (600, 1200), (300, 500), (600, 1200)])


def test_frcnn_postprocess_single_class_variant(ops, cuda_device):
    _frcnn_case(ops, cuda_device, [1000, 800], 1, 54, 3.0, [(600, 1200), (600, 1200)])


def test_frcnn_postprocess_vs_reference_faithful_oracle(ops, cuda_device):
    """Against the oracle that uses ATen's own exp/softmax (<= 1 ulp different): boxes/scores within 1e-5,
    detection (row, class) sets identical up to threshold-straddling rarities."""
    ref_spec, out, (cls, dl, plist) = _frcnn_case(ops, cuda_device, [2000], 8, 55, 4.0, [(600, 1200)])
    ref = o.box_predictor_inference(cls, dl, plist, [(600, 1200)], 0.05, 0.5, 100)[0]
    k = out["count"].cpu().tolist()[0]
    a = set(zip(ref["kept_rows"].tolist(), ref["pred_classes"].tolist()))
    b = set(zip(out["rows"][0, :k].cpu().tolist(), out["classes"][0, :k].cpu().tolist()))
    assert len(a ^ b) <= 2
    # boxes / scores of the detections both sides kept: 1e-5 relative, whether or not a flip occurred
    got_keys = list(zip(out["rows"][0, :k].cpu().tolist(), out["classes"][0, :k].cpu().tolist()))
    ref_keys = list(zip(ref["kept_rows"].tolist(), ref["pred_classes"].tolist()))
    pos = {v: j for j, v in enumerate(got_keys)}
    ri = [j for j, v in enumerate(ref_keys) if v in pos]
    gi = [pos[ref_keys[j]] for j in ri]
    assert len(ri) >= len(ref_keys) - 2
    _close(out["boxes"][0][gi], ref["pred_boxes"][ri], rtol=1e-5, atol_scale=1e-6)
    _close(out["scores"][0][gi], ref["scores"][ri], rtol=1e-5, atol_scale=0)


def test_frcnn_postprocess_vs_reference_executed_fixture(ops, cuda_device):
    """tests/golden/ref_exec.npz holds what the REFERENCE'S OWN functions returned (fast_rcnn.py:88-142,
    source_free_adaptive_teacher.py:150-183, executed by tests/golden/make_golden_ref.py) for head outputs decoded with ATen
    exp / softmax.  The CUDA path runs from the same head outputs: identical detections and pseudo-label sets (rows, classes),
    boxes / scores within 1e-5 -- up to the measured, rare 1-ulp flips (tests/test_gpu_flip_rate.py), none on this fixture."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_exec.npz"))
    rows = g["frcnn_rows"].tolist()
    sizes = [tuple(int(v) for v in g[f"frcnn_{i}_image_size"]) for i in range(len(rows))]
    t = lambda k: torch.from_numpy(g[k])  # noqa: E731
    out = ops.frcnn_postprocess(t("frcnn_cls").to(cuda_device), t("frcnn_deltas").to(cuda_device), t("frcnn_proposals").to(cuda_device),
                                rows, sizes, pseudo_thresh=0.8)
    cnt, pc = out["count"].cpu().tolist(), out["pseudo_count"].cpu().tolist()
    total_pl = 0
    for i in range(len(rows)):
        k = cnt[i]
        assert k == len(g[f"frcnn_{i}_out_scores"])
        assert torch.equal(out["rows"][i, :k].cpu(), t(f"frcnn_{i}_out_kept_rows")) and torch.equal(out["classes"][i, :k].cpu(), t(f"frcnn_{i}_out_pred_classes"))
        _close(out["boxes"][i, :k], t(f"frcnn_{i}_out_pred_boxes"), rtol=1e-5, atol_scale=1e-6)
        _close(out["scores"][i, :k], t(f"frcnn_{i}_out_scores"), rtol=1e-5, atol_scale=0)
        assert pc[i] == len(g[f"frcnn_{i}_pl_scores"])                                    # pseudo-label set = reference's threshold_bbox
        assert torch.equal(out["classes"][i, :pc[i]].cpu(), t(f"frcnn_{i}_pl_gt_classes"))
        _close(out["boxes"][i, :pc[i]], t(f"frcnn_{i}_pl_gt_boxes"), rtol=1e-5, atol_scale=1e-6)
        total_pl += pc[i]
    assert total_pl >= 20
    # EMA against the reference's _update_teacher_model + load_state_dict (bit-exact, incl. the int64 buffer)
    names = [k[len("ema_s_"):] for k in g.files if k.startswith("ema_s_")]
    for tag, rate in (("a", 0.9996), ("b", 0.999696), ("c", 0.0)):
        sd = {n: t("ema_s_" + n).to(cuda_device) for n in names}
        td = {n: t("ema_t_" + n).to(cuda_device) for n in names}
        ops.EmaPlan([(sd[n], td[n]) for n in names]).step(rate)
        for n in names:
            want = t(f"ema_out_{tag}_{n}")
            assert (_bits_equal(td[n], want) if want.dtype == torch.float32 else torch.equal(td[n].cpu(), want)), (tag, n)


def test_threshold_select(ops, cuda_device):
    g = torch.Generator().manual_seed(61)
    v = torch.rand(5, 700, generator=g)
    counts = torch.tensor([700, 0, 1, 333, 512], dtype=torch.int32)
    idx, cnt = ops.threshold_select(v.to(cuda_device), counts.to(cuda_device), 0.8)
    for s in range(5):
        ref = (v[s, :counts[s]] > 0.8).nonzero().flatten()
        assert cnt[s].item() == ref.numel() and torch.equal(idx[s, :ref.numel()].cpu(), ref)


# ------------------------------------------------------------------------------------------------ BatchNorm / AdaBN
@pytest.fixture(params=["two_phase", "fused_l2"])
def bn_path(request, ops):
    """Both BatchNorm implementations: statistics kernel + finalize/apply kernel, and the single cooperative launch that serves
    activations <= ops.BN_FUSED_MAX_BYTES (NCHW) from L2."""
    old = ops.BN_FUSED_MAX_BYTES
    ops.BN_FUSED_MAX_BYTES = 0 if request.param == "two_phase" else 1 << 40
    yield request.param
    ops.BN_FUSED_MAX_BYTES = old


@pytest.mark.parametrize("shape", [(2, 64, 75, 150), (2, 512, 37, 75), (1, 128, 64, 96), (3, 24, 17, 19), (2, 3, 200, 331)])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_bn_train_forward(ops, cuda_device, shape, layout, bn_path):
    g = torch.Generator().manual_seed(71)
    x = torch.randn(shape, generator=g) * 3 + torch.linspace(-50, 50, shape[1]).view(1, -1, 1, 1)
    bn = torch.nn.BatchNorm2d(shape[1])
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=g); bn.bias.uniform_(-1, 1, generator=g)
        bn.running_mean.normal_(generator=g); bn.running_var.uniform_(0.5, 2.0, generator=g)
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    bn.train()
    with torch.no_grad():
        yref = bn(x)
    d = cuda_device
    xd = x.to(d)
    if layout == "nhwc":
        xd = xd.contiguous(memory_format=torch.channels_last)
    rm, rv = rm0.to(d), rv0.to(d); nbt = torch.zeros((), dtype=torch.int64, device=d)
    y = ops.bn_train_forward(xd, bn.weight.detach().to(d), bn.bias.detach().to(d), rm, rv, nbt, 0.1, 1e-5)
    _close(rm, bn.running_mean, rtol=1e-5, atol_scale=1e-6)
    _close(rv, bn.running_var, rtol=1e-5, atol_scale=0)
    _close(y, yref, rtol=1e-5, atol_scale=1e-5)
    assert nbt.item() == 1
    yr = ops.bn_train_forward(xd, bn.weight.detach().to(d), bn.bias.detach().to(d), None, None, None, 0.1, 1e-5, fuse_relu=True)
    _close(yr, torch.relu(yref), rtol=1e-5, atol_scale=1e-5)
    if layout == "nchw":      # the path under test really ran
        ops.timers.start()
        ops.bn_train_forward(xd, None, None, None, None, None)
        tags = set(ops.timers.stop())
        assert tags == ({"bn_train_fused"} if bn_path == "fused_l2" else {"bn_partial_stats", "bn_finalize_apply"}), tags
    # conv bias folded in + in place
    cb = torch.randn(shape[1], generator=g)
    bn2 = torch.nn.BatchNorm2d(shape[1]).train()
    with torch.no_grad():
        yref2 = torch.relu(bn2(x + cb.view(1, -1, 1, 1)))
    rm2, rv2 = torch.zeros(shape[1], device=d), torch.ones(shape[1], device=d)
    xin = xd.clone()
    y2 = ops.bn_train_forward(xin, None, None, rm2, rv2, None, 0.1, 1e-5, fuse_relu=True, inplace=True, pre_bias=cb.to(d))
    assert y2.data_ptr() == xin.data_ptr()
    _close(y2, yref2, rtol=1e-5, atol_scale=1e-5)
    _close(rm2, bn2.running_mean, rtol=1e-5, atol_scale=1e-6); _close(rv2, bn2.running_var, rtol=1e-5, atol_scale=0)


@pytest.mark.parametrize("shape", [(2, 64, 76, 152), (2, 32, 75, 150), (1, 16, 37, 75), (2, 8, 5, 3)])
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_bn_fused_conv_bias_relu_maxpool(ops, cuda_device, shape, layout):
    """conv bias + BN(train) + ReLU + MaxPool2d(2, 2) in the two BN kernels vs the unfused torch-CPU chain
    (reference vgg.py:15-19).  Running statistics must be those of fl(x + bias)."""
    g = torch.Generator().manual_seed(81)
    N, C, H, W = shape
    x = torch.randn(shape, generator=g) * 2
    cb = torch.randn(C, generator=g) * 5
    bn = torch.nn.BatchNorm2d(C)
    with torch.no_grad():
        bn.weight.uniform_(-1.5, 1.5, generator=g); bn.bias.uniform_(-1, 1, generator=g)     # negative scales: max must follow the affine map
        bn.running_mean.normal_(generator=g); bn.running_var.uniform_(0.5, 2.0, generator=g)
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    bn.train()
    with torch.no_grad():
        full = torch.relu(bn(x + cb.view(1, -1, 1, 1)))
        pooled = torch.nn.functional.max_pool2d(full, 2, 2)
    d = cuda_device
    xd = x.to(d)
    if layout == "nhwc":
        xd = xd.contiguous(memory_format=torch.channels_last)
    for pool, want in ((False, full), (True, pooled)):
        rm, rv = rm0.to(d), rv0.to(d); nbt = torch.zeros((), dtype=torch.int64, device=d)
        y = ops.bn_train_forward(xd, bn.weight.detach().to(d), bn.bias.detach().to(d), rm, rv, nbt, 0.1, 1e-5, fuse_relu=True,
                                 pre_bias=cb.to(d), fuse_maxpool=pool)
        assert y.shape == want.shape
        _close(y, want, rtol=1e-5, atol_scale=1e-5)
        _close(rm, bn.running_mean, rtol=1e-5, atol_scale=1e-6)
        _close(rv, bn.running_var, rtol=1e-5, atol_scale=0)
    # pre_bias == None must equal pre_bias == 0 bit for bit
    y0 = ops.bn_train_forward(xd, None, None, None, None, None, fuse_relu=False)
    y1 = ops.bn_train_forward(xd, None, None, None, None, None, fuse_relu=False, pre_bias=torch.zeros(C, device=d))
    assert torch.equal(y0, y1)


def test_vgg_stage_fusion_matches_unfused_modules(cuda_device):
    """modeling/vgg.py::_Stage hands conv-bias / ReLU / max-pool to the BN kernels; the result must match the plain
    nn.Sequential evaluation of the same modules (cuDNN BN) within fp32 tolerance, including the state_dict side effects."""
    import copy
    import sfod_b200
    from sfod_b200 import config, modeling
    torch.manual_seed(5)
    cfg = config.vgg_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
    bb = modeling.vgg_backbone(cfg)
    with torch.no_grad():
        for m in bb.modules():
            if isinstance(m, torch.nn.Conv2d):
                m.bias.normal_(0, 0.5)
    ref = copy.deepcopy(bb).to(cuda_device).train()
    bb = bb.to(cuda_device).train()
    x = torch.randn(2, 3, 96, 160, device=cuda_device)
    tf = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            got = bb(x)                                   # native path (train + no_grad)
            want = {}
            h = x
            for name, stage in zip(ref._stage_names, ref.stages):
                h = torch.nn.Sequential.forward(stage, h)  # plain module-by-module evaluation
                want[name] = h
    finally:
        torch.backends.cudnn.allow_tf32 = tf
    for k in want:
        assert got[k].shape == want[k].shape
        _close(got[k], want[k], rtol=1e-4, atol_scale=1e-4)
    for (k, a), (_, b) in zip(bb.state_dict().items(), ref.state_dict().items()):
        if "running" in k:
            _close(a, b, rtol=1e-4, atol_scale=1e-5)
        if k.endswith("num_batches_tracked"):
            assert a.item() == b.item() == 1


# ------------------------------------------------------------------------------------------------ fused pairwise_iou + Matcher
@pytest.mark.parametrize("M,N", [(0, 100), (1, 1), (5, 1000), (37, 9990), (600, 2000)])
@pytest.mark.parametrize("cfg", [([0.3, 0.7], [0, -1, 1], True), ([0.5], [0, 1], False), ([0.5, 0.5], [0, -1, 1], True)],
                         ids=["rpn", "roi_heads", "degenerate_interval"])
def test_iou_match_equals_pairwise_iou_plus_matcher(ops, cuda_device, M, N, cfg):
    """SURVEY.md 8f rank 1: labels / matches are integers and must be bit-exact, the matched IoU value as well (same
    separately rounded arithmetic as detectron2's pairwise_iou)."""
    from sfod_b200.modeling.matcher import Matcher
    from sfod_b200.structures import Boxes, pairwise_iou
    thresholds, labels, lowq = cfg
    g = torch.Generator().manual_seed(1000 + M + N)
    def rand_boxes(n):
        ctr = torch.rand(n, 2, generator=g) * torch.tensor([1200.0, 600.0])
        wh = torch.rand(n, 2, generator=g) ** 2 * 400 + 2
        return torch.cat([ctr - wh / 2, ctr + wh / 2], 1)
    gt, bx = rand_boxes(M), rand_boxes(N)
    if M >= 5:
        bx[: min(N, 50)] = gt[torch.randint(0, M, (min(N, 50),), generator=g)]          # exact copies: IoU 1 and ties between gts
        gt[1] = gt[0]                                                                   # duplicate gt: first maximal index wins
        gt[2] = torch.tensor([5000.0, 5000.0, 5010.0, 5010.0])                          # overlaps nothing: its maximum is 0
        bx[-1] = torch.tensor([10.0, 10.0, 10.0, 30.0])                                 # degenerate prediction
    m = Matcher(thresholds, labels, allow_low_quality_matches=lowq)
    mqm = o.pairwise_iou(gt, bx)                                   # the oracle's restatement (pinned against torchvision's Matcher)
    ref_matches, ref_labels = o.matcher(mqm, thresholds, labels, lowq)
    pm, pl = m(pairwise_iou(Boxes(gt), Boxes(bx)))                 # and the package's torch pair agree with it
    assert torch.equal(pm, ref_matches) and torch.equal(pl, ref_labels)
    got_matches, got_labels, got_vals = ops.iou_match(gt.to(cuda_device), bx.to(cuda_device), thresholds, labels, lowq)
    assert torch.equal(got_matches.cpu(), ref_matches)
    assert torch.equal(got_labels.cpu(), ref_labels)
    if M > 0:
        assert torch.equal(got_vals.cpu(), mqm.max(dim=0).values)
    # the Matcher method used by the plugins dispatches to the same call
    mm, ml = m.match_boxes(Boxes(gt.to(cuda_device)), Boxes(bx.to(cuda_device)))
    assert torch.equal(mm.cpu(), ref_matches) and torch.equal(ml.cpu(), ref_labels)


# ------------------------------------------------------------------------------------------------ image preprocessing
@pytest.mark.parametrize("dtype", [torch.uint8, torch.float32])
def test_normalize_pad_equals_preprocess_image(ops, cuda_device, dtype):
    """SURVEY.md 8f rank 3 (normalise / pad / batch): bit-exact against `(x - mean) / std` + ImageList.from_tensors."""
    from sfod_b200.structures import ImageList
    g = torch.Generator().manual_seed(5)
    mean, std = (103.530, 116.280, 123.675), (57.375, 57.120, 58.395)
    tm, ts = torch.tensor(mean).view(-1, 1, 1), torch.tensor(std).view(-1, 1, 1)
    def img(h, w):
        t = torch.randint(0, 256, (3, h, w), generator=g, dtype=torch.uint8)
        return t if dtype == torch.uint8 else t.float() + torch.rand(3, h, w, generator=g)
    # a list of differently sized images, padded to a multiple of 32 (odd widths: scalar path)
    ims = [img(37, 53), img(64, 40), img(50, 61)]
    ref = ImageList.from_tensors([(x - tm) / ts for x in ims], 32)
    got, sizes = ops.normalize_pad([x.to(cuda_device) for x in ims], mean, std, 32)
    assert sizes == ref.image_sizes and got.shape == ref.tensor.shape
    assert _bits_equal(got.cpu(), ref.tensor)
    # an equally sized batch (vector path), NCHW and channels-last storage
    b = torch.stack([img(48, 64) for _ in range(4)])
    refb = (b - tm) / ts
    for cl in (False, True):
        gotb, sizesb = ops.normalize_pad(b.to(cuda_device), mean, std, 0, channels_last=cl)
        assert sizesb == [(48, 64)] * 4
        assert gotb.is_contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format)
        assert _bits_equal(gotb.cpu().contiguous(), refb)


# ------------------------------------------------------------------------------------------------ BN v2: residual fusion, frozen statistics
@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("relu", [True, False])
def test_bn_residual_add_relu_fusion(ops, cuda_device, layout, relu, bn_path):
    """Tail of a detectron2 BottleneckBlock (conv3+norm; out += shortcut; relu_) in one pass, vs nn.BatchNorm2d on the CPU:
    output and running statistics to 1e-5 relative."""
    g = torch.Generator().manual_seed(81)
    shape = (2, 36, 19, 23)          # HW not a multiple of 4: head / tail paths of the vector kernel
    x = torch.randn(shape, generator=g) * 2 + torch.linspace(-20, 20, shape[1]).view(1, -1, 1, 1)
    r = torch.randn(shape, generator=g)
    bn = torch.nn.BatchNorm2d(shape[1])
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5, generator=g); bn.bias.uniform_(-1, 1, generator=g)
        bn.running_mean.normal_(generator=g); bn.running_var.uniform_(0.5, 2.0, generator=g)
    dv = lambda t: t.to(cuda_device)  # noqa: E731
    rm, rv, nbt = dv(bn.running_mean.clone()), dv(bn.running_var.clone()), dv(bn.num_batches_tracked.clone())
    fmt = torch.channels_last if layout == "nhwc" else torch.contiguous_format
    got = ops.bn_train_forward(dv(x).contiguous(memory_format=fmt), dv(bn.weight.detach()), dv(bn.bias.detach()), rm, rv, nbt,
                               fuse_relu=relu, residual=dv(r).contiguous(memory_format=fmt))
    bn.train()
    with torch.no_grad():
        ref = bn(x) + r
        ref = torch.relu(ref) if relu else ref
    _close(got, ref)
    _close(rm, bn.running_mean); _close(rv, bn.running_var)
    assert nbt.item() == 1
    # frozen statistics (detectron2 FrozenBatchNorm2d / eval mode) with the same fusions
    bn.eval()
    with torch.no_grad():
        ref = bn(x) + r
        ref = torch.relu(ref) if relu else ref
    got = ops.bn_frozen_forward(dv(x).contiguous(memory_format=fmt), dv(bn.weight.detach()), dv(bn.bias.detach()), dv(bn.running_mean),
                                dv(bn.running_var), bn.eps, fuse_relu=relu, residual=dv(r).contiguous(memory_format=fmt))
    _close(got, ref)
    got = ops.bn_frozen_forward(dv(x).contiguous(memory_format=fmt), dv(bn.weight.detach()), dv(bn.bias.detach()), dv(bn.running_mean),
                                dv(bn.running_var), bn.eps, fuse_relu=relu)
    with torch.no_grad():
        ref = torch.relu(bn(x)) if relu else bn(x)
    _close(got, ref)


def test_r101_c4_backbone_every_norm_layer_vs_cpu(cuda_device):
    """BASELINE config [4]: the ResNet-101-C4 backbone (detectron2 key layout, RESNETS.NORM "BN", FREEZE_AT 2) in the teacher's
    mode -- train() under no_grad.  Every one of its 94 norm layers runs on the native kernels (83 train-mode BatchNorms with
    the ReLU / residual-add fusions, 11 frozen ones); each is checked against nn.BatchNorm2d / F.batch_norm on the CPU GIVEN THE
    SAME INPUT (the convolution output captured on the GPU), so that cuDNN-vs-ATen convolution differences do not blur the
    comparison: fused output and both running statistics to 1e-5 relative."""
    import copy
    from sfod_b200 import config, modeling
    from sfod_b200.modeling.resnet import FrozenBatchNorm2d
    a, b = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
    try:
        cfg = config.r101_c4_source_free_cfg()
        torch.manual_seed(5)
        bb = modeling.build_resnet_backbone(cfg)
        g = torch.Generator().manual_seed(6)
        with torch.no_grad():
            for m in bb.modules():          # non-trivial affine parameters and statistics everywhere
                if isinstance(m, (torch.nn.BatchNorm2d, FrozenBatchNorm2d)):
                    m.weight.uniform_(0.5, 1.5, generator=g); m.bias.uniform_(-0.5, 0.5, generator=g)
                    m.running_mean.normal_(0, 0.1, generator=g); m.running_var.uniform_(0.5, 1.5, generator=g)
        ref_state = copy.deepcopy(bb.state_dict())
        bb.to(cuda_device).train()
        norms = [(n, m) for n, m in bb.named_modules() if isinstance(m, (torch.nn.BatchNorm2d, FrozenBatchNorm2d))]
        assert len(norms) == 94 and sum(isinstance(m, FrozenBatchNorm2d) for _, m in norms) == 11
        cap = {}

        def pre(name):
            def hook(mod, args, kwargs):
                cap[name] = dict(x=args[0].detach().clone().cpu(), relu=kwargs.get("fuse_relu", False),
                                 res=None if kwargs.get("residual") is None else kwargs["residual"].detach().clone().cpu())
            return hook

        def post(name):
            def hook(mod, args, kwargs, out):
                cap[name]["y"] = out.detach().clone().cpu()
            return hook
        hs = []
        for n, m in norms:
            hs.append(m.register_forward_pre_hook(pre(n), with_kwargs=True)); hs.append(m.register_forward_hook(post(n), with_kwargs=True))
        x = torch.randn(2, 3, 160, 224, generator=g) * 50
        l0 = sfod_b200.ops.launch_count()
        with torch.no_grad():
            out = bb(x.to(cuda_device))
        assert sfod_b200.ops.launch_count() - l0 >= 83 + 11 * 2              # every norm layer went through the library (>= 1 launch each)
        for h in hs:
            h.remove()
        assert out["res4"].shape == (2, 1024, 10, 14)
        gpu_state = {k: v.cpu() for k, v in bb.state_dict().items()}
        for n, m in norms:
            c = cap[n]
            w, bias = ref_state[n + ".weight"], ref_state[n + ".bias"]
            rm, rv = ref_state[n + ".running_mean"].clone(), ref_state[n + ".running_var"].clone()
            frozen = isinstance(m, FrozenBatchNorm2d)
            y = torch.nn.functional.batch_norm(c["x"], rm, rv, w, bias, not frozen, 0.1, 1e-5)
            if c["res"] is not None:
                y = y + c["res"]
            if c["relu"]:
                y = torch.relu(y)
            _close(c["y"], y)
            _close(gpu_state[n + ".running_mean"], rm); _close(gpu_state[n + ".running_var"], rv)
            if not frozen:
                assert gpu_state[n + ".num_batches_tracked"].item() == 1
        # conv3 of every bottleneck carries the residual + ReLU fusion; shortcuts carry neither
        assert all(cap[n]["res"] is not None and cap[n]["relu"] for n, _ in norms if n.endswith("conv3.norm"))
        assert all(cap[n]["res"] is None and not cap[n]["relu"] for n, _ in norms if n.endswith("shortcut.norm"))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = a, b


# ------------------------------------------------------------------------------------------------ batched subsample_labels (8f rank 1)
def _perm_from_hash(ops, seed, seg, cand):
    """The permutation `randperm(len(cand))` must return for detectron2's subsample_labels to reproduce the kernel: candidates
    ordered by (hash, index)."""
    h = ops.sample_hash(seed, seg, cand.numpy())
    order = np.lexsort((cand.numpy(), h))
    return torch.from_numpy(order.astype(np.int64))


def test_subsample_labels_batched_equals_detectron2_with_the_same_permutation(ops, cuda_device):
    """sfod_subsample_labels vs oracle.subsample_labels (detectron2's) fed the permutation the kernel's counter-based keys
    define: identical index lists (order included), for ROI-head style labels (bg = 8, ignore = -1) and RPN style ({-1, 0, 1},
    bg = 0), segments with no / few / many positives, empty segments, 34 200 anchors."""
    g = torch.Generator().manual_seed(91)
    def roi_seg(n, p_fg, p_ign):
        u = torch.rand(n, generator=g)
        lab = torch.full((n,), 8, dtype=torch.int64)
        lab[u < p_fg] = torch.randint(0, 8, (int((u < p_fg).sum()),), generator=g)
        lab[u > 1 - p_ign] = -1
        return lab
    cases = [
        (8, 512, 0.25, [roi_seg(2003, 0.3, 0.05), roi_seg(2000, 0.01, 0.0), roi_seg(2000, 0.0, 0.0), roi_seg(37, 0.5, 0.2),
                        torch.full((50,), -1, dtype=torch.int64), torch.zeros(0, dtype=torch.int64), roi_seg(700, 1.0, 0.0)]),
        (0, 256, 0.5, [(torch.rand(34200, generator=g) < q).to(torch.int64) - (torch.rand(34200, generator=g) < 0.1).to(torch.int64) * 0
                       for q in (0.01, 0.0005, 0.3)]),
    ]
    for bg, num_samples, frac, segs in cases:
        if bg == 0:   # RPN labels: 1 positive, 0 negative, -1 ignore
            segs = [torch.where(torch.rand(s.numel(), generator=g) < 0.2, torch.full_like(s, -1), s) for s in segs]
        seed = 0xC0FFEE1234 + bg
        lab = torch.cat(segs)
        sampled, counts = ops.subsample_labels_batched(lab.to(cuda_device), [s.numel() for s in segs], num_samples, frac, bg, seed)
        sampled, counts = sampled.cpu(), counts.cpu().tolist()
        for i, s in enumerate(segs):
            calls = []
            def randperm(n, device=None, _i=i, _s=s):
                cand = ((_s != -1) & (_s != bg)).nonzero().flatten() if not calls else (_s == bg).nonzero().flatten()
                calls.append(1)
                assert cand.numel() == n
                return _perm_from_hash(ops, seed, _i, cand)
            pos, neg = o.subsample_labels(s, num_samples, frac, bg, randperm=randperm)
            assert counts[i] == [pos.numel(), neg.numel()], (i, counts[i], pos.numel(), neg.numel())
            assert torch.equal(sampled[i, :pos.numel()], pos) and torch.equal(sampled[i, pos.numel():pos.numel() + neg.numel()], neg)
            assert (sampled[i, pos.numel() + neg.numel():] == -1).all()


def test_subsample_labels_batched_is_uniform(ops, cuda_device):
    """Every candidate is selected with probability k / n (binomial 5-sigma band over 4000 independent keys)."""
    n, k, trials = 200, 20, 4000
    lab = torch.zeros(n, dtype=torch.int64).repeat(trials)            # all negatives, bg = 0
    sampled, counts = ops.subsample_labels_batched(lab.to(cuda_device), [n] * trials, k, 0.0, 0, 99)
    assert (counts.cpu() == torch.tensor([0, k])).all()
    freq = torch.bincount(sampled.cpu().flatten(), minlength=n).double()
    p = k / n
    sigma = (trials * p * (1 - p)) ** 0.5
    assert (freq - trials * p).abs().max() < 5 * sigma
    # first position uniform too (random ORDER, not just a random subset)
    first = torch.bincount(sampled[:, 0].cpu(), minlength=n).double()
    assert (first - trials / n).abs().max() < 6 * (trials / n) ** 0.5


# ------------------------------------------------------------------------------------------------ strong augmentation (8f rank 3)
def _aug_images(N=3, H=97, W=131, seed=7):
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(0, 256, (N, 3, H, W), dtype=torch.uint8, generator=g)
    x[0, :, :10, :10] = 0; x[0, :, 10:20, :10] = 255; x[0, :, 20:30, :10] = 77        # flat patches (maxc == minc in rgb2hsv)
    return x


def _tv_jitter(img, p):
    import torchvision.transforms.functional as TF
    for o, f in zip(p["order"], p["factors"]):
        img = (TF.adjust_brightness, TF.adjust_contrast, TF.adjust_saturation, TF.adjust_hue)[o](img, f)
    if p.get("grayscale"):
        img = TF.rgb_to_grayscale(img, num_output_channels=3)
    return img


def test_color_jitter_bit_exact_vs_pil(ops, cuda_device):
    """ColorJitter(0.4, 0.4, 0.4, 0.1) + RandomGrayscale of reference daod/data/detection_utils.py:13-16 through torchvision's PIL
    path -- what the reference executes, because its mapper hands PIL images to
    the transforms (reference daod/data/mappers/two_crop_augmentation_mapper.py:141-157): ImageEnhance.Brightness / Contrast /
    Color (Image.blend), convert("L"), convert("HSV").  ops.color_jitter is bit-equal, for every op alone at the
    extreme factors (incl. hue +-0.5 and factors outside [0, 1], where Image.blend clips) and for full random sequences with
    RandomGrayscale; also bit-equal to the CPU restatement (oracle/pil_cpu.py)."""
    from PIL import Image
    from oracle import pil_cpu
    x = _aug_images(3, 97, 131, 21)
    x[2] = (x[2] // 12 + 100)                                     # low-contrast image: contrast / saturation extrapolation clips
    g = torch.Generator().manual_seed(4)
    recs = []
    for o in range(4):
        lo, hi = [(0.6, 1.4), (0.6, 1.4), (0.6, 1.4), (-0.1, 0.1)][o]
        for f in (lo, hi, (lo + hi) / 2 + 0.0123) + ((0.0, 1.0, 2.5) if o < 3 else (-0.5, 0.5, 0.0)):
            recs.append(dict(order=[o], factors=[f]))
    for _ in range(15):
        order = torch.randperm(4, generator=g).tolist()
        vals = [float(torch.empty(1).uniform_(0.6, 1.4, generator=g)) for _ in range(3)] + [float(torch.empty(1).uniform_(-0.1, 0.1, generator=g))]
        recs.append(dict(order=order, factors=[vals[k] for k in order], grayscale=bool(torch.rand(1, generator=g) < 0.3)))
    recs += [dict(order=[], factors=[], grayscale=True), dict(order=[], factors=[])]
    for r0 in range(0, len(recs), 3):
        batch = recs[r0:r0 + 3]
        imgs = x[:len(batch)]
        got = ops.color_jitter(imgs.to(cuda_device), batch).cpu()
        for n, p in enumerate(batch):
            hwc = imgs[n].permute(1, 2, 0).contiguous().numpy()
            want = torch.from_numpy(np.array(_tv_jitter(Image.fromarray(hwc, "RGB"), p))).permute(2, 0, 1)
            assert torch.equal(got[n], want), (p, int((got[n].int() - want.int()).abs().max()), int((got[n] != want).sum()))
            assert np.array_equal(pil_cpu.color_jitter(hwc, p["order"], p["factors"], bool(p.get("grayscale"))), want.permute(1, 2, 0).numpy())


def test_gaussian_blur_pil_bit_exact(ops, cuda_device):
    """ops.gaussian_blur_pil == PIL.ImageFilter.GaussianBlur(radius=sigma), bit for bit: the blur of the reference's strong
    augmentation (reference daod/data/transforms/augmentations.py:18-21).  Image sizes that are not multiples of the 32-pixel tile,
    images narrower than the halo, the reference's sigma range and beyond, RandomApply misses; also against the CPU restatement
    (oracle/pil_cpu.py) and through engine.strong_augment."""
    from PIL import Image, ImageFilter
    from oracle import pil_cpu
    g = torch.Generator().manual_seed(17)
    for (H, W), sigmas in (((97, 131), [0.1, 0.77, 2.0, None, 1.3]), ((600, 1200), [1.9, None]), ((5, 7), [2.0, 0.4]), ((33, 4), [5.5, 9.7]),
                           ((1, 40), [1.0]), ((64, 64), [0.0, 3.3])):
        x = torch.randint(0, 256, (len(sigmas), 3, H, W), dtype=torch.uint8, generator=g)
        got = ops.gaussian_blur_pil(x.to(cuda_device), sigmas).cpu()
        for n, sg in enumerate(sigmas):
            if sg is None or sg == 0.0:
                assert torch.equal(got[n], x[n])
                continue
            hwc = x[n].permute(1, 2, 0).contiguous().numpy()
            want = torch.from_numpy(np.array(Image.fromarray(hwc, "RGB").filter(ImageFilter.GaussianBlur(radius=sg)))).permute(2, 0, 1)
            assert torch.equal(got[n], want), ((H, W), sg, int((got[n].int() - want.int()).abs().max()), int((got[n] != want).sum()))
            if H * W <= 20000:
                assert np.array_equal(pil_cpu.gaussian_blur(hwc, sg), want.permute(1, 2, 0).numpy())
    with pytest.raises(ValueError):
        ops.gaussian_blur_pil(torch.zeros(1, 3, 8, 8, dtype=torch.uint8, device=cuda_device), [40.0])
    # the strong augmentation blurs with it
    from sfod_b200 import engine
    x = torch.randint(0, 256, (2, 3, 60, 90), dtype=torch.uint8, generator=g)
    params = [{"order": [], "factors": [], "grayscale": False, "sigma": 1.25, "rects": []}, {"order": [], "factors": [], "grayscale": False, "sigma": None, "rects": []}]
    aug = engine.strong_augment(x.to(cuda_device), params=params).cpu()
    want = torch.from_numpy(np.array(Image.fromarray(x[0].permute(1, 2, 0).contiguous().numpy(), "RGB").filter(ImageFilter.GaussianBlur(radius=1.25)))).permute(2, 0, 1)
    assert torch.equal(aug[0], want) and torch.equal(aug[1], x[1])


def test_random_erase_equals_totensor_erase_topil(ops, cuda_device):
    """3 x RandomErasing(value="random") between ToTensor and ToPILImage (reference daod/data/detection_utils.py:18-33) with the
    SAME noise: bit-exact, including the wrap-around of byte(255 * v) for v outside [0, 1] and overlapping rectangles; with the
    device generator: pixels outside the rectangles untouched, the fill looks like wrapped N(0, 255^2) noise."""
    import torchvision.transforms.functional as TF
    x = _aug_images(2, 80, 120, 9)
    rects = [[(5, 7, 30, 40), (20, 30, 25, 50), (0, 0, 3, 3)], [(10, 10, 60, 100)]]
    g = torch.Generator().manual_seed(11)
    noise = torch.randn(2, 4, 3, 80, 120, generator=g)
    got = ops.random_erase_(x.clone().to(cuda_device), rects, noise=noise.to(cuda_device)).cpu()
    for n in range(2):
        t = x[n].to(torch.float32).div(255)                        # ToTensor
        for k, (i, j, h, w) in enumerate(rects[n]):
            t = TF.erase(t, i, j, h, w, noise[n, k, :, i:i + h, j:j + w])
        want = t.mul(255).byte()                                   # ToPILImage
        assert torch.equal(got[n], want), int((got[n] != want).sum())
    dev = ops.random_erase_(x.clone().to(cuda_device), rects, seed=1234).cpu()
    mask = torch.zeros(2, 80, 120, dtype=torch.bool)
    for n in range(2):
        for (i, j, h, w) in rects[n]:
            mask[n, i:i + h, j:j + w] = True
    m3 = mask.unsqueeze(1).expand(-1, 3, -1, -1)
    assert torch.equal(dev[~m3], x[~m3])
    fill = dev[m3].float()
    assert abs(fill.mean().item() - 127.5) < 4 and 65 < fill.std().item() < 82             # ~uniform bytes
    again = ops.random_erase_(x.clone().to(cuda_device), rects, seed=1234).cpu()
    assert torch.equal(again, dev)                                                           # counter-based: reproducible


def test_strong_augment_equals_the_reference_chain_on_pil_images(cuda_device):
    """The WHOLE strong augmentation of reference daod/data/detection_utils.py:7-37 as its mapper runs it
    (two_crop_augmentation_mapper.py:141-157: PIL image in, PIL image out) -- ColorJitter ops in the drawn order and
    RandomGrayscale on the PIL image, PIL GaussianBlur(radius=sigma), ToTensor, the RandomErasing rectangles filled with the
    drawn noise, ToPILImage -- against engine.strong_augment with the SAME decisions and noise: bit-equal for every image of a
    batch drawn with the reference's probabilities (seeded until every branch occurs)."""
    import torchvision.transforms.functional as TF
    from PIL import Image, ImageFilter
    from sfod_b200 import engine
    N, H, W = 12, 96, 160
    x = _aug_images(N, H, W, 31)
    g = torch.Generator().manual_seed(2025)
    params = engine.draw_strong_augmentation_params(N, H, W, g)
    assert any(p["order"] for p in params) and any(p["grayscale"] for p in params) and any(p["sigma"] is not None for p in params)
    assert any(len(p["rects"]) >= 2 for p in params) and any(not p["order"] for p in params)
    noise = torch.randn(N, 4, 3, H, W, generator=g)
    got = engine.strong_augment(x.to(cuda_device), params=params, noise=noise.to(cuda_device)).cpu()
    for n, p in enumerate(params):
        img = Image.fromarray(x[n].permute(1, 2, 0).contiguous().numpy(), "RGB")
        img = _tv_jitter(img, p)                                                             # ColorJitter + RandomGrayscale (PIL path)
        if p["sigma"] is not None:
            img = img.filter(ImageFilter.GaussianBlur(radius=p["sigma"]))                   # reference augmentations.py:18-21
        t = TF.to_tensor(img)
        for k, (i, j, h, w) in enumerate(p["rects"]):
            t = TF.erase(t, i, j, h, w, noise[n, k, :, i:i + h, j:j + w])
        want = torch.from_numpy(np.array(TF.to_pil_image(t))).permute(2, 0, 1)
        assert torch.equal(got[n], want), (n, p, int((got[n] != want).sum()))


def test_strong_augment_pipeline(cuda_device):
    from sfod_b200 import engine
    x = _aug_images(6, 120, 200, 13).to(cuda_device)
    g = torch.Generator().manual_seed(99)
    params = engine.draw_strong_augmentation_params(6, 120, 200, g)
    y = engine.strong_augment(x, params=params, seed=5)
    assert y.shape == x.shape and y.dtype == torch.uint8 and y.data_ptr() != x.data_ptr()
    y2 = engine.strong_augment(x, params=params, seed=5)
    assert torch.equal(y, y2)
    for n, p in enumerate(params):
        if not p["order"] and not p["grayscale"] and p["sigma"] is None and not p["rects"]:
            assert torch.equal(y[n], x[n])
