"""GPU tests at BASELINE.json's FULL sizes, through size-independent properties (the CPU oracle would take minutes there):
NMS idempotence / cleanliness / order, RPN selection invariants on 8 x 34 200 R101 anchors, ROIAlign linearity and the
forward/backward adjoint identity on 16 000 ROIs, EMA fixed points on the 47.6 M-element VGG state, BatchNorm statistics on
8 x 64 x 600 x 1200 activations, Fast R-CNN post-processing invariants on 8 x 2000 proposals."""
import pytest
import torch
import torchvision

import sfod_b200  # noqa: F401
from sfod_b200 import config, engine, modeling, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops(cuda_device):
    return sfod_b200.ops


def _max_offdiag_iou(boxes):
    iou = torchvision.ops.box_iou(boxes, boxes)
    iou.fill_diagonal_(0)
    return float(iou.max()) if boxes.shape[0] > 1 else 0.0


@pytest.mark.parametrize("n,kind", [(12000, "low"), (34200, "high")])
def test_nms_full_size_properties(ops, cuda_device, n, kind):
    b, s = synth.boxes_low_suppression(synth.R101, n, 7) if kind == "low" else synth.boxes_high_suppression(n, 7, clusters=900)
    b, s = b.to(cuda_device), s.to(cuda_device)
    keep = ops.nms(b, s, 0.7)
    ks = s[keep]
    assert torch.all(ks[:-1] >= ks[1:]), "kept indices must be score-descending"
    assert keep.unique().numel() == keep.numel()
    kb = b[keep]
    assert _max_offdiag_iou(kb[:6000]) <= 0.7 + 1e-5, "no kept pair may overlap above the threshold"
    again = ops.nms(kb, ks, 0.7)                                    # idempotence: the kept set survives a second pass unchanged
    assert torch.equal(again, torch.arange(keep.numel(), device=cuda_device))
    # completeness: every dropped box is suppressed by some kept box with a higher (or equal, lower-index) score
    dropped = torch.ones(b.shape[0], dtype=torch.bool, device=cuda_device)
    dropped[keep] = False
    di = dropped.nonzero().flatten()[:3000]
    iou = torchvision.ops.box_iou(b[di], kb)
    higher = (ks[None, :] > s[di][:, None]) | ((ks[None, :] == s[di][:, None]) & (keep[None, :] < di[:, None]))
    assert bool(((iou > 0.7 - 1e-5) & higher).any(dim=1).all())


def test_rpn_select_r101_batch8_properties(ops, cuda_device):
    cfg = synth.R101
    N = 8
    logits, deltas, cell, anchors = synth.rpn_head_outputs(cfg, N, 99)
    lg, dl = logits.to(cuda_device), deltas.to(cuda_device)
    sizes = [(600, 1200)] * 7 + [(512, 1000)]
    boxes, out_lg, src, cnt, invalid = ops.rpn_select(lg, dl, sizes, cell_anchors=cell, feat_hw=(cfg["H"], cfg["W"]), stride=cfg["stride"],
                                                      pre_nms_topk=12000, post_nms_topk=2000)
    assert invalid.sum().item() == 0
    for i in range(N):
        k = int(cnt[i])
        assert 0 < k <= 2000
        bi, li, si = boxes[i, :k], out_lg[i, :k], src[i, :k]
        assert torch.all(li[:-1] >= li[1:]) and si.unique().numel() == k
        assert torch.equal(lg[i][si], li), "objectness logits must be the gathered head outputs"
        h, w = sizes[i]
        assert bi[:, 0::2].min() >= 0 and bi[:, 0::2].max() <= w and bi[:, 1::2].min() >= 0 and bi[:, 1::2].max() <= h
        assert torch.all((bi[:, 2] > bi[:, 0]) & (bi[:, 3] > bi[:, 1]))
        assert _max_offdiag_iou(bi) <= 0.7 + 1e-6
        # top-k: every selected logit is among the 12 000 largest of the image
        kth = torch.topk(lg[i], 12000).values[-1]
        assert li.min() >= kth
        assert torch.all(boxes[i, k:] == 0) and torch.all(src[i, k:] == -1)


def test_roi_align_linearity_and_adjoint_full_size(ops, cuda_device):
    cfg = synth.V
    N, R = 8, 16000
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, cfg["C"], cfg["H"], cfg["W"], generator=g).to(cuda_device)
    y = torch.randn(N, cfg["C"], cfg["H"], cfg["W"], generator=g).to(cuda_device)
    rois = synth.random_rois(N, R, 4).to(cuda_device)
    f = lambda t: ops.roi_align(t, rois, (7, 7), 1 / 32, 0, True)
    fx, fy = f(x), f(y)
    lin = f(2.5 * x - 0.75 * y)
    ref = 2.5 * fx - 0.75 * fy
    assert float((lin - ref).abs().max()) <= 1e-5 * float(ref.abs().max()) + 1e-6            # linear operator (1e-5 relative fp32)
    ones = f(torch.ones_like(x))
    inside = (rois[:, 1] > 40) & (rois[:, 2] > 40) & (rois[:, 3] < 1100) & (rois[:, 4] < 540)
    assert float((ones[inside] - 1).abs().max()) <= 1e-5                                     # partition of unity inside the map
    # adjoint identity <A x, g> == <x, A^T g> ties the backward kernel to the forward kernel
    xr = x[:, :, :, :].clone().requires_grad_(True)
    rs = rois[:4096]
    out = ops.roi_align(xr, rs, (7, 7), 1 / 32, 0, True)
    gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(5)).to(cuda_device)
    out.backward(gout)
    lhs = float((out.detach().double() * gout.double()).sum())
    rhs = float((xr.grad.double() * x.double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1.0) + 1e-2 * 1e-3


def test_ema_fixed_points_on_vgg_state(ops, cuda_device):
    torch.manual_seed(1)
    cfg = config.vgg_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
    teacher = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg).to(cuda_device)
    student = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg).to(cuda_device)
    t0 = {k: v.clone() for k, v in teacher.state_dict().items()}
    ema = engine.TeacherEMA(student, teacher, 1)
    ema.step(1.0)                                   # s*0 + t*1: the teacher is a fixed point
    assert ema.numel == 47636547
    for k, v in teacher.state_dict().items():
        assert torch.equal(v, t0[k]), k
    ema.step(0.0)                                   # s*1 + t*0: the teacher becomes the student
    for (k, v), (_, sv) in zip(teacher.state_dict().items(), student.state_dict().items()):
        assert torch.equal(v, sv), k
    # one 0.9996 step from t0 equals the reference expression evaluated by torch on the GPU (same fp32 ops: bit-exact)
    teacher.load_state_dict(t0)
    ema.step(0.9996)
    for (k, v), (_, sv) in zip(teacher.state_dict().items(), student.state_dict().items()):
        want = (sv * (1 - 0.9996) + t0[k] * 0.9996).to(v.dtype)
        assert torch.equal(v, want), k


def test_bn_statistics_full_size_abi_v2(ops, cuda_device):
    N, C, H, W = 8, 64, 600, 1200
    g = torch.Generator(device=cuda_device).manual_seed(2)
    x = torch.randn(N, C, H, W, device=cuda_device, generator=g) * 2 + torch.linspace(-30, 30, C, device=cuda_device).view(1, C, 1, 1)
    rm = torch.zeros(C, device=cuda_device); rv = torch.ones(C, device=cuda_device); nbt = torch.zeros((), dtype=torch.int64, device=cuda_device)
    y = ops.bn_train_forward(x, None, None, rm, rv, nbt, 0.1, 1e-5)
    mean64 = x.double().mean(dim=(0, 2, 3)); var64 = x.double().var(dim=(0, 2, 3), unbiased=True)
    assert torch.allclose(rm.double(), 0.1 * mean64, rtol=1e-5, atol=1e-6)                   # 1e-5 relative fp32 (BASELINE.json)
    assert torch.allclose(rv.double(), 0.9 + 0.1 * var64, rtol=1e-5)
    ym = y.double().mean(dim=(0, 2, 3)); yv = y.double().var(dim=(0, 2, 3), unbiased=False)
    assert float(ym.abs().max()) < 1e-4 and float((yv - 1).abs().max()) < 1e-4              # normalised output
    # statistics of the whole batch == merge of the two half batches (the quantity the multi-GPU all-reduce sums)
    L = sfod_b200._lib.lib()
    def raw(t):
        st = torch.empty(L.sfod_bn_stats_bytes(C) // 8, dtype=torch.float64, device=cuda_device)
        sfod_b200._lib.check(L.sfod_bn_partial_stats(t.data_ptr(), None, 0, t.shape[0], C, H * W, st.data_ptr(), None,
                                                     torch.cuda.current_stream().cuda_stream))
        return st[: 2 * C].clone()
    whole, a, b = raw(x), raw(x[:4].contiguous()), raw(x[4:].contiguous())
    assert torch.allclose(whole, a + b, rtol=1e-6, atol=1e-3)     # <= 64-term fp32 partials with different pivots, fp64 above


def test_frcnn_postprocess_full_size_properties(ops, cuda_device):
    N, Rn, K = 8, 2000, 8
    cls, dl = synth.box_head_outputs(N * Rn, K, 11, 4.0)
    props = synth.random_rois(1, N * Rn, 12)[:, 1:].contiguous()
    out = ops.frcnn_postprocess(cls.to(cuda_device), dl.to(cuda_device), props.to(cuda_device), [Rn] * N, [(600, 1200)] * N,
                                pseudo_thresh=0.8)
    for i in range(N):
        k, p = int(out["count"][i]), int(out["pseudo_count"][i])
        assert 0 < k <= 100 and 0 <= p <= k
        sc, cl, bx = out["scores"][i, :k], out["classes"][i, :k], out["boxes"][i, :k]
        assert torch.all(sc[:-1] >= sc[1:]) and torch.all(sc > 0.05) and cl.min() >= 0 and cl.max() < K
        assert p == int((sc > 0.8).sum()), "pseudo-label set = prefix of detections above the threshold"
        assert bx[:, 0::2].min() >= 0 and bx[:, 0::2].max() <= 1200 and bx[:, 1::2].max() <= 600
        for c in cl.unique():
            assert _max_offdiag_iou(bx[cl == c]) <= 0.5 + 1e-6          # per-class NMS-clean
        rows = out["rows"][i, :k]
        probs = torch.softmax(cls[i * Rn:(i + 1) * Rn].to(cuda_device), -1)
        assert torch.allclose(probs[rows, cl], sc, rtol=1e-5, atol=1e-7)


_NCCL_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SFOD_ROOT"])
import sfod_b200
from sfod_b200 import modeling, engine
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
g = torch.Generator().manual_seed(5)
full = torch.randn(4, 32, 40, 56, generator=g) * 3 + 1.5                 # the concatenated batch of both ranks
b, e = engine.shard_range(4, rank, 2)
bn = modeling.SfodBatchNorm2d(32, process_group=True).cuda().train()
ref = torch.nn.BatchNorm2d(32).train()
with torch.no_grad():
    y = bn(full[b:e].cuda())
    yref = ref(full)
assert torch.allclose(bn.running_mean.cpu(), ref.running_mean, rtol=1e-5, atol=1e-6), "running_mean"
assert torch.allclose(bn.running_var.cpu(), ref.running_var, rtol=1e-5), "running_var"
assert torch.allclose(y.cpu(), yref[b:e], rtol=1e-5, atol=1e-5), "normalised output"
dist.barrier()
if rank == 0:
    print("NCCL_BN_OK")
dist.destroy_process_group()
"""


def test_adabn_statistic_allreduce_nccl_two_gpus(tmp_path):
    """SURVEY.md 8e collective (2): with a process group, every rank normalises with the statistics of the concatenated
    batch; parity is defined against nn.BatchNorm2d on the concatenated batch (single process, CPU)."""
    import os, subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "worker.py"
    script.write_text(_NCCL_WORKER)
    env = dict(os.environ, SFOD_ROOT=root, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", str(script)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and "NCCL_BN_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


@pytest.mark.parametrize("world", [3, 6])   # all 8 slots are exercised by the 8-process bench self-check (profiles/r2s_*)
def test_peer_statistic_exchange_local_ring_matches_concatenated_batch(cuda_device, world):
    """The NVLink peer-memory all-reduce of the BN statistics (sfod_bn_finalize_apply with a comm), with the ranks emulated as
    streams of ONE GPU (their inboxes are plain allocations in this process): every rank must end with the running statistics
    and the normalised output of nn.BatchNorm2d on the concatenated batch, the exchanged totals must be bit-identical on all
    ranks, and repeated exchanges (slot parity, device-side epoch counter) must keep working without a host reset."""
    from sfod_b200 import modeling
    from sfod_b200.engine.p2p import PeerStatExchange
    from sfod_b200 import ops
    C_ = 48
    tail_default = ops.BN_P2P_TAIL_PUSH
    peers = PeerStatExchange.local_ring(world, cuda_device)
    try:
        g = torch.Generator().manual_seed(11)
        streams = [torch.cuda.Stream(cuda_device) for _ in range(world)]
        bns = [modeling.SfodBatchNorm2d(C_, process_group=peers[r]).to(cuda_device).train() for r in range(world)]
        ref = torch.nn.BatchNorm2d(C_).train()
        for it in range(5):                                               # odd and even epochs
            ops.BN_P2P_TAIL_PUSH = int(it not in (2, 3))                  # payload delivered by the statistics kernel / by the finalize kernel
            parts = [torch.randn(2 + (r == 1), C_, 20, 28, generator=g) * (r + 1) + 0.5 * r for r in range(world)]   # ragged shards
            dparts = [p.to(cuda_device) for p in parts]
            if it == 4:                                                   # channels-last statistics pass (delivery always by the finalize kernel)
                dparts = [p.contiguous(memory_format=torch.channels_last) for p in dparts]
            torch.cuda.synchronize()
            ys = [None] * world
            for r in range(world):
                with torch.cuda.stream(streams[r]), torch.no_grad():
                    ys[r] = bns[r](dparts[r], fuse_relu=(it % 2 == 1))
            torch.cuda.synchronize()
            with torch.no_grad():
                yref = ref(torch.cat(parts))
                if it % 2 == 1:
                    yref = torch.relu(yref)
            o = 0
            for r in range(world):
                n = parts[r].shape[0]
                assert torch.allclose(ys[r].cpu(), yref[o:o + n], rtol=1e-5, atol=1e-5), (it, r)
                o += n
                assert torch.allclose(bns[r].running_mean.cpu(), ref.running_mean, rtol=1e-5, atol=1e-6)
                assert torch.allclose(bns[r].running_var.cpu(), ref.running_var, rtol=1e-5)
                assert torch.equal(bns[r].running_mean, bns[0].running_mean) and torch.equal(bns[r].running_var, bns[0].running_var)
                assert int(bns[r].num_batches_tracked) == it + 1
        for r in range(world):
            assert peers[r].status() == (5, 0)                            # 5 exchanges, no timeout
    finally:
        ops.BN_P2P_TAIL_PUSH = tail_default
        for p in peers:
            p.close()


def test_peer_statistic_exchange_single_rank_equals_plain_path(cuda_device):
    """world = 1 degenerates to the plain two-phase BatchNorm (bit for bit)."""
    from sfod_b200 import modeling
    from sfod_b200.engine.p2p import PeerStatExchange
    (peer,) = PeerStatExchange.local_ring(1, cuda_device)
    try:
        x = torch.randn(3, 16, 33, 41, device=cuda_device) * 2 + 1
        a = modeling.SfodBatchNorm2d(16, process_group=peer).to(cuda_device).train()
        b = modeling.SfodBatchNorm2d(16, process_group=True).to(cuda_device).train()   # no process group initialised: local statistics, two-phase path
        with torch.no_grad():
            ya, yb = a(x), b(x)
        assert torch.equal(ya, yb) and torch.equal(a.running_mean, b.running_mean) and torch.equal(a.running_var, b.running_var)
    finally:
        peer.close()


_P2P_WORKER = _NCCL_WORKER.replace("bn = modeling.SfodBatchNorm2d(32, process_group=True).cuda().train()",
                                   "from sfod_b200.engine.p2p import PeerStatExchange\n"
                                   "peer = PeerStatExchange.from_process_group()\n"
                                   "bn = modeling.SfodBatchNorm2d(32, process_group=peer).cuda().train()") \
    .replace('    print("NCCL_BN_OK")', '    print("NCCL_BN_OK")\nassert peer.status() == (2, 0)\npeer.close()')


def test_adabn_statistic_exchange_peer_memory_two_gpus(tmp_path):
    """The same contract as the NCCL test above for the product path: IPC-mapped inboxes of two processes on two GPUs."""
    import os, subprocess, sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "worker.py"
    script.write_text(_P2P_WORKER)
    env = dict(os.environ, SFOD_ROOT=root, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29534", str(script)], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and "NCCL_BN_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
