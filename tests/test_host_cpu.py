"""CPU tests (no GPU) of the C-ABI library surface and of the host-side logic.

* libsfod_b200.so loads and exports every symbol include/sfod_b200.h declares; its host-only entry points (version, status
  strings, workspace-size queries, EMA plan builder) behave; no kernel is launched.
* The product never imports ``oracle/`` and refuses CPU tensors (no fallback).
* detectron2-shaped structures, registries, config and the trainer-level host logic (state-dict key matching, sharding).
* world_size-2 ``gloo`` run of the multi-GPU host logic: image sharding and the AdaBN (sum, sum^2, count) reduction.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest
import torch

import sfod_b200  # noqa: F401
from sfod_b200 import _lib, config, engine, modeling, ops, registry
from sfod_b200.engine.ema import match_state_dicts
from sfod_b200.structures import Boxes, ImageList, Instances, pairwise_iou

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ C ABI
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "sfod_b200.h")).read()
    declared = set(re.findall(r"\b(sfod_[a-z0-9_]+)\s*\(", header))
    declared -= {"sfod_status", "sfod_layout", "sfod_dtype"}
    assert len(declared) >= 24
    lib = C.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in include/sfod_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    # exported symbols are exactly the ABI (everything else is hidden)
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert {e for e in exported if e.startswith("sfod_")} == declared


def test_host_only_entry_points():
    L = _lib.lib()
    launches = L.sfod_debug_launch_count()                      # non-zero when GPU tests ran earlier in this process
    assert L.sfod_abi_version() == 1
    # the ctypes mirrors of the parameter structs have the C layout (sizeof as compiled into the library)
    for which, mirror in enumerate((_lib.EmaTensor, _lib.RpnParams, _lib.FrcnnParams, _lib.P2PComm, _lib.JitterParams, _lib.EraseParams)):
        assert L.sfod_abi_sizeof(which) == C.sizeof(mirror), (which, mirror.__name__, L.sfod_abi_sizeof(which), C.sizeof(mirror))
    assert L.sfod_abi_sizeof(99) == 0
    assert L.sfod_status_string(0) == b"ok" and L.sfod_status_string(2) == b"workspace too small"
    assert L.sfod_nms_workspace_bytes(0) == 256 and L.sfod_nms_workspace_bytes(9990) > 9990 * 157 * 8
    rec = (128 + 8 * 18) * 4                                                                           # per-ROI table record (kRecHead + 8 H floats)
    assert L.sfod_roi_align_fwd_workspace_bytes(8, 512, 18, 37, 16000, 0, 0) >= 8 * 512 * 18 * 37 * 4 + 16000 * rec   # NCHW in -> NHWC copy + records
    cls = 16000 * 16 * 4                                                                               # cost-class lists of the L2 forward
    assert 16000 * rec <= L.sfod_roi_align_fwd_workspace_bytes(8, 512, 18, 37, 16000, 1, 0) <= 16000 * rec + cls + 1024
    assert L.sfod_roi_align_fwd_workspace_bytes(8, 512, 18, 37, 16000, 0, 1) == 256                 # exact kernel reads NCHW directly
    assert L.sfod_bn_stats_bytes(512) >= 512 * 4 * 8
    # peer-memory statistic exchange: inbox = header + 2 parities x 8 ranks x (2 * 2048 + 1 rounded up) 16-byte (value, tag) elements; argument checks
    # happen before any CUDA call
    assert L.sfod_p2p_max_channels() == 2051 and L.sfod_p2p_inbox_bytes() == 256 + 2 * 8 * 4104 * 16
    comm = _lib.P2PComm(); comm.rank, comm.world = 0, 2
    comm.inbox[0] = 0x1000                                                                                # inbox[1] missing
    a = [None] * 4 + [0, 8, 64, 20, 20, 0x2000]
    tail = [None] * 5 + [0.1, 1e-5, 0, 0, None, None, None]
    assert L.sfod_bn_exchange_finalize_apply(*a, C.byref(comm), *tail) == 1
    comm.inbox[1] = 0x3000; comm.world = 9
    assert L.sfod_bn_exchange_finalize_apply(*a, C.byref(comm), *tail) == 1
    comm.world = 2
    a[6] = 2052                                                                                           # C beyond the payload slot
    assert L.sfod_bn_exchange_finalize_apply(*a, C.byref(comm), *tail) == 3
    assert L.sfod_p2p_status(C.byref(_lib.P2PComm()), None, None) == 1 and L.sfod_p2p_open(None, None) == 1
    p = _lib.RpnParams(); p.N, p.HWA, p.pre_nms_topk, p.post_nms_topk = 8, 9990, 12000, 2000
    assert L.sfod_rpn_select_workspace_bytes(C.byref(p)) > 8 * 9990 * 157 * 8
    # EMA plan: 16384-element chunks, built on the host
    arr = (_lib.EmaTensor * 2)()
    arr[0].student, arr[0].teacher, arr[0].numel, arr[0].dtype = 0x1000, 0x2000, 40000, 0
    arr[1].student, arr[1].teacher, arr[1].numel, arr[1].dtype = 0x9000, 0xA000, 1, 1
    n = L.sfod_ema_plan_chunks(arr, 2)
    assert n == 4
    buf = (C.c_char * L.sfod_ema_plan_bytes(n))()
    assert L.sfod_ema_plan_build(arr, 2, buf, len(buf)) == 0
    assert L.sfod_ema_plan_build(arr, 2, buf, 8) == 2           # SFOD_ERR_WORKSPACE_TOO_SMALL
    arr[1].dtype = 7
    assert L.sfod_ema_plan_build(arr, 2, buf, len(buf)) == 3    # SFOD_ERR_UNSUPPORTED
    assert L.sfod_debug_launch_count() == launches              # nothing was launched by any of the above


def test_product_never_imports_oracle_and_has_no_cpu_fallback():
    pkg = os.path.join(ROOT, "simple-sfod_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f"{f} imports the oracle"
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.nms(torch.zeros(3, 4), torch.zeros(3), 0.5)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.roi_align(torch.zeros(1, 4, 8, 8), torch.zeros(1, 5), 7)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        modeling.Box2BoxTransform((1, 1, 1, 1)).apply_deltas(torch.zeros(2, 4), torch.zeros(2, 4))


# ------------------------------------------------------------------------------------------------ structures / registries / config
def test_structures_follow_detectron2():
    b = Boxes(torch.tensor([[-5.0, 2.0, 30.0, 50.0], [4.0, 4.0, 4.0, 9.0]]))
    b.clip((40, 20))
    assert b.tensor.tolist() == [[0.0, 2.0, 20.0, 40.0], [4.0, 4.0, 4.0, 9.0]]
    assert b.nonempty().tolist() == [True, False] and b.area().tolist() == [760.0, 0.0]
    assert len(Boxes.cat([b, b])) == 4 and len(Boxes(torch.zeros(0))) == 0
    inst = Instances((40, 20))
    inst.pred_boxes = b
    inst.scores = torch.tensor([0.9, 0.1])
    assert len(inst) == 2 and inst.has("scores") and inst[inst.scores > 0.5].pred_boxes.tensor.shape == (1, 4)
    with pytest.raises(AssertionError):
        inst.pred_classes = torch.zeros(3)
    with pytest.raises(AttributeError):
        inst.nope
    assert len(Instances.cat([inst, inst])) == 4
    il = ImageList.from_tensors([torch.ones(3, 10, 12), torch.ones(3, 8, 16)], size_divisibility=32)
    assert il.tensor.shape == (2, 3, 32, 32) and il.image_sizes == [(10, 12), (8, 16)] and il[1].shape == (3, 8, 16)
    iou = pairwise_iou(Boxes(torch.tensor([[0.0, 0, 10, 10]])), Boxes(torch.tensor([[0.0, 0, 10, 5], [20.0, 20, 30, 30]])))
    assert iou.tolist() == [[0.5, 0.0]]


def test_registries_and_config():
    cfg = config.vgg_source_free_cfg()
    assert cfg.MODEL.PROPOSAL_GENERATOR.NAME == "PseudoLabRPN" and cfg.MODEL.RPN.PRE_NMS_TOPK_TRAIN == 12000
    assert cfg.MODEL.RPN.POST_NMS_TOPK_TEST == 1000 and cfg.SEMISUPNET.BBOX_THRESHOLD == 0.8 and cfg.MODEL.ROI_HEADS.NUM_CLASSES == 8
    assert registry.PROPOSAL_GENERATOR_REGISTRY.get("PseudoLabRPN") is modeling.PseudoLabRPN
    assert registry.ROI_HEADS_REGISTRY.get("SourceFreeAdaptiveTeacherStandardROIHeads") is modeling.SourceFreeAdaptiveTeacherStandardROIHeads
    with pytest.raises(KeyError):
        registry.ROI_HEADS_REGISTRY.get("NoSuchHeads")
    cfg.MODEL.DEVICE = "cpu"
    m = registry.build_model(cfg)
    sd = m.state_dict()
    assert sum(v.numel() for v in sd.values()) == 47636547 and sum(p.numel() for p in m.parameters()) == 47628086   # SURVEY.md App. C
    # reference state_dict keys (vgg.py stage slicing, d2 module names)
    for k in ("backbone.vgg0.0.weight", "backbone.vgg4.7.running_var", "proposal_generator.rpn_head.anchor_deltas.bias",
              "roi_heads.box_head.fc2.weight", "roi_heads.box_predictor.bbox_pred.weight", "DC_img.classifier.bias",
              "DC_ins.da_ins_fc3_level_vgg4.weight"):
        assert k in sd, k
    assert m.backbone.output_shape()["vgg4"].stride == 32 and m.proposal_generator.anchor_generator.num_anchors == [15]
    assert m.roi_heads.box_predictor.bbox_pred.out_features == 32 and m.roi_heads.box_head.fc1.in_features == 25088
    r = config.r101_c4_source_free_cfg()
    assert r.MODEL.ANCHOR_GENERATOR.SIZES == [[64, 128, 256, 512]] and r.MODEL.ROI_BOX_HEAD.FC_DIM == 2048
    # CPU forward of the BN module defers to nn.BatchNorm2d (native path only for CUDA train/no_grad)
    bn = modeling.SfodBatchNorm2d(4)
    ref = torch.nn.BatchNorm2d(4)
    x = torch.randn(2, 4, 5, 5)
    assert torch.equal(bn(x), ref(x)) and torch.equal(bn.running_var, ref.running_var)


def test_ema_key_matching_and_sharding_host_logic():
    t = {"a": torch.zeros(2), "b": torch.zeros(1)}
    s = {"module.a": torch.ones(2), "module.b": torch.ones(1), "module.extra": torch.ones(1)}
    pairs = match_state_dicts(s, t, strip_module_prefix=True)
    assert [k for k, _, _ in pairs] == ["a", "b"] and pairs[0][1] is s["module.a"] and pairs[0][2] is t["a"]
    with pytest.raises(Exception, match="b is not found in student model"):
        match_state_dicts({"a": torch.ones(2)}, t, False)
    assert engine.images_per_rank(8, 4) == 2
    with pytest.raises(AssertionError):
        engine.images_per_rank(8, 3)
    cover = []
    for r in range(3):
        b, e = engine.shard_range(10, r, 3)
        cover += list(range(b, e))
    assert cover == list(range(10))
    # reset_bn_stats semantics (reference base.py:318-323)
    m = torch.nn.Sequential(torch.nn.Conv2d(3, 4, 1), torch.nn.BatchNorm2d(4))
    m[1].running_mean.fill_(3.0)
    engine.recursive_traversal(m)
    assert isinstance(m[1].running_mean, torch.nn.Parameter) and not m[1].running_mean.requires_grad
    assert m[1].running_mean.sum() == 0 and m[1].running_var.sum() == 4 and "1.running_mean" in m.state_dict()
    modeling.convert_batchnorm(m)
    assert isinstance(m[1], modeling.SfodBatchNorm2d) and isinstance(m[1].running_mean, torch.nn.Parameter)


# ------------------------------------------------------------------------------------------------ world_size 2 (gloo)
_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SFOD_ROOT"])
import sfod_b200
from sfod_b200 import engine
from sfod_b200.engine.adabn_dist import allreduce_bn_stats, finalize_stats_host
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
g = torch.Generator().manual_seed(123)
full = torch.randn(6, 5, 7, 9, generator=g, dtype=torch.float64) * 3 + 2       # the concatenated batch of both ranks
b, e = engine.shard_range(full.shape[0], rank, world)
mine = full[b:e]
stats = torch.stack([mine.sum(dim=(0, 2, 3)), (mine * mine).sum(dim=(0, 2, 3))], dim=1).reshape(-1)   # (C, 2) layout of the kernel
payload = torch.cat([stats, torch.tensor([float(mine.numel() // 5)], dtype=torch.float64)])
total = allreduce_bn_stats(payload, 5)
mean, var = finalize_stats_host(payload, 5, total)
ref_mean = full.mean(dim=(0, 2, 3)); ref_var = full.var(dim=(0, 2, 3), unbiased=False)
assert total == 6 * 7 * 9, total
assert torch.allclose(mean, ref_mean, rtol=1e-12, atol=1e-12) and torch.allclose(var, ref_var, rtol=1e-10), (mean, ref_mean)
# the sync-free variant (round 2): the global count stays inside the payload, where phase 2 of the kernels reads it
from sfod_b200.engine.adabn_dist import allreduce_bn_stats_device
payload2 = torch.cat([stats, torch.tensor([float(mine.numel() // 5)], dtype=torch.float64)])
assert allreduce_bn_stats_device(payload2, 5) is None
assert torch.equal(payload2, payload) and payload2[10].item() == 6 * 7 * 9
# the shim's detectron2.utils.comm is rank-aware (ADVICE r1): one main process, gather / all_gather of picklable objects
from sfod_b200 import d2shim
d2shim.install(force=True)
import detectron2.utils.comm as comm
assert comm.get_world_size() == world and comm.get_rank() == rank and comm.is_main_process() == (rank == 0)
got = comm.gather({"rank": rank}, dst=0)
assert (got == [{"rank": 0}, {"rank": 1}]) if rank == 0 else (got == [])
assert comm.all_gather(rank * 10) == [0, 10]
comm.synchronize()
d2shim.uninstall()
# the peer-memory exchange cannot exist without GPUs: construction must fail on EVERY rank with the same collective sequence
# (no rank may be left waiting in a collective or, on a GPU box, polling for a payload that never comes)
from sfod_b200.engine.p2p import PeerStatExchange
if not torch.cuda.is_available():
    try:
        PeerStatExchange.from_process_group(device="cuda:0")
        raise SystemExit("PeerStatExchange must not come up without a GPU")
    except RuntimeError as e:
        assert "peer memory is not usable" in str(e) and "rank 0" in str(e) and "rank 1" in str(e), str(e)
dist.barrier()
if rank == 0:
    print("GLOO_OK")
'''


def test_world_size_2_gloo_sharding_and_bn_stat_reduction(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, SFOD_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29517", str(script)], capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0 and "GLOO_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_pseudo_label_export_formats():
    """SURVEY.md 8f rank 4: COCO result json of detections, prediction_to_gt (score >= 0.7, ids from 1), detector_postprocess."""
    inst = Instances((600, 1200))
    inst.pred_boxes = Boxes(torch.tensor([[10.0, 20.0, 110.0, 220.0], [0.0, 0.0, 1200.0, 600.0], [5.0, 5.0, 6.0, 6.0]]))
    inst.scores = torch.tensor([0.9, 0.75, 0.3])
    inst.pred_classes = torch.tensor([2, 0, 7])
    res = engine.instances_to_coco_json(inst, 42)
    assert res[0] == {"image_id": 42, "category_id": 2, "bbox": [10.0, 20.0, 100.0, 200.0], "score": pytest.approx(0.9)}
    assert [r["category_id"] for r in engine.instances_to_coco_json(inst, 1, id_map={0: 24, 2: 26, 7: 33})] == [26, 24, 33]
    assert engine.instances_to_coco_json(inst[inst.scores > 2], 1) == []
    ds = {"images": [{"id": 42}], "categories": [], "annotations": [{"id": 99}]}
    out = engine.prediction_to_gt(res, ds, 0.7)
    assert [a["id"] for a in out["annotations"]] == [1, 2] and out["annotations"][1]["bbox"] == [0.0, 0.0, 1200.0, 600.0]
    assert "score" not in out["annotations"][0] and ds["annotations"] == [{"id": 99}]          # input untouched
    assert len(engine.prediction_to_gt([{"image_id": 1, "bbox": [0, 0, 1, 1], "category_id": 1, "score": 0.7}], ds)["annotations"]) == 1   # >= keeps 0.7
    pp = engine.detector_postprocess(inst, 1024, 2048)                                       # Cityscapes 1024x2048 <- 600x1200
    assert pp.image_size == (1024, 2048) and torch.allclose(pp.pred_boxes.tensor[0], torch.tensor([10.0, 20, 110, 220]) * (2048 / 1200))
    assert len(pp) == 3


def test_matcher_and_preprocessing_host_paths():
    """Host side of the two 8f widenings: `Matcher.match_boxes` keeps detectron2's two-step result on CPU tensors (the
    fused kernel is the CUDA path), argument errors are raised before any launch, and the native operators refuse CPU
    tensors instead of falling back."""
    from oracle import d2_cpu as oracle
    from sfod_b200.modeling.matcher import Matcher
    g = torch.Generator().manual_seed(11)
    gt = torch.rand(7, 4, generator=g) * 200; gt[:, 2:] += gt[:, :2]
    bx = torch.rand(300, 4, generator=g) * 200; bx[:, 2:] += bx[:, :2]
    for th, lb, lq in (([0.3, 0.7], [0, -1, 1], True), ([0.5], [0, 1], False)):
        m = Matcher(th, lb, allow_low_quality_matches=lq)
        a = m.match_boxes(Boxes(gt), Boxes(bx))
        b = m(pairwise_iou(Boxes(gt), Boxes(bx)))
        r = oracle.matcher(oracle.pairwise_iou(gt, bx), th, lb, lq)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[0], r[0]) and torch.equal(a[1], r[1])
    assert L_ws(0) == 256 and L_ws(1000) >= 4000
    with pytest.raises(RuntimeError):
        ops.iou_match(gt, bx, [0.5], [0, 1])                     # CPU tensors: no fallback
    with pytest.raises(RuntimeError):
        ops.normalize_pad(torch.zeros(2, 3, 8, 8, dtype=torch.uint8), (1.0, 2.0, 3.0), (1.0, 1.0, 1.0))
    # host-side validation of the C entry points (no device work is reached)
    L = _lib.lib()
    th = (C.c_float * 2)(0.7, 0.3)                               # thresholds must ascend
    lb = (C.c_int * 3)(0, -1, 1)
    assert L.sfod_iou_match(None, None, 0, 0, th, lb, 2, 0, None, None, None, None, 0, None) == 0      # N == 0: nothing to do
    assert L.sfod_iou_match(None, 16, 0, 4, th, lb, 2, 0, 16, 16, None, None, 0, None) == 1            # descending thresholds
    assert L.sfod_iou_match(None, 16, 0, 4, th, lb, 9, 0, 16, 16, None, None, 0, None) == 1            # too many thresholds
    mean = (C.c_float * 3)(1, 2, 3)
    assert L.sfod_normalize_pad(None, 2, 0, 0, 3, 8, 8, mean, mean, 8, 8, 0, None, None) == 0          # N == 0
    assert L.sfod_normalize_pad(16, 2, 192, 1, 3, 8, 8, mean, mean, 4, 8, 0, 16, None) == 1            # padded size < image size
    assert L.sfod_normalize_pad(16, 1, 192, 1, 3, 8, 8, mean, mean, 8, 8, 0, 16, None) == 1            # int64 images are not accepted
    assert L.sfod_normalize_pad(16, 2, 192, 1, 9, 8, 8, mean, mean, 8, 8, 0, 16, None) == 1            # more channels than supported


def L_ws(m):
    return _lib.lib().sfod_iou_match_workspace_bytes(m)


def test_resnet101_c4_backbone_layout_and_cpu_forward_matches_oracle():
    """BASELINE config [4]: detectron2's ResNet-101-C4 key layout (a detectron2 checkpoint loads unchanged), FREEZE_AT 2
    (stem + res2 -> FrozenBatchNorm2d: 11 of the 94 norm layers), and the module's plain-torch mode (CPU) equals the oracle's
    functional restatement bit for bit, in train (running statistics updated) and eval mode."""
    import torch
    from oracle import teacher_cpu
    from sfod_b200 import config, modeling
    from sfod_b200.modeling.resnet import FrozenBatchNorm2d
    cfg = config.r101_c4_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
    torch.manual_seed(0)
    bb = modeling.build_resnet_backbone(cfg)
    keys = list(bb.state_dict().keys())
    assert keys[:5] == ["stem.conv1.weight", "stem.conv1.norm.weight", "stem.conv1.norm.bias", "stem.conv1.norm.running_mean",
                        "stem.conv1.norm.running_var"]                              # frozen stem: no num_batches_tracked
    assert "res2.0.shortcut.norm.running_var" in keys and "res3.0.conv1.norm.num_batches_tracked" in keys
    assert "res4.22.conv3.norm.weight" in keys and not any(k.startswith("res5") for k in keys)
    assert sum(isinstance(m, FrozenBatchNorm2d) for m in bb.modules()) == 11
    assert sum(isinstance(m, torch.nn.BatchNorm2d) for m in bb.modules()) == 83
    assert not bb.stem.conv1.weight.requires_grad and not bb.res2[0].conv1.weight.requires_grad and bb.res3[0].conv1.weight.requires_grad
    assert bb.output_shape()["res4"].stride == 16 and bb.output_shape()["res4"].channels == 1024
    assert bb.res3[0].conv1.stride == (2, 2) and bb.res3[0].conv2.stride == (1, 1)   # STRIDE_IN_1X1
    x = torch.randn(2, 3, 64, 96, generator=torch.Generator().manual_seed(1))
    for training in (True, False):
        sd = {"backbone." + k: v.clone() for k, v in bb.state_dict().items()}
        bb.train(training)
        with torch.no_grad():
            got = bb(x)["res4"]
        want = teacher_cpu.resnet_c4_forward(sd, x, training)
        assert torch.equal(got, want)
        for k, v in bb.state_dict().items():
            assert torch.equal(v, sd["backbone." + k]), k
    # the whole detector of config [4] builds; checkpoint keys carry detectron2's prefixes
    model = modeling.SourceFreeAdaptiveTeacherGeneralizedRCNN(cfg)
    sdk = model.state_dict().keys()
    assert "backbone.res4.22.conv3.norm.running_mean" in sdk and "roi_heads.box_head.fc1.weight" in sdk
    assert model.roi_heads.box_head.fc1.weight.shape == (2048, 1024 * 7 * 7) and model.proposal_generator.anchor_generator.num_anchors[0] == 12


def test_strong_augmentation_parameter_draws_follow_the_reference_distributions():
    """Host half of SURVEY.md 8f rank 3: decisions drawn as reference daod/data/detection_utils.py:7-37 specifies
    (RandomApply 0.8 / RandomGrayscale 0.2 / blur 0.5 / erasers 0.7, 0.5, 0.3; factor and rectangle ranges)."""
    import torch
    from sfod_b200 import engine
    g = torch.Generator().manual_seed(1)
    ps = engine.draw_strong_augmentation_params(4000, 600, 1200, g)
    frac = lambda f: sum(1 for p in ps if f(p)) / len(ps)  # noqa: E731
    assert abs(frac(lambda p: bool(p["order"])) - 0.8) < 0.03 and abs(frac(lambda p: p["grayscale"]) - 0.2) < 0.03
    assert abs(frac(lambda p: p["sigma"] is not None) - 0.5) < 0.03
    assert abs(sum(len(p["rects"]) for p in ps) / len(ps) - (0.7 + 0.5 + 0.3)) < 0.06
    for p in ps:
        assert sorted(p["order"]) in ([], [0, 1, 2, 3])
        for o, f in zip(p["order"], p["factors"]):
            lo, hi = [(0.6, 1.4), (0.6, 1.4), (0.6, 1.4), (-0.1, 0.1)][o]
            assert lo <= f <= hi
        assert p["sigma"] is None or 0.1 <= p["sigma"] <= 2.0
        for (i, j, h, w) in p["rects"]:
            assert 0 <= i and i + h <= 600 and 0 <= j and j + w <= 1200 and 0.015 * 720000 <= h * w <= 0.21 * 720000


def test_box_decode_and_probs_are_differentiable_when_a_gradient_is_requested():
    """ADVICE r1: detectron2's predict_boxes / predict_probs are differentiable (giou/diou losses, bpc_loss on convert_bbox_scores
    outputs); with autograd on, the mirror runs the same formula as torch ops instead of the (backward-less) kernels."""
    import torch
    from oracle import d2_cpu as o
    from sfod_b200.modeling import Box2BoxTransform
    g = torch.Generator().manual_seed(0)
    boxes = torch.rand(20, 4, generator=g) * 100; boxes[:, 2:] += boxes[:, :2] + 1
    deltas = (torch.randn(20, 32, generator=g) * 0.5).requires_grad_(True)
    t = Box2BoxTransform(weights=(10.0, 10.0, 5.0, 5.0))
    out = t.apply_deltas(deltas, boxes)
    assert out.requires_grad and torch.equal(out.detach(), o.apply_deltas(deltas.detach(), boxes, (10.0, 10.0, 5.0, 5.0)))
    out.sum().backward()
    assert deltas.grad is not None and torch.isfinite(deltas.grad).all() and deltas.grad.abs().sum() > 0


def test_head_layout_helper_inverts_the_reference_flatten():
    """The GPU tests of ``head_layout = 1`` build (N, A, H, W) / (N, 4A, H, W) inputs from flattened ones with
    ``test_gpu_kernels._head_layout``; that helper must be the exact inverse of the flatten of reference rpn.py:28-41
    (``RPN._flatten_head_outputs`` here, checked against the reference's own text in test_reference_plugins_cpu), so that the
    native-layout tests exercise the index mapping real head outputs have."""
    import importlib.util
    import types
    spec = importlib.util.spec_from_file_location("_gpu_kernel_tests", os.path.join(ROOT, "tests", "test_gpu_kernels.py"))
    tk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tk)
    from sfod_b200.modeling.proposal_generator import RPN
    g = torch.Generator().manual_seed(5)
    N, A, H, W = 2, 3, 4, 5
    logits4 = torch.randn(N, A, H, W, generator=g)
    deltas4 = torch.randn(N, 4 * A, H, W, generator=g)

    class _AG:
        box_dim = 4
    stub = types.SimpleNamespace(anchor_generator=_AG())
    flat_l, flat_d = RPN._flatten_head_outputs(stub, [logits4], [deltas4])
    assert flat_l[0].shape == (N, H * W * A) and flat_d[0].shape == (N, H * W * A, 4)
    # flattened index i = (h * W + w) * A + a  <->  logits4[n, a, h, w]; deltas4[n, 4a + k, h, w]
    n, a, h, w, k = 1, 2, 3, 4, 1
    i = (h * W + w) * A + a
    assert flat_l[0][n, i] == logits4[n, a, h, w] and flat_d[0][n, i, k] == deltas4[n, 4 * a + k, h, w]
    back_l, back_d = tk._head_layout(dict(H=H, W=W), flat_l[0], flat_d[0])
    assert torch.equal(back_l, logits4) and torch.equal(back_d, deltas4)

