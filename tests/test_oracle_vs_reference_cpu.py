"""Pins oracle/d2_cpu.py against the REFERENCE'S OWN on-disk functions, executed here on the CPU (SURVEY.md 8c).

tests/ref_exec.py imports / compiles the reference's functions from $SFOD_REFERENCE_ROOT (nothing is copied) and runs them with
``Boxes`` / ``Instances`` of the shim and detectron2 0.6's ``batched_nms`` one-liner over the installed torchvision CPU kernel.
Every comparison below is bit-exact (``torch.equal``): the oracle restates the same torch calls in the same order.
Skipped where the reference sources are absent: there the committed fixture tests/golden/ref_exec.npz --
generated from these same reference functions by tests/golden/make_golden_ref.py -- takes over (second half of this file).
"""
import os
import sys
from collections import OrderedDict

import numpy as np
import pytest
import torch
from torch import nn

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ref_exec  # noqa: E402
from oracle import d2_cpu as o  # noqa: E402
from sfod_b200 import synth  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_reference = pytest.mark.skipif(not ref_exec.available(), reason="original project sources not available (SFOD_REFERENCE_ROOT)")


@pytest.fixture(scope="module")
def R():
    with ref_exec.Reference() as r:
        yield r


def head_case(rows, K, seed, logit_std=4.0, delta_std=1.0, nonfinite=False):
    """(boxes (R,4K), scores (R,K+1)) the way d2's predict_boxes / predict_probs produce them (ATen exp / softmax)."""
    n = sum(rows)
    cls, dl = synth.box_head_outputs(n, K, seed, logit_std, delta_std)
    props = synth.random_rois(1, n, seed + 1)[:, 1:].contiguous()
    boxes = o.apply_deltas(dl, props, (10.0, 10.0, 5.0, 5.0))
    scores = torch.softmax(cls, -1)
    if nonfinite and n > 7:
        boxes[3, 1] = float("inf"); scores[5, 0] = float("nan"); boxes[7, 2] = float("-inf")
    return cls, dl, props, list(boxes.split(rows)), list(scores.split(rows))


def same(a: dict, b: dict, keys):
    for k in keys:
        assert torch.equal(a[k], b[k]), k
    assert tuple(a["image_size"]) == tuple(b["image_size"])


DET_KEYS = ("pred_boxes", "scores", "pred_classes", "kept_rows")
CASES = [  # rows per image, K, seed, logit std, delta std, image sizes, non-finite rows
    ([2000], 8, 101, 4.0, 1.0, [(600, 1200)], False),            # ~4 000 candidates: per-class NMS strategy of torchvision
    ([300, 0, 57], 8, 102, 4.0, 1.0, [(600, 1200), (600, 1200), (300, 500)], False),   # <= 1000: coordinate trick; an empty image
    ([2000], 8, 103, 0.05, 0.1, [(600, 1200)], False),           # random-init-like: all 16 000 candidates pass 0.05
    ([1200], 1, 104, 3.0, 1.0, [(600, 1200)], False),            # single class (class-agnostic-shaped boxes)
    ([600, 500], 8, 105, 4.0, 1.0, [(600, 1200), (576, 1100)], True),  # non-finite rows are dropped first
]


# ================================================================================================ live: reference executed here
@needs_reference
@pytest.mark.parametrize("case", CASES, ids=[f"seed{c[2]}" for c in CASES])
def test_fast_rcnn_inference_single_image_equals_reference(R, case):
    """reference daod/modeling/roi_heads/fast_rcnn.py:88-142 == oracle fast_rcnn_inference_single_image."""
    rows, K, seed, ls, ds, sizes, nonfinite = case
    _, _, _, boxes, scores = head_case(rows, K, seed, ls, ds, nonfinite)
    for b, s, sz in zip(boxes, scores, sizes):
        ref = R.fast_rcnn_inference_single_image(b.clone(), s.clone(), sz, 0.05, 0.5, 100)
        ours = o.fast_rcnn_inference_single_image(b.clone(), s.clone(), sz, 0.05, 0.5, 100)
        if nonfinite:                      # the reference reports rows of the FILTERED tensor; the oracle maps them back
            valid = (torch.isfinite(b).all(1) & torch.isfinite(s).all(1)).nonzero().flatten()
            ref["kept_rows"] = valid[ref["kept_rows"]]
        same(ref, ours, DET_KEYS)
        # topk < 0 returns everything that survives NMS
        ref_all = R.fast_rcnn_inference_single_image(b.clone(), s.clone(), sz, 0.05, 0.5, -1)
        ours_all = o.fast_rcnn_inference_single_image(b.clone(), s.clone(), sz, 0.05, 0.5, -1)
        # (torchvision's final sort over the kept scores is unstable on exact score ties -- SURVEY.md B-4; the oracle breaks ties
        #  by index, so beyond the scores themselves the comparison is on the SET of (row, class) detections)
        assert torch.equal(ref_all["scores"], ours_all["scores"])
        rows_ref = ref_all["kept_rows"] if not nonfinite else valid[ref_all["kept_rows"]]
        assert sorted(zip(rows_ref.tolist(), ref_all["pred_classes"].tolist())) == sorted(zip(ours_all["kept_rows"].tolist(), ours_all["pred_classes"].tolist()))


@needs_reference
@pytest.mark.parametrize("case", CASES[:3], ids=[f"seed{c[2]}" for c in CASES[:3]])
def test_convert_bbox_scores_equals_reference(R, case):
    """reference source_free_fast_rcnn.py:15-36,82-147 (decode + clip, ``scores > 0``, no NMS) == oracle."""
    rows, K, seed, ls, ds, sizes, _ = case
    cls, dl, props, boxes, scores = head_case(rows, K, seed, ls, ds)
    for b, s, sz in zip(boxes, scores, sizes):
        same(R.fast_rcnn_inference_single_image_new(b.clone(), s.clone(), sz), o.convert_bbox_scores_single_image(b.clone(), s.clone(), sz), DET_KEYS)

    # the whole method, with detectron2's predict_boxes / predict_probs (not on disk) supplied by the oracle's restatement
    class Stub:
        test_score_thresh, test_nms_thresh, test_topk_per_image = 0.05, 0.5, 100
        predict_boxes = staticmethod(lambda predictions, proposals: o.predict_boxes(predictions[1], [p.proposal_boxes.tensor for p in proposals]))
        predict_probs = staticmethod(lambda predictions, proposals: o.predict_probs(predictions[0], [len(p) for p in proposals]))
    cls_ = R.sf_fast_rcnn.SourceFreeFastRCNNOutputLayers
    Stub.fast_rcnn_inference_new = lambda self, *a: cls_.fast_rcnn_inference_new(self, *a)
    Stub.fast_rcnn_inference_single_image_new = lambda self, *a: cls_.fast_rcnn_inference_single_image_new(self, *a)
    proposals = []
    for p, sz in zip(props.split(rows), sizes):
        inst = R.Instances(sz); inst.proposal_boxes = R.Boxes(p); proposals.append(inst)
    insts, kept = cls_.convert_bbox_scores(Stub(), (cls, dl), proposals)
    for inst, rows_i, b, s, sz in zip(insts, kept, boxes, scores, sizes):
        want = o.convert_bbox_scores_single_image(b.clone(), s.clone(), sz)
        got = R.from_instances(inst); got["kept_rows"] = rows_i
        same(got, want, DET_KEYS)


@needs_reference
def test_threshold_bbox_and_process_pseudo_label_equal_reference(R):
    """reference source_free_adaptive_teacher.py:150-183, 256-280 (and the identical adaptive_teacher.py:116-149)."""
    _, _, _, boxes, scores = head_case([2000, 900], 8, 111)
    dets = [o.fast_rcnn_inference_single_image(b, s, (600, 1200), 0.05, 0.5, 100) for b, s in zip(boxes, scores)]
    assert sum(int((d["scores"] > 0.8).sum()) for d in dets) > 10          # a non-empty pseudo-label set
    t, t_at = R.trainer(), R.TrainerAT()
    for thr in (0.8, 0.5, 0.999999, 0.0):
        for d in dets:
            want = o.threshold_bbox(d, thr, "roih")
            for tr in (t, t_at):
                got = R.from_instances(tr.threshold_bbox(R.to_instances({k: v for k, v in d.items() if k != "kept_rows"}), thres=thr, proposal_type="roih"))
                same(got, want, ("gt_boxes", "gt_classes", "scores"))
        ref_list, ref_n = t.process_pseudo_label([R.to_instances({k: v for k, v in d.items() if k != "kept_rows"}) for d in dets], thr, "roih", "thresholding")
        our_list, our_n = o.process_pseudo_label(dets, thr, "roih")
        assert ref_n == our_n
        for a, b in zip(ref_list, our_list):
            same(R.from_instances(a), b, ("gt_boxes", "gt_classes", "scores"))
    # RPN branch: objectness_logits > thres
    g = torch.Generator().manual_seed(5)
    prop = dict(image_size=(600, 1200), proposal_boxes=torch.rand(300, 4, generator=g) * 500, objectness_logits=torch.randn(300, generator=g))
    got = R.from_instances(t.threshold_bbox(R.to_instances(prop), thres=0.3, proposal_type="rpn"))
    same(got, o.threshold_bbox(prop, 0.3, "rpn"), ("gt_boxes", "objectness_logits"))
    with pytest.raises(ValueError, match="Unkown pseudo label boxes methods"):
        t.process_pseudo_label([R.to_instances(prop)], 0.5, "rpn", "")
    with pytest.raises(ValueError, match="Unkown pseudo label boxes methods"):
        o.process_pseudo_label([prop], 0.5, "rpn", "")


@needs_reference
def test_adaptive_threshold_path_equals_reference(R):
    """reference adaptive_confidence.py:6-33 and source_free_adaptive_teacher.py:185-254, 282-310 (``.cuda()`` neutralised)."""
    _, _, _, boxes, scores = head_case([1500, 1500, 1500], 8, 121)
    dets = [o.fast_rcnn_inference_single_image(b, s, (600, 1200), 0.05, 0.5, 100) for b, s in zip(boxes, scores)]
    insts = lambda: [R.to_instances({k: v for k, v in d.items() if k != "kept_rows"}) for d in dets]  # noqa: E731
    acc = torch.tensor([1.0, 0.3, 1.0, 0.9, 0.05, 0.6, 0.0, 0.45])

    class Cfg:                                    # the two keys count_label_prediction reads
        class MODEL:
            class ROI_HEADS:
                NUM_CLASSES = 8
        class SEMISUPNET:
            BBOX_THRESHOLD = 0.8
    with ref_exec.cpu_is_the_device():
        t = R.trainer(cfg=Cfg, classwise_acc=acc.clone(), threshold=0.8)
        # mask of the criterion itself
        for d in dets:
            assert torch.equal(t.self_training_criterion(d["scores"], d["pred_classes"]), o.adaptive_confidence_mask(d["scores"], d["pred_classes"], 0.8, acc))
        for method, as_gt in (("adaptive_thresholding", True), ("prediction_thresholding", False)):
            ref_list, ref_n = t.process_pseudo_label(insts(), 0.8, "roih", method)
            keys = ("gt_boxes", "gt_classes", "scores") if as_gt else ("pred_boxes", "pred_classes", "scores")
            tot = 0
            for a, d in zip(ref_list, dets):
                want = o.adaptive_threshold_bbox(d, 0.8, acc, as_gt=as_gt)
                same(R.from_instances(a), want, keys)
                tot += len(want["scores"])
            assert ref_n == tot / len(dets) and tot > 0
        # class histogram of a batch, reserve matrix -> new per-class accuracy
        reserve = t.count_label_prediction(insts())
        assert torch.equal(reserve, o.count_label_prediction(dets, 8, 0.8)) and reserve.sum() > 0
        t.reserve_matrix = torch.stack([reserve, reserve * 2, torch.zeros(8)])
        t.update_adaptive_threshold()
        assert torch.equal(t.self_training_criterion.classwise_acc, o.update_adaptive_threshold(torch.stack([reserve, reserve * 2, torch.zeros(8)])))
        # the criterion's own update() (bincount / max)
        labels = torch.cat([d["pred_classes"] for d in dets])
        t.self_training_criterion.update(labels)
        sigma = labels.bincount(minlength=8)
        assert torch.equal(t.self_training_criterion.classwise_acc, sigma / sigma.max())


def _small_models(seed):
    torch.manual_seed(seed)
    def make():
        return nn.Sequential(OrderedDict(conv=nn.Conv2d(3, 8, 3), bn=nn.BatchNorm2d(8), inner=nn.Sequential(nn.Linear(4, 5), nn.BatchNorm2d(3))))
    s, t = make(), make()
    s.train(); t.train()
    with torch.no_grad():
        s.bn.num_batches_tracked += 1000; t.bn.num_batches_tracked += 7
        s.bn.running_mean.normal_(); t.bn.running_var.uniform_(0.5, 2)
    return s, t


@needs_reference
@pytest.mark.parametrize("keep_rate", [0.9996, 0.999696, 0.0, 1.0])
def test_update_teacher_model_equals_reference(R, keep_rate):
    """reference source_free_adaptive_teacher.py:583-603 (== adaptive_teacher.py:339-358): formula, int64 buffers, DDP prefix,
    missing-key exception; the result is what load_state_dict then copies into the teacher."""
    for cls in (R.Trainer, R.TrainerAT):
        student, teacher = _small_models(7)
        s_sd = {k: v.clone() for k, v in student.state_dict().items()}
        t_sd = {k: v.clone() for k, v in teacher.state_dict().items()}
        tr = cls(); tr.model, tr.model_teacher = student, teacher
        tr._update_teacher_model(keep_rate=keep_rate)
        want = o.update_teacher_model(s_sd, t_sd, keep_rate)
        o.load_state_dict_like(t_sd, want)
        got = teacher.state_dict()
        assert list(got) == list(t_sd)
        for k in got:
            assert got[k].dtype == t_sd[k].dtype and torch.equal(got[k], t_sd[k]), k
        assert got["bn.num_batches_tracked"].dtype == torch.int64
    # DDP: student keys carry the "module." prefix when world_size > 1
    student, teacher = _small_models(8)
    wrapped = nn.Sequential(OrderedDict(module=student))
    s_sd = {k: v.clone() for k, v in wrapped.state_dict().items()}
    t_sd = {k: v.clone() for k, v in teacher.state_dict().items()}
    tr = R.Trainer(); tr.model, tr.model_teacher = wrapped, teacher
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(R.comm, "get_world_size", lambda: 2)
        tr._update_teacher_model(keep_rate=keep_rate)
    want = o.update_teacher_model(s_sd, t_sd, keep_rate, ddp_prefix=True)
    o.load_state_dict_like(t_sd, want)
    for k, v in teacher.state_dict().items():
        assert torch.equal(v, t_sd[k]), k
    # a teacher key that the student lacks
    teacher.add_module("extra", nn.Linear(2, 2))
    tr = R.Trainer(); tr.model, tr.model_teacher = student, teacher
    with pytest.raises(Exception, match="extra.weight is not found in student model"):
        tr._update_teacher_model(keep_rate=keep_rate)
    with pytest.raises(Exception, match="extra.weight is not found in student model"):
        o.update_teacher_model(student.state_dict(), teacher.state_dict(), keep_rate)


@needs_reference
def test_reset_bn_stats_equals_reference(R, capsys):
    """reference base.py:318-328: running statistics become fresh non-trainable Parameters (0, 1); num_batches_tracked is NOT reset."""
    a, _ = _small_models(9)
    b, _ = _small_models(9)
    R.recursive_traversal(a); R.recursive_traversal(a)
    o.recursive_traversal(b); o.recursive_traversal(b)
    capsys.readouterr()                                    # the reference prints every BN module
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb)
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    for m1, m2 in zip(a.modules(), b.modules()):
        if isinstance(m1, nn.BatchNorm2d):
            assert isinstance(m1.running_mean, nn.Parameter) and isinstance(m2.running_mean, nn.Parameter)
            assert not m1.running_mean.requires_grad and not m2.running_var.requires_grad
            assert m1.running_mean.abs().sum() == 0 and (m1.running_var == 1).all()
    assert sa["bn.num_batches_tracked"].item() == 1000
    # the product's mirror does the same
    from sfod_b200.engine import adabn
    c, _ = _small_models(9)
    adabn.recursive_traversal(c); adabn.recursive_traversal(c)
    for k, v in c.state_dict().items():
        assert torch.equal(v, sa[k]), k


@needs_reference
def test_pseudolab_rpn_flatten_equals_reference(R):
    """reference rpn.py:25-58 executed with its own class: the tensors it hands to ``predict_proposals`` are the oracle's
    ``rpn_flatten_head_outputs`` of the head outputs, and the anchors are the oracle's grid."""
    import importlib
    import types
    import detectron2.modeling as d2m
    from sfod_b200 import config
    from sfod_b200.structures import ImageList
    pkg = types.ModuleType("refexec_pg"); pkg.__path__ = [os.path.join(ref_exec.REF_ROOT, "daod/modeling/proposal_generator")]
    sys.modules["refexec_pg"] = pkg
    importlib.import_module("refexec_pg.rpn")
    cfg = config.vgg_source_free_cfg(); cfg.MODEL.DEVICE = "cpu"
    torch.manual_seed(1)
    from sfod_b200.structures import ShapeSpec
    rpn = d2m.build_proposal_generator(cfg, {"vgg4": ShapeSpec(channels=512, stride=32)})
    assert type(rpn).__module__ == "refexec_pg.rpn"
    seen = {}

    def capture(anchors, logits, deltas, image_sizes):
        seen.update(anchors=anchors, logits=logits, deltas=deltas, image_sizes=image_sizes)
        return ["proposals"]
    rpn.predict_proposals = capture
    feats = {"vgg4": torch.randn(2, 512, 5, 7)}
    rpn.eval()
    out, losses = rpn(ImageList(torch.zeros(2, 3, 160, 224), [(160, 224), (150, 200)]), feats, None, compute_loss=False)
    assert out == ["proposals"] and losses == {}
    obj, dl = rpn.rpn_head([feats["vgg4"]])
    want_l, want_d = o.rpn_flatten_head_outputs(obj, dl)
    assert torch.equal(seen["logits"][0], want_l[0]) and torch.equal(seen["deltas"][0], want_d[0])
    assert seen["deltas"][0].shape == (2, 5 * 7 * 15, 4) and seen["image_sizes"] == [(160, 224), (150, 200)]
    anchors = seen["anchors"][0]
    anchors = anchors.tensor if hasattr(anchors, "tensor") else anchors
    assert torch.equal(anchors, o.grid_anchors((5, 7), 32, o.generate_cell_anchors()))


# ================================================================================================ fixture: reference outputs that travel
@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "ref_exec.npz"))


def test_oracle_reproduces_reference_executed_fixture(gold):
    """tests/golden/ref_exec.npz was written by tests/golden/make_golden_ref.py FROM THE REFERENCE'S FUNCTIONS; the oracle must
    reproduce it bit for bit wherever the tests run (this one also runs on the GPU box)."""
    t = lambda k: torch.from_numpy(gold[k])  # noqa: E731
    n_img = int(gold["frcnn_n_images"])
    for i in range(n_img):
        sz = tuple(int(v) for v in gold[f"frcnn_{i}_image_size"])
        got = o.fast_rcnn_inference_single_image(t(f"frcnn_{i}_boxes"), t(f"frcnn_{i}_scores"), sz, 0.05, 0.5, 100)
        for k in DET_KEYS:
            assert torch.equal(got[k], t(f"frcnn_{i}_out_{k}")), (i, k)
        pl = o.threshold_bbox(got, 0.8, "roih")
        for k in ("gt_boxes", "gt_classes", "scores"):
            assert torch.equal(pl[k], t(f"frcnn_{i}_pl_{k}")), (i, k)
        conv = o.convert_bbox_scores_single_image(t(f"frcnn_{i}_boxes"), t(f"frcnn_{i}_scores"), sz)
        # the reference's scores of this path are the input scores at its kept (row, class) pairs, so only the pairs are stored
        conv_scores = t(f"frcnn_{i}_scores")[t(f"frcnn_{i}_conv_kept_rows"), t(f"frcnn_{i}_conv_pred_classes")]
        for k in DET_KEYS:
            assert torch.equal(conv[k], conv_scores if k == "scores" else t(f"frcnn_{i}_conv_{k}")), (i, k)
        ad = o.adaptive_threshold_bbox(got, 0.8, t("adaptive_acc"))
        for k in ("gt_boxes", "gt_classes", "scores"):
            assert torch.equal(ad[k], t(f"frcnn_{i}_adaptive_{k}")), (i, k)
    assert sum(len(gold[f"frcnn_{i}_pl_scores"]) for i in range(n_img)) >= 20      # the pseudo-label sets are not empty
    # EMA (incl. the int64 buffer) for three keep rates
    s_sd = OrderedDict((k[len("ema_s_"):], t(k)) for k in gold.files if k.startswith("ema_s_"))
    for tag, rate in (("a", 0.9996), ("b", 0.999696), ("c", 0.0)):
        t_sd = OrderedDict((k[len("ema_t_"):], t(k).clone()) for k in gold.files if k.startswith("ema_t_"))
        o.load_state_dict_like(t_sd, o.update_teacher_model(s_sd, t_sd, rate))
        for k, v in t_sd.items():
            assert torch.equal(v, t(f"ema_out_{tag}_{k}")), (tag, k)
    dets = [dict(scores=t(f"frcnn_{i}_out_scores"), pred_classes=t(f"frcnn_{i}_out_pred_classes")) for i in range(n_img)]
    assert torch.equal(o.count_label_prediction(dets, 8, 0.8), t("reserve_count"))
    assert torch.equal(o.update_adaptive_threshold(t("reserve_matrix").clone()), t("classwise_acc_new"))


@needs_reference
def test_prediction_to_gt_equals_the_reference_script_executed(tmp_path):
    """SURVEY.md 8f rank 4: the reference converts detections into the fixed-pseudo-label annotation file with a SCRIPT
    (cityscapes-to-coco-conversion/prediction_to_gt.py).  The script's own text is executed here with its three hard-coded paths
    redirected to temporary files (nothing is copied), and the json it writes must equal engine.prediction_to_gt's, entry by
    entry -- including the `score < 0.7` boundary, the running ids and the untouched rest of the dataset dict."""
    import json
    import re
    from sfod_b200 import engine
    src_path = os.path.join(ref_exec.REF_ROOT, "cityscapes-to-coco-conversion", "prediction_to_gt.py")
    src = open(src_path).read()
    rng = np.random.default_rng(5)
    preds = [{"image_id": int(rng.integers(1, 40)), "bbox": [float(v) for v in rng.uniform(0, 500, 4).round(2)],
              "category_id": int(rng.integers(1, 9)), "score": float(s)}
             for s in list(rng.uniform(0.05, 1.0, 300)) + [0.7, 0.7000000001, 0.6999999999]]
    dataset = {"images": [{"id": i, "file_name": f"{i}.png", "height": 600, "width": 1200} for i in range(1, 40)],
               "categories": [{"id": k, "name": f"c{k}"} for k in range(1, 9)], "annotations": [{"id": 99, "old": True}], "info": {"x": 1}}
    p_in, d_in, out = tmp_path / "preds.json", tmp_path / "dataset.json", tmp_path / "out.json"
    p_in.write_text(json.dumps(preds)); d_in.write_text(json.dumps(dataset))
    # the uncommented open() calls, in order: predictions (read), dataset (read), output (write)
    paths = iter([str(p_in), str(d_in), str(out)])
    lines = []
    for line in src.splitlines():
        if not line.lstrip().startswith("#") and "open(" in line:
            line = re.sub(r"open\('[^']*'", lambda m: "open(%r" % next(paths), line, count=1)
        lines.append(line)
    exec(compile("\n".join(lines), src_path, "exec"), {"__name__": "__ref_script__"})
    want = json.loads(out.read_text())
    got = engine.prediction_to_gt(preds, dataset, 0.7)
    assert got == want and len(want["annotations"]) == sum(p["score"] >= 0.7 for p in preds) and want["annotations"][0]["id"] == 1
    assert want["images"] == dataset["images"] and want["info"] == dataset["info"]
