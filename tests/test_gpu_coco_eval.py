"""COCO box AP on the device (ops.coco_box_eval through engine.COCOBoxEvaluator) against the oracle restatement of pycocotools'
COCOeval: precision / recall / scores arrays np.array_equal, summary stats and per-class APs ==."""
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import coco_eval_cpu as o
from sfod_b200 import config, engine, registry
from sfod_b200.engine.export import detector_postprocess, instances_to_coco_json
from sfod_b200.structures import Boxes, Instances
from coco_eval_cases import dense_case, known_answer_cases, synthetic_case, to_results

pytestmark = pytest.mark.gpu


def names(gt):
    return [c["name"] for c in sorted(gt["categories"], key=lambda c: c["id"])]


def device_outputs(dets, dev, image_size=(600, 1200), output_size=None):
    inputs, outputs = [], []
    for img, b, s, c in dets:
        inst = Instances(image_size)
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.to(dev)), s.to(dev), c.to(dev)
        inp = {"image_id": img}
        if output_size is not None:
            inp["height"], inp["width"] = output_size
        inputs.append(inp)
        outputs.append({"instances": inst})
    return inputs, outputs


def assert_same(got, want):
    for k in ("precision", "recall", "scores", "stats"):
        assert np.array_equal(got[k], want[k]), k
    assert got["bbox"].keys() == want["bbox"].keys()
    for k, v in want["bbox"].items():
        assert got["bbox"][k] == v or (math.isnan(v) and math.isnan(got["bbox"][k])), k


def evaluate_both(gt, dets, dev, split=1, image_size=(600, 1200), output_size=None):
    """(device evaluator: its result dict merged with its ``eval`` arrays, oracle on the detector_postprocess-ed results)."""
    ev = engine.COCOBoxEvaluator(gt)
    inputs, outputs = device_outputs(dets, dev, image_size, output_size)
    step = max(1, len(inputs) // split)
    for i in range(0, len(inputs), step):
        ev.process(inputs[i:i + step], outputs[i:i + step])
    got = ev.evaluate()
    assert set(got) == {"bbox"}
    want = o.evaluate_bbox(gt, to_results(gt, dets, image_size, output_size or image_size), names(gt))
    return {**ev.eval, **got}, want


@pytest.mark.parametrize("name", sorted(known_answer_cases()))
def test_known_answer_cases_equal_oracle(name, cuda_device):
    gt, dets = known_answer_cases()[name]
    got, want = evaluate_both(gt, dets, cuda_device)
    assert_same(got, want)


@pytest.mark.parametrize("seed,crowd,id_zero", [(0, 0.05, False), (1, 0.05, False), (2, 0.3, False), (3, 0.05, True)])
def test_synthetic_datasets_equal_oracle(seed, crowd, id_zero, cuda_device):
    gt, dets = synthetic_case(seed, 60, 5, 30, 130, crowd_frac=crowd, id_zero=id_zero)
    got, want = evaluate_both(gt, dets, cuda_device, split=4)
    assert_same(got, want)


def test_foggy_cityscapes_val_sized_dataset_equals_oracle(cuda_device):
    gt, dets = synthetic_case(11, 500, 8, 60, 100)
    got, want = evaluate_both(gt, dets, cuda_device, split=250)
    assert_same(got, want)
    assert 0 < got["bbox"]["AP"] < 100 and all(np.isfinite(got["bbox"]["AP-" + n]) for n in names(gt))


def test_iou_recomputed_when_the_table_does_not_fit(cuda_device):
    """100 detections x 50 gt in one (image, category): 5000 IoU pairs, beyond the 4096-entry shared-memory table."""
    gt, dets = dense_case()
    assert len(dets[0][1]) * len(gt["annotations"]) > 4096
    got, want = evaluate_both(gt, dets, cuda_device)
    assert_same(got, want)
    assert got["bbox"]["AP50"] > 0


def test_detections_are_rescaled_to_the_input_size(cuda_device):
    """Detections in the network frame (600 x 1200) of inputs whose height / width are 1024 x 2048: evaluated in the
    input's frame, as detectron2's detector_postprocess leaves them (scale, clip, empty boxes dropped)."""
    gt, dets = synthetic_case(21, 40, 4, 20, 60)
    sx, sy = 2048 / 1200, 1024 / 600
    for a in gt["annotations"]:
        x, y, w, h = a["bbox"]
        a["bbox"] = [x * sx, y * sy, w * sx, h * sy]
        a["area"] *= sx * sy
    # a few boxes reaching past the image and one collapsing to zero width after the clip
    img, b, s, c = dets[0]
    b = b.clone()
    b[0, 2] += 400.0
    b[1, 0], b[1, 2] = 1250.0, 1300.0
    dets[0] = (img, b, s, c)
    got, want = evaluate_both(gt, dets, cuda_device, split=3, output_size=(1024, 2048))
    assert_same(got, want)
    assert got["bbox"]["AP50"] > 10                     # without the rescale almost nothing would match


def test_several_records_of_one_image_are_concatenated(cuda_device):
    """loadRes takes the result list as it is: an image processed twice contributes both sets of detections, in order."""
    gt, dets = synthetic_case(5, 10, 3, 10, 40)
    dets = dets + [(img, b[::2], s[::2], c[::2]) for img, b, s, c in dets[:4]]
    got, want = evaluate_both(gt, dets, cuda_device)
    assert_same(got, want)


def test_unknown_image_id_raises(cuda_device):
    gt, dets = known_answer_cases()["perfect"]
    ev = engine.COCOBoxEvaluator(gt)
    inputs, outputs = device_outputs([(99,) + tuple(dets[0][1:])], cuda_device)
    ev.process(inputs, outputs)
    with pytest.raises(ValueError, match="coco set"):
        ev.evaluate()


@pytest.fixture(scope="module")
def teacher_eval(cuda_device):
    torch.manual_seed(42)
    cfg = config.vgg_source_free_cfg()
    cfg.MODEL.DEVICE = "cuda"
    return registry.build_model(cfg).eval(), cfg.MODEL.ROI_HEADS.NUM_CLASSES


def _synth_loader(dev, n=6, batch=2, out_hw=(544, 816)):
    """Images of 320 x 480 whose original size (the evaluation frame) is ``out_hw``, as a test loader's resize leaves them."""
    g = torch.Generator().manual_seed(17)
    ims = [torch.randint(0, 256, (3, 320, 480), dtype=torch.uint8, generator=g).to(dev) for _ in range(n)]
    ids = [10 + 3 * i for i in range(n)]
    return [[{"image": ims[j], "image_id": ids[j], "height": out_hw[0], "width": out_hw[1]} for j in range(i, min(n, i + batch))]
            for i in range(0, n, batch)], ids


class _Tee:
    def __init__(self, inner):
        self.inner, self.seen = inner, []

    def reset(self):
        self.inner.reset()

    def process(self, inputs, outputs):
        self.seen.append((inputs, outputs))
        self.inner.process(inputs, outputs)

    def evaluate(self):
        return self.inner.evaluate()


def test_end_to_end_teacher_equals_oracle(teacher_eval, cuda_device):
    model, K = teacher_eval
    loader, ids = _synth_loader(cuda_device)
    # ground truth: jittered copies of the teacher's own detections (so that matches happen) plus some crowd regions
    with torch.no_grad():
        first = [model(b) for b in loader]
    rng = np.random.default_rng(3)
    anns, aid = [], 1
    for batch, outs in zip(loader, first):
        for inp, out in zip(batch, outs):
            inst = detector_postprocess(out["instances"], inp["height"], inp["width"])
            for k, d in enumerate(instances_to_coco_json(inst, inp["image_id"])[:40:2]):
                x, y, w, h = (float(v) * (1 + rng.normal(0, 0.05)) for v in d["bbox"])
                anns.append({"id": aid, "image_id": inp["image_id"], "bbox": [x, y, w, h], "category_id": 100 + d["category_id"],
                             "iscrowd": int(k % 9 == 8), "area": w * h * 0.8})
                aid += 1
    gt = {"images": [{"id": i} for i in ids], "categories": [{"id": 100 + k, "name": f"k{k}"} for k in range(K)], "annotations": anns}
    tee = _Tee(engine.COCOBoxEvaluator(gt))
    got = engine.inference_on_dataset(model, loader, tee)
    assert set(got) == {"bbox"} and all(isinstance(v, float) for v in got["bbox"].values())   # what EvalHook accepts
    # the oracle sees the outputs as detectron2's GeneralizedRCNN.inference(do_postprocess=True) returns them
    results = [r for inputs, outputs in tee.seen for inp, out in zip(inputs, outputs)
               for r in instances_to_coco_json(detector_postprocess(out["instances"], inp["height"], inp["width"]), inp["image_id"],
                                               {k: 100 + k for k in range(K)})]
    assert len(results) > 0 and len(anns) > 0
    want = o.evaluate_bbox(gt, results, [f"k{k}" for k in range(K)])
    assert_same({**tee.inner.eval, **got}, want)
    assert got["bbox"]["AP50"] > 0                      # the gt are jittered copies of the rescaled detections


def test_process_does_not_synchronise_and_evaluate_once(teacher_eval, cuda_device):
    model, K = teacher_eval
    loader, ids = _synth_loader(cuda_device)
    gt = {"images": [{"id": i} for i in ids], "categories": [{"id": k, "name": str(k)} for k in range(K)],
          "annotations": [{"id": 1, "image_id": ids[0], "bbox": [10.0, 10.0, 100.0, 80.0], "category_id": 0, "iscrowd": 0, "area": 8000.0}]}
    ev = engine.COCOBoxEvaluator(gt)
    with torch.no_grad():
        outs = [model(b) for b in loader]
    for b, out in zip(loader, outs):           # warm-up: workspace, pinned staging, ground truth on the device
        ev.process(b, out)
    ev.evaluate()
    ev.reset()
    with torch.no_grad():
        outs = [model(b) for b in loader]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            for b, out in zip(loader, outs):
                ev.process(b, out)
            n_process = len([x for x in w if "synchroniz" in str(x.message).lower()])
            ev.evaluate()
            n_total = len([x for x in w if "synchroniz" in str(x.message).lower()])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert n_process == 0 and n_total == 1, [str(x.message)[:120] for x in w]
