"""COCO box-evaluation cases shared by tests/test_coco_eval_cpu.py (oracle known answers) and tests/test_gpu_coco_eval.py
(device vs oracle).  A case is (ground-truth COCO dict, detections) where the detections are per-image tuples
(image_id, boxes XYXY fp32 (n, 4), scores fp32 (n,), class indices int64 (n,)) -- what a detector's Instances hold.  The
oracle sees them as ``instances_to_coco_json`` writes them (XYWH computed in fp32, class index -> category id)."""
from __future__ import annotations

from typing import Dict, List, Tuple

import numpy as np
import torch

Det = Tuple[int, torch.Tensor, torch.Tensor, torch.Tensor]


def gt_dict(images, anns, cats=(1,)) -> dict:
    return {"images": [{"id": i, "height": 600, "width": 1200} for i in images],
            "categories": [{"id": c, "name": f"c{c}"} for c in cats],
            "annotations": [dict(a) for a in anns]}


def ann(id, image_id, bbox, category_id=1, iscrowd=0, area=None) -> dict:
    return {"id": id, "image_id": image_id, "bbox": [float(v) for v in bbox], "category_id": category_id, "iscrowd": iscrowd,
            "area": float(bbox[2] * bbox[3] if area is None else area)}


def det(image_id, xywh, scores, classes=None) -> Det:
    b = torch.tensor(xywh, dtype=torch.float32).reshape(-1, 4)
    b[:, 2] += b[:, 0]
    b[:, 3] += b[:, 1]
    s = torch.tensor(scores, dtype=torch.float32).reshape(-1)
    c = torch.zeros(len(s), dtype=torch.int64) if classes is None else torch.tensor(classes, dtype=torch.int64)
    return image_id, b, s, c


def to_results(gt: dict, dets: List[Det], image_size=(600, 1200), output_size=None) -> List[dict]:
    """The detections as detectron2's COCOEvaluator hands them to loadRes (export.instances_to_coco_json).  With
    ``output_size`` = (height, width) they first go through export.detector_postprocess from the network frame
    ``image_size``, as GeneralizedRCNN.inference(do_postprocess=True) applies it."""
    from sfod_b200.engine.export import detector_postprocess, instances_to_coco_json
    from sfod_b200.structures import Boxes, Instances
    id_map = {n: c for n, c in enumerate(sorted(c["id"] for c in gt["categories"]))}
    out = []
    for img, b, s, c in dets:
        inst = Instances(image_size)
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.cpu()), s.cpu(), c.cpu()
        if output_size is not None:
            inst = detector_postprocess(inst, output_size[0], output_size[1])
        out += instances_to_coco_json(inst, img, id_map)
    return out


# ---------------------------------------------------------------------------------------------- known-answer cases
def known_answer_cases() -> Dict[str, Tuple[dict, List[Det]]]:
    c = {}
    c["perfect"] = (gt_dict([1], [ann(1, 1, [10, 10, 50, 50])]), [det(1, [10, 10, 50, 50], [0.9])])
    # d1 -> g1 (tp), d2 duplicate of g1 (fp), d3 -> g2 (tp)
    c["duplicate"] = (gt_dict([1], [ann(1, 1, [10, 10, 50, 50]), ann(2, 1, [200, 200, 40, 40])]),
                      [det(1, [[10, 10, 50, 50], [10, 10, 50, 50], [200, 200, 40, 40]], [0.9, 0.8, 0.7])])
    # one real gt and a crowd region: the three detections inside the crowd are all absorbed by it (ignored)
    c["crowd"] = (gt_dict([1], [ann(1, 1, [10, 10, 50, 50]), ann(2, 1, [300, 300, 200, 200], iscrowd=1)]),
                  [det(1, [[10, 10, 50, 50], [310, 310, 50, 50], [400, 400, 60, 60], [320, 420, 40, 40]], [0.5, 0.9, 0.8, 0.7])])
    # the ignored gt (crowd, listed first) overlaps the detection better than the regular gt: evaluateImg scans the
    # non-ignored gt first, takes the regular one and then `break`s at the first ignored gt
    c["ignored_order"] = (gt_dict([1], [ann(1, 1, [100, 100, 100, 100], iscrowd=1), ann(2, 1, [100, 100, 80, 80])]),
                          [det(1, [100, 100, 95, 95], [0.9])])
    # a gt whose annotation id is 0: dtMatches holds 0, so accumulate counts the match as a false positive
    c["gt_id_zero"] = (gt_dict([1], [ann(0, 1, [10, 10, 50, 50])]), [det(1, [10, 10, 50, 50], [0.9])])
    # 120 detections of one (image, category): only the 100 best count; the one true positive is ranked 110th
    xs = [[1000 + (i % 10) * 10, 500 + (i // 10) * 2, 5, 5] for i in range(120)]
    sc = [1.0 - 0.001 * i for i in range(120)]
    xs[110] = [10, 10, 50, 50]
    c["over_100"] = (gt_dict([1], [ann(1, 1, [10, 10, 50, 50])]), [det(1, xs, sc)])
    # equal scores: across images the image order decides, within an image the result-list order
    c["score_ties"] = (gt_dict([1, 2], [ann(1, 1, [10, 10, 50, 50]), ann(2, 2, [10, 10, 50, 50])]),
                       [det(2, [[10, 10, 50, 50], [600, 10, 50, 50]], [0.5, 0.5]), det(1, [[600, 10, 50, 50], [10, 10, 50, 50]], [0.5, 0.5])])
    # gt areas exactly 32^2 and 96^2 sit in two area ranges each (inclusive bounds); detection areas too
    c["area_bounds"] = (gt_dict([1], [ann(1, 1, [10, 10, 32, 32]), ann(2, 1, [100, 100, 96, 96])]),
                        [det(1, [[10, 10, 32, 32], [100, 100, 96, 96]], [0.9, 0.8])])
    # category 7 has no gt: its cells stay -1 and AP-c7 is NaN; the detection of class 1 (category 7) is a false positive
    c["category_without_gt"] = (gt_dict([1], [ann(1, 1, [10, 10, 50, 50], 3)], cats=(3, 7)),
                                [det(1, [[10, 10, 50, 50], [10, 10, 50, 50]], [0.9, 0.8], [0, 1])])
    # image 2 has gt but no detection: it still counts towards npig
    c["image_without_detections"] = (gt_dict([1, 2], [ann(1, 1, [10, 10, 50, 50]), ann(2, 2, [10, 10, 50, 50])]),
                                     [det(1, [10, 10, 50, 50], [0.9])])
    return c


# ---------------------------------------------------------------------------------------------- synthetic datasets
def synthetic_case(seed: int, n_images: int, n_cats: int, max_gt: int, max_dets: int, crowd_frac: float = 0.05,
                   id_zero: bool = False) -> Tuple[dict, List[Det]]:
    """Seeded dataset: gt with crowd regions, annotation areas that differ from w*h (polygon areas) and a spread of sizes
    around the 32^2 / 96^2 bounds; detections = jittered gt (sometimes of the wrong class) + false positives, scores on a
    0.02 grid so that ties occur within and across images.  Image ids are shuffled, category ids are not contiguous."""
    rng = np.random.default_rng(seed)
    img_ids = [int(v) for v in rng.permutation(np.arange(1, 3 * n_images + 1))[:n_images]]
    cat_ids = [int(5 + 3 * k) for k in range(n_cats)]
    anns, dets = [], []
    aid = 0 if id_zero else 1
    for img in img_ids:
        g = int(rng.integers(0, max_gt + 1))
        boxes = []
        for _ in range(g):
            side = float(np.exp(rng.uniform(np.log(8), np.log(300))))
            w = round(side * rng.uniform(0.5, 1.5), 2)
            h = round(side * rng.uniform(0.5, 1.5), 2)
            x, y = round(rng.uniform(0, 1200 - w), 2), round(rng.uniform(0, 600 - h), 2)
            k = int(rng.integers(0, n_cats))
            crowd = int(rng.random() < crowd_frac)
            area = w * h * rng.uniform(0.6, 1.0) if rng.random() < 0.8 else w * h
            anns.append(ann(aid, img, [x, y, w, h], cat_ids[k], crowd, area))
            aid += 1
            boxes.append((x, y, w, h, k))
        xywh, sc, cl = [], [], []
        for (x, y, w, h, k) in boxes:
            for _ in range(int(rng.integers(0, 3))):
                j = rng.normal(0, 0.08, 4)
                xywh.append([x + j[0] * w, y + j[1] * h, w * (1 + j[2]), h * (1 + j[3])])
                sc.append(float(np.round(rng.uniform(0.05, 1.0) / 0.02) * 0.02))
                cl.append(k if rng.random() < 0.9 else int(rng.integers(0, n_cats)))
        for _ in range(int(rng.integers(0, max(1, max_dets // 4)))):
            w, h = float(rng.uniform(4, 200)), float(rng.uniform(4, 200))
            xywh.append([float(rng.uniform(0, 1100)), float(rng.uniform(0, 500)), w, h])
            sc.append(float(np.round(rng.uniform(0.05, 1.0) / 0.02) * 0.02))
            cl.append(int(rng.integers(0, n_cats)))
        xywh, sc, cl = xywh[:max_dets], sc[:max_dets], cl[:max_dets]
        if xywh:
            order = np.argsort(-np.asarray(sc), kind="stable")      # a detector emits score order
            dets.append(det(img, [xywh[i] for i in order], [sc[i] for i in order], [cl[i] for i in order]))
    return gt_dict(img_ids, anns, cat_ids), dets


def dense_case(seed: int = 0, n_gt: int = 50, n_dets: int = 100) -> Tuple[dict, List[Det]]:
    """One (image, category) with n_gt x n_dets IoU pairs (5000 by default): more than the device keeps as a shared-memory
    table (4096), so the matching recomputes every IoU.  Overlapping gt, some of them crowd, and jittered duplicates."""
    rng = np.random.default_rng(seed)
    anns, gts = [], []
    for g in range(n_gt):
        w, h = float(rng.uniform(20, 120)), float(rng.uniform(20, 120))
        x, y = float(rng.uniform(0, 400)), float(rng.uniform(0, 300))
        anns.append(ann(g + 1, 1, [x, y, w, h], 1, int(g % 11 == 10), w * h * float(rng.uniform(0.7, 1.0))))
        gts.append((x, y, w, h))
    xywh = []
    for d in range(n_dets):
        x, y, w, h = gts[int(rng.integers(0, n_gt))]
        j = rng.normal(0, 0.1, 4)
        xywh.append([x + j[0] * w, y + j[1] * h, w * (1 + j[2]), h * (1 + j[3])])
    sc = np.sort(np.round(rng.uniform(0.05, 1.0, n_dets) / 0.02) * 0.02)[::-1]
    return gt_dict([1], anns), [det(1, xywh, sc.tolist())]
