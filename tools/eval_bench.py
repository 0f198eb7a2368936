"""Times COCO box evaluation at the Foggy-Cityscapes-val shape (500 images, 8 classes, 100 detections per image, up to 60 gt per
image): the device call (ops.coco_box_eval: match + sort + accumulate, CUDA events, repeated), the whole
COCOBoxEvaluator.evaluate() (packing + call + the one device->host copy + summarize, wall clock), and the same evaluation on the
host by the numpy restatement of pycocotools (oracle/coco_eval_cpu.py) and by pycocotools when it is importable.
Prints one JSON line (and writes it to --out); the GPU name and power limit are part of the record."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import coco_eval_cpu as o  # noqa: E402
from sfod_b200 import engine, ops  # noqa: E402
from sfod_b200.engine import evaluation as E  # noqa: E402
from sfod_b200.structures import Boxes, Instances  # noqa: E402


def dataset(seed: int, n_images: int, n_cats: int, max_gt: int, n_dets: int):
    rng = np.random.default_rng(seed)
    anns, per_image = [], []
    for img in range(1, n_images + 1):
        g = int(rng.integers(1, max_gt + 1))
        wh = np.exp(rng.uniform(np.log(8), np.log(300), (g, 2)))
        xy = rng.uniform(0, 1, (g, 2)) * (np.array([2048, 1024]) - wh)
        cat = rng.integers(0, n_cats, g)
        for j in range(g):
            anns.append({"id": len(anns) + 1, "image_id": img, "bbox": [*xy[j], *wh[j]], "category_id": int(cat[j]) + 1,
                         "iscrowd": int(rng.random() < 0.05), "area": float(wh[j, 0] * wh[j, 1] * rng.uniform(0.6, 1.0))})
        src = rng.integers(0, g, n_dets)
        jit = rng.normal(0, 0.1, (n_dets, 4))
        b = np.concatenate([xy[src] + jit[:, :2] * wh[src], wh[src] * (1 + jit[:, 2:])], 1)
        fp = rng.random(n_dets) < 0.4
        b[fp, :2] = rng.uniform(0, 1800, (fp.sum(), 2))
        cls = np.where(rng.random(n_dets) < 0.9, cat[src], rng.integers(0, n_cats, n_dets))
        sc = np.sort(np.round(rng.uniform(0.05, 1, n_dets) / 0.01) * 0.01)[::-1].copy()
        xyxy = torch.tensor(b, dtype=torch.float32)
        xyxy[:, 2:] += xyxy[:, :2]
        per_image.append((img, xyxy, torch.tensor(sc, dtype=torch.float32), torch.tensor(cls, dtype=torch.int64)))
    gt = {"images": [{"id": i} for i in range(1, n_images + 1)], "categories": [{"id": k + 1, "name": f"c{k}"} for k in range(n_cats)],
          "annotations": anns}
    return gt, per_image


def gpu_record() -> dict:
    rec = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        rec["nvidia_smi"] = q.stdout.strip()
    except Exception as e:  # pragma: no cover
        rec["nvidia_smi"] = f"unavailable: {e}"
    return rec


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=500)
    ap.add_argument("--classes", type=int, default=8)
    ap.add_argument("--dets", type=int, default=100)
    ap.add_argument("--max-gt", type=int, default=60)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    gt, dets = dataset(0, a.images, a.classes, a.max_gt, a.dets)
    ev = engine.COCOBoxEvaluator(gt)
    inputs, outputs = [], []
    for img, b, s, c in dets:
        inst = Instances((1024, 2048))
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.to(dev)), s.to(dev), c.to(dev)
        inputs.append({"image_id": img})
        outputs.append({"instances": inst})
    ev.process(inputs, outputs)
    got = ev.evaluate()   # the arrays stay in ev.eval
    # device time of the library call alone, on the packed inputs evaluate() builds
    g = ev._gt_on(dev)
    P = a.dets
    boxes = torch.stack([E._xyxy_to_xywh(b) for _, b, _, _ in dets]).to(dev)
    scores = torch.stack([s for _, _, s, _ in dets]).to(dev)
    classes = torch.stack([c for _, _, _, c in dets]).to(dev)
    counts = torch.full((a.images,), P, dtype=torch.int32, device=dev)
    args = (ev._gt_offsets, g["boxes"], g["area"], g["iscrowd"], g["ids"], g["cats"], boxes, scores, classes, counts, a.classes,
            E.IOU_THRS, E.REC_THRS, E.AREA_RNG, E.MAX_DETS)
    for _ in range(3):
        ops.coco_box_eval(*args)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(a.reps):
        ev0.record()
        ops.coco_box_eval(*args)
        ev1.record()
        ev1.synchronize()
        ms.append(ev0.elapsed_time(ev1))
    launches0 = ops.launch_count()
    ops.coco_box_eval(*args)
    launches = ops.launch_count() - launches0
    wall = []
    for _ in range(5):
        torch.cuda.synchronize()
        t = time.perf_counter()
        ev.evaluate()
        wall.append((time.perf_counter() - t) * 1e3)
    # the oracle sees what detectron2's inference(do_postprocess=True) would return: clipped to the 1024 x 2048 frame, empty dropped
    results = [r for inp, out in zip(inputs, outputs)
               for r in engine.instances_to_coco_json(engine.detector_postprocess(out["instances"], 1024, 2048), inp["image_id"],
                                                      {k: k + 1 for k in range(a.classes)})]
    t = time.perf_counter()
    want = o.evaluate_bbox(gt, results)
    oracle_ms = (time.perf_counter() - t) * 1e3
    rec = {**gpu_record(), "shape": {"images": a.images, "classes": a.classes, "dets_per_image": a.dets, "max_gt_per_image": a.max_gt,
                                     "n_gt": len(gt["annotations"]), "n_dets": len(results)},
           "device_call_ms": {"median": float(np.median(ms)), "min": float(np.min(ms)), "reps": a.reps},
           "launches_per_call": launches,
           "evaluate_wall_ms": {"median": float(np.median(wall)), "min": float(np.min(wall))},
           "oracle_numpy_host_ms": oracle_ms,
           "equal_to_oracle": bool(all(np.array_equal(ev.eval[k], want[k]) for k in ("precision", "recall", "scores", "stats"))),
           "AP": got["bbox"]["AP"], "AP50": got["bbox"]["AP50"]}
    try:
        from pycocotools.coco import COCO
        from pycocotools.cocoeval import COCOeval
        cg = COCO()
        cg.dataset = gt
        cg.createIndex()
        t = time.perf_counter()
        P_ = COCOeval(cg, cg.loadRes(results), "bbox")
        P_.evaluate(); P_.accumulate()
        rec["pycocotools_host_ms"] = (time.perf_counter() - t) * 1e3
    except ImportError:
        rec["pycocotools_host_ms"] = None
    line = json.dumps(rec)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
