"""COCO box AP of a detector's outputs (SURVEY.md 8f row f-5): detectron2's ``COCOEvaluator`` (iou_type "bbox") and
``inference_on_dataset``, as the reference uses them (reference daod/evaluation/; test_refinement at
daod/engine/trainers/base.py:300, the --eval-only runs of train_net*.py, EvalHook).

``COCOeval.evaluate`` + ``accumulate`` run on the device in one library call (``ops.coco_box_eval``, bit-equal to pycocotools);
``summarize`` and detectron2's ``_derive_coco_results`` run here on the host in numpy over the arrays the device returned, so
their summation order is pycocotools' own.  ``process`` keeps the detections on the device without synchronising; ``evaluate``
packs them, makes one library call and one device->host copy.  In a distributed run every rank's detections are gathered
onto the main rank first, as detectron2's ``COCOEvaluator(distributed=True)`` does.
"""
from __future__ import annotations

import json
import os
from typing import Dict, List, Optional, Sequence, Union

import numpy as np
import torch
import torch.distributed as dist

from .. import ops
from .export import _xyxy_to_xywh

# pycocotools Params (iouType "bbox"), computed exactly as there
IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
MAX_DETS = [1, 10, 100]
AREA_RNG = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
AREA_RNG_LBL = ["all", "small", "medium", "large"]
METRICS = ["AP", "AP50", "AP75", "APs", "APm", "APl"]

_UNKNOWN_IMAGE = "Results do not correspond to current coco set: detections on an image the ground truth does not list"


def summarize(precision: np.ndarray, recall: np.ndarray) -> np.ndarray:
    """COCOeval.summarize (_summarizeDets) without the printing: the 12 COCO stats, -1 where nothing is defined."""
    def _summarize(ap=1, iouThr=None, areaRng="all", maxDets=100):
        aind = [i for i, aRng in enumerate(AREA_RNG_LBL) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(MAX_DETS) if mDet == maxDets]
        s = precision if ap == 1 else recall
        if iouThr is not None:
            s = s[np.where(iouThr == IOU_THRS)[0]]
        s = s[:, :, :, aind, mind] if ap == 1 else s[:, :, aind, mind]
        return -1 if len(s[s > -1]) == 0 else np.mean(s[s > -1])

    stats = np.zeros((12,))
    stats[0] = _summarize(1)
    stats[1] = _summarize(1, iouThr=.5, maxDets=MAX_DETS[2])
    stats[2] = _summarize(1, iouThr=.75, maxDets=MAX_DETS[2])
    for i, lbl in enumerate(("small", "medium", "large")):
        stats[3 + i] = _summarize(1, areaRng=lbl, maxDets=MAX_DETS[2])
    for i, m in enumerate(MAX_DETS):
        stats[6 + i] = _summarize(0, maxDets=m)
    for i, lbl in enumerate(("small", "medium", "large")):
        stats[9 + i] = _summarize(0, areaRng=lbl, maxDets=MAX_DETS[2])
    return stats


def derive_coco_results(stats: Optional[np.ndarray], precision: Optional[np.ndarray], class_names: Optional[Sequence[str]]) -> Dict[str, float]:
    """detectron2 COCOEvaluator._derive_coco_results for "bbox": percentages, NaN where COCOeval gives -1, per-class AP
    ("AP-<name>": mean precision over the IoU and recall thresholds, area "all", 100 detections).  ``stats`` None = the model
    produced no detection at all."""
    if stats is None:
        return {metric: float("nan") for metric in METRICS}
    results = {metric: float(stats[idx] * 100 if stats[idx] >= 0 else "nan") for idx, metric in enumerate(METRICS)}
    if class_names is None or len(class_names) <= 1:
        return results
    assert len(class_names) == precision.shape[2]
    for idx, name in enumerate(class_names):
        p = precision[:, :, idx, 0, -1]
        p = p[p > -1]
        ap = np.mean(p) if p.size else float("nan")
        results["AP-" + name] = float(ap * 100)
    return results


class COCOBoxEvaluator:
    """detectron2's ``DatasetEvaluator`` protocol (``reset`` / ``process(inputs, outputs)`` / ``evaluate``) for COCO box AP.

    ``coco_gt``: the ground truth as a COCO-format dict or the path of its json.  Images and categories are those it lists;
    a predicted class index c stands for the c-th category in ascending id order (detectron2's contiguous ids of a COCO json).
    ``class_names`` defaults to the category names in that order.  ``evaluate`` returns detectron2's
    ``{"bbox": {"AP", "AP50", "AP75", "APs", "APm", "APl", "AP-<name>", ...}}`` and leaves COCOeval's arrays and the 12
    summary stats in ``self.eval`` (per-class AP50: ``self.eval["precision"][0, :, :, 0, -1].mean(axis=0)``).  A detection on an
    image the ground truth does not list makes ``evaluate`` raise, as ``COCO.loadRes`` does.

    ``distributed`` (detectron2's keyword): when ``torch.distributed`` is initialised with more than one rank, ``evaluate``
    gathers the detections of every rank of the default group onto rank 0, in rank order, and evaluates them there; the other
    ranks return ``{}`` and leave ``self.eval`` all None.  Every rank must call ``evaluate``, and every rank raises when the
    evaluation fails.  With ``distributed=False`` each process evaluates what it processed itself.

    ``output_dir``: rank 0 also writes ``output_dir/coco_instances_results.json``, detectron2's COCO result list (the kept
    detections in processing order and, distributed, rank order; boxes XYWH in the input's frame; dataset category ids), the
    list ``engine.prediction_to_gt`` turns into pseudo-labels."""

    def __init__(self, coco_gt: Union[dict, str], class_names: Optional[Sequence[str]] = None, *, distributed: bool = True,
                 output_dir: Optional[str] = None):
        self._distributed = distributed
        self._output_dir = output_dir
        if isinstance(coco_gt, (str, bytes)) or hasattr(coco_gt, "__fspath__"):
            with open(coco_gt) as f:
                coco_gt = json.load(f)
        cats = sorted(coco_gt["categories"], key=lambda c: c["id"])
        self.cat_ids = [c["id"] for c in cats]
        self.img_ids = sorted({im["id"] for im in coco_gt["images"]})
        self.class_names = list(class_names) if class_names is not None else [str(c.get("name", c["id"])) for c in cats]
        if len(self.class_names) != len(self.cat_ids):
            raise ValueError(f"{len(self.class_names)} class names for {len(self.cat_ids)} categories")
        self._img_index = {i: n for n, i in enumerate(self.img_ids)}
        cat_index = {c: n for n, c in enumerate(self.cat_ids)}
        per_image: List[list] = [[] for _ in self.img_ids]
        for a in coco_gt.get("annotations", []):
            n = self._img_index.get(a["image_id"])
            if n is not None and a["category_id"] in cat_index:
                per_image[n].append(a)
        anns = [a for lst in per_image for a in lst]
        self._gt_offsets = np.cumsum([0] + [len(lst) for lst in per_image]).tolist()
        self._gt_host = dict(
            boxes=torch.tensor([[float(v) for v in a["bbox"]] for a in anns], dtype=torch.float64).reshape(-1, 4),
            area=torch.tensor([float(a["area"]) for a in anns], dtype=torch.float64),
            iscrowd=torch.tensor([bool(a.get("iscrowd", 0)) for a in anns], dtype=torch.uint8),
            ids=torch.tensor([int(a["id"]) for a in anns], dtype=torch.int64),
            cats=torch.tensor([cat_index[a["category_id"]] for a in anns], dtype=torch.int64))
        self._gt_dev: Dict[torch.device, Dict[str, torch.Tensor]] = {}
        self.eval: Dict[str, Optional[np.ndarray]] = {}
        self.reset()

    def reset(self) -> None:
        self._records = []

    def process(self, inputs, outputs) -> None:
        """Keeps each image's detections on the device, without host synchronisation, in the frame of the input's
        ``height`` / ``width``: ``detector_postprocess`` (scale, clip, drop empty boxes) is applied here as detectron2's
        ``GeneralizedRCNN.inference(do_postprocess=True)`` applies it, because this package's meta-architecture returns its
        detections in the resized network frame.  On outputs that are already post-processed it is the identity (scale 1,
        boxes inside the image, none empty).  Empty boxes are kept as a device mask instead of being cut out.  Boxes are then
        stored as fp32 XYWH (``export._xyxy_to_xywh``).  A detector's padded batch that nobody has looked at yet stays padded,
        with its device-side counts."""
        for inp, out in zip(inputs, outputs):
            inst = out["instances"]
            src = inst.packed_source() if hasattr(inst, "packed_source") else None
            if src is not None:
                batch, i = src
                boxes, scores, classes, count = batch.boxes[i], batch.scores[i], batch.classes[i], batch.count[i:i + 1]
            else:
                boxes, scores, classes, count = inst.pred_boxes.tensor, inst.scores, inst.pred_classes, len(inst)
            height, width = inp.get("height", inst.image_size[0]), inp.get("width", inst.image_size[1])
            boxes, keep = _postprocess_boxes(boxes.detach().to(torch.float32), inst.image_size, height, width)
            self._records.append((inp["image_id"], _xyxy_to_xywh(boxes), scores.detach().to(torch.float32), classes.detach().to(torch.int64),
                                  count, keep))

    def _gt_on(self, dev: torch.device) -> Dict[str, torch.Tensor]:
        g = self._gt_dev.get(dev)
        if g is None:
            g = {k: v.pin_memory().to(dev, non_blocking=True) if v.numel() else v.to(dev) for k, v in self._gt_host.items()}
            self._gt_dev[dev] = g
        return g

    def evaluate(self):
        """-> ``{"bbox": {"AP", "AP50", "AP75", "APs", "APm", "APl", "AP-<name>", ...}}`` (detectron2's result: a nested dict of
        floats, as ``EvalHook`` requires), ``{}`` when nothing was processed.  COCOeval's arrays stay on the evaluator:
        ``self.eval = {"precision": (T, R, K, A, M), "recall": (T, K, A, M), "scores": (T, R, K, A, M), "stats": (12,)}``
        (numpy; all None when there was not a single detection, as detectron2 then skips COCOeval).  Distributed: the result on
        rank 0, ``{}`` on the other ranks."""
        self.eval = {"precision": None, "recall": None, "scores": None, "stats": None}
        gather = self._distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        records = self._gather_records() if gather else self._records
        if not records:                                  # other ranks (None), or nothing processed anywhere
            return {}                                    # detectron2: "did not receive valid predictions"
        dev = records[0][1].device
        if dev.type != "cuda":
            raise RuntimeError("COCOBoxEvaluator evaluates on the GPU (no CPU fallback); got detections on " + str(dev))
        K = len(self.cat_ids)
        packed = self._pack(dev, records)
        T, R, A, M = len(IOU_THRS), len(REC_THRS), len(AREA_RNG), len(MAX_DETS)
        n_out = ops.coco_eval_out_numel(T, R, K, A, M)
        buf = torch.empty(n_out + 2, dtype=torch.float64, device=dev)
        buf[n_out] = packed["n_results"]                 # loadRes' result list: every kept detection
        buf[n_out + 1] = packed["n_unknown"]             # ... of them on images outside the ground truth
        g = self._gt_on(dev)
        ops.coco_box_eval(self._gt_offsets, g["boxes"], g["area"], g["iscrowd"], g["ids"], g["cats"], packed["boxes"], packed["scores"],
                          packed["classes"], packed["counts"], K, IOU_THRS, REC_THRS, AREA_RNG, MAX_DETS, out=buf)
        res = buf.cpu().numpy()                          # the one device->host copy
        if res[n_out + 1] > 0:
            raise ValueError(_UNKNOWN_IMAGE)
        if self._output_dir is not None and (not dist.is_available() or not dist.is_initialized() or dist.get_rank() == 0):
            self._write_results(records)
        if res[n_out] == 0:                              # detectron2 skips COCOeval without a single detection
            return {"bbox": derive_coco_results(None, None, self.class_names)}
        n1 = T * R * K * A * M
        precision = res[:n1].reshape(T, R, K, A, M)
        recall = res[2 * n1:n_out].reshape(T, K, A, M)
        stats = summarize(precision, recall)
        self.eval = {"precision": precision, "recall": recall, "scores": res[n1:2 * n1].reshape(T, R, K, A, M), "stats": stats}
        return {"bbox": derive_coco_results(stats, precision, self.class_names)}

    def _gather_records(self) -> Optional[list]:
        """Every rank's records, in rank order then processing order, on rank 0 (the list ``itertools.chain(*comm.gather(...))``
        leaves in detectron2), None on the other ranks.  Every rank enters the same two collectives whatever it holds:

        1. ``all_gather_object`` of the host-known metadata: (image id, width) per record and the device of detections that
           are not on a GPU.  Every rank then raises the same error for a condition that fails the evaluation;
        2. ``all_gather`` of one padded fp32 (n_max, 7) tensor per rank: XYWH, score, class index, kept flag per entry
           (``_entries``, computed on the device: no count is read on the host).

        Every rank holds the whole gathered list afterwards, so a kept detection on an image outside the ground truth, which
        fails the evaluation on rank 0 (``loadRes``), makes the other ranks raise the same error too."""
        rank, world = dist.get_rank(), dist.get_world_size()
        recs = self._records
        not_gpu = next((str(r[1].device) for r in recs if r[1].device.type != "cuda"), None)
        meta = [None] * world
        dist.all_gather_object(meta, ([(r[0], r[1].shape[0]) for r in recs], not_gpu))
        for r, (_, dev) in enumerate(meta):
            if dev is not None:
                raise RuntimeError(f"COCOBoxEvaluator evaluates on the GPU (no CPU fallback); got detections on {dev} on rank {r}")
        if not any(m for m, _ in meta):
            return [] if rank == 0 else None
        self._row_width([x for m, _ in meta for x in m])        # raises on every rank
        n_max = max(1, max(sum(w for _, w in m) for m, _ in meta))
        dev = recs[0][1].device if recs else torch.device("cuda", torch.cuda.current_device())
        mine = _entries(recs, dev)
        payload = torch.zeros(n_max, 7, dtype=torch.float32, device=dev)
        payload[:mine.shape[0]] = mine
        parts = [torch.empty_like(payload) for _ in range(world)]
        dist.all_gather(parts, payload)
        gathered = []
        for (m, _), part in zip(meta, parts):
            offsets = np.cumsum([0] + [w for _, w in m]).tolist()
            for (img, w), o in zip(m, offsets):
                e = part[o:o + w]
                gathered.append((img, e[:, :4], e[:, 4], e[:, 5].to(torch.int64), w, e[:, 6] > 0))
        if rank == 0:
            return gathered
        unknown = [r[5] for r in gathered if r[0] not in self._img_index]
        if unknown and bool(torch.cat(unknown).any()):
            raise ValueError(_UNKNOWN_IMAGE)
        return None

    def _write_results(self, records) -> None:
        """``output_dir/coco_instances_results.json``: the kept detections of ``records`` as detectron2's COCOEvaluator writes
        them, the values ``export.instances_to_coco_json(export.detector_postprocess(...), image_id, id_map)`` gives."""
        rows = _entries(records, records[0][1].device).cpu()      # the json's one device->host copy
        image_ids = [r[0] for r in records for _ in range(r[1].shape[0])]
        kept = (rows[:, 6] > 0).tolist()
        boxes, scores, classes = rows[:, :4].tolist(), rows[:, 4].tolist(), rows[:, 5].to(torch.int64).tolist()
        results = [{"image_id": img, "category_id": self.cat_ids[classes[k]], "bbox": boxes[k], "score": scores[k]}
                   for k, img in enumerate(image_ids) if kept[k]]
        os.makedirs(self._output_dir, exist_ok=True)
        with open(os.path.join(self._output_dir, "coco_instances_results.json"), "w") as f:
            json.dump(results, f)

    def _row_width(self, meta) -> int:
        """P of ``_pack`` for records given as (image id, width): the sum of the record widths of the widest ground-truth image."""
        row_width = [0] * max(len(self.img_ids), 1)
        for img, w in meta:
            n = self._img_index.get(img, -1)
            if n >= 0:
                row_width[n] += w
        P = max(1, max(row_width))
        if P > 1024:
            raise ValueError(f"{P} detections for one image: at most 1024 are supported")
        return P

    def _pack(self, dev: torch.device, recs) -> Dict[str, torch.Tensor]:
        """The processed detections in the library's layout, built on the device without reading any count on the host.

        The library wants one padded row of P slots per ground-truth image (ascending image id) with the image's detections in
        result-list order at the front, and a device-side count per row.  The records hold padded rows whose valid length
        (``count``) and kept entries (``keep``: inside the count and not emptied by the post-processing) are only known on the
        device.  So every entry of every record gets a destination slot computed on the device:

        1. records are put in image order (stable: several records of one image keep their processing order, as loadRes
           concatenates them) and their entries concatenated into one flat list;
        2. ``placed`` = the entry is kept and its image is in the ground truth; its slot within its image's row = number of
           placed entries before it in the flat list minus that number at the first entry of the image's records
           (``start``), i.e. an exclusive prefix sum restarted per image;
        3. entries that are not placed go to one spare column (column P of row 0) that is cut off afterwards, so
           ``index_copy_`` may write there several times without effect.

        Example, P = 3: image 0 has records A (2 slots, count 1) and B (2 slots, count 2); flat entries A0 A1 B0 B1, placed
        1 0 1 1, exclusive prefix 0 1 1 2, start of image 0 = entry 0 -> slots 0 - 1 2; A1 goes to the spare column; row 0 =
        [A0, B0, B1], count 3.  P is the sum of the record widths of the widest image (known on the host)."""
        I = len(self.img_ids)
        img_of = [self._img_index.get(r[0], -1) for r in recs]
        order = sorted(range(len(recs)), key=lambda r: (img_of[r] < 0, img_of[r]))
        widths = [recs[r][1].shape[0] for r in order]
        P = self._row_width([(r[0], r[1].shape[0]) for r in recs])
        # per flat entry (host-known): its record, its index within the record, its image (-1: unknown), the start of its group
        rec_e = np.repeat(np.arange(len(order)), widths)
        idx_e = np.concatenate([np.arange(w) for w in widths])
        offsets = np.concatenate([[0], np.cumsum(widths)])
        group_start = []
        for j, r in enumerate(order):
            same = j > 0 and img_of[r] >= 0 and img_of[order[j - 1]] == img_of[r]
            group_start.append(group_start[j - 1] if same else int(offsets[j]))
        img_e = np.repeat([img_of[r] for r in order], widths)
        start_e = np.repeat(group_start, widths)
        host_count = [recs[r][4] if isinstance(recs[r][4], int) else 0 for r in order]
        host = torch.from_numpy(np.concatenate([rec_e, idx_e, img_e, start_e, host_count]).astype(np.int64))
        n = len(rec_e)
        rec_e, idx_e, img_e, start_e, host_count = torch.split(host.pin_memory().to(dev, non_blocking=True), [n, n, n, n, len(order)])
        zero = torch.zeros(1, dtype=torch.int32, device=dev)
        count = torch.cat([zero if isinstance(recs[r][4], int) else recs[r][4].to(torch.int32) for r in order]).to(torch.int64) + host_count
        kept = (idx_e < count[rec_e]) & torch.cat([recs[r][5] for r in order])
        known = img_e >= 0
        placed = (kept & known).to(torch.int64)
        before = torch.cumsum(placed, 0) - placed
        slot = before - before[start_e]
        dest = torch.where(placed.bool(), img_e * (P + 1) + slot, torch.full_like(slot, P))
        rows = max(I, 1) * (P + 1)
        out = {}
        for name, col, width in (("boxes", 1, 4), ("scores", 2, 1), ("classes", 3, 1)):
            src = torch.cat([recs[r][col] for r in order])
            buf = torch.zeros((rows, width) if width > 1 else (rows,), dtype=src.dtype, device=dev).index_copy_(0, dest, src)
            out[name] = buf.view(max(I, 1), P + 1, *buf.shape[1:])[:I, :P].contiguous()
        out["counts"] = torch.zeros(max(I, 1), dtype=torch.int64, device=dev).index_add_(0, img_e.clamp(min=0), placed)[:I].to(torch.int32)
        out["n_results"] = kept.sum()
        out["n_unknown"] = (kept & ~known).sum()
        return out


def _entries(records, dev: torch.device) -> torch.Tensor:
    """(n, 7) fp32 on ``dev``, one row per entry of ``records`` in order: XYWH, score, class index, kept (1 / 0: inside the
    record's count and not emptied by the post-processing).  Class indices are < 2^24, so exact in fp32; the class of an
    entry that is not kept is written as 0."""
    rows = []
    for _, boxes, scores, classes, count, keep in records:
        kept = (torch.arange(boxes.shape[0], device=boxes.device) < count) & keep
        rows.append(torch.cat([boxes, scores[:, None], torch.where(kept, classes, 0)[:, None].to(torch.float32),
                               kept[:, None].to(torch.float32)], dim=1))
    return torch.cat(rows) if rows else torch.zeros((0, 7), dtype=torch.float32, device=dev)


def _postprocess_boxes(boxes, image_size, height, width):
    """``export.detector_postprocess`` on an (n, 4) XYXY fp32 device tensor without host reads: the same scale factors
    (Python floats) and ``Boxes.scale`` / ``clip`` / ``nonempty`` arithmetic, the empty boxes returned as a mask (``Boxes.clip``'s
    finiteness assert, a host read, is left out)."""
    if isinstance(width, torch.Tensor):
        width, height = float(width), float(height)
    scale_x, scale_y = width / image_size[1], height / image_size[0]
    h, w = int(height), int(width)
    b = boxes.clone()
    b[:, 0::2] *= scale_x
    b[:, 1::2] *= scale_y
    b = torch.stack((b[:, 0].clamp(min=0, max=w), b[:, 1].clamp(min=0, max=h), b[:, 2].clamp(min=0, max=w), b[:, 3].clamp(min=0, max=h)), dim=-1)
    return b, ((b[:, 2] - b[:, 0]) > 0) & ((b[:, 3] - b[:, 1]) > 0)


def inference_on_dataset(model, data_loader, evaluator):
    """detectron2.evaluation.inference_on_dataset without the timing log: eval mode, no_grad, ``process`` every batch,
    ``evaluate`` once (``{}`` when it returns None)."""
    evaluator.reset()
    was_training = model.training
    model.eval()
    try:
        with torch.no_grad():
            for inputs in data_loader:
                outputs = model(inputs)
                evaluator.process(inputs, outputs)
    finally:
        model.train(was_training)
    results = evaluator.evaluate()
    return {} if results is None else results
