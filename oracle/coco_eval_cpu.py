"""Literal numpy restatement of pycocotools 2.0 ``COCOeval`` for ``iouType="bbox"`` (test infrastructure only).

Restated: ``COCO`` (the index, ``getAnnIds`` / ``getCatIds`` / ``getImgIds`` / ``loadAnns``, ``loadRes`` for box results),
``maskApi.c::bbIou`` (the loop order and the fp64 operation order; ``fmin`` / ``fmax`` are C's, NaN-ignoring), and
``COCOeval._prepare`` / ``computeIoU`` / ``evaluateImg`` / ``accumulate`` / ``summarize``, statement by statement, plus
detectron2's ``COCOEvaluator._derive_coco_results`` for the ``bbox`` task.  pycocotools itself is not a dependency: the
known-answer tests pin this file, and a test compares it against pycocotools where that is importable.
"""
from __future__ import annotations

import copy
import itertools
from collections import defaultdict
from typing import Dict, List, Optional, Sequence

import numpy as np


class COCO:
    def __init__(self, dataset: Optional[dict] = None):
        self.dataset = dataset if dataset is not None else {}
        self.createIndex()

    def createIndex(self):
        anns, cats, imgs = {}, {}, {}
        imgToAnns = defaultdict(list)
        for ann in self.dataset.get("annotations", []):
            imgToAnns[ann["image_id"]].append(ann)
            anns[ann["id"]] = ann
        for img in self.dataset.get("images", []):
            imgs[img["id"]] = img
        for cat in self.dataset.get("categories", []):
            cats[cat["id"]] = cat
        self.anns, self.imgToAnns, self.imgs, self.cats = anns, imgToAnns, imgs, cats

    def getAnnIds(self, imgIds=(), catIds=()):
        lists = [self.imgToAnns[imgId] for imgId in imgIds if imgId in self.imgToAnns]
        anns = list(itertools.chain.from_iterable(lists))
        anns = anns if len(catIds) == 0 else [ann for ann in anns if ann["category_id"] in catIds]
        return [ann["id"] for ann in anns]

    def getCatIds(self):
        return [cat["id"] for cat in self.dataset["categories"]]

    def getImgIds(self):
        return list(self.imgs.keys())

    def loadAnns(self, ids):
        return [self.anns[i] for i in ids]

    def loadRes(self, anns: List[dict]) -> "COCO":
        res = COCO()
        res.dataset["images"] = [img for img in self.dataset["images"]]
        anns = copy.deepcopy(anns)
        assert type(anns) == list, "results in not an array of objects"
        annsImgIds = [ann["image_id"] for ann in anns]
        assert set(annsImgIds) == (set(annsImgIds) & set(self.getImgIds())), "Results do not correspond to current coco set"
        assert "bbox" in anns[0] and not anns[0]["bbox"] == []
        res.dataset["categories"] = copy.deepcopy(self.dataset["categories"])
        for id, ann in enumerate(anns):
            bb = ann["bbox"]
            ann["area"] = bb[2] * bb[3]
            ann["id"] = id + 1
            ann["iscrowd"] = 0
        res.dataset["annotations"] = anns
        res.createIndex()
        return res


def bb_iou(dt: np.ndarray, gt: np.ndarray, iscrowd: Sequence[int]) -> np.ndarray:
    """maskApi.c::bbIou: (D, G) fp64, XYWH boxes."""
    D, G = len(dt), len(gt)
    o = np.zeros((D, G), dtype=np.float64)
    if D == 0 or G == 0:
        return o
    dt = np.asarray(dt, dtype=np.float64).reshape(D, 4)
    gt = np.asarray(gt, dtype=np.float64).reshape(G, 4)
    dx, dy, dw, dh = (dt[:, i:i + 1] for i in range(4))
    gx, gy, gw, gh = (gt[None, :, i] for i in range(4))
    ga = gw * gh
    da = dw * dh
    with np.errstate(invalid="ignore", divide="ignore"):
        w = np.fmin(dw + dx, gw + gx) - np.fmax(dx, gx)
        h = np.fmin(dh + dy, gh + gy) - np.fmax(dy, gy)
        i = w * h
        crowd = np.asarray(iscrowd, dtype=bool)[None, :]
        u = np.where(crowd, da, da + ga - i)
        val = i / u
    keep = ~(w <= 0) & ~(h <= 0)
    o[keep] = val[keep]
    return o


class Params:
    def __init__(self):
        self.imgIds = []
        self.catIds = []
        self.iouThrs = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
        self.recThrs = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
        self.maxDets = [1, 10, 100]
        self.areaRng = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
        self.areaRngLbl = ["all", "small", "medium", "large"]
        self.useCats = 1


class COCOeval:
    def __init__(self, cocoGt: COCO, cocoDt: COCO):
        self.cocoGt, self.cocoDt = cocoGt, cocoDt
        self.evalImgs = []
        self.eval = {}
        self._gts = defaultdict(list)
        self._dts = defaultdict(list)
        self.params = Params()
        self.stats = []
        self.ious = {}
        self.params.imgIds = sorted(cocoGt.getImgIds())
        self.params.catIds = sorted(cocoGt.getCatIds())

    def _prepare(self):
        p = self.params
        gts = self.cocoGt.loadAnns(self.cocoGt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        dts = self.cocoDt.loadAnns(self.cocoDt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        for gt in gts:
            gt["ignore"] = gt["ignore"] if "ignore" in gt else 0
            gt["ignore"] = "iscrowd" in gt and gt["iscrowd"]
        self._gts = defaultdict(list)
        self._dts = defaultdict(list)
        for gt in gts:
            self._gts[gt["image_id"], gt["category_id"]].append(gt)
        for dt in dts:
            self._dts[dt["image_id"], dt["category_id"]].append(dt)
        self.evalImgs = defaultdict(list)
        self.eval = {}

    def evaluate(self):
        p = self.params
        p.imgIds = list(np.unique(p.imgIds))
        p.catIds = list(np.unique(p.catIds))
        p.maxDets = sorted(p.maxDets)
        self.params = p
        self._prepare()
        catIds = p.catIds
        self.ious = {(imgId, catId): self.computeIoU(imgId, catId) for imgId in p.imgIds for catId in catIds}
        maxDet = p.maxDets[-1]
        self.evalImgs = [self.evaluateImg(imgId, catId, areaRng, maxDet)
                         for catId in catIds for areaRng in p.areaRng for imgId in p.imgIds]
        self._paramsEval = copy.deepcopy(self.params)

    def computeIoU(self, imgId, catId):
        p = self.params
        gt = self._gts[imgId, catId]
        dt = self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return []
        inds = np.argsort([-d["score"] for d in dt], kind="mergesort")
        dt = [dt[i] for i in inds]
        if len(dt) > p.maxDets[-1]:
            dt = dt[0:p.maxDets[-1]]
        g = [g["bbox"] for g in gt]
        d = [d["bbox"] for d in dt]
        iscrowd = [int(o["iscrowd"]) for o in gt]
        if len(d) == 0 or len(g) == 0:
            return []
        return bb_iou(d, g, iscrowd)

    def evaluateImg(self, imgId, catId, aRng, maxDet):
        p = self.params
        gt = self._gts[imgId, catId]
        dt = self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return None
        for g in gt:
            if g["ignore"] or (g["area"] < aRng[0] or g["area"] > aRng[1]):
                g["_ignore"] = 1
            else:
                g["_ignore"] = 0
        gtind = np.argsort([g["_ignore"] for g in gt], kind="mergesort")
        gt = [gt[i] for i in gtind]
        dtind = np.argsort([-d["score"] for d in dt], kind="mergesort")
        dt = [dt[i] for i in dtind[0:maxDet]]
        iscrowd = [int(o["iscrowd"]) for o in gt]
        ious = self.ious[imgId, catId][:, gtind] if len(self.ious[imgId, catId]) > 0 else self.ious[imgId, catId]
        T = len(p.iouThrs)
        G = len(gt)
        D = len(dt)
        gtm = np.zeros((T, G))
        dtm = np.zeros((T, D))
        gtIg = np.array([g["_ignore"] for g in gt])
        dtIg = np.zeros((T, D))
        if not len(ious) == 0:
            for tind, t in enumerate(p.iouThrs):
                for dind, d in enumerate(dt):
                    iou = min([t, 1 - 1e-10])
                    m = -1
                    for gind, g in enumerate(gt):
                        if gtm[tind, gind] > 0 and not iscrowd[gind]:
                            continue
                        if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                            break
                        if ious[dind, gind] < iou:
                            continue
                        iou = ious[dind, gind]
                        m = gind
                    if m == -1:
                        continue
                    dtIg[tind, dind] = gtIg[m]
                    dtm[tind, dind] = gt[m]["id"]
                    gtm[tind, m] = d["id"]
        a = np.array([d["area"] < aRng[0] or d["area"] > aRng[1] for d in dt]).reshape((1, len(dt)))
        dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
        return {"image_id": imgId, "category_id": catId, "aRng": aRng, "maxDet": maxDet,
                "dtIds": [d["id"] for d in dt], "gtIds": [g["id"] for g in gt], "dtMatches": dtm, "gtMatches": gtm,
                "dtScores": [d["score"] for d in dt], "gtIgnore": gtIg, "dtIgnore": dtIg}

    def accumulate(self):
        p = self.params
        T = len(p.iouThrs)
        R = len(p.recThrs)
        K = len(p.catIds) if p.useCats else 1
        A = len(p.areaRng)
        M = len(p.maxDets)
        precision = -np.ones((T, R, K, A, M))
        recall = -np.ones((T, K, A, M))
        scores = -np.ones((T, R, K, A, M))
        _pe = self._paramsEval
        catIds = _pe.catIds if _pe.useCats else [-1]
        setK = set(catIds)
        setA = set(map(tuple, _pe.areaRng))
        setM = set(_pe.maxDets)
        setI = set(_pe.imgIds)
        k_list = [n for n, k in enumerate(p.catIds) if k in setK]
        m_list = [m for n, m in enumerate(p.maxDets) if m in setM]
        a_list = [n for n, a in enumerate(map(lambda x: tuple(x), p.areaRng)) if a in setA]
        i_list = [n for n, i in enumerate(p.imgIds) if i in setI]
        I0 = len(_pe.imgIds)
        A0 = len(_pe.areaRng)
        for k, k0 in enumerate(k_list):
            Nk = k0 * A0 * I0
            for a, a0 in enumerate(a_list):
                Na = a0 * I0
                for m, maxDet in enumerate(m_list):
                    E = [self.evalImgs[Nk + Na + i] for i in i_list]
                    E = [e for e in E if e is not None]
                    if len(E) == 0:
                        continue
                    dtScores = np.concatenate([e["dtScores"][0:maxDet] for e in E])
                    inds = np.argsort(-dtScores, kind="mergesort")
                    dtScoresSorted = dtScores[inds]
                    dtm = np.concatenate([e["dtMatches"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    dtIg = np.concatenate([e["dtIgnore"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    gtIg = np.concatenate([e["gtIgnore"] for e in E])
                    npig = np.count_nonzero(gtIg == 0)
                    if npig == 0:
                        continue
                    tps = np.logical_and(dtm, np.logical_not(dtIg))
                    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                    tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
                    fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
                    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                        tp = np.array(tp)
                        fp = np.array(fp)
                        nd = len(tp)
                        rc = tp / npig
                        pr = tp / (fp + tp + np.spacing(1))
                        q = np.zeros((R,))
                        ss = np.zeros((R,))
                        if nd:
                            recall[t, k, a, m] = rc[-1]
                        else:
                            recall[t, k, a, m] = 0
                        pr = pr.tolist()
                        q = q.tolist()
                        for i in range(nd - 1, 0, -1):
                            if pr[i] > pr[i - 1]:
                                pr[i - 1] = pr[i]
                        inds = np.searchsorted(rc, p.recThrs, side="left")
                        try:
                            for ri, pi in enumerate(inds):
                                q[ri] = pr[pi]
                                ss[ri] = dtScoresSorted[pi]
                        except Exception:
                            pass
                        precision[t, :, k, a, m] = np.array(q)
                        scores[t, :, k, a, m] = np.array(ss)
        self.eval = {"params": p, "counts": [T, R, K, A, M], "precision": precision, "recall": recall, "scores": scores}

    def summarize(self):
        self.stats = summarize(self.eval["precision"], self.eval["recall"], self.params)


def summarize(precision: np.ndarray, recall: np.ndarray, p: Optional[Params] = None) -> np.ndarray:
    """COCOeval.summarize -> _summarizeDets: the 12 stats (without the printing)."""
    p = p or Params()

    def _summarize(ap=1, iouThr=None, areaRng="all", maxDets=100):
        aind = [i for i, aRng in enumerate(p.areaRngLbl) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(p.maxDets) if mDet == maxDets]
        if ap == 1:
            s = precision
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            s = recall
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, aind, mind]
        if len(s[s > -1]) == 0:
            mean_s = -1
        else:
            mean_s = np.mean(s[s > -1])
        return mean_s

    stats = np.zeros((12,))
    stats[0] = _summarize(1)
    stats[1] = _summarize(1, iouThr=.5, maxDets=p.maxDets[2])
    stats[2] = _summarize(1, iouThr=.75, maxDets=p.maxDets[2])
    stats[3] = _summarize(1, areaRng="small", maxDets=p.maxDets[2])
    stats[4] = _summarize(1, areaRng="medium", maxDets=p.maxDets[2])
    stats[5] = _summarize(1, areaRng="large", maxDets=p.maxDets[2])
    stats[6] = _summarize(0, maxDets=p.maxDets[0])
    stats[7] = _summarize(0, maxDets=p.maxDets[1])
    stats[8] = _summarize(0, maxDets=p.maxDets[2])
    stats[9] = _summarize(0, areaRng="small", maxDets=p.maxDets[2])
    stats[10] = _summarize(0, areaRng="medium", maxDets=p.maxDets[2])
    stats[11] = _summarize(0, areaRng="large", maxDets=p.maxDets[2])
    return stats


def derive_coco_results(stats: Optional[np.ndarray], precisions: Optional[np.ndarray], class_names: Optional[Sequence[str]]) -> Dict[str, float]:
    """detectron2 COCOEvaluator._derive_coco_results for iou_type "bbox" (stats None: no predictions at all)."""
    metrics = ["AP", "AP50", "AP75", "APs", "APm", "APl"]
    if stats is None:
        return {metric: float("nan") for metric in metrics}
    results = {metric: float(stats[idx] * 100 if stats[idx] >= 0 else "nan") for idx, metric in enumerate(metrics)}
    if class_names is None or len(class_names) <= 1:
        return results
    assert len(class_names) == precisions.shape[2]
    for idx, name in enumerate(class_names):
        precision = precisions[:, :, idx, 0, -1]
        precision = precision[precision > -1]
        ap = np.mean(precision) if precision.size else float("nan")
        results["AP-" + name] = float(ap * 100)
    return results


def evaluate_bbox(coco_gt: dict, results: List[dict], class_names: Optional[Sequence[str]] = None) -> dict:
    """COCOEvaluator's bbox path end to end: {"bbox": metrics, "precision", "recall", "scores", "stats"} (arrays None when
    there are no results, as detectron2 skips COCOeval then)."""
    gt = COCO(copy.deepcopy(coco_gt))
    if len(results) == 0:
        return {"bbox": derive_coco_results(None, None, class_names), "precision": None, "recall": None, "scores": None, "stats": None}
    dt = gt.loadRes(results)
    E = COCOeval(gt, dt)
    E.evaluate()
    E.accumulate()
    E.summarize()
    return {"bbox": derive_coco_results(E.stats, E.eval["precision"], class_names), "precision": E.eval["precision"],
            "recall": E.eval["recall"], "scores": E.eval["scores"], "stats": E.stats}
