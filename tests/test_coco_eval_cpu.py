"""COCO box AP on the host: the oracle's known answers (oracle/coco_eval_cpu.py, pycocotools' COCOeval restated), the C ABI's
refusals before any launch, and ops.coco_box_eval's refusal of CPU tensors."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import coco_eval_cpu as o
from sfod_b200 import _lib, ops
from coco_eval_cases import known_answer_cases, synthetic_case, to_results

EPS = np.spacing(1)
E1 = 1.0 / (0.0 + 1.0 + EPS)          # precision of one true positive and no false positive
REC = o.Params().recThrs
CASES = known_answer_cases()


def run(name):
    gt, dets = CASES[name]
    return o.evaluate_bbox(gt, to_results(gt, dets), [c["name"] for c in sorted(gt["categories"], key=lambda c: c["id"])])


def test_params_are_pycocotools():
    p = o.Params()
    assert len(p.iouThrs) == 10 and len(p.recThrs) == 101 and p.maxDets == [1, 10, 100]
    assert p.areaRng == [[0, 1e10], [0, 1024], [1024, 9216], [9216, 1e10]]


def test_perfect_match():
    r = run("perfect")
    assert np.all(r["precision"][:, :, 0, 0, :] == E1) and np.all(r["recall"][:, 0, 0, :] == 1.0)
    assert np.all(r["precision"][:, :, 0, 1] == -1) and np.all(r["precision"][:, :, 0, 3] == -1)    # a medium box only
    assert r["stats"][0] == np.mean(np.full(1010, E1)) and r["stats"][3] == -1 and math.isnan(r["bbox"]["APs"])


def test_duplicate_detection_is_one_false_positive():
    r = run("duplicate")
    e2 = 2.0 / (1.0 + 2.0 + EPS)                       # tp = [1, 1, 2], fp = [0, 1, 1]; envelope [E1, e2, e2]
    want = np.where(REC <= 0.5, E1, e2)
    assert np.array_equal(r["precision"][0, :, 0, 0, 2], want) and r["recall"][0, 0, 0, 2] == 1.0
    assert np.array_equal(r["scores"][0, :, 0, 0, 2], np.where(REC <= 0.5, np.float32(0.9), np.float32(0.7)).astype(np.float64))
    assert r["recall"][0, 0, 0, 0] == 0.5                # maxDet 1: the first detection only


def test_crowd_absorbs_several_detections():
    r = run("crowd")
    # order d2, d3, d4 (ignored: matched to the crowd region), d1 (true positive)
    assert np.all(r["precision"][:, :, 0, 0, 2] == E1) and np.all(r["recall"][:, 0, 0, 2] == 1.0)
    assert r["scores"][0, 0, 0, 0, 2] == np.float32(0.9) and np.all(r["scores"][0, 1:, 0, 0, 2] == 0.5)


def test_ignored_gt_order_and_break():
    r = run("ignored_order")
    # IoU with the regular gt 6400/9025 = 0.709: matched up to t = 0.70; above, the crowd gt takes it (ignored)
    assert np.all(r["precision"][:5, :, 0, 0, 2] == E1) and np.all(r["recall"][:5, 0, 0, 2] == 1.0)
    assert np.all(r["precision"][5:, :, 0, 0, 2] == 0) and np.all(r["recall"][5:, 0, 0, 2] == 0)


def test_gt_id_zero_counts_as_false_positive():
    r = run("gt_id_zero")
    assert np.all(r["precision"][:, :, 0, 0, :] == 0) and np.all(r["recall"][:, 0, 0, :] == 0) and r["stats"][0] == 0
    assert np.all(r["precision"][:, :, 0, 1, :] == -1)  # small: the gt is out of range, the unmatched-by-id detection ignored


def test_only_100_detections_per_image_and_category():
    r = run("over_100")
    assert np.all(r["precision"][:, :, 0, 0, 2] == 0) and np.all(r["recall"][:, 0, 0, 2] == 0)
    gt, dets = CASES["over_100"]
    ev = o.COCOeval(o.COCO(gt), o.COCO(gt).loadRes(to_results(gt, dets)))
    ev.evaluate()
    assert len(ev.evalImgs[0]["dtIds"]) == 100


def test_score_ties_follow_image_then_list_order():
    r = run("score_ties")
    # [img1 fp, img1 tp, img2 tp, img2 fp]: rc = [0, .5, 1, 1], envelope starts at 2 / (3 + eps)
    assert np.all(r["precision"][0, :, 0, 0, 2] == 2.0 / (1.0 + 2.0 + EPS))
    assert np.all(r["scores"][0, :, 0, 0, 2] == 0.5)


def test_area_range_bounds_are_inclusive():
    r = run("area_bounds")
    assert np.all(r["precision"][:, :, 0, 1, 2] == E1) and np.all(r["precision"][:, :, 0, 3, 2] == E1)
    assert np.all(r["precision"][:, :, 0, 2, 2] == 1.0)      # medium holds both: pr = [E1, 2 / (2 + eps)] and 2 + eps rounds to 2
    assert np.all(r["recall"][:, 0, :, 2] == 1.0)


def test_category_without_gt_is_nan():
    r = run("category_without_gt")
    assert np.all(r["precision"][:, :, 1] == -1) and np.all(r["recall"][:, 1] == -1)
    assert math.isnan(r["bbox"]["AP-c7"]) and r["bbox"]["AP-c3"] == float(np.mean(np.full(1010, E1)) * 100)


def test_image_without_detections_counts_its_gt():
    r = run("image_without_detections")
    assert r["recall"][0, 0, 0, 2] == 0.5
    assert np.array_equal(r["precision"][0, :, 0, 0, 2], np.where(REC <= 0.5, E1, 0.0))


def test_unknown_image_id_raises():
    gt, dets = CASES["perfect"]
    res = to_results(gt, dets)
    res[0]["image_id"] = 99
    with pytest.raises(AssertionError):
        o.evaluate_bbox(gt, res)


def test_oracle_matches_pycocotools_when_available():
    pytest.importorskip("pycocotools")
    from pycocotools.coco import COCO
    from pycocotools.cocoeval import COCOeval
    cases = list(CASES.values()) + [synthetic_case(s, 30, 4, 12, 40) for s in range(3)]
    for gt, dets in cases:
        res = to_results(gt, dets)
        want = o.evaluate_bbox(gt, res)
        cg = COCO()
        cg.dataset = {k: [dict(x) for x in v] for k, v in gt.items()}
        cg.createIndex()
        E = COCOeval(cg, cg.loadRes([dict(x) for x in res]), "bbox")
        E.evaluate(); E.accumulate(); E.summarize()
        assert np.array_equal(E.eval["precision"], want["precision"]) and np.array_equal(E.eval["recall"], want["recall"])
        assert np.array_equal(E.eval["scores"], want["scores"]) and np.array_equal(np.asarray(E.stats), want["stats"])


# ------------------------------------------------------------------------------------------------ C ABI and operator refusals
def _params(I=4, K=8, P=100):
    p = _lib.CocoEvalParams()
    p.n_images, p.n_categories, p.dt_stride = I, K, P
    p.n_iou_thrs, p.n_rec_thrs, p.n_area_rngs, p.n_max_dets = 10, 101, 4, 3
    for i, v in enumerate((1, 10, 100)):
        p.max_dets[i] = v
    return p


def test_coco_eval_refuses_before_any_launch():
    L = _lib.lib()
    launches = L.sfod_debug_launch_count()
    need = L.sfod_coco_eval_workspace_bytes(C.byref(_params()))
    assert need >= 4 * 100 * (4 * 4 + 1) + 512 * 8
    offs = (C.c_int64 * 5)(0, 3, 3, 7, 9)
    ptr = dict(offs=offs, gb=0x10000, ga=0x20000, gc=0x30000, gi=0x40000, gk=0x50000, db=0x60000, ds=0x70000, dc=0x80000, dn=0x90000,
               pr=0xA0000, sc=0xB0000, rc=0xC0000, ws=0xD0000, nbytes=need)

    def call(p=None, **over):
        a = {**ptr, **over}
        pp = C.byref(p if p is not None else _params()) if p != "null" else None
        return L.sfod_coco_eval(pp, a["offs"], a["gb"], a["ga"], a["gc"], a["gi"], a["gk"], a["db"], a["ds"], a["dc"], a["dn"],
                                a["pr"], a["sc"], a["rc"], a["ws"], a["nbytes"], None)

    def with_(**f):
        p = _params()
        for k, v in f.items():
            if k == "max_dets":
                for i, m in enumerate(v):
                    p.max_dets[i] = m
            else:
                setattr(p, k, v)
        return p

    assert call("null") == 1
    assert call(with_(n_images=-1)) == 1 and call(with_(n_categories=0)) == 1 and call(with_(dt_stride=0)) == 1
    assert call(with_(max_dets=(1, 0, 100))) == 1 and call(with_(n_rec_thrs=0)) == 1
    assert call(with_(n_categories=255)) == 3 and call(with_(dt_stride=1025)) == 3 and call(with_(n_iou_thrs=17)) == 3
    assert call(with_(n_area_rngs=5)) == 3 and call(with_(max_dets=(1, 10, 129))) == 3
    assert call(with_(n_images=1 << 14, dt_stride=1024)) == 3                          # image * P + rank beyond 24 bits
    assert call(offs=None) == 1 and call(pr=None) == 1 and call(dn=None) == 1 and call(db=None) == 1
    assert call(offs=(C.c_int64 * 5)(0, 3, 2, 7, 9)) == 1                            # gt not sorted by image
    assert call(offs=(C.c_int64 * 5)(1, 3, 3, 7, 9)) == 1
    assert call(offs=(C.c_int64 * 5)(0, 3, 1028, 1030, 1031)) == 3                  # 1025 gt in one image
    assert call(gb=None) == 1
    assert call(db=0x60004) == 4                                                      # SFOD_ERR_ALIGNMENT
    assert call(nbytes=need - 1) == 2 and call(ws=None) == 2                          # SFOD_ERR_WORKSPACE_TOO_SMALL
    assert L.sfod_coco_eval_workspace_bytes(C.byref(with_(n_categories=0))) == 0
    assert L.sfod_debug_launch_count() == launches


def test_coco_box_eval_refuses_cpu_tensors():
    f64, i64 = torch.zeros(1, 4, dtype=torch.float64), torch.zeros(1, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.coco_box_eval([0, 1], f64, f64[:, 0], torch.zeros(1, dtype=torch.uint8), i64, i64, torch.zeros(1, 1, 4), torch.zeros(1, 1),
                          torch.zeros(1, 1, dtype=torch.int64), torch.zeros(1, dtype=torch.int32), 1, o.Params().iouThrs,
                          o.Params().recThrs, o.Params().areaRng, [1, 10, 100])
