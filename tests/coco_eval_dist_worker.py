"""Worker of tests/test_gpu_coco_eval_distributed.py, started by ``torch.distributed.run``:
``python -m torch.distributed.run --nproc-per-node=N tests/coco_eval_dist_worker.py <gloo|nccl> <output directory>``.

The ranks evaluate one synthetic dataset (coco_eval_cases.synthetic_case) with ``engine.COCOBoxEvaluator``:

* ranks 0 and N-1 process the two halves of its detections (``engine.shard_range``); in a world of three, rank 1 processes
  nothing;
* rank 0's inputs carry height / width 1024 x 2048 for detections in the 600 x 1200 network frame (its ground truth is
  scaled to that frame);
* rank N-1 processes the last image of rank 0's half a second time, and the outputs of the VGG teacher on four small
  synthetic images (padded batches with device-side counts, ``packed_source``).

Rank 0's result must equal the oracle restatement of pycocotools on the rank-ordered result list and a single-process
evaluator fed the same outputs in rank order, and its json must equal that list; the other ranks return {} and write
nothing.  Then two failing evaluations: a detection on an image outside the ground truth on rank 1 only, and detections on
the CPU on rank 0 only, must make every rank raise.  Under gloo all ranks share cuda:0; under NCCL rank r uses cuda:r."""
from __future__ import annotations

import json
import math
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from coco_eval_cases import synthetic_case  # noqa: E402
from oracle import coco_eval_cpu as o  # noqa: E402
from sfod_b200 import config, engine, registry  # noqa: E402
from sfod_b200.engine.export import detector_postprocess, instances_to_coco_json, prediction_to_gt  # noqa: E402
from sfod_b200.structures import Boxes, Instances  # noqa: E402

RESULTS = "coco_instances_results.json"


def plain_outputs(dets, dev, output_size=None):
    inputs, outputs = [], []
    for img, b, s, c in dets:
        inst = Instances((600, 1200))
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.to(dev)), s.to(dev), c.to(dev)
        inp = {"image_id": img}
        if output_size is not None:
            inp["height"], inp["width"] = output_size
        inputs.append(inp)
        outputs.append({"instances": inst})
    return inputs, outputs


def teacher_batches(dev, ids):
    """The VGG teacher (random weights, seed 42) on 320 x 480 images whose evaluation frame is 544 x 816, two per batch.  Its
    detections stay padded device batches (``defer_host_read``, as in the benchmark's teacher step)."""
    torch.manual_seed(42)
    cfg = config.vgg_source_free_cfg()
    cfg.MODEL.DEVICE = str(dev)
    model = registry.build_model(cfg).eval()
    model.roi_heads.box_predictor.defer_host_read = True
    g = torch.Generator().manual_seed(17)
    ims = [torch.randint(0, 256, (3, 320, 480), dtype=torch.uint8, generator=g).to(dev) for _ in ids]
    batches = []
    with torch.no_grad():
        for i in range(0, len(ids), 2):
            inputs = [{"image": ims[j], "image_id": ids[j], "height": 544, "width": 816} for j in range(i, i + 2)]
            batches.append((inputs, model(inputs)))
    return batches


def same(got, want):
    """Result dicts equal, NaN equal to NaN (categories without any detection or ground truth)."""
    assert got.keys() == want.keys(), (got.keys(), want.keys())
    for k, v in want.items():
        assert got[k] == v or (math.isnan(v) and math.isnan(got[k])), (k, got[k], v)


def raises_everywhere(ev, exc, match):
    try:
        ev.evaluate()
    except exc as e:
        assert match in str(e), str(e)
        return
    raise AssertionError(f"rank {dist.get_rank()}: evaluate() did not raise {exc.__name__}")


def main():
    backend, out_root = sys.argv[1], sys.argv[2]
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]) if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, **({"device_id": dev} if backend == "nccl" else {}))
    last = world - 1

    K = 8                                                               # the VGG configuration's classes
    gt, dets = synthetic_case(7, 24, K, 12, 40)
    halves = [engine.shard_range(len(dets), j, 2) for j in range(2)]
    sx, sy = 2048 / 1200, 1024 / 600
    rank0_images = {d[0] for d in dets[halves[0][0]:halves[0][1]]}
    for a in gt["annotations"]:
        if a["image_id"] in rank0_images:
            x, y, w, h = a["bbox"]
            a["bbox"], a["area"] = [x * sx, y * sy, w * sx, h * sy], a["area"] * sx * sy
    teacher_ids = [9001, 9002, 9003, 9004]
    gt["images"] += [{"id": i, "height": 544, "width": 816} for i in teacher_ids]
    id_map = {k: c for k, c in enumerate(sorted(c["id"] for c in gt["categories"]))}
    names = [c["name"] for c in sorted(gt["categories"], key=lambda c: c["id"])]

    batches = []                                                        # this rank's (inputs, outputs), in processing order
    if rank == 0:
        b, e = halves[0]
        batches.append(plain_outputs(dets[b:e], dev, (1024, 2048)))
    if rank == last:
        b, e = halves[1]
        batches.append(plain_outputs(dets[b:e], dev))
        img, bx, s, c = dets[halves[0][1] - 1]                          # rank 0's last image, processed here too
        batches.append(plain_outputs([(img, bx[::2], s[::2], c[::2])], dev, (1024, 2048)))
        teacher = teacher_batches(dev, teacher_ids)
        assert all(out["instances"].packed_source() is not None for _, outs in teacher for out in outs)
        batches += teacher

    out_dir = os.path.join(out_root, f"rank{rank}")
    ev = engine.COCOBoxEvaluator(gt, output_dir=out_dir)
    for inputs, outputs in batches:
        ev.process(inputs, outputs)
    got = ev.evaluate()

    # every rank's outputs, as plain host tensors, on rank 0 for the references
    mine = []
    for inputs, outputs in batches:
        for inp, out in zip(inputs, outputs):
            inst = out["instances"]
            mine.append(({k: inp[k] for k in ("image_id", "height", "width") if k in inp}, inst.image_size,
                         inst.pred_boxes.tensor.cpu(), inst.scores.cpu(), inst.pred_classes.cpu()))
    every = [None] * world
    dist.all_gather_object(every, mine)

    if rank == 0:
        single = engine.COCOBoxEvaluator(gt, distributed=False, output_dir=os.path.join(out_root, "single"))
        results = []
        for inp, size, b, s, c in (x for part in every for x in part):
            inst = Instances(size)
            inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.to(dev)), s.to(dev), c.to(dev)
            single.process([inp], [{"instances": inst}])
            pp = detector_postprocess(inst, inp.get("height", size[0]), inp.get("width", size[1]))
            results += instances_to_coco_json(pp, inp["image_id"], id_map)
        assert {r["image_id"] for r in results} & set(teacher_ids), "the teacher produced no detection"
        want = o.evaluate_bbox(gt, results, names)
        ref = single.evaluate()
        for k in ("precision", "recall", "scores", "stats"):
            assert np.array_equal(ev.eval[k], want[k]), k
            assert np.array_equal(ev.eval[k], single.eval[k]), k
        same(got["bbox"], want["bbox"])
        same(got["bbox"], ref["bbox"])
        assert got.keys() == {"bbox"} and 0 < got["bbox"]["AP"] < 100
        with open(os.path.join(out_dir, RESULTS)) as f:
            written = json.load(f)
        with open(os.path.join(out_root, "single", RESULTS)) as f:
            assert json.load(f) == written
        assert written == results and len(results) > 0
        assert prediction_to_gt(written, gt) == prediction_to_gt(results, gt)
    else:
        assert got == {} and all(v is None for v in ev.eval.values())
        assert not os.path.exists(os.path.join(out_dir, RESULTS))

    # a detection on an image the ground truth does not list, on rank 1 only: every rank raises loadRes' error
    ev = engine.COCOBoxEvaluator(gt, output_dir=os.path.join(out_root, f"unknown{rank}"))
    if rank == 0:
        ev.process(*plain_outputs(dets[:2], dev))
    if rank == 1:
        img, b, s, c = dets[2]
        ev.process(*plain_outputs([(10 ** 7, b, s, c)], dev))
    raises_everywhere(ev, ValueError, "coco set")
    assert not os.path.exists(os.path.join(out_root, f"unknown{rank}", RESULTS))

    # detections on the CPU on rank 0 only: every rank raises
    ev = engine.COCOBoxEvaluator(gt)
    if rank == 0:
        ev.process(*plain_outputs(dets[:2], torch.device("cpu")))
    if rank == last:
        ev.process(*plain_outputs(dets[2:4], dev))
    raises_everywhere(ev, RuntimeError, "cpu on rank 0")

    dist.barrier()
    print(f"COCO_DIST_OK {rank}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
