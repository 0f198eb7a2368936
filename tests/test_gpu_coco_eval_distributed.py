"""COCO box AP across the ranks of a distributed run (engine.COCOBoxEvaluator, distributed=True): rank 0 evaluates the
detections of every rank in rank order, equal to the oracle and to a single-process evaluator fed the same outputs, and
writes detectron2's coco_instances_results.json; failures raise on every rank (tests/coco_eval_dist_worker.py).  Single
process: output_dir writes the same result list and changes nothing else."""
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch

from sfod_b200 import engine
from sfod_b200.engine.export import detector_postprocess, instances_to_coco_json, prediction_to_gt
from sfod_b200.structures import Boxes, Instances
from coco_eval_cases import synthetic_case

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_worker(tmp_path, backend, nproc, port):
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
                        "--master-port", str(port), os.path.join(ROOT, "tests", "coco_eval_dist_worker.py"), backend, str(tmp_path)],
                       capture_output=True, text=True, env=env, timeout=600)
    # the end of each rank's own output: the rank that failed first is not the last one to write
    per_rank = "".join(f"\n--- rank {k}:\n" + "\n".join([ln for ln in r.stderr.splitlines() if ln.startswith(f"[rank{k}]")][-30:])
                       for k in range(nproc))
    assert r.returncode == 0, r.stdout[-2000:] + per_rank + r.stderr[-2000:]
    for rank in range(nproc):
        assert f"COCO_DIST_OK {rank}" in r.stdout, r.stdout[-2000:] + per_rank


def test_three_ranks_gloo_on_one_gpu(tmp_path, cuda_device):
    run_worker(tmp_path, "gloo", 3, 29541)


def test_two_ranks_nccl_on_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    run_worker(tmp_path, "nccl", 2, 29542)


def _outputs(dets, dev, output_size):
    inputs, outputs = [], []
    for img, b, s, c in dets:
        inst = Instances((600, 1200))
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b.to(dev)), s.to(dev), c.to(dev)
        inputs.append({"image_id": img, "height": output_size[0], "width": output_size[1]})
        outputs.append({"instances": inst})
    return inputs, outputs


def _evaluate_counting_syncs(ev, inputs, outputs):
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            for i in range(0, len(inputs), 5):
                ev.process(inputs[i:i + 5], outputs[i:i + 5])
            got = ev.evaluate()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    return got, len([x for x in w if "synchroniz" in str(x.message).lower()])


def test_single_process_output_dir_writes_the_result_list(tmp_path, cuda_device):
    """The json is detectron2's result list (instances_to_coco_json of the post-processed outputs, in processing order, a
    re-processed image included); the evaluation is the same with and without output_dir, at one more device->host copy."""
    gt, dets = synthetic_case(9, 30, 5, 20, 80)
    dets = dets + [(img, b[1::2], s[1::2], c[1::2]) for img, b, s, c in dets[:3]]
    img, b, s, c = dets[0]
    b = b.clone()
    b[0, 0], b[0, 2] = 1250.0, 1300.0                                   # empty after the clip: not written
    dets[0] = (img, b, s, c)
    inputs, outputs = _outputs(dets, cuda_device, (1024, 2048))
    plain = engine.COCOBoxEvaluator(gt)
    ev = engine.COCOBoxEvaluator(gt, output_dir=str(tmp_path / "out"))
    for e in (plain, ev):                                               # warm-up: ground truth on the device, pinned staging
        e.process(inputs, outputs)
        e.evaluate()
        e.reset()
    want, syncs_plain = _evaluate_counting_syncs(plain, inputs, outputs)
    got, syncs = _evaluate_counting_syncs(ev, inputs, outputs)
    assert set(got) == {"bbox"} and got["bbox"].keys() == want["bbox"].keys() and syncs_plain == 1 and syncs == 2
    for k, v in want["bbox"].items():
        assert got["bbox"][k] == v or (np.isnan(v) and np.isnan(got["bbox"][k])), k
    for k in ("precision", "recall", "scores", "stats"):
        assert np.array_equal(ev.eval[k], plain.eval[k]), k
    id_map = {k: cid for k, cid in enumerate(ev.cat_ids)}
    results = [r for inp, out in zip(inputs, outputs)
               for r in instances_to_coco_json(detector_postprocess(out["instances"], inp["height"], inp["width"]), inp["image_id"], id_map)]
    with open(tmp_path / "out" / "coco_instances_results.json") as f:
        written = json.load(f)
    assert written == results and len(results) < sum(len(d[2]) for d in dets)
    assert prediction_to_gt(written, gt) == prediction_to_gt(results, gt)


def test_single_process_output_dir_without_records(tmp_path, cuda_device):
    gt, _ = synthetic_case(9, 5, 2, 3, 5)
    ev = engine.COCOBoxEvaluator(gt, output_dir=str(tmp_path / "out"))
    assert ev.evaluate() == {} and not (tmp_path / "out").exists()
