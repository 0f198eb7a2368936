"""engine.COCOBoxEvaluator in a gloo world of two CPU processes: the ranks exchange their error conditions before any tensor
collective, so detections on the CPU of one rank make every rank raise (no rank is left waiting in a collective), and a
world in which nobody processed anything returns {} everywhere."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["SFOD_ROOT"])
sys.path.insert(0, os.path.join(os.environ["SFOD_ROOT"], "tests"))
from sfod_b200 import engine
from sfod_b200.structures import Boxes, Instances
from coco_eval_cases import synthetic_case
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
gt, dets = synthetic_case(4, 8, 3, 6, 20)
out_dir = os.path.join(os.environ["OUT_DIR"], f"rank{rank}")

# nothing processed on any rank: {} everywhere, nothing written
ev = engine.COCOBoxEvaluator(gt, output_dir=out_dir)
assert ev.evaluate() == {} and all(v is None for v in ev.eval.values())

# rank 0 processes detections on the CPU, rank 1 processes nothing: both raise the same error
ev.reset()
if rank == 0:
    for img, b, s, c in dets:
        inst = Instances((600, 1200))
        inst.pred_boxes, inst.scores, inst.pred_classes = Boxes(b), s, c
        ev.process([{"image_id": img}], [{"instances": inst}])
try:
    ev.evaluate()
    raise SystemExit(f"rank {rank}: evaluate() must raise")
except RuntimeError as e:
    assert "no CPU fallback" in str(e) and "cpu on rank 0" in str(e), str(e)
assert not os.path.exists(os.path.join(out_dir, "coco_instances_results.json"))
dist.barrier()
print(f"COCO_DIST_CPU_OK {rank}")
dist.destroy_process_group()
'''


def test_world_size_2_gloo_cpu_detections_raise_on_every_rank(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, SFOD_ROOT=ROOT, OUT_DIR=str(tmp_path), MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29543", str(script)], capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert "COCO_DIST_CPU_OK 0" in r.stdout and "COCO_DIST_CPU_OK 1" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
