"""Writes tests/golden/ref_exec.npz: inputs and outputs of the REFERENCE'S OWN functions, executed on the CPU from the sources
under $SFOD_REFERENCE_ROOT (tests/ref_exec.py: nothing is copied, the code that runs is the reference's text).

    SFOD_REFERENCE_ROOT=<checkout of the original project> python tests/golden/make_golden_ref.py

Functions executed (reference file:line):
  daod/modeling/roi_heads/fast_rcnn.py:88-142            fast_rcnn_inference_single_image_with_mcd   -> frcnn_*_out_*
  daod/modeling/roi_heads/source_free_fast_rcnn.py:82-147 fast_rcnn_inference_single_image_new        -> frcnn_*_conv_*
  daod/engine/trainers/source_free_adaptive_teacher.py:150-183 threshold_bbox (roih, 0.8)             -> frcnn_*_pl_*
  ...:185-228 adaptive_threshold_bbox with adaptive_confidence.py:21-33                              -> frcnn_*_adaptive_*
  ...:282-310 count_label_prediction / update_adaptive_threshold                                    -> reserve_count, classwise_acc_new
  ...:583-603 _update_teacher_model + load_state_dict                                                -> ema_out_*
Inputs: Fast R-CNN head outputs of sfod_b200.synth (seeded), decoded with ATen exp / softmax as detectron2's predict_boxes /
predict_probs do; the stored ``boxes`` / ``scores`` are the inputs of the on-disk functions, ``cls`` / ``deltas`` / ``proposals``
are kept as well so that the CUDA path can be run from the head outputs (tests/test_gpu_kernels.py).
"""
import os
import sys
from collections import OrderedDict

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import ref_exec  # noqa: E402
from oracle import d2_cpu as o  # noqa: E402  (only apply_deltas: detectron2's decode is not on disk)
from sfod_b200 import synth  # noqa: E402


def main():
    torch.set_num_threads(1)
    out = {}
    rows, sizes = [600, 300, 1300], [(600, 1200), (576, 1100), (600, 1200)]
    cls, dl = synth.box_head_outputs(sum(rows), 8, 301, 2.2, 1.0)
    props = synth.random_rois(1, sum(rows), 302)[:, 1:].contiguous()
    boxes = o.apply_deltas(dl, props, (10.0, 10.0, 5.0, 5.0)).split(rows)
    scores = torch.softmax(cls, -1).split(rows)
    acc = torch.tensor([1.0, 0.3, 1.0, 0.9, 0.05, 0.6, 0.0, 0.45])
    out["frcnn_n_images"] = np.int64(len(rows))
    out["frcnn_cls"], out["frcnn_deltas"], out["frcnn_proposals"], out["frcnn_rows"] = cls.numpy(), dl.numpy(), props.numpy(), np.array(rows)
    out["adaptive_acc"] = acc.numpy()

    class Cfg:
        class MODEL:
            class ROI_HEADS:
                NUM_CLASSES = 8
        class SEMISUPNET:
            BBOX_THRESHOLD = 0.8

    with ref_exec.Reference() as R, ref_exec.cpu_is_the_device():
        tr = R.trainer(cfg=Cfg, classwise_acc=acc.clone(), threshold=0.8)
        dets = []
        for i, (b, s, sz) in enumerate(zip(boxes, scores, sizes)):
            out[f"frcnn_{i}_boxes"], out[f"frcnn_{i}_scores"], out[f"frcnn_{i}_image_size"] = b.numpy(), s.numpy(), np.array(sz)
            det = R.fast_rcnn_inference_single_image(b.clone(), s.clone(), sz, 0.05, 0.5, 100)
            for k in ("pred_boxes", "scores", "pred_classes", "kept_rows"):
                out[f"frcnn_{i}_out_{k}"] = det[k].numpy()
            inst = R.to_instances({k: v for k, v in det.items() if k != "kept_rows"})
            dets.append(inst)
            pl = R.from_instances(tr.threshold_bbox(inst, thres=0.8, proposal_type="roih"))
            ad = R.from_instances(tr.adaptive_threshold_bbox(inst, thres=0.8, proposal_type="roih"))
            for k in ("gt_boxes", "gt_classes", "scores"):
                out[f"frcnn_{i}_pl_{k}"] = pl[k].numpy()
                out[f"frcnn_{i}_adaptive_{k}"] = ad[k].numpy()
            conv = R.fast_rcnn_inference_single_image_new(b.clone(), s.clone(), sz)
            # its scores are s[kept_rows, pred_classes] bit for bit (a gather, no NMS): not stored, which keeps the file under 1 MB
            assert torch.equal(conv["scores"], s[conv["kept_rows"], conv["pred_classes"]])
            for k in ("pred_boxes", "pred_classes", "kept_rows"):
                out[f"frcnn_{i}_conv_{k}"] = conv[k].numpy()
        reserve = tr.count_label_prediction(dets)
        out["reserve_count"] = reserve.numpy()
        tr.reserve_matrix = torch.stack([reserve, reserve * 3, torch.ones(8)])
        out["reserve_matrix"] = tr.reserve_matrix.clone().numpy()
        tr.update_adaptive_threshold()
        out["classwise_acc_new"] = tr.self_training_criterion.classwise_acc.numpy()

        def make(seed):
            torch.manual_seed(seed)
            m = nn.Sequential(OrderedDict(conv=nn.Conv2d(3, 16, 3), bn=nn.BatchNorm2d(16), fc=nn.Linear(33, 17)))
            with torch.no_grad():
                m.bn.running_mean.normal_(); m.bn.running_var.uniform_(0.5, 2.0); m.bn.num_batches_tracked += 1000 + seed
            return m
        student = make(1)
        for k, v in student.state_dict().items():
            out[f"ema_s_{k}"] = v.clone().numpy()
        for k, v in make(2).state_dict().items():
            out[f"ema_t_{k}"] = v.clone().numpy()
        for tag, rate in (("a", 0.9996), ("b", 0.999696), ("c", 0.0)):
            teacher = make(2)
            t = R.Trainer(); t.model, t.model_teacher = student, teacher
            t._update_teacher_model(keep_rate=rate)
            for k, v in teacher.state_dict().items():
                out[f"ema_out_{tag}_{k}"] = v.clone().numpy()
    np.savez_compressed(os.path.join(HERE, "ref_exec.npz"), **out)
    n_pl = sum(len(out[f"frcnn_{i}_pl_scores"]) for i in range(len(rows)))
    print(f"wrote ref_exec.npz: {len(out)} arrays, {n_pl} pseudo-labels over {len(rows)} images")


if __name__ == "__main__":
    main()
