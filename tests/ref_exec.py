"""Executes the REFERENCE's own on-disk functions of the hot path on the CPU (test infrastructure).

The reference cannot be imported as a package here (detectron2 / fvcore / yacs are not installable), but the functions that
state the hot path's semantics are plain torch once three names resolve: ``Boxes`` / ``Instances`` (provided by
``sfod_b200.d2shim``, a detectron2 namespace backed by this package's structures), ``batched_nms`` (detectron2 0.6
``layers/nms.py``: ``torchvision.ops.boxes.batched_nms(boxes.float(), scores, idxs, iou_threshold)`` -- bound here to the
installed torchvision CPU kernel) and ``comm.get_world_size``.  Module-level sources are imported from where they lie under
$SFOD_REFERENCE_ROOT; trainer METHODS live in modules whose imports cannot be satisfied (DefaultTrainer, checkpointing, data
loaders), so their ``def`` nodes are cut out of the parsed file and compiled in a small namespace -- the code that runs is the
reference's text, byte for byte, and nothing is copied into this repository.  ``.cuda()`` calls inside those functions are
neutralised (identity) for the duration of a call so that the CPU is the device.

Used by tests/test_oracle_vs_reference_cpu.py (oracle/d2_cpu.py == reference, live) and tests/golden/make_golden_ref.py (writes
tests/golden/ref_exec.npz, the fixture that stands in for the reference wherever its sources are absent).
"""
from __future__ import annotations

import ast
import contextlib
import importlib
import importlib.util
import os
import sys
import types
from collections import OrderedDict
from unittest import mock

import numpy as np
import torch
import torchvision
from torch import nn

# A checkout of the original project (the directory holding daod/); the tests that execute it skip without one.
REF_ROOT = os.environ.get("SFOD_REFERENCE_ROOT", "")
TRAINER = os.path.join(REF_ROOT, "daod/engine/trainers/source_free_adaptive_teacher.py")
TRAINER_AT = os.path.join(REF_ROOT, "daod/engine/trainers/adaptive_teacher.py")
BASE = os.path.join(REF_ROOT, "daod/engine/trainers/base.py")
ADAPTIVE = os.path.join(REF_ROOT, "daod/modeling/adaptive_thresh/adaptive_confidence.py")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_ROOT, "daod"))


def d2_batched_nms(boxes, scores, idxs, iou_threshold):
    """detectron2 0.6 layers.nms.batched_nms (SURVEY.md A-4)."""
    assert boxes.shape[-1] == 4
    return torchvision.ops.boxes.batched_nms(boxes.float(), scores, idxs, iou_threshold)


@contextlib.contextmanager
def cpu_is_the_device():
    with mock.patch.object(torch.Tensor, "cuda", lambda self, *a, **k: self):
        yield


def _cut(path: str, names, cls: str | None = None) -> ast.Module:
    """The ``def`` nodes called ``names`` (module level, or inside class ``cls``) of the file at ``path``."""
    with open(path) as f:
        tree = ast.parse(f.read(), filename=path)
    scope = tree.body
    if cls is not None:
        scope = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    found = [n for n in scope if isinstance(n, ast.FunctionDef) and n.name in names]
    missing = set(names) - {n.name for n in found}
    assert not missing, f"{path}: {missing} not found"
    return found


def _compile_methods(path: str, cls: str, names, namespace: dict, new_name: str):
    """A class ``new_name`` holding the reference methods ``names`` of ``cls`` (compiled from the reference file, with its
    file name and line numbers, in ``namespace``)."""
    body = _cut(path, names, cls)
    node = ast.ClassDef(name=new_name, bases=[], keywords=[], body=body, decorator_list=[], lineno=body[0].lineno, col_offset=0,
                        end_lineno=body[-1].end_lineno, end_col_offset=0)
    if "type_params" in ast.ClassDef._fields:
        node.type_params = []
    mod = ast.Module(body=[node], type_ignores=[])
    ast.fix_missing_locations(mod)
    exec(compile(mod, path, "exec"), namespace)
    return namespace[new_name]


def _compile_functions(path: str, names, namespace: dict):
    mod = ast.Module(body=_cut(path, names), type_ignores=[])
    exec(compile(mod, path, "exec"), namespace)
    return [namespace[n] for n in names]


class Reference:
    """Handles to the reference's functions, live from REF_ROOT.  Use as a context manager (installs / removes the shim)."""

    def __enter__(self):
        import sfod_b200  # noqa: F401
        from sfod_b200 import d2shim
        self._had = {k: v for k, v in sys.modules.items() if k.split(".")[0] == "detectron2"}
        self._d2shim = d2shim
        assert d2shim.install(force=True)
        import detectron2.layers as d2l
        d2l.batched_nms = d2_batched_nms                     # the CPU kernel the reference binds to, through d2's one-liner
        from detectron2.structures import Boxes, Instances
        import detectron2.utils.comm as comm
        self.Boxes, self.Instances, self.comm = Boxes, Instances, comm
        pkg = types.ModuleType("refexec_rh")
        pkg.__path__ = [os.path.join(REF_ROOT, "daod/modeling/roi_heads")]   # the package's real __init__ is not executed
        sys.modules["refexec_rh"] = pkg
        self.fast_rcnn = importlib.import_module("refexec_rh.fast_rcnn")                       # daod/modeling/roi_heads/fast_rcnn.py
        self.sf_fast_rcnn = importlib.import_module("refexec_rh.source_free_fast_rcnn")        # .../source_free_fast_rcnn.py
        assert self.fast_rcnn.__file__.startswith(REF_ROOT) and self.fast_rcnn.batched_nms is d2_batched_nms
        spec = importlib.util.spec_from_file_location("refexec_adaptive_confidence", ADAPTIVE)
        self.adaptive = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(self.adaptive)
        ns = {"torch": torch, "np": np, "Instances": Instances, "Boxes": Boxes, "OrderedDict": OrderedDict, "comm": comm, "nn": nn}
        self.Trainer = _compile_methods(
            TRAINER, "SourceFreeAdaptiveTeacherTrainer",
            ["threshold_bbox", "adaptive_threshold_bbox", "prediction_threshold_bbox", "process_pseudo_label", "count_label_prediction",
             "update_adaptive_threshold", "_update_teacher_model"], dict(ns), "RefSourceFreeTrainerMethods")
        self.TrainerAT = _compile_methods(TRAINER_AT, "AdaptiveTeacherTrainer", ["threshold_bbox", "_update_teacher_model"], dict(ns),
                                          "RefAdaptiveTeacherTrainerMethods")
        self.reset_bn_stats, self.recursive_traversal = _compile_functions(BASE, ["reset_bn_stats", "recursive_traversal"], dict(ns))
        return self

    def __exit__(self, *exc):
        self._d2shim.uninstall()
        for k in [k for k in sys.modules if k.startswith("refexec_")]:
            del sys.modules[k]
        sys.modules.update(self._had)

    # ------------------------------------------------------------------ convenience wrappers (dict in / dict out, like the oracle)
    def to_instances(self, d: dict):
        inst = self.Instances(tuple(d["image_size"]))
        for k, v in d.items():
            if k == "image_size":
                continue
            inst.set(k, self.Boxes(v) if k.endswith("_boxes") else v)
        return inst

    @staticmethod
    def from_instances(inst) -> dict:
        out = {"image_size": tuple(inst.image_size)}
        for k, v in inst.get_fields().items():
            out[k] = v.tensor if hasattr(v, "tensor") else v
        return out

    def fast_rcnn_inference_single_image(self, boxes, scores, image_shape, score_thresh, nms_thresh, topk):
        """reference daod/modeling/roi_heads/fast_rcnn.py:88-142."""
        inst, rows = self.fast_rcnn.fast_rcnn_inference_single_image_with_mcd(boxes, scores, image_shape, score_thresh, nms_thresh, topk, 0)
        out = self.from_instances(inst)
        out["kept_rows"] = rows
        return out

    def fast_rcnn_inference_single_image_new(self, boxes, scores, image_shape):
        """reference daod/modeling/roi_heads/source_free_fast_rcnn.py:82-147 (``self`` is unused by the method)."""
        fn = self.sf_fast_rcnn.SourceFreeFastRCNNOutputLayers.fast_rcnn_inference_single_image_new
        inst, rows = fn(None, boxes, scores, image_shape, 0.05, 0.5, 100, None)
        out = self.from_instances(inst)
        out["kept_rows"] = rows
        return out

    def trainer(self, cfg=None, classwise_acc=None, threshold=None, num_classes=8, model=None, model_teacher=None, reserve_matrix=None):
        """An object carrying the reference trainer's methods and only the attributes those methods read."""
        t = self.Trainer()
        t.cfg, t.model, t.model_teacher, t.reserve_matrix = cfg, model, model_teacher, reserve_matrix
        if threshold is not None:
            with cpu_is_the_device():
                t.self_training_criterion = self.adaptive.AdaptiveConfidenceBasedSelfTrainingLoss(threshold, num_classes)
            if classwise_acc is not None:
                t.self_training_criterion.classwise_acc = classwise_acc
        return t
