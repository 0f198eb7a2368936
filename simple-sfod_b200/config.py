"""Minimal yacs-style config carrying the detectron2 0.6 defaults the hot path reads (SURVEY.md A-8) plus
the keys the reference adds (reference daod/config.py:8-141).  ``get_cfg()`` returns the defaults;
``vgg_source_free_cfg()`` / ``r101_c4_source_free_cfg()`` apply the overrides of the two shipped mean-teacher
YAMLs (reference configs/faster_rcnn_VGG_cityscapes_foggy_adaptive_teacher_source_free.yaml:1-79 and
configs/r101_c4_cs_foggy_adaptive_teacher_source_free.yaml); ``merge_from_file`` accepts those YAMLs directly.
"""
from __future__ import annotations

import copy
from typing import Any, Dict


class CfgNode(dict):
    """Attribute-access nested dict (yacs.config.CfgNode subset: clone / merge_from_file / merge_from_list)."""

    def __init__(self, init: Dict[str, Any] = None):
        super().__init__()
        for k, v in (init or {}).items():
            self[k] = CfgNode(v) if isinstance(v, dict) and not isinstance(v, CfgNode) else v

    def __getattr__(self, name: str) -> Any:
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    def __setattr__(self, name: str, value: Any) -> None:
        self[name] = value

    def clone(self) -> "CfgNode":
        return copy.deepcopy(self)

    def merge_from_dict(self, other: Dict[str, Any]) -> None:
        for k, v in other.items():
            if isinstance(v, dict):
                if k not in self or not isinstance(self[k], CfgNode):
                    self[k] = CfgNode()
                self[k].merge_from_dict(v)
            else:
                self[k] = v

    def merge_from_file(self, path: str) -> None:
        import yaml
        with open(path) as f:
            self.merge_from_dict(yaml.safe_load(f) or {})

    def merge_from_list(self, opts) -> None:
        assert len(opts) % 2 == 0
        for key, val in zip(opts[0::2], opts[1::2]):
            node = self
            parts = key.split(".")
            for p in parts[:-1]:
                node = node[p]
            node[parts[-1]] = val


_DEFAULTS = {
    "VERSION": 2,
    "SEED": -1,
    "MODEL": {
        "DEVICE": "cuda",
        "META_ARCHITECTURE": "GeneralizedRCNN",
        "MASK_ON": False,
        "PIXEL_MEAN": [103.530, 116.280, 123.675],
        "PIXEL_STD": [1.0, 1.0, 1.0],
        "BACKBONE": {"NAME": "build_resnet_backbone", "FREEZE_AT": 2},
        "PROPOSAL_GENERATOR": {"NAME": "RPN", "MIN_SIZE": 0},
        "ANCHOR_GENERATOR": {"NAME": "DefaultAnchorGenerator", "SIZES": [[32, 64, 128, 256, 512]],
                             "ASPECT_RATIOS": [[0.5, 1.0, 2.0]], "ANGLES": [[-90, 0, 90]], "OFFSET": 0.0},
        "RPN": {"HEAD_NAME": "StandardRPNHead", "IN_FEATURES": ["res4"], "BOUNDARY_THRESH": -1,
                "IOU_THRESHOLDS": [0.3, 0.7], "IOU_LABELS": [0, -1, 1], "BATCH_SIZE_PER_IMAGE": 256,
                "POSITIVE_FRACTION": 0.5, "BBOX_REG_LOSS_TYPE": "smooth_l1", "BBOX_REG_LOSS_WEIGHT": 1.0,
                "BBOX_REG_WEIGHTS": (1.0, 1.0, 1.0, 1.0), "SMOOTH_L1_BETA": 0.0, "LOSS_WEIGHT": 1.0,
                "PRE_NMS_TOPK_TRAIN": 12000, "PRE_NMS_TOPK_TEST": 6000, "POST_NMS_TOPK_TRAIN": 2000,
                "POST_NMS_TOPK_TEST": 1000, "NMS_THRESH": 0.7, "CONV_DIMS": [-1]},
        "ROI_HEADS": {"NAME": "Res5ROIHeads", "NUM_CLASSES": 80, "IN_FEATURES": ["res4"], "IOU_THRESHOLDS": [0.5],
                      "IOU_LABELS": [0, 1], "BATCH_SIZE_PER_IMAGE": 512, "POSITIVE_FRACTION": 0.25,
                      "SCORE_THRESH_TEST": 0.05, "NMS_THRESH_TEST": 0.5, "PROPOSAL_APPEND_GT": True,
                      "LOSS": "CrossEntropy"},
        "ROI_BOX_HEAD": {"NAME": "", "BBOX_REG_LOSS_TYPE": "smooth_l1", "BBOX_REG_LOSS_WEIGHT": 1.0,
                         "BBOX_REG_WEIGHTS": (10.0, 10.0, 5.0, 5.0), "SMOOTH_L1_BETA": 0.0, "POOLER_RESOLUTION": 14,
                         "POOLER_SAMPLING_RATIO": 0, "POOLER_TYPE": "ROIAlignV2", "NUM_FC": 0, "FC_DIM": 1024,
                         "NUM_CONV": 0, "CONV_DIM": 256, "NORM": "", "CLS_AGNOSTIC_BBOX_REG": False,
                         "TRAIN_ON_PRED_BOXES": False, "USE_FED_LOSS": False, "USE_SIGMOID_CE": False},
        "RESNETS": {"DEPTH": 50, "OUT_FEATURES": ["res4"], "NORM": "FrozenBN"},
    },
    "INPUT": {"MIN_SIZE_TRAIN": (800,), "MIN_SIZE_TRAIN_SAMPLING": "choice", "MAX_SIZE_TRAIN": 1333, "MIN_SIZE_TEST": 800,
              "MAX_SIZE_TEST": 1333, "RANDOM_FLIP": "horizontal", "FORMAT": "BGR"},
    "VIS_PERIOD": 0,
    "TEST": {"DETECTIONS_PER_IMAGE": 100},
    "SOLVER": {"IMS_PER_BATCH": 16, "IMS_PER_BATCH_TARGET": 16},
    # keys added by the reference (daod/config.py)
    "SEMISUPNET": {"BBOX_THRESHOLD": 0.7, "PSEUDO_BBOX_SAMPLE": "thresholding", "TEACHER_UPDATE_ITER": 1,
                   "BURN_UP_STEP": 12000, "EMA_KEEP_RATE": 0.0, "DIS_TYPE": "res4", "INS_DC": False},
    "ADAPTIVE_THRESHOLD": {"ENABLED": False, "WARM_UP": 100, "RESERVE": 500},
    "VGG": {"BN": True},
}


def get_cfg() -> CfgNode:
    return CfgNode(copy.deepcopy(_DEFAULTS))


def vgg_source_free_cfg() -> CfgNode:
    """faster_rcnn_VGG_cityscapes_foggy_adaptive_teacher_source_free.yaml (model-relevant keys)."""
    cfg = get_cfg()
    cfg.merge_from_dict({
        "MODEL": {"META_ARCHITECTURE": "SourceFreeAdaptiveTeacherGeneralizedRCNN",
                  "BACKBONE": {"NAME": "build_vgg_backbone"},
                  "ROI_HEADS": {"IN_FEATURES": ["vgg4"], "NAME": "SourceFreeAdaptiveTeacherStandardROIHeads", "NUM_CLASSES": 8},
                  "ROI_BOX_HEAD": {"NAME": "FastRCNNConvFCHead", "NUM_FC": 2, "POOLER_RESOLUTION": 7},
                  "RPN": {"IN_FEATURES": ["vgg4"], "PRE_NMS_TOPK_TEST": 6000, "POST_NMS_TOPK_TEST": 1000},
                  "PROPOSAL_GENERATOR": {"NAME": "PseudoLabRPN"}},
        "INPUT": {"MIN_SIZE_TRAIN": (600,), "MIN_SIZE_TEST": 600},
        "SOLVER": {"IMS_PER_BATCH": 1, "IMS_PER_BATCH_TARGET": 1},
        "SEMISUPNET": {"BBOX_THRESHOLD": 0.8, "TEACHER_UPDATE_ITER": 1, "BURN_UP_STEP": 2000, "EMA_KEEP_RATE": 0.9996,
                       "DIS_TYPE": "vgg4", "INS_DC": True},
        "SEED": 42, "VGG": {"BN": True},
    })
    return cfg


def r101_c4_source_free_cfg() -> CfgNode:
    """r101_c4_cs_foggy_adaptive_teacher_source_free.yaml (model-relevant keys)."""
    cfg = get_cfg()
    cfg.merge_from_dict({
        "MODEL": {"META_ARCHITECTURE": "SourceFreeAdaptiveTeacherGeneralizedRCNN",
                  "RESNETS": {"DEPTH": 101, "NORM": "BN"},
                  "ROI_HEADS": {"NAME": "SourceFreeAdaptiveTeacherStandardROIHeads", "NUM_CLASSES": 8, "BATCH_SIZE_PER_IMAGE": 256},
                  "ROI_BOX_HEAD": {"NAME": "FastRCNNConvFCHead", "NUM_FC": 2, "FC_DIM": 2048, "POOLER_RESOLUTION": 7},
                  "ANCHOR_GENERATOR": {"SIZES": [[64, 128, 256, 512]]},
                  "RPN": {"PRE_NMS_TOPK_TEST": 6000, "POST_NMS_TOPK_TEST": 1000, "BATCH_SIZE_PER_IMAGE": 256},
                  "PROPOSAL_GENERATOR": {"NAME": "PseudoLabRPN"}},
        "INPUT": {"MIN_SIZE_TRAIN": (600,), "MIN_SIZE_TEST": 600},
        "SEMISUPNET": {"BBOX_THRESHOLD": 0.8, "EMA_KEEP_RATE": 0.9996},
    })
    return cfg
