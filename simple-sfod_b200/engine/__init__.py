"""Host-side mirror of the trainer-level hot-path functions of the reference (reference daod/engine/trainers/*)."""
from .pseudo_label import process_pseudo_label, threshold_bbox  # noqa: F401
from .ema import TeacherEMA, update_teacher_model  # noqa: F401
from .adabn import adabn_refinement, recursive_traversal, reset_bn_stats, test_refinement  # noqa: F401
from .sharding import images_per_rank, shard_range  # noqa: F401
from .adaptive_threshold import (AdaptiveConfidenceBasedSelfTrainingLoss, adaptive_threshold_bbox, count_label_prediction,  # noqa: F401
                                 prediction_threshold_bbox, update_adaptive_threshold)
from .export import (batch_to_coco_json, detector_postprocess, instances_to_coco_json, load_pseudo_label_annotations,  # noqa: F401
                     prediction_to_gt)
from .hooks import HookBase, TeacherEMAHook, TrainerBase  # noqa: F401
from .augment import draw_params as draw_strong_augmentation_params, strong_augment  # noqa: F401
from .augment import apply_weak_to_boxes, draw_weak_params, weak_augment  # noqa: F401
from .evaluation import COCOBoxEvaluator, inference_on_dataset  # noqa: F401
