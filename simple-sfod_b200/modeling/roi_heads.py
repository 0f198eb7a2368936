"""ROI-heads plugins of the reference on the sm_100a kernels.

``SourceFreeAdaptiveTeacherStandardROIHeads`` (reference daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:25-215),
its eval sibling (``..._eval.py:25-128``) and ``AdaptiveTeacherStandardROIHeads`` (reference adaptive_teacher_roi_heads.py:22-187)
share one body: ROIPooler -> box head -> predictor, then either ``box_predictor.inference`` (the pseudo-labelling
path: pooling, decode, per-class NMS, top-k all run in libsfod_b200) or the training losses.  Proposal labelling /
sampling and the losses (the student's training step, SURVEY.md 8f rank 1) are restated from detectron2 0.6 and the
reference in plain torch; in that mode the library contributes ROIAlign forward AND backward (autograd) and the decode
kernels.  Without autograd and in strict fp32 (``matmul.allow_tf32`` off) the box-head FCs run on the library's 3xTF32
tensor-core kernel (``ops.linear_3xtf32``: fp32-level accuracy, see ``FastRCNNConvFCHead.forward``); the student's training
step and TF32 math keep them on cuBLAS.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np
import torch
from torch import Tensor, nn

from ..registry import ROI_BOX_HEAD_REGISTRY, ROI_HEADS_REGISTRY
from ..structures import Boxes, ImageList, Instances, ShapeSpec, pairwise_iou
from ..utils.events import get_event_storage
from .fast_rcnn import FastRCNNOutputLayers, SourceFreeFastRCNNOutputLayers, packed_proposal_batch
from .matcher import Matcher, add_ground_truth_to_proposals, subsample_labels
from .poolers import ROIPooler


@ROI_BOX_HEAD_REGISTRY.register()
class FastRCNNConvFCHead(nn.Sequential):
    """detectron2 FastRCNNConvFCHead (conv layers optional, then FCs with ReLU); c2_xavier / c2_msra init."""

    def __init__(self, cfg_or_shape, input_shape: Optional[ShapeSpec] = None, *, conv_dims: List[int] = None,
                 fc_dims: List[int] = None, conv_norm: str = ""):
        super().__init__()
        if hasattr(cfg_or_shape, "MODEL"):
            cfg = cfg_or_shape
            conv_dims = [cfg.MODEL.ROI_BOX_HEAD.CONV_DIM] * cfg.MODEL.ROI_BOX_HEAD.NUM_CONV
            fc_dims = [cfg.MODEL.ROI_BOX_HEAD.FC_DIM] * cfg.MODEL.ROI_BOX_HEAD.NUM_FC
            conv_norm = cfg.MODEL.ROI_BOX_HEAD.NORM
        else:
            input_shape = cfg_or_shape
        conv_dims, fc_dims = list(conv_dims or []), list(fc_dims or [])
        assert len(conv_dims) + len(fc_dims) > 0
        assert conv_norm == "", "normalised conv heads are not used by any shipped config"
        self._output_size = (input_shape.channels, input_shape.height, input_shape.width)
        self.conv_norm_relus, self.fcs = [], []
        for k, conv_dim in enumerate(conv_dims):
            conv = nn.Conv2d(self._output_size[0], conv_dim, kernel_size=3, padding=1)
            nn.init.kaiming_normal_(conv.weight, mode="fan_out", nonlinearity="relu")
            nn.init.constant_(conv.bias, 0)
            self.add_module("conv{}".format(k + 1), conv)
            self.add_module("conv_relu{}".format(k + 1), nn.ReLU())
            self.conv_norm_relus.append(conv)
            self._output_size = (conv_dim, self._output_size[1], self._output_size[2])
        for k, fc_dim in enumerate(fc_dims):
            if k == 0:
                self.add_module("flatten", nn.Flatten())
            fc = nn.Linear(int(np.prod(self._output_size)), fc_dim)
            nn.init.kaiming_uniform_(fc.weight, a=1)  # c2_xavier_fill
            nn.init.constant_(fc.bias, 0)
            self.add_module("fc{}".format(k + 1), fc)
            self.add_module("fc_relu{}".format(k + 1), nn.ReLU())
            self.fcs.append(fc)
            self._output_size = fc_dim

    def forward(self, x: Tensor) -> Tensor:
        """Without autograd, on CUDA fp32 input and with ``matmul.allow_tf32`` off (strict fp32), every FC + ReLU runs as one
        ``ops.linear_3xtf32`` call (tensor cores, fp32-level accuracy).  Otherwise -- the student's training step, TF32 math,
        CPU -- the layers run as the ``nn.Sequential`` they are."""
        if not self._native_fcs(x):
            return super().forward(x)
        from .. import ops
        for k, conv in enumerate(self.conv_norm_relus):
            x = getattr(self, "conv_relu{}".format(k + 1))(conv(x))
        x = torch.flatten(x, 1)
        for fc in self.fcs:   # every fc is followed by its ReLU
            x = ops.linear_3xtf32(x, fc.weight, fc.bias, relu=True)
        return x

    def _native_fcs(self, x: Tensor) -> bool:
        if not self.fcs or not x.is_cuda or x.dtype != torch.float32 or torch.backends.cuda.matmul.allow_tf32:
            return False
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return False
        from .. import ops
        return all(ops.linear_3xtf32_supported(fc.in_features, fc.out_features) for fc in self.fcs)

    @property
    def output_shape(self) -> ShapeSpec:
        o = self._output_size
        return ShapeSpec(channels=o) if isinstance(o, int) else ShapeSpec(channels=o[0], height=o[1], width=o[2])


def build_box_head(cfg, input_shape: ShapeSpec):
    """detectron2.modeling.roi_heads.box_head.build_box_head."""
    return ROI_BOX_HEAD_REGISTRY.get(cfg.MODEL.ROI_BOX_HEAD.NAME)(cfg, input_shape)


class _StandardROIHeadsBase(nn.Module):
    """The slice of detectron2 StandardROIHeads the reference's subclasses rely on (box branch only: MASK_ON False)."""

    predictor_cls = FastRCNNOutputLayers

    def __init__(self, cfg=None, input_shape: Dict[str, ShapeSpec] = None, *, box_in_features: List[str] = None,
                 box_pooler: ROIPooler = None, box_head: nn.Module = None, box_predictor: nn.Module = None,
                 num_classes: int = None, batch_size_per_image: int = 512, positive_fraction: float = 0.25,
                 proposal_append_gt: bool = True, train_on_pred_boxes: bool = False, proposal_matcher: Matcher = None):
        super().__init__()
        if cfg is not None:
            proposal_matcher = Matcher(cfg.MODEL.ROI_HEADS.IOU_THRESHOLDS, cfg.MODEL.ROI_HEADS.IOU_LABELS, allow_low_quality_matches=False)
            parts = self._init_box_head(cfg, input_shape)
            box_in_features, box_pooler = parts["box_in_features"], parts["box_pooler"]
            box_head, box_predictor = parts["box_head"], parts["box_predictor"]
            num_classes = cfg.MODEL.ROI_HEADS.NUM_CLASSES
            batch_size_per_image = cfg.MODEL.ROI_HEADS.BATCH_SIZE_PER_IMAGE
            positive_fraction = cfg.MODEL.ROI_HEADS.POSITIVE_FRACTION
            proposal_append_gt = cfg.MODEL.ROI_HEADS.PROPOSAL_APPEND_GT
            train_on_pred_boxes = cfg.MODEL.ROI_BOX_HEAD.TRAIN_ON_PRED_BOXES
        self.in_features = self.box_in_features = box_in_features
        self.box_pooler, self.box_head, self.box_predictor = box_pooler, box_head, box_predictor
        self.num_classes = num_classes
        self.batch_size_per_image, self.positive_fraction = batch_size_per_image, positive_fraction
        self.proposal_append_gt, self.train_on_pred_boxes = proposal_append_gt, train_on_pred_boxes
        self.proposal_matcher = proposal_matcher or Matcher([0.5], [0, 1], allow_low_quality_matches=False)

    @classmethod
    def _init_box_head(cls, cfg, input_shape):
        """reference source_free_adaptive_teacher_roi_heads.py:28-66 (ROIPooler built at :42-47)."""
        in_features = cfg.MODEL.ROI_HEADS.IN_FEATURES
        pooler_resolution = cfg.MODEL.ROI_BOX_HEAD.POOLER_RESOLUTION
        pooler_scales = tuple(1.0 / input_shape[k].stride for k in in_features)
        sampling_ratio = cfg.MODEL.ROI_BOX_HEAD.POOLER_SAMPLING_RATIO
        pooler_type = cfg.MODEL.ROI_BOX_HEAD.POOLER_TYPE
        in_channels = [input_shape[f].channels for f in in_features]
        assert len(set(in_channels)) == 1, in_channels
        in_channels = in_channels[0]
        box_pooler = ROIPooler(output_size=pooler_resolution, scales=pooler_scales, sampling_ratio=sampling_ratio,
                               pooler_type=pooler_type)
        box_head = build_box_head(cfg, ShapeSpec(channels=in_channels, height=pooler_resolution, width=pooler_resolution))
        if cfg.MODEL.ROI_HEADS.LOSS == "CrossEntropy":
            box_predictor = cls.predictor_cls(cfg, box_head.output_shape)
        else:
            raise ValueError("Unknown ROI head loss.")
        return {"box_in_features": in_features, "box_pooler": box_pooler, "box_head": box_head, "box_predictor": box_predictor}

    def _sample_proposals(self, matched_idxs: Tensor, matched_labels: Tensor, gt_classes: Tensor):
        """d2 ROIHeads._sample_proposals."""
        has_gt = gt_classes.numel() > 0
        if has_gt:
            gt_classes = gt_classes[matched_idxs]
            gt_classes[matched_labels == 0] = self.num_classes   # background
            gt_classes[matched_labels == -1] = -1                # ignore
        else:
            gt_classes = torch.zeros_like(matched_idxs) + self.num_classes
        sampled_fg_idxs, sampled_bg_idxs = subsample_labels(gt_classes, self.batch_size_per_image, self.positive_fraction, self.num_classes)
        sampled_idxs = torch.cat([sampled_fg_idxs, sampled_bg_idxs], dim=0)
        return sampled_idxs, gt_classes[sampled_idxs]

    _sample_calls = 0   # advances the counter-based sampling key of the batched path (one value per call)

    def _sampling_seed(self) -> int:
        type(self)._sample_calls += 1
        return (torch.initial_seed() * 0x9E3779B97F4A7C15 + type(self)._sample_calls) & ((1 << 64) - 1)

    @torch.no_grad()
    def label_and_sample_proposals(self, proposals: List[Instances], targets: List[Instances], branch: str = "") -> List[Instances]:
        """reference source_free_adaptive_teacher_roi_heads.py:165-215.  On CUDA the whole batch is labelled and sampled with
        one fused matcher call per image (no sync), ONE sampler launch for all images and ONE device->host read of the
        (num_fg, num_bg) counts -- the reference's loop synchronises ~4 times per image (two ``nonzero`` in subsample_labels,
        two ``.item()`` for the logged counts).  Elsewhere (CPU tensors) the per-image torch steps run as in detectron2."""
        gt_boxes = [x.gt_boxes for x in targets]
        if self.proposal_append_gt:
            proposals = add_ground_truth_to_proposals(gt_boxes, proposals)
        if len(proposals) and proposals[0].proposal_boxes.tensor.is_cuda and hasattr(self.proposal_matcher, "match_boxes"):
            return self._label_and_sample_batched(proposals, targets, branch)
        proposals_with_gt, num_fg_samples, num_bg_samples = [], [], []
        for proposals_per_image, targets_per_image in zip(proposals, targets):
            has_gt = len(targets_per_image) > 0
            if hasattr(self.proposal_matcher, "match_boxes"):   # fused pairwise_iou + Matcher on the device
                matched_idxs, matched_labels = self.proposal_matcher.match_boxes(targets_per_image.gt_boxes, proposals_per_image.proposal_boxes)
            else:
                matched_idxs, matched_labels = self.proposal_matcher(
                    pairwise_iou(targets_per_image.gt_boxes, proposals_per_image.proposal_boxes))
            sampled_idxs, gt_classes = self._sample_proposals(matched_idxs, matched_labels, targets_per_image.gt_classes)
            proposals_per_image = proposals_per_image[sampled_idxs]
            proposals_per_image.gt_classes = gt_classes
            if has_gt:
                sampled_targets = matched_idxs[sampled_idxs]
                for (trg_name, trg_value) in targets_per_image.get_fields().items():
                    if trg_name.startswith("gt_") and not proposals_per_image.has(trg_name):
                        proposals_per_image.set(trg_name, trg_value[sampled_targets])
            else:
                proposals_per_image.gt_boxes = Boxes(targets_per_image.gt_boxes.tensor.new_zeros((len(sampled_idxs), 4)))
            num_bg_samples.append((gt_classes == self.num_classes).sum().item())
            num_fg_samples.append(gt_classes.numel() - num_bg_samples[-1])
            proposals_with_gt.append(proposals_per_image)
        storage = get_event_storage()
        storage.put_scalar("roi_head/num_target_fg_samples_" + branch, np.mean(num_fg_samples))
        storage.put_scalar("roi_head/num_target_bg_samples_" + branch, np.mean(num_bg_samples))
        return proposals_with_gt

    def _label_and_sample_batched(self, proposals: List[Instances], targets: List[Instances], branch: str) -> List[Instances]:
        from .. import ops
        matched, classes = [], []
        for proposals_per_image, targets_per_image in zip(proposals, targets):
            matched_idxs, matched_labels = self.proposal_matcher.match_boxes(targets_per_image.gt_boxes, proposals_per_image.proposal_boxes)
            if len(targets_per_image) > 0:                       # d2 ROIHeads._sample_proposals, labelling half
                gt_classes = targets_per_image.gt_classes[matched_idxs]
                gt_classes = torch.where(matched_labels == 0, torch.full_like(gt_classes, self.num_classes), gt_classes)
                gt_classes = torch.where(matched_labels == -1, torch.full_like(gt_classes, -1), gt_classes)
            else:
                gt_classes = torch.zeros_like(matched_idxs) + self.num_classes
            matched.append(matched_idxs)
            classes.append(gt_classes)
        lengths = [int(c.numel()) for c in classes]
        sampled, counts = ops.subsample_labels_batched(torch.cat(classes), lengths, self.batch_size_per_image, self.positive_fraction,
                                                       self.num_classes, self._sampling_seed())
        host = counts.cpu().tolist()                              # the ONE device->host read of the batch
        out, num_fg_samples, num_bg_samples = [], [], []
        for i, (proposals_per_image, targets_per_image) in enumerate(zip(proposals, targets)):
            nfg, nbg = host[i]
            sampled_idxs = sampled[i, : nfg + nbg]
            gt_classes = classes[i][sampled_idxs]
            proposals_per_image = proposals_per_image[sampled_idxs]
            proposals_per_image.gt_classes = gt_classes
            if len(targets_per_image) > 0:
                sampled_targets = matched[i][sampled_idxs]
                for (trg_name, trg_value) in targets_per_image.get_fields().items():
                    if trg_name.startswith("gt_") and not proposals_per_image.has(trg_name):
                        proposals_per_image.set(trg_name, trg_value[sampled_targets])
            else:
                proposals_per_image.gt_boxes = Boxes(targets_per_image.gt_boxes.tensor.new_zeros((len(sampled_idxs), 4)))
            num_fg_samples.append(nfg); num_bg_samples.append(nbg)
            out.append(proposals_per_image)
        storage = get_event_storage()
        storage.put_scalar("roi_head/num_target_fg_samples_" + branch, np.mean(num_fg_samples))
        storage.put_scalar("roi_head/num_target_bg_samples_" + branch, np.mean(num_bg_samples))
        return out

    def _wants_loss(self, compute_loss: bool, compute_val_loss: bool) -> bool:
        return (self.training and compute_loss) or compute_val_loss

    def forward(self, images: ImageList, features: Dict[str, Tensor], proposals: List[Instances],
                targets: Optional[List[Instances]] = None, compute_loss=True, branch="", compute_val_loss=False):
        """reference source_free_adaptive_teacher_roi_heads.py:68-106."""
        del images
        if self.training and compute_loss:
            assert targets
            proposals = self.label_and_sample_proposals(proposals, targets, branch=branch)
        elif compute_val_loss:
            assert targets
            tmp = self.proposal_append_gt
            self.proposal_append_gt = False
            proposals = self.label_and_sample_proposals(proposals, targets, branch=branch)
            self.proposal_append_gt = tmp
        del targets
        if self._wants_loss(compute_loss, compute_val_loss):
            out = self._forward_box(features, proposals, compute_loss, compute_val_loss, branch)
            return (proposals, out[0]) + tuple(out[2:])      # (proposals, losses, box_features[, instance_proposals])
        pred_instances, predictions = self._forward_box(features, proposals, compute_loss, compute_val_loss, branch)
        return pred_instances, predictions

    def _box_predictions(self, features: Dict[str, Tensor], proposals: List[Instances]):
        feats = [features[f] for f in self.box_in_features]
        pb = packed_proposal_batch(proposals) if (not torch.is_grad_enabled() and len(feats) == 1) else None
        if pb is not None:
            # Sync-free inference path: pool the padded (N, P) proposal batch as it left the RPN kernel (rows beyond an
            # image's count are zero boxes whose outputs are ignored downstream through the device-side counts).
            N, P = pb.boxes.shape[:2]
            idx = torch.arange(N, device=pb.boxes.device, dtype=pb.boxes.dtype).repeat_interleave(P).unsqueeze(1)
            rois = torch.cat([idx, pb.boxes.reshape(N * P, 4)], dim=1)
            box_features = self.box_pooler._pool_level(feats[0], rois, self.box_pooler.scales[0])
            box_features = self.box_head(box_features)
            return box_features, self.box_predictor(box_features)
        box_features = self.box_pooler(feats, [x.proposal_boxes for x in proposals])  # reference ...roi_heads.py:117
        box_features = self.box_head(box_features)
        return box_features, self.box_predictor(box_features)

    def _forward_box(self, features: Dict[str, Tensor], proposals: List[Instances], compute_loss: bool = True,
                     compute_val_loss: bool = False, branch: str = ""):
        box_features, predictions = self._box_predictions(features, proposals)
        if self._wants_loss(compute_loss, compute_val_loss):
            losses = self.box_predictor.losses(predictions, proposals)
            return self._after_losses(losses, predictions, box_features, proposals)
        pred_instances, _ = self.box_predictor.inference(predictions, proposals)  # reference ...roi_heads.py:161
        return pred_instances, predictions

    def _replace_proposals_by_predictions(self, predictions, proposals: List[Instances]) -> None:
        with torch.no_grad():
            pred_boxes = self.box_predictor.predict_boxes_for_gt_classes(predictions, proposals)
            for proposals_per_image, pred_boxes_per_image in zip(proposals, pred_boxes):
                proposals_per_image.proposal_boxes = Boxes(pred_boxes_per_image)

    def _after_losses(self, losses, predictions, box_features, proposals):
        """reference source_free_adaptive_teacher_roi_heads.py:139-158: proposals are replaced by the boxes predicted for
        their GT class (unconditionally), then the dense per-class instances for bpc_loss are produced."""
        self._replace_proposals_by_predictions(predictions, proposals)
        instance_proposals, _ = self.box_predictor.convert_bbox_scores(predictions, proposals)
        return losses, predictions, box_features, instance_proposals


@ROI_HEADS_REGISTRY.register()
class SourceFreeAdaptiveTeacherStandardROIHeads(_StandardROIHeadsBase):
    predictor_cls = SourceFreeFastRCNNOutputLayers


@ROI_HEADS_REGISTRY.register()
class SourceFreeAdaptiveTeacherEvalStandardROIHeads(_StandardROIHeadsBase):
    """reference ..._roi_heads_eval.py:25-128: identical, except that the loss switches ignore ``self.training``."""
    predictor_cls = SourceFreeFastRCNNOutputLayers

    def _wants_loss(self, compute_loss: bool, compute_val_loss: bool) -> bool:
        return bool(compute_loss or compute_val_loss)

    def forward(self, images, features, proposals, targets=None, compute_loss=True, branch="", compute_val_loss=False):
        del images
        if compute_loss:
            assert targets
            proposals = self.label_and_sample_proposals(proposals, targets, branch=branch)
        del targets
        if self._wants_loss(compute_loss, compute_val_loss):
            out = self._forward_box(features, proposals, compute_loss, compute_val_loss, branch)
            return (proposals, out[0]) + tuple(out[2:])
        return self._forward_box(features, proposals, compute_loss, compute_val_loss, branch)


@ROI_HEADS_REGISTRY.register()
class AdaptiveTeacherStandardROIHeads(_StandardROIHeadsBase):
    """reference adaptive_teacher_roi_heads.py:22-187 (plain FastRCNNOutputLayers predictor; the loss branch returns
    ``(losses, predictions, box_features)`` and only replaces the proposals when ``train_on_pred_boxes``, :119-133)."""
    predictor_cls = FastRCNNOutputLayers

    def _after_losses(self, losses, predictions, box_features, proposals):
        if self.train_on_pred_boxes:
            self._replace_proposals_by_predictions(predictions, proposals)
        return losses, predictions, box_features
