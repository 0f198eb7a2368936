"""ResNet-C4 backbone with detectron2's module layout and state_dict keys (``build_resnet_backbone``, the default
``MODEL.BACKBONE.NAME`` that reference configs/r101_c4_cs_foggy_adaptive_teacher_source_free.yaml:1-23 and
configs/r_101_c4_cs_foggy_adabn.yaml inherit: ``RESNETS.DEPTH 101``, ``NORM "BN"``, ``OUT_FEATURES ["res4"]``,
``STRIDE_IN_1X1 True``, ``BACKBONE.FREEZE_AT 2``).

Keys: ``stem.conv1.{weight, norm.*}``, ``res{2,3,4}.{i}.{shortcut, conv1, conv2, conv3}.{weight, norm.*}`` -- a detectron2
checkpoint loads unchanged.  The convolutions stay on cuDNN (BASELINE.json north_star); what this module adds is the
normalisation path of the teacher / AdaBN forwards (train() under no_grad):

* ``conv -> BN -> ReLU`` runs the two native BN kernels (statistics 4 B/element, fused normalise+ReLU in place 8 B/element);
* the bottleneck tail ``conv3 -> BN``, ``out += shortcut``, ``relu_`` -- three elementwise passes (28 B/element) in
  detectron2's ``BottleneckBlock.forward`` -- is ONE pass (``residual`` fusion of ``sfod_bn_finalize_apply``, 12 B/element);
* the frozen stem and res2 (``FREEZE_AT 2`` turns their 11 norm layers into ``FrozenBatchNorm2d``) use the same fused pass with
  coefficients from the running statistics (``sfod_bn_frozen_apply``).

Any other mode (autograd for the student, CPU) runs plain torch modules with identical arithmetic order.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
from torch import Tensor, nn
from torch.nn import functional as F

from .. import ops
from ..registry import BACKBONE_REGISTRY
from ..structures import ShapeSpec
from .batch_norm import SfodBatchNorm2d


class FrozenBatchNorm2d(nn.Module):
    """detectron2.layers.FrozenBatchNorm2d: fixed statistics and affine parameters, all buffers (no num_batches_tracked)."""

    _version = 3

    def __init__(self, num_features: int, eps: float = 1e-5):
        super().__init__()
        self.num_features, self.eps = num_features, eps
        self.register_buffer("weight", torch.ones(num_features))
        self.register_buffer("bias", torch.zeros(num_features))
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features) - eps)

    def _native_ok(self, x: Tensor) -> bool:
        return not torch.is_grad_enabled() and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4

    def forward(self, x: Tensor, fuse_relu: bool = False, inplace: bool = False, residual: Optional[Tensor] = None) -> Tensor:
        if self._native_ok(x):
            return ops.bn_frozen_forward(x, self.weight, self.bias, self.running_mean, self.running_var, self.eps,
                                         fuse_relu=fuse_relu, inplace=inplace, residual=residual)
        if x.requires_grad:
            scale = self.weight * (self.running_var + self.eps).rsqrt()
            bias = self.bias - self.running_mean * scale
            y = x * scale.reshape(1, -1, 1, 1).to(x.dtype) + bias.reshape(1, -1, 1, 1).to(x.dtype)
        else:
            y = F.batch_norm(x, self.running_mean, self.running_var, self.weight, self.bias, training=False, eps=self.eps)
        if residual is not None:
            y = y + residual
        return F.relu(y) if fuse_relu else y

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        state_dict.pop(prefix + "num_batches_tracked", None)     # a BatchNorm2d checkpoint loads into the frozen layer
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)

    @classmethod
    def convert_frozen_batchnorm(cls, module: nn.Module) -> nn.Module:
        """detectron2: replace every BatchNorm2d below ``module`` by a FrozenBatchNorm2d with the same tensors' values."""
        res = module
        if isinstance(module, nn.modules.batchnorm._BatchNorm):
            res = cls(module.num_features, module.eps)
            if module.affine:
                res.weight.data = module.weight.data.clone().detach()
                res.bias.data = module.bias.data.clone().detach()
            res.running_mean.data = module.running_mean.data
            res.running_var.data = module.running_var.data
        else:
            for name, child in module.named_children():
                new_child = cls.convert_frozen_batchnorm(child)
                if new_child is not child:
                    module.add_module(name, new_child)
        return res


def get_norm(norm: str, out_channels: int) -> Optional[nn.Module]:
    """detectron2.layers.get_norm for the two values the shipped configs use."""
    if not norm:
        return None
    if norm == "BN":
        return SfodBatchNorm2d(out_channels)
    if norm == "FrozenBN":
        return FrozenBatchNorm2d(out_channels)
    raise NotImplementedError(f"RESNETS.NORM {norm!r}: the shipped configs use 'BN' (and detectron2's default 'FrozenBN')")


class Conv2d(nn.Conv2d):
    """detectron2.layers.Conv2d: a convolution that owns its norm layer (``.norm``), applied after the convolution."""

    def __init__(self, *args, norm: Optional[nn.Module] = None, **kwargs):
        super().__init__(*args, **kwargs)
        self.norm = norm

    def conv(self, x: Tensor) -> Tensor:
        return F.conv2d(x, self.weight, self.bias, self.stride, self.padding, self.dilation, self.groups)

    def forward(self, x: Tensor, fuse_relu: bool = False, residual: Optional[Tensor] = None) -> Tensor:
        """conv -> norm [-> + residual] [-> ReLU].  The elementwise tail goes to the norm layer's fused kernel when it can
        take it (train()/no_grad BatchNorm, FrozenBatchNorm under no_grad); otherwise the same steps run in plain torch."""
        z = self.conv(x)
        n = self.norm
        if n is not None and hasattr(n, "_native_ok") and n._native_ok(z):
            return n(z, fuse_relu=fuse_relu, inplace=True, residual=residual)      # z is private to this call
        if n is not None:
            z = n(z)
        if residual is not None:
            z = z + residual
        return F.relu(z) if fuse_relu else z


def _msra_fill(conv: nn.Conv2d) -> None:
    nn.init.kaiming_normal_(conv.weight, mode="fan_out", nonlinearity="relu")
    if conv.bias is not None:
        nn.init.constant_(conv.bias, 0)


class CNNBlockBase(nn.Module):
    def __init__(self, in_channels: int, out_channels: int, stride: int):
        super().__init__()
        self.in_channels, self.out_channels, self.stride = in_channels, out_channels, stride

    def freeze(self):
        for p in self.parameters():
            p.requires_grad = False
        FrozenBatchNorm2d.convert_frozen_batchnorm(self)
        return self


class BasicStem(CNNBlockBase):
    """detectron2 BasicStem: 7x7/2 conv + norm + ReLU, then 3x3/2 max-pool."""

    def __init__(self, in_channels: int = 3, out_channels: int = 64, norm: str = "BN"):
        super().__init__(in_channels, out_channels, 4)
        self.conv1 = Conv2d(in_channels, out_channels, kernel_size=7, stride=2, padding=3, bias=False, norm=get_norm(norm, out_channels))
        _msra_fill(self.conv1)

    def forward(self, x: Tensor) -> Tensor:
        x = self.conv1(x, fuse_relu=True)
        return F.max_pool2d(x, kernel_size=3, stride=2, padding=1)


class BottleneckBlock(CNNBlockBase):
    """detectron2 BottleneckBlock (1x1 -> 3x3 -> 1x1, optional projection shortcut, stride on the first 1x1 when
    ``stride_in_1x1``).  forward: relu(conv1) -> relu(conv2) -> conv3; out += shortcut; relu."""

    def __init__(self, in_channels: int, out_channels: int, *, bottleneck_channels: int, stride: int = 1, num_groups: int = 1,
                 norm: str = "BN", stride_in_1x1: bool = False, dilation: int = 1):
        super().__init__(in_channels, out_channels, stride)
        if in_channels != out_channels:
            self.shortcut = Conv2d(in_channels, out_channels, kernel_size=1, stride=stride, bias=False, norm=get_norm(norm, out_channels))
        else:
            self.shortcut = None
        stride_1x1, stride_3x3 = (stride, 1) if stride_in_1x1 else (1, stride)
        self.conv1 = Conv2d(in_channels, bottleneck_channels, kernel_size=1, stride=stride_1x1, bias=False,
                            norm=get_norm(norm, bottleneck_channels))
        self.conv2 = Conv2d(bottleneck_channels, bottleneck_channels, kernel_size=3, stride=stride_3x3, padding=1 * dilation, bias=False,
                            groups=num_groups, dilation=dilation, norm=get_norm(norm, bottleneck_channels))
        self.conv3 = Conv2d(bottleneck_channels, out_channels, kernel_size=1, bias=False, norm=get_norm(norm, out_channels))
        for layer in [self.conv1, self.conv2, self.conv3, self.shortcut]:
            if layer is not None:
                _msra_fill(layer)

    def forward(self, x: Tensor) -> Tensor:
        out = self.conv1(x, fuse_relu=True)
        out = self.conv2(out, fuse_relu=True)
        shortcut = self.shortcut(x) if self.shortcut is not None else x
        return self.conv3(out, fuse_relu=True, residual=shortcut)


class ResNet(nn.Module):
    """detectron2 ResNet restricted to what ``build_resnet_backbone`` builds for the C4 configs."""

    def __init__(self, stem: nn.Module, stages: List[List[CNNBlockBase]], out_features: List[str], freeze_at: int = 0):
        super().__init__()
        self.stem = stem
        current_stride = stem.stride
        self._out_feature_strides = {"stem": current_stride}
        self._out_feature_channels = {"stem": stem.out_channels}
        self.stage_names, self.stages = [], []
        for i, blocks in enumerate(stages):
            name = "res" + str(i + 2)
            stage = nn.Sequential(*blocks)
            self.add_module(name, stage)
            self.stage_names.append(name)
            self.stages.append(stage)
            current_stride = int(current_stride * int(torch.tensor([k.stride for k in blocks]).prod()))
            self._out_feature_strides[name] = current_stride
            self._out_feature_channels[name] = blocks[-1].out_channels
        self._out_features = out_features
        self.freeze(freeze_at)

    @property
    def size_divisibility(self) -> int:
        return 0

    def output_shape(self) -> Dict[str, ShapeSpec]:
        return {n: ShapeSpec(channels=self._out_feature_channels[n], stride=self._out_feature_strides[n]) for n in self._out_features}

    def forward(self, x: Tensor) -> Dict[str, Tensor]:
        assert x.dim() == 4, f"ResNet takes an input of shape (N, C, H, W). Got {x.shape} instead!"
        outputs = {}
        x = self.stem(x)
        if "stem" in self._out_features:
            outputs["stem"] = x
        for name, stage in zip(self.stage_names, self.stages):
            x = stage(x)
            if name in self._out_features:
                outputs[name] = x
        return outputs

    def freeze(self, freeze_at: int = 0):
        """detectron2 ResNet.freeze: stem for freeze_at >= 1, res2 for >= 2, ...; frozen blocks lose their gradients and their
        BatchNorm layers become FrozenBatchNorm2d."""
        if freeze_at >= 1:
            self.stem.freeze()
        for idx, stage in enumerate(self.stages, start=2):
            if freeze_at >= idx:
                for block in stage.children():
                    block.freeze()
        return self


def make_stage(num_blocks: int, first_stride: int, in_channels: int, out_channels: int, bottleneck_channels: int, norm: str,
               stride_in_1x1: bool) -> List[CNNBlockBase]:
    blocks = []
    for i in range(num_blocks):
        blocks.append(BottleneckBlock(in_channels, out_channels, bottleneck_channels=bottleneck_channels,
                                      stride=first_stride if i == 0 else 1, norm=norm, stride_in_1x1=stride_in_1x1))
        in_channels = out_channels
    return blocks


@BACKBONE_REGISTRY.register()
def build_resnet_backbone(cfg, input_shape=None):
    """detectron2.modeling.backbone.build_resnet_backbone for depth 50 / 101 / 152 bottleneck nets up to the last stage named
    in RESNETS.OUT_FEATURES (C4: res4)."""
    r = cfg.MODEL.RESNETS
    norm = r.NORM
    depth = r.DEPTH
    out_features = list(r.OUT_FEATURES)
    in_channels = input_shape.channels if input_shape is not None and input_shape.channels else len(cfg.MODEL.PIXEL_MEAN)
    stem = BasicStem(in_channels=in_channels, out_channels=r.get("STEM_OUT_CHANNELS", 64), norm=norm)
    if depth not in (50, 101, 152):
        raise NotImplementedError("only the bottleneck depths 50 / 101 / 152 are provided (the shipped configs use 101)")
    num_blocks_per_stage = {50: [3, 4, 6, 3], 101: [3, 4, 23, 3], 152: [3, 8, 36, 3]}[depth]
    num_groups, width_per_group = r.get("NUM_GROUPS", 1), r.get("WIDTH_PER_GROUP", 64)
    if num_groups != 1:
        raise NotImplementedError("grouped bottlenecks (ResNeXt) are not used by any shipped config")
    bottleneck_channels = num_groups * width_per_group
    in_ch, out_ch = r.get("STEM_OUT_CHANNELS", 64), r.get("RES2_OUT_CHANNELS", 256)
    stride_in_1x1 = r.get("STRIDE_IN_1X1", True)
    out_stage_idx = [{"res2": 2, "res3": 3, "res4": 4, "res5": 5}[f] for f in out_features if f != "stem"]
    max_stage_idx = max(out_stage_idx)
    stages = []
    for idx, stage_idx in enumerate(range(2, max_stage_idx + 1)):
        first_stride = 1 if idx == 0 else 2
        stages.append(make_stage(num_blocks_per_stage[idx], first_stride, in_ch, out_ch, bottleneck_channels, norm, stride_in_1x1))
        in_ch = out_ch
        out_ch *= 2
        bottleneck_channels *= 2
    return ResNet(stem, stages, out_features=out_features, freeze_at=cfg.MODEL.BACKBONE.FREEZE_AT)
