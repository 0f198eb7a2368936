"""Cross-rank reduction of the AdaBN statistics (SURVEY.md 8e, collective (2)).

The statistics kernel leaves, per BN layer, a (C, 2) fp64 table of (sum x, sum x^2) on every rank; appending the rank's
element count gives a 2C+1 payload whose SUM all-reduce makes every rank normalise with the statistics of the concatenated
batch.  NCCL on the GPUs (one tiny all-reduce per layer over NVLink), gloo in the CPU tests; the payload layout is the
only contract between the kernel and the collective.  The reference itself keeps per-rank statistics
(``broadcast_buffers=False``, reference daod/engine/trainers/source_free_adaptive_teacher.py:69-73), which is the default.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.distributed as dist
from torch import Tensor


def allreduce_bn_stats(payload: Tensor, num_channels: int, group=None) -> float:
    """In-place SUM all-reduce of [sum_0, sumsq_0, ..., sum_{C-1}, sumsq_{C-1}, count]; returns the global count."""
    assert payload.dtype == torch.float64 and payload.numel() >= 2 * num_channels + 1
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(payload[: 2 * num_channels + 1], op=dist.ReduceOp.SUM, group=group)
    return float(payload[2 * num_channels].item())


def allreduce_bn_stats_device(payload: Tensor, num_channels: int, group=None) -> None:
    """The same all-reduce without leaving the device: the global count stays in ``payload[2C]`` and is read there by
    ``sfod_bn_finalize_apply`` -- no ``.item()``, so a multi-GPU AdaBN / teacher forward enqueues all
    of its BN layers without a single host synchronisation."""
    assert payload.dtype == torch.float64 and payload.numel() >= 2 * num_channels + 1
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(payload[: 2 * num_channels + 1], op=dist.ReduceOp.SUM, group=group)


def finalize_stats_host(payload: Tensor, num_channels: int, total: float) -> Tuple[Tensor, Tensor]:
    """Host-side restatement of phase 2's first step (mean, biased variance in fp64); used by the gloo tests."""
    st = payload[: 2 * num_channels].reshape(num_channels, 2)
    mean = st[:, 0] / total
    var = (st[:, 1] / total - mean * mean).clamp_(min=0)
    return mean, var
