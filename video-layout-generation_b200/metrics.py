"""Accuracy of predicted layouts: per-class IoU, mIoU and pixel accuracy from confusion matrices counted on the device.

The reference's `Trainer.validate` (src/trainer.py:289-379) and `generate_sequence` (:453-476) only dump
`torch.argmax(seg, 1)`; `LayoutIoU` scores those predictions against the ground-truth labels, per rollout step for the
autoregressive case:

    iou = vlg_b200.LayoutIoU(n_classes=20, steps=8)
    imgs, labels = vlg_b200.rollout(img, label, flow_fn, steps=8)
    for t, lab in enumerate(labels):
        iou.update(lab, gt[t], step=t)          # one kernel launch, no synchronisation
    iou.sync()                                  # data-parallel: one all-reduce of the counts
    res = iou.compute()                         # res.miou[t]: mIoU of rollout step t
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch

from . import parallel
from ._cabi import VlgError
from .ops import _confusion_into


class IoUResult(NamedTuple):
    iou: torch.Tensor         # [steps, K] float64; NaN where a class is absent from both target and prediction
    miou: torch.Tensor        # [steps] float64: mean over the classes that are not NaN
    pixel_acc: torch.Tensor   # [steps] float64: correctly predicted pixels / counted pixels
    confusion: torch.Tensor   # [steps, K, K] int64: rows = target class, columns = predicted class


class LayoutIoU:
    """Accumulates `steps` confusion matrices of K classes in int64 `counts` [steps, K*K + 1] (the last column counts
    pixels skipped for a label outside [0, K)).  `update` adds on the device and, after its first call, neither
    allocates nor synchronises, so it can run inside `CapturedStep`.  `compute`, `sync` and `reset` also work on counts
    held on the CPU."""

    def __init__(self, n_classes: int = 20, steps: int = 1, ignore_index: int = -100):
        if steps < 1:
            raise VlgError("steps must be >= 1")
        self.n_classes, self.steps, self.ignore_index = n_classes, steps, ignore_index
        self.counts = torch.zeros(steps, n_classes * n_classes + 1, dtype=torch.int64)

    def update(self, pred: torch.Tensor, target: torch.Tensor, step: int = 0):
        """Adds the confusion counts of `pred` (int64 [N,H,W] class ids or [N,K,H,W] fp32 / bf16 scores) against
        `target` (int64 [N,H,W]) to row `step`.  The first call moves the counts to the device of `target`."""
        if not 0 <= step < self.steps:
            raise VlgError(f"step {step} outside [0, {self.steps})")
        if self.counts.device != target.device:
            self.counts = self.counts.to(target.device)
        _confusion_into(self.counts[step], pred, target, self.n_classes, ignore_index=self.ignore_index)

    def sync(self, group=None):
        """Sums the counts over the ranks of `group` in place (one all-reduce); nothing without a process group."""
        reduced = parallel.sync_counts(self.counts, group)
        if reduced is not self.counts:
            self.counts.copy_(reduced)

    def reset(self):
        """Zeroes the counts in place (a captured `update` keeps writing the same storage)."""
        self.counts.zero_()

    def compute(self) -> IoUResult:
        """Reads the counts to the host (synchronises) and derives IoU, mIoU and pixel accuracy per step.  Raises
        `VlgError` if any pixel was skipped for a target or predicted label outside [0, K)."""
        K = self.n_classes
        c = self.counts.cpu()
        skipped = c[:, K * K]
        if bool((skipped != 0).any()):
            raise VlgError(f"pixels with a target or predicted label outside [0, {K}) (and not ignore_index), per step: "
                           f"{skipped.tolist()}")
        conf = c[:, :K * K].reshape(self.steps, K, K)
        cf = conf.double()
        tp = torch.diagonal(cf, dim1=1, dim2=2)
        union = cf.sum(2) + cf.sum(1) - tp
        iou = torch.where(union > 0, tp / union.clamp_min(1), torch.full_like(tp, float("nan")))
        total = cf.sum((1, 2))
        pixel_acc = torch.where(total > 0, tp.sum(1) / total.clamp_min(1), torch.full_like(total, float("nan")))
        return IoUResult(iou=iou, miou=torch.nanmean(iou, 1), pixel_acc=pixel_acc, confusion=conf)
