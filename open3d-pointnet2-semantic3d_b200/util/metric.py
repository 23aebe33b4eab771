"""The reference's ConfusionMatrix (util/metric.py:7-124) with the matrix resident on the device.

  ConfusionMatrix(num_classes)
      .increment(gt_label, pd_label)                         metric.py:18-23
      .increment_from_list(gt_labels, pd_labels)             metric.py:25-30  (pn2_confusion_from_labels)
      .increment_from_logits(logits, labels, pred_out=None)  new: replaces the host copy + np.argmax + double loop
                                                             of train.py:246-251 / 307-312 (pn2_confusion_from_logits)
      .get_per_class_ious / get_mean_iou / get_accuracy / print_metrics   metric.py:32-124

The counting runs on the caller's current CUDA stream and never synchronises the host, so it can sit inside a
captured CUDA graph.  Reading the matrix (``confusion_matrix`` and the getters) copies it to the host and is the
only synchronising step.  The arithmetic of the getters is the reference's, operation for operation, on a host
``np.int64`` matrix: the module-level functions below take such a matrix, so results are equal, not merely close.
"""
from pprint import pprint

import numpy as np
import torch

from .._ffi import F32, I32, call, ptr


def get_per_class_ious(confusion_matrix):
    """IoU of classes 1..C-1 (metric.py:32-65): the gt == 0 row and the pd == 0 column are ignored, a union of
    0 counts as 1, and a non-zero column 0 prints a warning."""
    if any(confusion_matrix[:, 0] != 0):
        print("[Warn] Contains prediction of label 0:", confusion_matrix[:, 0])
    valid_confusion_matrix = confusion_matrix[1:, 1:]
    ious = []
    for c in range(len(valid_confusion_matrix)):
        intersection = valid_confusion_matrix[c, c]
        union = (np.sum(valid_confusion_matrix[c, :]) + np.sum(valid_confusion_matrix[:, c]) - intersection)
        if union == 0:
            union = 1
        ious.append(float(intersection) / union)
    return ious


def get_mean_iou(confusion_matrix):
    """metric.py:67-74."""
    per_class_ious = get_per_class_ious(confusion_matrix)
    return np.sum(per_class_ious) / len(per_class_ious)


def get_accuracy(confusion_matrix):
    """trace / sum of the [1:, 1:] block (metric.py:76-83); nan for an empty matrix."""
    valid_confusion_matrix = confusion_matrix[1:, 1:]
    return np.trace(valid_confusion_matrix) / np.sum(valid_confusion_matrix)


def print_metrics(confusion_matrix, labels=None):
    """The reference's printed report (metric.py:85-124), same layout."""
    num_classes = len(confusion_matrix)
    print("Confusion matrix:")
    if labels is None:
        labels = [str(val) for val in range(num_classes)]
    elif len(labels) != num_classes:
        raise ValueError("len(labels) != self.num_classes")
    column_width = max([len(x) for x in labels] + [7])
    empty_cell = " " * column_width
    print("    " + empty_cell, end=" ")
    for label in labels:
        print("%{0}s".format(column_width) % label, end=" ")
    print()
    for i, label in enumerate(labels):
        print("    %{0}s".format(column_width) % label, end=" ")
        for j in range(len(labels)):
            cell = "%{0}.0f".format(column_width) % confusion_matrix[i, j]
            print(cell, end=" ")
        print()
    print("IoU per class:")
    pprint(get_per_class_ious(confusion_matrix))
    print("mIoU (ignoring label 0):")
    print(get_mean_iou(confusion_matrix))
    print("Overall accuracy")
    print(get_accuracy(confusion_matrix))


def _labels_on(x, num_classes, device):
    """Labels as an int32 contiguous CUDA tensor, from a numpy array or a tensor (a tensor stays on the device).
    Wider integers are clamped to [-1, num_classes] first, so that no out-of-range label wraps into range."""
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(np.ascontiguousarray(np.asarray(x)))
    x = x.reshape(-1)
    if x.dtype != I32:
        x = x.to(device=device, non_blocking=True)
        if x.dtype.is_floating_point:
            raise ValueError("labels must be integers, got %s" % x.dtype)
        x = x.clamp(-1, num_classes).to(I32)
    return x.to(device).contiguous()


class ConfusionMatrix:
    """``num_classes`` x ``num_classes`` counts, row = ground truth, column = prediction, on a CUDA device.
    There is no CPU fallback: ``device`` must be a CUDA device."""

    MAX_CLASSES = 128  # pn2_confusion_* keep one block's histogram in shared memory

    def __init__(self, num_classes, device="cuda"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("ConfusionMatrix counts on a CUDA device (no CPU fallback); got %s" % device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.num_classes = int(num_classes)
        if not 1 <= self.num_classes <= self.MAX_CLASSES:
            raise ValueError("num_classes must be in [1, %d]" % self.MAX_CLASSES)
        self.valid_labels = set(range(self.num_classes))
        # [0:C*C] the matrix, [C*C] the dropped rows / pairs: one buffer, so reset() is one memset
        # (the kernels add into it as uint64: the same bits below 2^63)
        self._counts = torch.zeros(self.num_classes * self.num_classes + 1, dtype=torch.int64, device=self.device)

    # ---- device views --------------------------------------------------------------------------------
    @property
    def counts(self):
        """The (C, C) int64 device accumulator (a caller may all_reduce it across data-parallel ranks)."""
        c = self.num_classes
        return self._counts[:c * c].view(c, c)

    def _cm_ptr(self):
        return ptr(self._counts, torch.int64)

    def _skip_ptr(self):
        import ctypes
        return ctypes.c_void_p(self._counts.data_ptr() + 8 * self.num_classes * self.num_classes)

    # ---- counting (no host synchronisation) -------------------------------------------------------------
    def increment(self, gt_label, pd_label):
        if gt_label not in self.valid_labels:
            raise ValueError("Invalid value for gt_label")
        if pd_label not in self.valid_labels:
            raise ValueError("Invalid value for pd_label")
        self.increment_from_list(np.array([gt_label]), np.array([pd_label]))

    def increment_from_list(self, gt_labels, pd_labels):
        """Count (gt, pd) pairs; a pair with a label outside [0, num_classes) is dropped (sklearn's
        confusion_matrix(labels=range(C)), which the reference calls) and counted in ``skipped``."""
        gt = _labels_on(gt_labels, self.num_classes, self.device)
        pd = _labels_on(pd_labels, self.num_classes, self.device)
        if gt.numel() != pd.numel():
            raise ValueError("gt_labels and pd_labels differ in length: %d vs %d" % (gt.numel(), pd.numel()))
        call("pn2_confusion_from_labels", gt.numel(), self.num_classes, ptr(gt, I32), ptr(pd, I32),
             self._cm_ptr(), self._skip_ptr())

    def increment_from_logits(self, logits, labels, pred_out=None):
        """logits (..., C) float32 CUDA, labels (...) int32 CUDA: count (label, arg-max of the row) with numpy's
        arg-max rule (first maximum; the first NaN wins).  ``pred_out`` (...) int32 CUDA receives the arg-max."""
        if logits.shape[-1] != self.num_classes:
            raise ValueError("logits have %d classes, the matrix %d" % (logits.shape[-1], self.num_classes))
        rows = logits.numel() // self.num_classes
        if labels.numel() != rows or (pred_out is not None and pred_out.numel() != rows):
            raise ValueError("labels / pred_out must hold one entry per row of logits (%d)" % rows)
        call("pn2_confusion_from_logits", rows, self.num_classes, ptr(logits, F32), ptr(labels, I32),
             self._cm_ptr(), self._skip_ptr(), ptr(pred_out, I32, allow_none=True))

    def reset(self):
        """Zero the counts in place (the buffer a captured graph holds stays valid)."""
        self._counts.zero_()

    # ---- host side (synchronises) -----------------------------------------------------------------------
    @property
    def confusion_matrix(self):
        return self.counts.cpu().numpy()

    @property
    def skipped(self):
        """Rows / pairs dropped because their label lies outside [0, num_classes)."""
        return int(self._counts[-1].item())

    def get_per_class_ious(self):
        return get_per_class_ious(self.confusion_matrix)

    def get_mean_iou(self):
        return get_mean_iou(self.confusion_matrix)

    def get_accuracy(self):
        return get_accuracy(self.confusion_matrix)

    def print_metrics(self, labels=None):
        if labels is not None and len(labels) != self.num_classes:
            raise ValueError("len(labels) != self.num_classes")
        print_metrics(self.confusion_matrix, labels)
