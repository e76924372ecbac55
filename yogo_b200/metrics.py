"""Evaluation metrics on the GPU: the confusion matrix with background errors, per-class precision / recall and COCO
mAP / mAR, accumulated on the device from the batched matching (``format_preds_and_labels_batch``).

Counterpart of the reference's ``yogo test`` metrics (``Metrics.update`` -> ``format_preds_and_labels_v2`` ->
torchmetrics).  ROC and calibration error are not computed (DESIGN.md).  The kernels live in csrc/metrics.cu;
tools/coco_eval_np.py restates them in numpy."""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Sequence

import numpy as np
import torch

from . import _lib as L
from .utils.prediction_formatting import _lsap_status_check, _match_batch

IOU_THRESHOLDS = np.linspace(0.5, 0.95, 10)   # COCOeval.Params.iouThrs
RECALL_POINTS = np.linspace(0.0, 1.00, 101)   # COCOeval.Params.recThrs
MAX_DETS = (1, 10, 100)                       # COCOeval.Params.maxDets
_OBJECTNESS_THRESH = 0.5                      # the matching's threshold, as the reference's test path
_MAX_CLASSES = 27


def _doubles(a: np.ndarray):
    return (C.c_double * len(a))(*[float(x) for x in a])


def _mean(s: np.ndarray) -> float:
    s = s[s > -1]
    return float(np.mean(s)) if s.size else -1.0


class Metrics:
    """Accumulates evaluation metrics of a model's predictions over batches, on the device.

    ``update(preds, labels)`` takes a batch of predictions (B, 5+C, Sy, Sx) and labels (B, 6, Sy, Sx) on one CUDA device,
    matches them exactly like ``format_preds_and_labels_batch`` (objectness 0.5, NMS 0.5, xyxy,
    ``min_class_confidence_threshold``) and adds the batch to the state, which stays on that device.  ``update``
    synchronises with the host only where the matching does (twice per call).  A label class outside [0, C) raises
    ``ValueError`` naming the image, and the batch is not added.

    ``compute()`` returns CPU values (one device->host copy):

    - ``confusion``: int64 (C+1, C+1) with background (last row / column), else (C, C); rows are the true class,
      columns the predicted class - the matrix of ``PredictionLabelMatch.convert_background_errors(C + 1)`` rows;
    - ``precision`` / ``recall``: float64, one per row of the confusion matrix, 0 where the denominator is 0;
    - with ``include_mAP``: ``map``, ``map_50``, ``map_75``, ``mar_1``, ``mar_10``, ``mar_100`` (floats, -1 without any
      label), ``map_per_class`` and ``mar_100_per_class`` (float64 (C,), -1 for a class without labels), and COCOeval's
      ``coco_precision`` (T=10, R=101, C, 3 maxDets) and ``coco_recall`` (T, C, 3) arrays (area "all");
    - ``num_images``.

    COCO evaluation uses the objectness as the detection score and the argmax of the class columns as its class.
    """

    def __init__(self, classes: Sequence[str], min_class_confidence_threshold: float = 0.0, include_mAP: bool = True,
                 include_background: bool = True):
        self.classes = list(classes)
        self.num_classes = len(self.classes)
        if not 1 <= self.num_classes <= _MAX_CLASSES:
            raise ValueError(f"{self.num_classes} classes; between 1 and {_MAX_CLASSES} are supported")
        self.min_class_confidence_threshold = float(min_class_confidence_threshold)
        self.include_mAP = bool(include_mAP)
        self.include_background = bool(include_background)
        self._iou_thrs = _doubles(IOU_THRESHOLDS)
        self._rec_thrs = _doubles(RECALL_POINTS)
        self.reset()

    def reset(self) -> None:
        """Forget every update; the state moves to the device of the next one."""
        self._device = None
        self._confusion = None
        self._gt_count = None
        self._records, self._keys = [], []
        self._num_images = 0

    @property
    def _side(self) -> int:
        return self.num_classes + (1 if self.include_background else 0)

    def update(self, preds: torch.Tensor, labels: torch.Tensor) -> None:
        if preds.ndim != 4 or preds.shape[1] != 5 + self.num_classes:
            raise ValueError(f"expected predictions (B, {5 + self.num_classes}, Sy, Sx) for {self.num_classes} classes, "
                             f"got {tuple(preds.shape)}")
        if labels.device != preds.device:
            raise ValueError(f"predictions on {preds.device} and labels on {labels.device}: both must be on one device")
        if self._device is not None and preds.device != self._device:
            raise ValueError(f"the metric state is on {self._device}, this batch on {preds.device}")
        L.require_cuda(preds, "predictions")
        with torch.cuda.device(preds.device):
            self._update(preds, labels)

    def _update(self, preds: torch.Tensor, labels: torch.Tensor) -> None:
        r = _match_batch(preds, labels, _OBJECTNESS_THRESH, self.min_class_confidence_threshold)   # synchronisation 1
        B, D, Sy, Sx = preds.shape
        if B == 0:
            return
        lib, dev, st, C_ = L.lib(), r.rows.device, L.stream(), self.num_classes
        m = r.match
        desc, goff = r.table, r.table[4 * B:]
        confusion = torch.zeros(self._side * self._side, dtype=torch.int64, device=dev)
        label_status = torch.empty(B, dtype=torch.int32, device=dev)
        L.check(lib.yg_confusion_batch(m.preds.data_ptr(), m.labels.data_ptr(), m.missed_labels.data_ptr(),
                                       m.extra_predictions.data_ptr(), B, C_, int(self.include_background), desc.data_ptr(),
                                       goff.data_ptr(), r.status.data_ptr(), label_status.data_ptr(), confusion.data_ptr(), st))
        if self.include_mAP:
            n_rec = int(r.m_host.sum())
            records = torch.empty((max(n_rec, 1), 4), dtype=torch.int32, device=dev)
            keys = torch.empty(max(n_rec, 1), dtype=torch.int64, device=dev)
            gt_count = torch.zeros(C_, dtype=torch.int64, device=dev)
            L.check(lib.yg_coco_match_batch(r.rows.data_ptr(), r.label_rows.data_ptr(), B, Sy * Sx, C_, int(r.n_host.max()),
                                            int(r.m_host.max()), desc.data_ptr(), goff.data_ptr(), self._num_images,
                                            self._iou_thrs, records.data_ptr(), keys.data_ptr(), gt_count.data_ptr(), st))
        status = torch.cat([r.status, label_status]).cpu()   # synchronisation 2: the solver's and the label check's status
        _lsap_status_check(status[:B], "image")
        bad = np.flatnonzero(status[B:].numpy())
        if bad.size:
            raise ValueError(f"label class outside [0, {C_}) (image {int(bad[0])})")
        # the batch is valid: add it to the state
        if self._device is None:
            self._device = dev
            self._confusion = torch.zeros(self._side * self._side, dtype=torch.int64, device=dev)
            self._gt_count = torch.zeros(C_, dtype=torch.int64, device=dev)
        self._confusion += confusion
        if self.include_mAP:
            self._gt_count += gt_count
            self._records.append(records[:n_rec])
            self._keys.append(keys[:n_rec])
        self._num_images += B

    def compute(self) -> Dict[str, Any]:
        if self._device is None:
            raise RuntimeError("Metrics.compute() called before any update()")
        with torch.cuda.device(self._device):
            return self._compute()

    def _compute(self) -> Dict[str, Any]:
        C_, nb = self.num_classes, self._side
        T, R, M = len(IOU_THRESHOLDS), len(RECALL_POINTS), len(MAX_DETS)
        n_prec, n_rc = T * R * C_ * M, T * C_ * M
        out = torch.empty(nb * nb + (n_prec + n_rc if self.include_mAP else 0), dtype=torch.float64, device=self._device)
        out[: nb * nb].view(torch.int64).copy_(self._confusion)
        if self.include_mAP:
            if len(self._records) > 1:   # keep one buffer, so that the next compute() does not concatenate again
                self._records, self._keys = [torch.cat(self._records)], [torch.cat(self._keys)]
            records = self._records[0] if self._records else torch.empty((0, 4), dtype=torch.int32, device=self._device)
            keys = self._keys[0] if self._keys else torch.empty(0, dtype=torch.int64, device=self._device)
            sorted_keys, perm = torch.sort(keys, stable=True)
            prec = out[nb * nb: nb * nb + n_prec]
            L.check(L.lib().yg_coco_accumulate(records.data_ptr(), sorted_keys.data_ptr(), perm.data_ptr(), keys.numel(),
                                               self._gt_count.data_ptr(), C_, self._rec_thrs, prec.data_ptr(),
                                               out[nb * nb + n_prec:].data_ptr(), L.stream()))
        host = out.cpu().numpy()   # the one device -> host copy
        confusion = host[: nb * nb].view(np.int64).reshape(nb, nb).copy()
        diag, col, row = np.diag(confusion).astype(np.float64), confusion.sum(0), confusion.sum(1)
        res: Dict[str, Any] = {
            "confusion": torch.from_numpy(confusion),
            "precision": torch.from_numpy(np.where(col > 0, diag / np.maximum(col, 1), 0.0)),
            "recall": torch.from_numpy(np.where(row > 0, diag / np.maximum(row, 1), 0.0)),
            "num_images": self._num_images,
        }
        if self.include_mAP:
            precision = host[nb * nb: nb * nb + n_prec].reshape(T, R, C_, M).copy()
            recall = host[nb * nb + n_prec:].reshape(T, C_, M).copy()
            res.update({
                "map": _mean(precision[:, :, :, 2]),
                "map_50": _mean(precision[0, :, :, 2]),
                "map_75": _mean(precision[5, :, :, 2]),
                "mar_1": _mean(recall[:, :, 0]),
                "mar_10": _mean(recall[:, :, 1]),
                "mar_100": _mean(recall[:, :, 2]),
                "map_per_class": torch.from_numpy(np.array([_mean(precision[:, :, k, 2]) for k in range(C_)])),
                "mar_100_per_class": torch.from_numpy(np.array([_mean(recall[:, k, 2]) for k in range(C_)])),
                "coco_precision": torch.from_numpy(precision),
                "coco_recall": torch.from_numpy(recall),
            })
        return res
