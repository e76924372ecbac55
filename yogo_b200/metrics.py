"""Evaluation metrics on the GPU: the confusion matrix with background errors, per-class precision / recall and COCO
mAP / mAR, accumulated on the device from the batched matching (``format_preds_and_labels_batch``).

Counterpart of the reference's ``yogo test`` metrics (``Metrics.update`` -> ``format_preds_and_labels_v2`` ->
torchmetrics), with per-class ROC curves and the calibration error on request.  The kernels live in csrc/metrics.cu;
tools/coco_eval_np.py and tools/roc_ece_np.py restate them in numpy (contract: DESIGN.md 6.1)."""
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
_MAX_BINS = 255                               # csrc/metrics.cu MET_MAX_BINS


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
    - ``num_images``;
    - with ``include_roc`` (torchmetrics ``MulticlassROC(thresholds=None)``): ``roc``, one ``(fpr float64, tpr float64,
      thresholds float32)`` tuple per row of the confusion matrix (one-vs-rest, the point (0, 0) with threshold 1.0 first),
      and ``roc_auc`` (float64, the trapezoidal area; -1 for a class without positive or without negative rows);
    - with ``include_calibration`` (torchmetrics ``MulticlassCalibrationError(n_bins=calibration_bins, norm="l1")``):
      ``calibration_error`` (float, -1 without any row), ``calibration_bin_count`` (int64 (calibration_bins + 1,): a
      confidence of exactly 1.0 lands in the last bin), ``calibration_bin_confidence`` and ``calibration_bin_accuracy``
      (float64 means per bin, 0 for an empty bin) - what a reliability diagram needs.

    COCO evaluation uses the objectness as the detection score and the argmax of the class columns as its class.  ROC and
    calibration use the rows of ``convert_background_errors`` (without background the matched pairs) and their class
    columns as scores, softmaxed over the row in an update where any class value lies outside [0, 1]; a NaN score raises
    ``ValueError`` naming the image, and the batch is not added.  With both flags off, ``update`` and ``compute`` do
    exactly the work they do without them.
    """

    def __init__(self, classes: Sequence[str], min_class_confidence_threshold: float = 0.0, include_mAP: bool = True,
                 include_background: bool = True, include_roc: bool = False, include_calibration: bool = False,
                 calibration_bins: int = 15):
        self.classes = list(classes)
        self.num_classes = len(self.classes)
        if not 1 <= self.num_classes <= _MAX_CLASSES:
            raise ValueError(f"{self.num_classes} classes; between 1 and {_MAX_CLASSES} are supported")
        self.min_class_confidence_threshold = float(min_class_confidence_threshold)
        self.include_mAP = bool(include_mAP)
        self.include_background = bool(include_background)
        self.include_roc = bool(include_roc)
        self.include_calibration = bool(include_calibration)
        self.calibration_bins = int(calibration_bins)
        if not 1 <= self.calibration_bins <= _MAX_BINS:
            raise ValueError(f"calibration_bins = {calibration_bins}; between 1 and {_MAX_BINS} are supported")
        # torch.linspace's fp32 boundaries, computed on the host so that the kernel bins against the same bits
        bounds = torch.linspace(0, 1, self.calibration_bins + 1, dtype=torch.float32).numpy()
        self._bin_bounds = (C.c_float * len(bounds))(*[float(x) for x in bounds])
        self._iou_thrs = _doubles(IOU_THRESHOLDS)
        self._rec_thrs = _doubles(RECALL_POINTS)
        self.reset()

    def reset(self) -> None:
        """Forget every update; the state moves to the device of the next one."""
        self._device = None
        self._confusion = None
        self._gt_count = None
        self._records, self._keys = [], []
        self._scores, self._targets = [], []
        self._bins = None   # int64 (2, bins + 1) row counts and correct counts, float64 (bins + 1,) confidence sums
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
        checks = [r.status, label_status]
        if self.include_roc or self.include_calibration:
            scores, targets, bins, nan_status = self._score_rows(r, B)
            checks.append(nan_status)
        status = torch.cat(checks).cpu()   # synchronisation 2: the solver's, the label check's and the NaN check's status
        _lsap_status_check(status[:B], "image")
        bad = np.flatnonzero(status[B:2 * B].numpy())
        if bad.size:
            raise ValueError(f"label class outside [0, {C_}) (image {int(bad[0])})")
        bad = np.flatnonzero(status[2 * B:].numpy())
        if bad.size:
            raise ValueError(f"NaN class score (image {int(bad[0])})")
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
        if self.include_roc:
            self._scores.append(scores)
            self._targets.append(targets)
        if self.include_calibration:
            if self._bins is None:
                self._bins = [torch.zeros_like(b) for b in bins]
            for acc, b in zip(self._bins, bins):
                acc += b
        self._num_images += B

    def _score_rows(self, r, B: int):
        """Launch yg_score_rows_batch for one update: the score rows and targets (with ``include_roc``), the per-bin sums
        of the update and the per-image NaN status, all on the device and not yet added to the state."""
        m, dev, C_ = r.match, r.rows.device, self.num_classes
        n_matched, n_missed, n_extra = m.preds.shape[0], m.missed_labels.shape[0], m.extra_predictions.shape[0]
        n_rows = n_matched + n_missed + n_extra if self.include_background else n_matched
        nbin = self.calibration_bins + 1
        scores = targets = None
        if self.include_roc:
            scores = torch.empty((n_rows, self._side), dtype=torch.float32, device=dev)
            targets = torch.empty(n_rows, dtype=torch.int32, device=dev)
        counts = torch.empty((2, nbin), dtype=torch.int64, device=dev)
        conf = torch.empty(nbin, dtype=torch.float64, device=dev)
        flag = torch.empty(1, dtype=torch.int32, device=dev)
        nan_status = torch.empty(B, dtype=torch.int32, device=dev)
        partials = torch.empty(B * nbin * 16, dtype=torch.uint8, device=dev)
        L.check(L.lib().yg_score_rows_batch(
            m.preds.data_ptr(), m.labels.data_ptr(), m.missed_labels.data_ptr(), m.extra_predictions.data_ptr(), n_matched,
            n_extra, B, C_, int(self.include_background), r.table.data_ptr(), r.table[4 * B:].data_ptr(), r.status.data_ptr(),
            self._bin_bounds, self.calibration_bins, flag.data_ptr(), L.ptr(scores) if n_rows else None,
            L.ptr(targets) if n_rows else None, nan_status.data_ptr(), partials.data_ptr(), counts[0].data_ptr(),
            counts[1].data_ptr(), conf.data_ptr(), L.stream()))
        return scores, targets, (counts, conf), nan_status

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
        if self.include_roc:
            pieces, roc_lengths = self._roc_device()
            out = torch.cat([out] + pieces)
        if self.include_calibration:
            counts, conf = self._bins
            out = torch.cat([out, counts.reshape(-1).view(torch.float64), conf])
        host = out.cpu().numpy()   # the one device -> host copy (with ROC the second read)
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
            recall = host[nb * nb + n_prec: nb * nb + n_prec + n_rc].reshape(T, C_, M).copy()
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
        o = nb * nb + (n_prec + n_rc if self.include_mAP else 0)
        if self.include_roc:
            res["roc_auc"] = torch.from_numpy(host[o:o + nb].copy())
            o += nb
            res["roc"] = []
            for n in roc_lengths:
                fpr, tpr, thr = host[o:o + n], host[o + n:o + 2 * n], host[o + 2 * n:o + 3 * n].astype(np.float32)
                res["roc"].append((torch.from_numpy(fpr.copy()), torch.from_numpy(tpr.copy()), torch.from_numpy(thr)))
                o += 3 * n
        if self.include_calibration:
            nbin = self.calibration_bins + 1
            counts = host[o:o + 2 * nbin].view(np.int64).reshape(2, nbin)
            conf_sum = host[o + 2 * nbin:o + 3 * nbin]
            count, correct = counts[0].copy(), counts[1]
            den = np.maximum(count, 1)
            bin_conf = np.where(count > 0, conf_sum / den, 0.0)
            bin_acc = np.where(count > 0, correct / den, 0.0)
            total = int(count.sum())
            res.update({
                "calibration_error": float(np.sum(np.abs(bin_acc - bin_conf) * (count / total))) if total else -1.0,
                "calibration_bin_count": torch.from_numpy(count),
                "calibration_bin_confidence": torch.from_numpy(bin_conf),
                "calibration_bin_accuracy": torch.from_numpy(bin_acc),
            })
        return res

    def _roc_device(self):
        """Sort the class-major keys of every stored score and walk each class's segment (yg_roc_curves); reads the curve
        lengths (one device -> host read) and returns the float64 pieces [auc, then per class fpr, tpr, thresholds] to pack
        into the copy of compute(), and the lengths."""
        if len(self._scores) > 1:   # keep one buffer, so that the next compute() does not concatenate again
            self._scores, self._targets = [torch.cat(self._scores)], [torch.cat(self._targets)]
        nb, dev, lib = self._side, self._device, L.lib()
        scores = self._scores[0] if self._scores else torch.empty((0, nb), dtype=torch.float32, device=dev)
        targets = self._targets[0] if self._targets else torch.empty(0, dtype=torch.int32, device=dev)
        R = scores.shape[0]
        keys = torch.empty(nb * R, dtype=torch.int64, device=dev)
        L.check(lib.yg_roc_keys(scores.data_ptr(), R, nb, keys.data_ptr(), L.stream()))
        sorted_keys, perm = torch.sort(keys)
        fpr = torch.empty((nb, R + 1), dtype=torch.float64, device=dev)
        tpr = torch.empty((nb, R + 1), dtype=torch.float64, device=dev)
        thr = torch.empty((nb, R + 1), dtype=torch.float32, device=dev)
        lengths = torch.empty(nb, dtype=torch.int64, device=dev)
        auc = torch.empty(nb, dtype=torch.float64, device=dev)
        L.check(lib.yg_roc_curves(sorted_keys.data_ptr(), perm.data_ptr(), targets.data_ptr(), R, nb, fpr.data_ptr(),
                                  tpr.data_ptr(), thr.data_ptr(), lengths.data_ptr(), auc.data_ptr(), L.stream()))
        roc_lengths = lengths.cpu().tolist()   # the first device -> host read: sizes of the packed curves
        pieces = [auc]
        for k, n in enumerate(roc_lengths):
            pieces += [fpr[k, :n], tpr[k, :n], thr[k, :n].double()]
        return pieces, roc_lengths
