"""Plain numpy restatement of the ROC curves and the calibration error of yogo_b200.metrics.Metrics (torchmetrics
MulticlassROC(thresholds=None) and MulticlassCalibrationError(norm="l1") over the rows of convert_background_errors).

The kernels of csrc/metrics.cu mirror this file, and the GPU tests compare them against it.  The contract (DESIGN.md 6.1):
1. rows: matched pairs, missed labels as one-hot background rows, extra predictions (target = the background class); every
   prediction row gains a 0 background column.  Without background the matched pairs alone over the C class columns;
2. scores: the class columns; when any class value of one update's rows lies outside [0, 1] (NaN included), every row of
   that update is softmaxed over all its columns;
3. ROC of class k (one-vs-rest): sklearn's / torchmetrics' _binary_clf_curve with the point (0, 0) and threshold 1.0
   prepended; fpr = fps / fps[-1] and tpr = tps / tps[-1] in float64 (all 0 without negatives / positives); the AUC is
   the trapezoidal area, summed exactly in integers, -1 without positives or negatives;
4. calibration: confidence = row maximum, prediction = its first maximum, bin = bucketize(confidence, linspace(0, 1,
   n_bins + 1) in fp32, right=True) - 1, so a confidence of exactly 1.0 lands in the extra bin n_bins;
   ECE = sum over bins of |accuracy - confidence| * count / total."""
import numpy as np


def score_rows_np(preds, labels, missed, extra, num_classes, with_background=True):
    """One group of matched (preds, labels), missed-label and extra-prediction rows -> (scores float32 (R, nb), targets
    int64 (R,)) before the format rule, in matched / missed / extra order."""
    C = num_classes
    p = np.asarray(preds, np.float32).reshape(-1, 5 + C)
    t = np.asarray(labels, np.float32).reshape(-1, 6)[:, 5].astype(np.int64)
    if not with_background:
        return p[:, 5:].copy(), t
    ms = np.asarray(missed, np.float32).reshape(-1, 6)
    ex = np.asarray(extra, np.float32).reshape(-1, 5 + C)
    onehot = np.zeros((len(ms), C + 1), np.float32)
    onehot[:, C] = 1
    scores = np.concatenate([np.pad(p[:, 5:], ((0, 0), (0, 1))), onehot, np.pad(ex[:, 5:], ((0, 0), (0, 1)))])
    targets = np.concatenate([t, ms[:, 5].astype(np.int64), np.full(len(ex), C, np.int64)])
    return scores, targets


def apply_format_rule(scores):
    """Rule 2 for the rows of one update -> (scores, softmaxed): the softmax is computed in float64, rounded to fp32."""
    s = np.asarray(scores, np.float32)
    with np.errstate(invalid="ignore"):
        inside = bool(np.all((s >= 0) & (s <= 1)))
    if inside:
        return s, False
    x = s.astype(np.float64)
    e = np.exp(x - x.max(axis=1, keepdims=True))
    return (e / e.sum(axis=1, keepdims=True)).astype(np.float32), True


def roc_np(scores, positive):
    """One-vs-rest ROC of fp32 scores with boolean positives -> (fpr float64, tpr float64, thresholds float32, auc)."""
    s = np.asarray(scores, np.float32).reshape(-1) + np.float32(0)   # -0 -> +0: equal scores form one group
    y = np.asarray(positive, bool).reshape(-1)
    order = np.argsort(-s, kind="mergesort")
    s, y = s[order], y[order]
    last = np.r_[np.flatnonzero(np.diff(s)), s.size - 1] if s.size else np.zeros(0, np.int64)
    tps = np.r_[0, np.cumsum(y, dtype=np.int64)[last]]
    fps = np.r_[0, last + 1 - tps[1:]]
    thresholds = np.r_[np.float32(1), s[last]].astype(np.float32)
    P, F = int(tps[-1]), int(fps[-1])
    fpr = fps / F if F > 0 else np.zeros(fps.size)
    tpr = tps / P if P > 0 else np.zeros(tps.size)
    area = int(np.sum(np.diff(fps) * (tps[1:] + tps[:-1])))   # twice the area in units of 1 / (F * P)
    auc = float(area) / (2.0 * F * P) if P > 0 and F > 0 else -1.0
    return fpr.astype(np.float64), tpr.astype(np.float64), thresholds, auc


def roc_all_np(scores, targets):
    """Per class k of the score columns: roc_np(scores[:, k], targets == k) -> (list of curves, aucs float64)."""
    s = np.asarray(scores, np.float32)
    t = np.asarray(targets)
    curves = [roc_np(s[:, k], t == k) for k in range(s.shape[1])]
    return [c[:3] for c in curves], np.array([c[3] for c in curves], np.float64)


def calibration_bins_np(scores, targets, bounds):
    """Rule 4 with bounds = torch.linspace(0, 1, n_bins + 1).numpy() -> per bin (n_bins + 1 of them): row count (int64),
    correct count (int64), confidence sum (float64)."""
    s = np.asarray(scores, np.float32)
    t = np.asarray(targets)
    nbin = len(bounds)
    if s.shape[0] == 0:
        return np.zeros(nbin, np.int64), np.zeros(nbin, np.int64), np.zeros(nbin)
    conf = s.max(axis=1)
    correct = np.argmax(s, axis=1) == t
    b = np.searchsorted(np.asarray(bounds, np.float32), conf, side="right") - 1
    count = np.bincount(b, minlength=nbin).astype(np.int64)
    return count, np.bincount(b, weights=correct, minlength=nbin).astype(np.int64), np.bincount(b, weights=conf.astype(np.float64),
                                                                                                minlength=nbin)


def calibration_error_np(count, correct, conf_sum):
    """-> (L1 expected calibration error, mean confidence per bin, accuracy per bin); empty bins are 0, -1 without rows."""
    count = np.asarray(count, np.int64)
    den = np.maximum(count, 1)
    conf = np.where(count > 0, np.asarray(conf_sum, np.float64) / den, 0.0)
    acc = np.where(count > 0, np.asarray(correct, np.int64) / den, 0.0)
    total = int(count.sum())
    return (float(np.sum(np.abs(acc - conf) * (count / total))) if total else -1.0), conf, acc
