"""Plain numpy restatement of the metrics of yogo_b200.metrics.Metrics: the confusion matrix with per-class precision and
recall, and COCO's bbox evaluation (pycocotools COCOeval.evaluateImg / accumulate / _summarize with no crowd
annotations, area range "all" and maxDets (1, 10, 100)).

The kernels of csrc/metrics.cu mirror this file, and the GPU tests compare them against it.  The contract choices (see
DESIGN.md): the detection score is the objectness, the IoU is torchvision's box_iou in fp32 (compared as the fp32 value
promoted to double), detections are ranked per (image, class) by score with ties in row (NMS) order."""
import numpy as np

IOU_THRS = np.linspace(0.5, 0.95, 10)   # COCOeval: np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1)
REC_THRS = np.linspace(0.0, 1.00, 101)  # COCOeval: np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1)
MAX_DETS = (1, 10, 100)


# ----------------------------------------------------------------------------------------------------- confusion
def confusion_matrix_np(true, pred, n):
    """M[true, pred] += 1 for each pair: rows are the true class, columns the predicted class."""
    m = np.zeros((n, n), np.int64)
    np.add.at(m, (np.asarray(true, np.int64), np.asarray(pred, np.int64)), 1)
    return m


def confusion_from_converted(bg_preds, bg_labels, n):
    """The confusion matrix of PredictionLabelMatch.convert_background_errors rows: (int(label[5]), argmax(pred[5:]))."""
    true = np.asarray(bg_labels)[:, 5].astype(np.int64)
    pred = np.argmax(np.asarray(bg_preds)[:, 5:], axis=1)
    return confusion_matrix_np(true, pred, n)


def precision_recall_np(m):
    """Per-class precision M[k,k] / sum_i M[i,k] and recall M[k,k] / sum_j M[k,j]; 0 where the denominator is 0."""
    m = np.asarray(m, np.int64)
    diag, col, row = np.diag(m).astype(np.float64), m.sum(0), m.sum(1)
    return (np.where(col > 0, diag / np.maximum(col, 1), 0.0), np.where(row > 0, diag / np.maximum(row, 1), 0.0))


# ----------------------------------------------------------------------------------------------------- COCO
def box_iou_np(gt, dt):
    """(G, D) fp32 torchvision.ops.box_iou(gt, dt), operation by operation."""
    a = np.asarray(gt, np.float32).reshape(-1, 4)
    b = np.asarray(dt, np.float32).reshape(-1, 4)
    area1 = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1])
    area2 = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    lt = np.maximum(a[:, None, :2], b[None, :, :2])
    rb = np.minimum(a[:, None, 2:], b[None, :, 2:])
    wh = rb - lt
    wh = np.where(wh < 0, np.float32(0), wh)
    inter = wh[:, :, 0] * wh[:, :, 1]
    union = (area1[:, None] + area2[None, :]) - inter
    with np.errstate(divide="ignore", invalid="ignore"):
        return (inter / union).astype(np.float32)


def image_inputs(pred_rows, label_rows):
    """One image's kept xyxy prediction rows (n, 5+C) and label rows (g, 6) = [mask, x1, y1, x2, y2, class] in grid order
    -> (dt_boxes, dt_scores, dt_cls, gt_boxes, gt_cls): score = objectness, class = argmax of the class columns."""
    p = np.asarray(pred_rows, np.float32)
    g = np.asarray(label_rows, np.float32)
    return p[:, :4], p[:, 4], np.argmax(p[:, 5:], axis=1), g[:, 1:5], g[:, 5].astype(np.int64)


def evaluate_image(dt_boxes, dt_scores, dt_cls, gt_boxes, gt_cls, num_classes):
    """COCOeval.evaluateImg of one image for every class -> ({k: (scores (n,), matched (T, n) bool)} for the classes with
    detections, ground-truth count per class).  Detections are sorted by score (stable) and cut to 100; ground truths of
    the class are visited in order, and a detection takes the unmatched one of the highest IoU >= min(t, 1 - 1e-10), the
    later of equal IoUs."""
    dt_scores = np.asarray(dt_scores, np.float32)
    dt_cls, gt_cls = np.asarray(dt_cls), np.asarray(gt_cls)
    ious_all = box_iou_np(gt_boxes, dt_boxes)
    best0 = np.minimum(IOU_THRS, 1 - 1e-10)
    out = {}
    for k in np.unique(dt_cls):
        d = np.flatnonzero(dt_cls == k)
        d = d[np.argsort(-dt_scores[d], kind="mergesort")[: MAX_DETS[-1]]]
        g = np.flatnonzero(gt_cls == k)
        ious = ious_all[np.ix_(g, d)].astype(np.float64)
        gtm = np.zeros((len(IOU_THRS), g.size), bool)
        dtm = np.zeros((len(IOU_THRS), d.size), bool)
        if g.size:
            for i in range(d.size):
                ok = ~gtm & ~(ious[None, :, i] < best0[:, None])
                cand = np.where(ok, ious[None, :, i], -np.inf)
                j = g.size - 1 - np.argmax(cand[:, ::-1], axis=1)   # last of the highest
                hit = ok.any(1)
                gtm[hit, j[hit]] = True
                dtm[hit, i] = True
        out[int(k)] = (dt_scores[d], dtm)
    return out, np.bincount(gt_cls[(gt_cls >= 0) & (gt_cls < num_classes)], minlength=num_classes).astype(np.int64)


def accumulate(per_image, gt_counts, num_classes):
    """COCOeval.accumulate over the images in order -> precision (T, R, K, 3) and recall (T, K, 3), -1 for a class with
    no ground truth."""
    T, R = len(IOU_THRS), len(REC_THRS)
    precision = -np.ones((T, R, num_classes, len(MAX_DETS)))
    recall = -np.ones((T, num_classes, len(MAX_DETS)))
    for k in range(num_classes):
        npig = int(gt_counts[k])
        if npig == 0:
            continue
        entries = [e[k] for e in per_image if k in e]
        for mi, m in enumerate(MAX_DETS):
            scores = np.concatenate([s[:m] for s, _ in entries]) if entries else np.zeros(0, np.float32)
            dtm = np.concatenate([x[:, :m] for _, x in entries], 1) if entries else np.zeros((T, 0), bool)
            order = np.argsort(-scores, kind="mergesort")
            dtm = dtm[:, order]
            tp_sum = np.cumsum(dtm, axis=1).astype(dtype=float)
            fp_sum = np.cumsum(~dtm, axis=1).astype(dtype=float)
            for t in range(T):
                tp, fp = tp_sum[t], fp_sum[t]
                nd = len(tp)
                rc = tp / npig
                pr = tp / (fp + tp + np.spacing(1))
                recall[t, k, mi] = rc[-1] if nd else 0
                pr = np.maximum.accumulate(pr[::-1])[::-1] if nd else pr
                q = np.zeros(R)
                inds = np.searchsorted(rc, REC_THRS, side="left")
                valid = inds < nd
                q[valid] = pr[inds[valid]]
                precision[t, :, k, mi] = q
    return precision, recall


def _mean(s):
    s = s[s > -1]
    return float(np.mean(s)) if s.size else -1.0


def summarize(precision, recall):
    """COCOeval._summarize (area "all"): means over the entries > -1."""
    K = precision.shape[2]
    return {
        "map": _mean(precision[:, :, :, 2]),
        "map_50": _mean(precision[0, :, :, 2]),
        "map_75": _mean(precision[5, :, :, 2]),
        "mar_1": _mean(recall[:, :, 0]),
        "mar_10": _mean(recall[:, :, 1]),
        "mar_100": _mean(recall[:, :, 2]),
        "map_per_class": np.array([_mean(precision[:, :, k, 2]) for k in range(K)]),
        "mar_100_per_class": np.array([_mean(recall[:, k, 2]) for k in range(K)]),
    }


def coco_eval_np(images, num_classes):
    """images: per image (dt_boxes, dt_scores, dt_cls, gt_boxes, gt_cls) -> (precision, recall, summary dict)."""
    per_image, gt = [], np.zeros(num_classes, np.int64)
    for im in images:
        e, n = evaluate_image(*im, num_classes)
        per_image.append(e)
        gt += n
    precision, recall = accumulate(per_image, gt, num_classes)
    return precision, recall, summarize(precision, recall)
