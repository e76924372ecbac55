"""``format_preds`` - same interface as /root/reference/yogo/utils/prediction_formatting.py:23-93,
plus ``format_preds_batch`` which post-processes a whole batch in one kernel launch
(csrc/nms.cu) instead of one Python iteration + 8 ATen/torchvision calls per image.
Its consumers follow: ``format_preds_and_labels_v2`` / ``PredictionLabelMatch`` (evaluation matching,
prediction_formatting.py:166-330) and ``format_to_numpy`` (:96-156)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Literal, Optional, Sequence, Tuple, get_args

import numpy as np
import torch

from .. import _lib as L

BoxFormat = Literal["xyxy", "cxcywh"]


@L.on_device(lambda preds, *a, **k: preds)
def format_preds_batch(
    preds: torch.Tensor,
    obj_thresh: float = 0.5,
    iou_thresh: float = 0.5,
    box_format: BoxFormat = "cxcywh",
    min_class_confidence_threshold: float = 0.0,
) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    """preds (B, 5+C, Sy, Sx) on the GPU -> (rows (B, Sy*Sx, 5+C), keep_count (B,) int32,
    keep_index (B, Sy*Sx) int32, class_counts (C,) int64).  Image b's formatted predictions
    are ``rows[b, :keep_count[b]]`` in the reference's output order; everything stays on the
    device and nothing synchronises."""
    if preds.ndim != 4:
        raise ValueError(f"expected batched predictions (B, pred_shape, Sy, Sx), got {tuple(preds.shape)}")
    if box_format not in get_args(BoxFormat):
        raise ValueError(f"invalid box format {box_format}; valid box formats are {get_args(BoxFormat)}")
    L.require_cuda(preds, "predictions")
    lib = L.lib()
    B, D, Sy, Sx = preds.shape
    p = preds.detach().contiguous().float()
    dev = p.device
    keep_count = torch.empty(B, dtype=torch.int32, device=dev)
    rows = torch.empty((B, Sy * Sx, D), dtype=torch.float32, device=dev)
    keep_index = torch.empty((B, Sy * Sx), dtype=torch.int32, device=dev)
    counts = torch.empty(D - 5, dtype=torch.int64, device=dev)
    nbytes = lib.yg_format_preds_workspace(B, D - 5, Sy, Sx)
    ws = L.workspace.get("nms", nbytes, dev)
    L.check(lib.yg_format_preds_batch(p.data_ptr(), B, D - 5, Sy, Sx, float(obj_thresh), float(iou_thresh),
                                      1 if box_format == "xyxy" else 0, float(min_class_confidence_threshold),
                                      keep_count.data_ptr(), rows.data_ptr(), keep_index.data_ptr(),
                                      counts.data_ptr(), ws.data_ptr(), nbytes, L.stream()))
    return rows, keep_count, keep_index, counts


def format_preds(
    pred: torch.Tensor,
    obj_thresh: float = 0.5,
    iou_thresh: float = 0.5,
    box_format: BoxFormat = "cxcywh",
    min_class_confidence_threshold: float = 0.0,
) -> torch.Tensor:
    """Unbatched (pred_shape, Sy, Sx) -> (n, pred_shape) rows after objectness threshold,
    NMS (rows in descending NMS-score order) and the class-confidence filter."""
    if len(pred.shape) != 3:
        raise ValueError(
            "argument to format_pred should be unbatched result - "
            f"shape should be (pred_shape, Sy, Sx), got {pred.shape}"
        )
    elif box_format not in get_args(BoxFormat):
        raise ValueError(f"invalid box format {box_format}; valid box formats are {get_args(BoxFormat)}")
    rows, keep_count, _, _ = format_preds_batch(
        pred.unsqueeze(0), obj_thresh, iou_thresh, box_format, min_class_confidence_threshold
    )
    n = int(keep_count.item())
    return rows[0, :n].clone()


def split_formatted(rows: torch.Tensor, keep_count: torch.Tensor) -> List[torch.Tensor]:
    """Per-image views of a ``format_preds_batch`` result (one device->host read of the counts)."""
    counts = keep_count.tolist()
    return [rows[b, :n] for b, n in enumerate(counts)]


@L.on_device(lambda labels_xyxy, preds_xyxy: preds_xyxy)
def box_iou_cost(labels_xyxy: torch.Tensor, preds_xyxy: torch.Tensor) -> torch.Tensor:
    """(N, >=4) label rows and (M, >=4) prediction rows whose first four columns are xyxy -> (N, M) fp32 matrix
    ``1 - torchvision.ops.box_iou(labels, preds)`` (prediction_formatting.py:296-298), one launch, bit-identical."""
    L.require_cuda(labels_xyxy, "labels")
    L.require_cuda(preds_xyxy, "predictions")
    a = labels_xyxy.detach().float()
    b = preds_xyxy.detach().float()
    if a.stride(-1) != 1:
        a = a.contiguous()
    if b.stride(-1) != 1:
        b = b.contiguous()
    n, m = a.shape[0], b.shape[0]
    cost = torch.empty((n, m), dtype=torch.float32, device=a.device)
    L.check(L.lib().yg_box_iou_cost(a.data_ptr(), a.stride(0) if n else 4, n, b.data_ptr(), b.stride(0) if m else 4, m,
                                    cost.data_ptr(), L.stream()))
    return cost


@dataclass
class PredictionLabelMatch:
    """Result of matching predictions to labels (prediction_formatting.py:166-251): one-to-one matches, labels that
    no prediction claimed, and predictions that match no label."""

    preds: torch.Tensor
    labels: torch.Tensor
    missed_labels: Optional[torch.Tensor]
    extra_predictions: Optional[torch.Tensor]

    @staticmethod
    def concat(preds_and_labels: List["PredictionLabelMatch"]) -> "PredictionLabelMatch":
        missed = [p.missed_labels for p in preds_and_labels if p.missed_labels is not None]
        extra = [p.extra_predictions for p in preds_and_labels if p.extra_predictions is not None]
        return PredictionLabelMatch(
            preds=torch.cat([p.preds for p in preds_and_labels]),
            labels=torch.cat([p.labels for p in preds_and_labels]),
            missed_labels=torch.cat(missed, dim=0) if missed else None,
            extra_predictions=torch.cat(extra, dim=0) if extra else None,
        )

    def convert_background_errors(self, num_classes: int) -> "PredictionLabelMatch":
        """Missed labels become predictions of the background class (the LAST class) with objectness 1 on the label's box;
        extra predictions get a background label on their own box; every prediction row gains a zero background column
        (prediction_formatting.py:206-251).  Built with tensor ops instead of per-row Python lists."""
        dev, dt = self.preds.device, self.preds.dtype
        new_preds, new_labels = [], []
        if self.missed_labels is not None and self.missed_labels.shape[0] > 0:
            ml = self.missed_labels.to(dev)
            k = ml.shape[0]
            onehot = torch.zeros((k, num_classes), dtype=dt, device=dev)
            onehot[:, num_classes - 1] = 1
            new_preds.append(torch.cat([ml[:, 1:5].to(dt), torch.ones((k, 1), dtype=dt, device=dev), onehot], dim=1))
            new_labels.append(ml)
        if self.extra_predictions is not None and self.extra_predictions.shape[0] > 0:
            ep = self.extra_predictions.to(dev)
            k = ep.shape[0]
            new_preds.append(torch.cat([ep, torch.zeros((k, 1), dtype=ep.dtype, device=dev)], dim=1))
            lab = torch.cat([torch.ones((k, 1), dtype=ep.dtype, device=dev), ep[:, :4],
                             torch.full((k, 1), float(num_classes - 1), dtype=ep.dtype, device=dev)], dim=1)
            new_labels.append(lab.to(self.labels.dtype))
        if not new_preds:
            # the reference's torch.stack([]) raises here as well
            raise RuntimeError("stack expects a non-empty TensorList")
        preds = torch.cat([self.preds, torch.zeros((self.preds.shape[0], 1), dtype=dt, device=dev)], dim=1)
        return PredictionLabelMatch(
            preds=torch.cat([preds] + [p.to(dt) for p in new_preds]),
            labels=torch.cat([self.labels] + [l.to(self.labels.device) for l in new_labels]),
            missed_labels=None,
            extra_predictions=None,
        )


def format_preds_and_labels_v2(
    pred: torch.Tensor,
    label: torch.Tensor,
    objectness_thresh: float = 0.5,
    min_class_confidence_threshold: float = 0.0,
) -> PredictionLabelMatch:
    """Match one image's predictions with its labels (prediction_formatting.py:254-330): ``format_preds`` (xyxy, NMS 0.5),
    labelled cells in grid order, cost = 1 - pairwise IoU, Hungarian assignment, matched / missed / extra rows.
    The threshold + NMS and the cost matrix are one launch each; the assignment itself runs on the host in
    scipy exactly like the reference (the matrix is bit-identical, so the assignment is)."""
    from scipy.optimize import linear_sum_assignment

    pred = pred.squeeze()
    label = label.squeeze()
    if len(pred.shape) != 3:
        raise ValueError(
            "argument to format_pred should be unbatched result - "
            f"shape should be (pred_shape, Sy, Sx), got {pred.shape}"
        )
    formatted_preds = format_preds(
        pred, obj_thresh=objectness_thresh, iou_thresh=0.5, box_format="xyxy",
        min_class_confidence_threshold=min_class_confidence_threshold,
    )
    label_shape, Sy, Sx = label.shape
    labels = label.reshape(label_shape, Sx * Sy).T
    formatted_labels = labels[labels[:, 0].bool()].to(formatted_preds.device)
    M, N = formatted_preds.shape[0], formatted_labels.shape[0]
    cost = box_iou_cost(formatted_labels[:, 1:5], formatted_preds[:, :4]) if M and N else torch.ones((N, M))
    row_idxs, col_idxs = linear_sum_assignment(cost.cpu().numpy())
    dev = formatted_preds.device
    rows = torch.as_tensor(row_idxs, dtype=torch.long, device=dev)
    cols = torch.as_tensor(col_idxs, dtype=torch.long, device=dev)
    pred_free = torch.ones(M, dtype=torch.bool, device=dev)
    pred_free[cols] = False
    label_free = torch.ones(N, dtype=torch.bool, device=dev)
    label_free[rows] = False
    return PredictionLabelMatch(
        preds=formatted_preds[cols],
        labels=formatted_labels[rows],
        missed_labels=formatted_labels[label_free],
        extra_predictions=formatted_preds[pred_free],
    )


_LSAP_ERRORS = {1: "matrix contains invalid numeric entries", 2: "cost matrix is infeasible"}   # scipy's messages


def _lsap_status_check(status: torch.Tensor, what: str) -> None:
    """Raise scipy's ValueError for the first matrix the solver rejected (one device->host read)."""
    st = status.cpu().numpy()
    bad = np.flatnonzero(st)
    if bad.size:
        k = int(bad[0])
        raise ValueError(f"{_LSAP_ERRORS.get(int(st[k]), 'assignment failed')} ({what} {k})")


def _upload_int64(table: np.ndarray, dev: torch.device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(table, dtype=np.int64)).pin_memory().to(dev, non_blocking=True)


def _exclusive_cumsum(x: np.ndarray) -> np.ndarray:
    out = np.zeros_like(x)
    np.cumsum(x[:-1], out=out[1:])
    return out


def _lsap_plan(rows: np.ndarray, cols: np.ndarray) -> Tuple[np.ndarray, int]:
    """Descriptor table of yg_lsap_batch / yg_match_batch for matrices of the given shapes (include/yogo_b200.h): int64
    [n, 4] = cost offset, workspace offset (8-byte words), output offset, rows | cols << 32, then for yg_match_batch
    [n, 2] = offsets of each image's missed (rows - k) and extra (cols - k) rows, k = min(rows, cols).  Returns the flat
    table and the workspace size in 8-byte words."""
    lib = L.load()
    rows, cols = np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64)
    k = np.minimum(rows, cols)
    words = np.array([lib.yg_lsap_workspace_words(int(r), int(c)) for r, c in zip(rows, cols)], dtype=np.int64)
    desc = np.stack([_exclusive_cumsum(rows * cols), _exclusive_cumsum(words), _exclusive_cumsum(k), rows | (cols << 32)], 1)
    goff = np.stack([_exclusive_cumsum(rows - k), _exclusive_cumsum(cols - k)], 1)
    return np.concatenate([desc.reshape(-1), goff.reshape(-1)]), int(words.sum())


@L.on_device(lambda costs: costs[0] if len(costs) else None)
def linear_sum_assignment_batch(costs: Sequence[torch.Tensor]) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """``scipy.optimize.linear_sum_assignment`` of several 2-D fp32 CUDA matrices (shapes may differ) in one launch of
    the device solver (csrc/match.cu, one warp per matrix).  Returns int64 ``(row_ind, col_ind)`` per matrix on the
    matrices' device, identical to scipy's.  Raises scipy's ValueError, naming the matrix, for NaN or -inf entries and
    for a matrix whose +inf entries leave a row unassignable.  One host synchronisation (the solver status)."""
    costs = list(costs)
    if not costs:
        return []
    dev = costs[0].device
    for k, c in enumerate(costs):
        if c.ndim != 2:
            raise ValueError(f"expected a matrix (2-D array), got a {c.ndim} array (cost matrix {k})")
        L.require_cuda(c, "cost matrices")
        if c.device != dev:
            raise ValueError(f"cost matrix {k} is on {c.device}, cost matrix 0 on {dev}; all must be on one device")
        if c.dtype != torch.float32:
            raise ValueError(f"cost matrix {k} has dtype {c.dtype}; the solver takes torch.float32")
    lib = L.lib()
    n = len(costs)
    rows = np.array([c.shape[0] for c in costs], dtype=np.int64)
    cols = np.array([c.shape[1] for c in costs], dtype=np.int64)
    k = np.minimum(rows, cols)
    table, words = _lsap_plan(rows, cols)
    flat = torch.cat([c.detach().reshape(-1) for c in costs])
    out = torch.empty((2, max(int(k.sum()), 1)), dtype=torch.int64, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    ws = L.workspace.get("lsap", 8 * words, dev)
    desc = _upload_int64(table, dev)
    L.check(lib.yg_lsap_batch(flat.data_ptr(), desc.data_ptr(), n, ws.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                              status.data_ptr(), L.stream()))
    _lsap_status_check(status, "cost matrix")
    offs = _exclusive_cumsum(k)
    return [(out[0, o:o + m], out[1, o:o + m]) for o, m in zip(offs.tolist(), k.tolist())]


@dataclass
class _BatchMatch:
    """Everything the batched matching computes, before its solver status is read: the match and its per-image counts,
    and the intermediates that the metrics reuse (yogo_b200.metrics)."""

    match: PredictionLabelMatch
    counts: torch.Tensor       # (B, 3) int64 CPU: matched, missed, extra per image
    rows: torch.Tensor         # (B, Sy*Sx, 5+C) xyxy rows of format_preds_batch, image b's first keep_count[b] are kept
    keep_count: torch.Tensor   # (B,) int32
    label_rows: torch.Tensor   # (B, Sy*Sx, 6) labelled cells in grid order (yg_compact_labels), first n_labels[b] valid
    n_labels: torch.Tensor     # (B,) int32
    n_host: np.ndarray         # n_labels and keep_count on the host (int64)
    m_host: np.ndarray
    table: torch.Tensor        # device plan of _lsap_plan: desc (B x 4), then gather offsets (B x 2)
    status: torch.Tensor       # (B,) solver status on the device, not yet read


def _match_batch(preds: torch.Tensor, labels: torch.Tensor, objectness_thresh: float,
                 min_class_confidence_threshold: float) -> _BatchMatch:
    """The body of format_preds_and_labels_batch up to (not including) the read of the solver status."""
    if preds.ndim != 4:
        raise ValueError(f"expected batched predictions (B, pred_shape, Sy, Sx), got {tuple(preds.shape)}")
    if labels.ndim != 4 or labels.shape[0] != preds.shape[0] or labels.shape[1] != 6 or labels.shape[2:] != preds.shape[2:]:
        raise ValueError(f"expected batched labels (B, 6, Sy, Sx) matching predictions {tuple(preds.shape)}, got {tuple(labels.shape)}")
    L.require_cuda(preds, "predictions")
    L.require_cuda(labels, "labels")
    if labels.device != preds.device:
        raise ValueError(f"predictions on {preds.device} and labels on {labels.device}: both must be on one device")
    rows, keep_count, _, _ = format_preds_batch(preds, objectness_thresh, 0.5, "xyxy", min_class_confidence_threshold)
    lib = L.lib()
    B, D, Sy, Sx = preds.shape
    cells = Sy * Sx
    dev = rows.device
    lab = labels.detach().float().contiguous()
    label_rows = torch.empty((B, cells, 6), dtype=torch.float32, device=dev)
    n_labels = torch.empty(B, dtype=torch.int32, device=dev)
    L.check(lib.yg_compact_labels(lab.data_ptr(), B, Sy, Sx, label_rows.data_ptr(), n_labels.data_ptr(), L.stream()))
    cnt = torch.stack([n_labels, keep_count]).cpu().numpy().astype(np.int64)   # host synchronisation 1
    N, M = cnt[0], cnt[1]
    K = np.minimum(N, M)
    counts = torch.from_numpy(np.stack([K, N - K, M - K], 1).astype(np.int64)).reshape(B, 3)
    plan, words = _lsap_plan(N, M)
    table = _upload_int64(plan, dev)
    Kt, Nt, Mt = int(K.sum()), int(N.sum()), int(M.sum())
    costs = torch.empty(max(int((N * M).sum()), 1), dtype=torch.float32, device=dev)
    pairs = torch.empty((2, max(Kt, 1)), dtype=torch.int64, device=dev)
    status = torch.empty(max(B, 1), dtype=torch.int32, device=dev)
    ws = L.workspace.get("lsap", 8 * words, dev)
    out_preds = torch.empty((Kt, D), dtype=torch.float32, device=dev)
    out_labels = torch.empty((Kt, 6), dtype=torch.float32, device=dev)
    missed = torch.empty((Nt - Kt, 6), dtype=torch.float32, device=dev)
    extra = torch.empty((Mt - Kt, D), dtype=torch.float32, device=dev)
    L.check(lib.yg_match_batch(label_rows.data_ptr(), rows.data_ptr(), B, cells, D - 5, int(N.max(initial=0)), int(M.max(initial=0)),
                               table.data_ptr(), table[4 * B:].data_ptr(), costs.data_ptr(), ws.data_ptr(), pairs[0].data_ptr(),
                               pairs[1].data_ptr(), status.data_ptr(), out_preds.data_ptr(), out_labels.data_ptr(),
                               missed.data_ptr(), extra.data_ptr(), L.stream()))
    match = PredictionLabelMatch(preds=out_preds, labels=out_labels, missed_labels=missed, extra_predictions=extra)
    return _BatchMatch(match, counts, rows, keep_count, label_rows, n_labels, N, M, table, status[:B])


@L.on_device(lambda preds, *a, **k: preds)
def format_preds_and_labels_batch(
    preds: torch.Tensor,
    labels: torch.Tensor,
    objectness_thresh: float = 0.5,
    min_class_confidence_threshold: float = 0.0,
) -> Tuple[PredictionLabelMatch, torch.Tensor]:
    """``format_preds_and_labels_v2`` for a whole batch: preds (B, 5+C, Sy, Sx) and labels (B, 6, Sy, Sx) on one CUDA
    device -> (match, counts).  ``match`` is bit-identical to ``PredictionLabelMatch.concat`` of the per-image results
    (matched pairs in ascending label index, missed labels, extra predictions in NMS order, image after image);
    ``counts`` is a (B, 3) int64 CPU tensor of [matched, missed, extra] per image, for ``torch.split``.

    Threshold + NMS, label gather, cost matrices, assignment (the device solver of ``linear_sum_assignment_batch``) and the
    output gather are batched launches; the call synchronises twice whatever B is: once to read the per-image counts that
    size the outputs, once to read the solver status (scipy's ValueError is raised for an image with a NaN cost, e.g. a
    zero-area label and a zero-area prediction that do not overlap)."""
    r = _match_batch(preds, labels, objectness_thresh, min_class_confidence_threshold)
    if preds.shape[0]:
        _lsap_status_check(r.status, "image")   # host synchronisation 2
    return r.match, r.counts


def format_to_numpy(img_id: int, prediction_tensor, img_h: int, img_w: int, np_dtype=np.float32) -> np.ndarray:
    """One image's prediction tensor -> the (8 + C) x n array ``yogo infer --save-npy`` stores
    (prediction_formatting.py:96-156): image id, pixel-space corners, objectness, argmax class, its probability, all
    class probabilities.  Threshold + NMS run in the batched kernel; the rest is column arithmetic on n rows."""
    t = prediction_tensor if isinstance(prediction_tensor, torch.Tensor) else torch.from_numpy(np.asarray(prediction_tensor))
    if not t.is_cuda:
        t = t.to(torch.device("cuda", torch.cuda.current_device())) if torch.cuda.is_available() else t
    fp = format_preds(t, box_format="xyxy").cpu().numpy().T
    n = fp.shape[1]
    img_ids = np.ones(n).astype(np_dtype) * img_id
    tlx, tly, brx, bry = fp[0, :] * img_w, fp[1, :] * img_h, fp[2, :] * img_w, fp[3, :] * img_h
    objectness = fp[4, :].astype(np_dtype)
    all_confs = fp[5:, :].astype(np_dtype)
    pred_labels = np.argmax(all_confs, axis=0).astype(np.uint8)
    pred_probs = fp[5:, ][pred_labels, np.arange(n)]
    return np.vstack((img_ids, tlx, tly, brx, bry, objectness, pred_labels.astype(np_dtype), pred_probs.astype(np_dtype),
                      all_confs))
