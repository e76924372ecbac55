from .prediction_formatting import (  # noqa: F401
    PredictionLabelMatch,
    box_iou_cost,
    format_preds,
    format_preds_and_labels_batch,
    format_preds_and_labels_v2,
    format_preds_batch,
    format_to_numpy,
    linear_sum_assignment_batch,
    split_formatted,
)
