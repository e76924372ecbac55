"""yogo_b200 - B200-native implementation of the YOGO hot path behind the reference's Python API."""
from .model import YOGO  # noqa: F401
from .model_defns import MODELS, get_model_func, register_model  # noqa: F401
from .yogo_loss import YOGOLoss  # noqa: F401
from ._lib import get_fp32_tensor_cores, set_fp32_tensor_cores  # noqa: F401
from .utils import (  # noqa: F401
    PredictionLabelMatch, box_iou_cost, format_preds, format_preds_and_labels_batch, format_preds_and_labels_v2,
    format_preds_batch, format_to_numpy, linear_sum_assignment_batch,
)
from .infer import get_prediction_class_counts, count_cells_for_formatted_preds, predict, save_predictions  # noqa: F401
from .metrics import Metrics  # noqa: F401

__all__ = [
    "YOGO", "YOGOLoss", "MODELS", "get_model_func", "register_model", "format_preds", "format_preds_batch",
    "get_prediction_class_counts", "count_cells_for_formatted_preds", "predict", "save_predictions",
    "PredictionLabelMatch", "box_iou_cost", "format_preds_and_labels_v2", "format_to_numpy", "set_fp32_tensor_cores",
    "get_fp32_tensor_cores", "format_preds_and_labels_batch", "linear_sum_assignment_batch", "Metrics",
]
