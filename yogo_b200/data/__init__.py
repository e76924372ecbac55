"""Input side of the training step (SURVEY.md 8f N3): batch transforms, label rasterisation and the device-resident dataset."""
from .data_transforms import (  # noqa: F401
    DualInputId,
    DualInputModule,
    ImageTransformLabelIdentity,
    MultiArgSequential,
    RandomHorizontalFlipWithBBs,
    RandomVerticalFlipWithBBs,
    flip_batch,
)
from .yogo_dataset import LABEL_TENSOR_PRED_DIM_SIZE, format_labels_batch, format_labels_tensor  # noqa: F401
from .utils import collate_batch_robust  # noqa: F401
from .device_dataset import DeviceResidentDataset  # noqa: F401
