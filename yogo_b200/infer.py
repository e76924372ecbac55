"""Inference entry points of /root/reference/yogo/infer.py: the per-class counts (:60-124), the YOGO-format
prediction writer (:39-57) and the ``predict`` batch loop (:140-421) with the post-processing of a whole batch
in one launch instead of one Python iteration per image."""
from __future__ import annotations

import datetime
import json
import warnings
from pathlib import Path
from typing import List, Literal, Optional, Sequence, Union

import numpy as np
import torch

from .utils.prediction_formatting import format_preds_batch


def get_prediction_class_counts(
    batch_preds: torch.Tensor,
    obj_thresh=0.5,
    iou_thresh=0.5,
    min_class_confidence_threshold: float = 0,
) -> torch.Tensor:
    """Count predictions per argmax class over a batch (infer.py:60-87).  The reference loops
    over images on the CPU; here threshold + NMS + counting is one launch and the (C,) int64
    result is returned on the CPU like the reference's accumulator."""
    _, _, _, counts = format_preds_batch(
        batch_preds, obj_thresh=obj_thresh, iou_thresh=iou_thresh,
        min_class_confidence_threshold=min_class_confidence_threshold,
    )
    return counts.cpu()


def count_cells_for_formatted_preds(
    formatted_class_predictions: torch.Tensor,
    min_confidence_threshold: Optional[float] = None,
) -> torch.Tensor:
    """infer.py:90-124 - host-side helper on an already formatted (N, num_classes) tensor; tiny
    integer bookkeeping, kept in torch."""
    if not len(formatted_class_predictions.shape) == 2:
        raise ValueError(
            "expected formatted_class_predictions to be shape (N, num_classes); "
            f"got {formatted_class_predictions.shape}"
        )
    if min_confidence_threshold is not None:
        if min_confidence_threshold < 0 or min_confidence_threshold > 1:
            raise ValueError(f"min_confidence_threshold should be between 0 and 1; is {min_confidence_threshold}")
    else:
        min_confidence_threshold = 0
    _, n_classes = formatted_class_predictions.shape
    values, indices = formatted_class_predictions.max(dim=1)
    mask = values > min_confidence_threshold
    return torch.nn.functional.one_hot(indices[mask], num_classes=n_classes).sum(dim=0)


def save_predictions(fnames: Sequence, batch_preds: torch.Tensor, obj_thresh: float = 0.5, iou_thresh: float = 0.5) -> None:
    """infer.py:39-57: one text file per image, a line ``<argmax class> <xc> <yc> <w> <h>`` per kept prediction in
    ``format_preds`` order.  Threshold + NMS of the whole batch is one launch and one device->host copy."""
    rows, keep_count, _, _ = format_preds_batch(batch_preds, obj_thresh=obj_thresh, iou_thresh=iou_thresh)
    counts = keep_count.tolist()
    nmax = max(counts) if counts else 0
    host = rows[:, :nmax].cpu()
    for fname, n, r in zip(fnames, counts, host):
        lines = []
        for pred in r[:n]:
            cls = int(torch.argmax(pred[5:]))   # first maximum, like the reference's max(range(n), key=...)
            lines.append(f"{cls} {pred[0]} {pred[1]} {pred[2]} {pred[3]}")
        with open(fname, "w") as f:
            f.write("\n".join(lines))


class GraphedInference:
    """Eval forward + objectness threshold + NMS + per-class counts of one fixed batch shape as ONE CUDA-graph replay.

    The per-batch work of `predict` is ~20 kernel launches whose GPU time at small batch (one 772x1032 image: ~60 us) is far
    below the host cost of launching them one by one; replaying a captured graph removes that (B200_PROFILING: "capture
    launch-bound inner loops in CUDA graphs").  `__call__` copies the batch into the static input and returns the static
    outputs `(pred, rows, keep_count, keep_index, class_counts)` - valid until the next call."""

    def __init__(self, model, batch_shape, dtype=torch.uint8, obj_thresh: float = 0.5, iou_thresh: float = 0.5,
                 min_class_confidence_threshold: float = 0.0, box_format: str = "cxcywh", warmup: int = 2):
        dev = next(model.parameters()).device
        self.model = model
        self.static_in = torch.zeros(tuple(batch_shape), dtype=dtype, device=dev)
        kw = dict(obj_thresh=obj_thresh, iou_thresh=iou_thresh, box_format=box_format,
                  min_class_confidence_threshold=min_class_confidence_threshold)

        def body():
            with torch.no_grad():
                pred = model(self.static_in)
            return (pred,) + tuple(format_preds_batch(pred, **kw))

        with torch.cuda.device(dev):
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(max(1, warmup)):   # workspaces, packed weights, function attributes: all outside the capture
                    body()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.out = body()

    def __call__(self, images: torch.Tensor):
        self.static_in.copy_(images, non_blocking=True)
        self.graph.replay()
        return self.out


class GraphedForward:
    """Eval forward of one fixed batch shape as a CUDA-graph replay (the forward alone; `predict` applies whatever
    post-processing its flags ask for to the static output, which is valid until the next call)."""

    def __init__(self, model, batch_shape, dtype=torch.uint8, warmup: int = 2):
        dev = next(model.parameters()).device
        self.static_in = torch.zeros(tuple(batch_shape), dtype=dtype, device=dev)
        with torch.cuda.device(dev):
            s = torch.cuda.Stream(device=dev)
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s), torch.no_grad():
                for _ in range(max(1, warmup)):
                    model(self.static_in)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph), torch.no_grad():
                self.out = model(self.static_in)

    def __call__(self, images: torch.Tensor) -> torch.Tensor:
        self.static_in.copy_(images, non_blocking=True)
        self.graph.replay()
        return self.out


def _list_images(path_to_images: Path) -> List[Path]:
    p = Path(path_to_images)
    if p.is_file():
        return [p]
    if not p.is_dir():
        raise FileNotFoundError(f"{p} is neither an image nor a directory of images")
    return sorted(q for q in p.iterdir() if q.suffix.lower() in (".png", ".npy"))


def _read_image(path: Path) -> torch.Tensor:
    """(1, H, W) uint8 - grayscale PNG (torchvision.io) or a .npy array; decoding is I/O around the path."""
    if path.suffix.lower() == ".npy":
        a = torch.from_numpy(np.load(path))
        return a.reshape(1, *a.shape[-2:]).to(torch.uint8)
    from torchvision.io import ImageReadMode, read_image

    return read_image(str(path), ImageReadMode.GRAY)


# Files of `predict` are decoded in groups of this many images per SM (rounded up to whole batches): the inflate kernel
# runs one warp per image, so a group needs several warps per SM to hide the latency of its serial decode.  8 per SM
# (1184 images on a B200, about 2.5 GB of output, scratch and streams at 772x1032) measured as fast as 16 per SM in
# `predict`, whose rate is bound by the host work of each group (profiles/png_decode_bench.jsonl), at half the memory.
DECODE_IMAGES_PER_SM = 8


def _read_files(paths: Sequence[Path]) -> list:
    """Raw bytes of the PNG files (torchvision.io.read_file) and decoded .npy arrays, or the exception a read raised."""
    from torchvision.io import read_file

    items = []
    for q in paths:
        try:
            items.append(_read_image(q) if q.suffix.lower() == ".npy" else read_file(str(q)))
        except Exception as e:   # raised again when its batch is loaded, like the per-batch read of the reference
            items.append(e)
    return items


class _FolderDecoder:
    """Images of `paths` for `predict`, decoded on the GPU in groups of whole batches (data.png.decode_entries) while a
    small thread pool reads the next group's files.  `prepare(lo)` decodes the group that holds batch `lo`; an error
    there (out of memory, a failed launch) is not a file's error and propagates.  `batch(lo, hi)` then returns what
    ``torch.stack([_read_image(q) for q in paths[lo:hi]])`` returns, on `dev`, and raises what it raises."""

    def __init__(self, paths: Sequence[Path], dev: torch.device, batch_size: int):
        import math
        from concurrent.futures import ThreadPoolExecutor

        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        self.group = max(1, math.ceil(sms * DECODE_IMAGES_PER_SM / batch_size)) * batch_size
        self.paths, self.dev = list(paths), dev
        self.workers = 4
        self.pool = ThreadPoolExecutor(max_workers=self.workers)
        self.index = -1                    # group whose entries are held
        self.entries: list = []
        self.pending = self._submit(0)     # (group index, read futures)

    def _submit(self, g: int):
        paths = self.paths[g * self.group:(g + 1) * self.group]
        step = -(-len(paths) // self.workers) if paths else 1
        return g, [self.pool.submit(_read_files, paths[i:i + step]) for i in range(0, len(paths), step)]

    def prepare(self, lo: int) -> None:
        from torchvision.io import ImageReadMode, decode_image

        from .data.png import decode_entries

        g = lo // self.group
        if g == self.index:
            return
        self.index, self.entries = -1, []
        _, futs = self.pending if self.pending[0] == g else self._submit(g)
        items = [it for f in futs for it in f.result()]
        self.pending = self._submit(g + 1)
        pngs = [i for i, it in enumerate(items) if isinstance(it, torch.Tensor) and it.dim() == 1]
        decoded, _ = decode_entries([items[i] for i in pngs], self.dev, lambda x: decode_image(x, ImageReadMode.GRAY))
        entries = [it if isinstance(it, BaseException) else (it.unsqueeze(0).to(self.dev), 0) for it in items]
        for i, e in zip(pngs, decoded):
            entries[i] = e
        self.index, self.entries = g, entries

    def batch(self, lo: int, hi: int) -> torch.Tensor:
        from .data.png import stack_entries

        g = lo // self.group
        if g != self.index or (hi - 1) // self.group != g:
            raise AssertionError(f"batch [{lo}, {hi}) is not inside the prepared decode group {self.index}")
        return stack_entries(self.entries[lo - g * self.group:hi - g * self.group])

    def close(self) -> None:
        self.pool.shutdown(wait=True, cancel_futures=True)


@torch.no_grad()
def predict(
    path_to_pth: str,
    *,
    path_to_images: Optional[Path] = None,
    path_to_zarr: Optional[Path] = None,
    output_dir: Optional[str] = None,
    draw_boxes: bool = False,
    save_preds: bool = False,
    save_npy: bool = False,
    class_names: Optional[List[str]] = None,
    count_predictions: bool = False,
    batch_size: int = 64,
    obj_thresh: float = 0.5,
    iou_thresh: float = 0.5,
    vertical_crop_height: Optional[float] = None,
    use_tqdm: bool = False,
    device: Optional[Union[str, torch.device]] = None,
    output_img_ftype: Literal[".png", ".tif", ".tiff"] = ".png",
    requested_num_workers: Optional[int] = None,
    min_class_confidence_threshold: float = 0.0,
    half: bool = False,
    return_full_predictions: bool = False,
    images: Optional[torch.Tensor] = None,
) -> Optional[torch.Tensor]:
    """The ``yogo infer`` batch loop (infer.py:140-421) on the B200 path: checkpoint -> eval model, batches of uint8
    images -> forward -> batched threshold / NMS / counts, optional YOGO-format text files, ``.npy`` export and the full
    prediction tensor.  ``half`` selects bf16 compute (the reference's autocast), otherwise fp32.  ``images`` (N,1,H,W)
    uint8 is an in-memory alternative to ``path_to_images``.  Box drawing and zarr input are outside the path and raise."""
    from .model import YOGO
    from .utils.prediction_formatting import split_formatted

    if save_preds and draw_boxes:
        raise ValueError("cannot save predictions in YOGO format and draw_boxes at the same time")
    elif output_dir is not None and not (save_preds or draw_boxes or save_npy):
        warnings.warn(
            f"output dir is not None (is {output_dir}), but it will not be used "
            "since save_preds and draw_boxes are both false"
        )
    elif output_dir is not None:
        Path(output_dir).mkdir(exist_ok=True, parents=False)
    elif save_preds:
        raise ValueError("output_dir must not be None if save_preds is True")
    elif output_img_ftype not in [".png", ".tif", ".tiff"]:
        raise ValueError(
            "only .png, .tif, and .tiff are supported for output img " f"filetype; got {output_img_ftype}"
        )
    if draw_boxes:
        raise NotImplementedError("draw_boxes (matplotlib/PIL rendering) is outside the B200 hot path")
    if path_to_zarr is not None:
        raise NotImplementedError("zarr input is outside the B200 hot path; use path_to_images or images=")
    if (path_to_images is None) == (images is None):
        raise ValueError("exactly one of path_to_images and images must be given")

    dev = torch.device(device or "cuda")
    model, cfg = YOGO.from_pth(Path(path_to_pth), inference=True)
    model.eval()
    model.to(dev)
    model.compute_dtype = torch.bfloat16 if half else torch.float32

    img_h, img_w = model.get_img_size()
    crop_h = None
    if vertical_crop_height:
        crop_h = int((vertical_crop_height * img_h).round().item())
        model.resize_model(crop_h)
        img_h = torch.tensor(crop_h)
    in_h, in_w = int(model.img_size[0].item()), int(model.img_size[1].item())
    num_classes = int(model.num_classes.item())
    if class_names is not None and len(class_names) != num_classes:
        raise ValueError(f"expected {num_classes} class names, got {len(class_names)}")

    if images is not None:
        n_images = images.shape[0]
        fnames_all = [f"image_{i:06d}.png" for i in range(n_images)]
    else:
        paths = _list_images(Path(path_to_images))
        n_images = len(paths)
        fnames_all = [str(q) for q in paths]

    def load_batch(lo: int, hi: int) -> torch.Tensor:
        if images is not None:
            b = images[lo:hi]
        else:
            b = folder.batch(lo, hi)
        if crop_h is not None:   # CenterCrop((crop_h, img_w))
            top = int(round((b.shape[-2] - crop_h) / 2.0))
            b = b[..., top:top + crop_h, :]
        if b.shape[-2:] != (in_h, in_w):
            raise RuntimeError(f"image size {tuple(b.shape[-2:])} does not match the model's {(in_h, in_w)}")
        return b

    results = None
    np_results = []
    tot_counts = torch.zeros(num_classes, dtype=torch.int64, device=dev) if count_predictions else None
    pbar = None
    if use_tqdm:
        from tqdm import tqdm

        pbar = tqdm(unit="images", total=n_images)
    graphed: dict = {}
    normalize = bool(model.normalize_images)
    if normalize:
        model.set_fused_input_scale(1.0 / 255.0)   # uint8 batches: the /255 happens inside the first-layer kernel
    folder = _FolderDecoder(paths, dev, batch_size) if images is None else None
    try:
        for i, lo in enumerate(range(0, n_images, batch_size)):
            hi = min(lo + batch_size, n_images)
            if folder is not None:
                folder.prepare(lo)
            try:
                img_batch = load_batch(lo, hi)
            except RuntimeError as e:   # malformed images: warn and continue, like the reference
                warnings.warn(f"got error {e}; continuing")
                continue
            x = img_batch.to(dev, non_blocking=True)
            if normalize and x.dtype != torch.uint8:
                x = x.float() / 255.0
            # full batches replay the forward from a CUDA graph (a batch of one 772x1032 image is ~60 us of GPU work behind
            # ~250 us of launches); the ragged last batch runs eagerly
            if dev.type == "cuda" and tuple(x.shape) == (batch_size,) + tuple(x.shape[1:]) and n_images >= 2 * batch_size:
                key = (tuple(x.shape), x.dtype)
                if graphed.get("key") != key:
                    graphed["key"], graphed["fwd"] = key, GraphedForward(model, x.shape, x.dtype)
                res = graphed["fwd"](x)
            else:
                res = model(x)
            if results is None and return_full_predictions:
                results = torch.zeros((n_images, res.shape[1], res.shape[2], res.shape[3]))
            if save_preds:
                out_fnames = [Path(output_dir) / Path(f).with_suffix(".txt").name for f in fnames_all[lo:hi]]
                save_predictions(out_fnames, res, obj_thresh=obj_thresh, iou_thresh=iou_thresh)
            if save_npy:
                rows, keep_count, _, _ = format_preds_batch(res, box_format="xyxy")
                for j, r in enumerate(split_formatted(rows, keep_count)):
                    fp = r.cpu().numpy().T
                    n = fp.shape[1]
                    labels = np.argmax(fp[5:, :], axis=0).astype(np.uint8)
                    np_results.append(np.vstack((
                        np.ones(n).astype(np.float32) * (lo + j), fp[0, :] * in_w, fp[1, :] * int(img_h.item()),
                        fp[2, :] * in_w, fp[3, :] * int(img_h.item()), fp[4, :], labels.astype(np.float32),
                        fp[5:, ][labels, np.arange(n)], fp[5:, :])))
            if count_predictions:
                _, _, _, counts = format_preds_batch(
                    res, obj_thresh=obj_thresh, iou_thresh=iou_thresh,
                    min_class_confidence_threshold=min_class_confidence_threshold)
                tot_counts += counts
            if return_full_predictions:
                results[lo:hi, ...] = res.cpu()
            if pbar is not None:
                pbar.update(hi - lo)
    finally:
        if folder is not None:
            folder.close()
    if pbar is not None:
        pbar.close()

    if count_predictions:
        print(list(zip(class_names or range(num_classes), map(int, tot_counts.cpu()))))

    if save_npy:
        pred_tensors = np.hstack(np_results) if np_results else np.zeros((8 + num_classes, 0), dtype=np.float32)
        filename = Path(path_to_images).resolve().parent.stem if path_to_images else "predictions"
        base = Path(output_dir).resolve() if output_dir is not None else Path.cwd().resolve()
        fp_out = base / Path(filename).with_suffix(".npy")
        np.save(fp_out, pred_tensors)
        with open(fp_out.with_suffix(".json"), "w") as f:
            json.dump(dict(run_name=fp_out.with_suffix("").name,
                           model_name=torch.load(Path(path_to_pth), map_location="cpu").get("model_name", None),
                           obj_thresh=obj_thresh, iou_thresh=iou_thresh, vertical_crop_height_px=int(img_h.item()),
                           write_date=datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S")), f, indent=4)

    return results if return_full_predictions else None
