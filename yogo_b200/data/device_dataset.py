"""Device-resident training data: the dataset is decoded once into HBM and every batch of every epoch is built on the GPU.

The reference's training loop reads, decodes and collates every image of every epoch on the host (yogo_dataloader.py,
utils.py:49-63); at the step rate of this project that host work, not the GPU, bounds training on real data.  YOGO trains
many epochs over the same images and its only augmentations are the two whole-batch flips, so
``DeviceResidentDataset`` decodes the dataset once (spread over the ranks of a process group, completed with
all-gathers so that every rank holds the full store) and afterwards builds each batch with three kernels
(csrc/input.cu): the flip draw, the image gather + flip and the label build.  They read the epoch's index table and their
own state from device memory, so they run inside the captured training step (``DataParallelTrainer.steps_from_device``)
and the host does no per-step data work.

What it computes: batch i of epoch e is ``flip_batch(collate([dataset[j] for j in idx]), h, v)`` where ``idx`` is batch
i of the reference's ``DistributedSampler(shuffle=True, seed=seed, drop_last=False)`` with ``set_epoch(e)``, in batches
of ``batch_size`` with the ragged last batch kept, and ``(h, v)`` are drawn on the device with the flip modules' ``p``.
Deviations from the reference's DataLoader:
  * items the dataset returns as ``None`` (unreadable files) are left out once, at build time; the reference drops them
    from each batch instead, so its batches can be short.  Their count is in ``num_dropped`` and in a warning.
  * the flip decisions come from a device Philox stream, not from the host generator: the same distribution, other
    values (as for Dropout2d).
"""
from __future__ import annotations

import warnings
from typing import Iterator, List, Tuple

import torch
import torch.distributed as dist
from torch.utils.data import DataLoader, DistributedSampler, Subset

from .. import _lib as L
from .data_transforms import DualInputId, MultiArgSequential, RandomHorizontalFlipWithBBs, RandomVerticalFlipWithBBs

# device memory left free after the build for the training step itself (activations, gradients, optimizer state, graph
# pools): base_model at batch 64 uses a few GB; 8 GiB leaves room for larger models and batches
DEFAULT_RESERVE_BYTES = 8 << 30
RECORD_WORDS = 8          # int32 per labelled cell: cell index, the six channel values' bits, padding (32 bytes)
BUILD_CHUNK = 64          # items per DataLoader batch while decoding


def flip_probabilities(transforms) -> Tuple[float, float]:
    """`p` of the horizontal and vertical flip modules in `transforms` (what `collate_batch_robust` takes: None, one
    module or a MultiArgSequential).  Any other module raises NotImplementedError: the device path builds batches with
    these two flips only."""
    if transforms is None:
        return 0.0, 0.0
    mods = list(transforms) if isinstance(transforms, MultiArgSequential) else [transforms]
    ph = pv = None
    for m in mods:
        if isinstance(m, DualInputId):
            continue
        if isinstance(m, RandomHorizontalFlipWithBBs) and ph is None:
            ph = float(m.p)
        elif isinstance(m, RandomVerticalFlipWithBBs) and pv is None:
            pv = float(m.p)
        else:
            raise NotImplementedError(f"DeviceResidentDataset supports RandomHorizontalFlipWithBBs and "
                                      f"RandomVerticalFlipWithBBs (at most one of each), not {type(m).__name__}")
    for p in (ph, pv):
        if p is not None and not 0.0 <= p <= 1.0:
            raise ValueError(f"flip probability {p} outside [0, 1]")
    return ph or 0.0, pv or 0.0


class _Sized:
    def __init__(self, n: int):
        self.n = n

    def __len__(self) -> int:
        return self.n


def epoch_batches(n: int, world: int, rank: int, seed: int, epoch: int, batch_size: int) -> List[List[int]]:
    """Batches of rank `rank` in epoch `epoch`: torch's own DistributedSampler(shuffle=True, drop_last=False) over `n`
    items, chunked into `batch_size` with the ragged last batch kept (yogo_dataloader.py:249-264)."""
    sampler = DistributedSampler(_Sized(n), num_replicas=world, rank=rank, shuffle=True, seed=seed, drop_last=False)
    sampler.set_epoch(epoch)
    idx = list(sampler)
    return [idx[i:i + batch_size] for i in range(0, len(idx), batch_size)]


def store_bytes(n_slots: int, item_bytes: int, n_records: int, samples_per_rank: int, batch_size: int) -> int:
    """Device bytes of a store: images, label records, record offsets (int64 per slot + 1) and the index table (whole
    batches of int32)."""
    table = -(-samples_per_rank // batch_size) * batch_size
    return n_slots * item_bytes + n_records * RECORD_WORDS * 4 + (n_slots + 1) * 8 + table * 4


def check_capacity(needed: int, free: int, reserve: int = DEFAULT_RESERVE_BYTES) -> None:
    """ValueError when `needed` bytes do not fit into `free` device bytes minus `reserve` kept for training."""
    if needed > free - reserve:
        raise ValueError(f"the device-resident dataset needs {needed} bytes ({needed / 2**30:.2f} GiB) but the device has "
                         f"{free} bytes free ({free / 2**30:.2f} GiB), of which {reserve} are kept for training")


def compact_labels(labels: torch.Tensor) -> torch.Tensor:
    """(6, Sy, Sx) fp32 -> (k, 8) int32 records {cell, six channel bit patterns, 0} of the k cells with any non-zero bit,
    in cell order.  The label kernel writes +0.0 (mirrored) into every other cell, so the dense tensor round-trips exactly."""
    bits = labels.contiguous().view(torch.int32).reshape(6, -1)
    cells = (bits != 0).any(0).nonzero().squeeze(1)
    rec = torch.zeros(cells.numel(), RECORD_WORDS, dtype=torch.int32)
    rec[:, 0] = cells.to(torch.int32)
    rec[:, 1:7] = bits[:, cells].t()
    return rec


def _keep_list(batch):
    return batch


class DeviceResidentDataset:
    """Decoded images and compact labels of a map-style dataset on every rank's GPU; batches are built on the device.

    ``dataset[i]`` is ``(image (C, H, W) uint8 or fp32, labels (6, Sy, Sx) fp32)`` or None, as `collate_batch_robust`
    expects; every item must have the shape and dtype of the first.  `transforms` is the object the collate function
    takes (the two flip modules or none).  `reserve_bytes` of free device memory are kept for training; a dataset that
    does not fit beside them raises ValueError before its images are allocated."""

    def __init__(self, dataset, batch_size: int, transforms=None, device=None, process_group=None, seed: int = 0,
                 num_workers: int = 0, reserve_bytes: int = DEFAULT_RESERVE_BYTES):
        if batch_size < 1:
            raise ValueError(f"batch_size must be positive, got {batch_size}")
        self.p_hflip, self.p_vflip = flip_probabilities(transforms)
        self.batch_size = int(batch_size)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if self.device.type != "cuda":
            raise L.YogoB200Error(f"DeviceResidentDataset keeps its store on a CUDA device, got {self.device}")
        self.pg = process_group
        distributed = dist.is_available() and dist.is_initialized()
        self.world = dist.get_world_size(process_group) if distributed else 1
        self.rank = dist.get_rank(process_group) if distributed else 0
        self.seed = int(seed)
        self.reserve_bytes = int(reserve_bytes)
        self._images = self._records = self._rec_off = self._slots = self._table = None
        self._state = self._flags = None
        with torch.cuda.device(self.device):
            try:
                self._build(dataset, num_workers)
            except BaseException:
                self._images = self._records = self._rec_off = self._slots = self._table = None
                self._state = self._flags = None
                raise

    # ------------------------------------------------------------------ build
    def _build(self, dataset, num_workers: int) -> None:
        n_items = len(dataset)
        if n_items == 0:
            raise ValueError("DeviceResidentDataset: the dataset is empty")
        world, rank, dev = self.world, self.rank, self.device
        chunk = -(-n_items // world)                  # items decoded by each rank (the last ranks may get fewer)
        lo, hi = min(rank * chunk, n_items), min((rank + 1) * chunk, n_items)
        loader = DataLoader(Subset(dataset, range(lo, hi)), batch_size=BUILD_CHUNK, shuffle=False, num_workers=num_workers,
                            collate_fn=_keep_list)
        it = iter(loader)
        first = next(it, None) if hi > lo else None

        # shape of the first item of the lowest rank that has one, agreed on by every rank
        ref = None
        for item in first or []:
            if item is not None:
                ref = (tuple(item[0].shape), item[0].dtype, tuple(item[1].shape))
                break
        if world > 1:
            refs = [None] * world
            dist.all_gather_object(refs, ref, group=self.pg)
            ref = next((r for r in refs if r is not None), None)
        if ref is None:
            raise ValueError("DeviceResidentDataset: every item of the dataset is None")
        (C, H, W), idt, lshape = ref
        if idt not in (torch.uint8, torch.float32) or C not in (1, 3):
            raise ValueError(f"DeviceResidentDataset: images must be (C, H, W) uint8 or float32 with C in (1, 3), the first "
                             f"item is {tuple(ref[0])} {idt}")
        if len(lshape) != 3 or lshape[0] != 6:
            raise ValueError(f"DeviceResidentDataset: labels must be (6, Sy, Sx), the first item's are {lshape}")
        self.image_shape, self.image_dtype, self.grid = (C, H, W), idt, (lshape[1], lshape[2])
        item_bytes = C * H * W * (1 if idt == torch.uint8 else 4)
        n_slots = chunk * world
        samples = -(-n_items // world)
        # images and index tables are known now; label records are checked again once decoded
        check_capacity(store_bytes(n_slots, item_bytes, 0, samples, self.batch_size), torch.cuda.mem_get_info(dev)[0],
                       self.reserve_bytes)
        self._images = torch.zeros((n_slots, C, H, W), dtype=idt, device=dev)

        valid = torch.zeros(chunk, dtype=torch.uint8)
        records: List[torch.Tensor] = []
        counts = torch.zeros(chunk, dtype=torch.int64)
        pos = 0
        batch = first
        while batch is not None:
            imgs = torch.zeros((len(batch), C, H, W), dtype=idt)
            for j, item in enumerate(batch):
                k = lo + pos + j
                if item is None:
                    continue
                img, lab = item
                if not isinstance(img, torch.Tensor) or tuple(img.shape) != (C, H, W) or img.dtype != idt:
                    raise ValueError(f"DeviceResidentDataset: item {k} has image {tuple(getattr(img, 'shape', ()))} "
                                     f"{getattr(img, 'dtype', type(img))}, the first item's is {(C, H, W)} {idt}")
                if not isinstance(lab, torch.Tensor) or tuple(lab.shape) != lshape or lab.dtype != torch.float32:
                    raise ValueError(f"DeviceResidentDataset: item {k} has labels {tuple(getattr(lab, 'shape', ()))} "
                                     f"{getattr(lab, 'dtype', type(lab))}, the first item's are {lshape} float32")
                imgs[j] = img
                rec = compact_labels(lab)
                records.append(rec)
                counts[pos + j] = rec.shape[0]
                valid[pos + j] = 1
            s0 = rank * chunk + pos
            self._images[s0:s0 + len(batch)].copy_(imgs)
            pos += len(batch)
            batch = next(it, None)
        del it, loader
        recs = torch.cat(records) if records else torch.zeros((0, RECORD_WORDS), dtype=torch.int32)

        if world > 1:
            # images: in-place all-gather of the equal per-rank slot ranges; labels: variable-size, padded to the largest
            flat = self._images.view(torch.uint8).reshape(-1)
            part = chunk * item_bytes
            dist.all_gather_into_tensor(flat, flat[rank * part:(rank + 1) * part], group=self.pg)
            del flat
            meta = torch.cat([valid.to(torch.int64), counts]).to(dev)
            metas = torch.empty((world, 2 * chunk), dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(metas, meta, group=self.pg)
            metas = metas.cpu()
            valid, counts = metas[:, :chunk].reshape(-1).to(torch.uint8), metas[:, chunk:].reshape(-1)
            nrec = [int(metas[r, chunk:].sum()) for r in range(world)]
            check_capacity((sum(nrec) + max(nrec) * world) * RECORD_WORDS * 4, torch.cuda.mem_get_info(dev)[0],
                           self.reserve_bytes)
            pad = torch.zeros((max(nrec), RECORD_WORDS), dtype=torch.int32, device=dev)
            pad[:recs.shape[0]].copy_(recs)
            gathered = torch.empty((world, max(nrec), RECORD_WORDS), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(gathered, pad, group=self.pg)
            del pad
            self._records = torch.cat([gathered[r, :nrec[r]] for r in range(world)]) if sum(nrec) else \
                torch.zeros((1, RECORD_WORDS), dtype=torch.int32, device=dev)
            del gathered
        else:
            check_capacity(recs.numel() * 4, torch.cuda.mem_get_info(dev)[0], self.reserve_bytes)
            self._records = (recs if recs.numel() else torch.zeros((1, RECORD_WORDS), dtype=torch.int32)).to(dev)

        # per slot: record range (empty for None items and padding); sampler index -> slot
        valid = valid[:n_slots].bool()
        counts = counts[:n_slots] * valid
        off = torch.zeros(n_slots + 1, dtype=torch.int64)
        off[1:] = counts.cumsum(0)
        self._rec_off = off.to(dev)
        slots = valid.nonzero().squeeze(1)
        self.num_items = int(slots.numel())
        self.num_dropped = n_items - self.num_items
        if self.num_items == 0:
            raise ValueError("DeviceResidentDataset: every item of the dataset is None")
        if self.num_dropped:
            warnings.warn(f"DeviceResidentDataset: {self.num_dropped} of {n_items} items are None (unreadable) and are "
                          f"left out of every epoch")
        self._slots = slots.to(torch.int32)
        self.samples_per_rank = -(-self.num_items // self.world)
        # whole batches: the kernels of a short last batch never read past the table, whatever size they are asked for
        self._table = torch.zeros(self.num_batches() * self.batch_size, dtype=torch.int32, device=dev)
        self._state = torch.tensor([self.seed, 0, 0], dtype=torch.int64, device=dev)
        self._flags = torch.zeros(4, dtype=torch.int32, device=dev)
        self.nbytes = (self._images.numel() * self._images.element_size() + self._records.numel() * 4 +
                       self._rec_off.numel() * 8 + self._table.numel() * 4)
        self.epoch = None
        torch.cuda.synchronize(dev)

    # ------------------------------------------------------------------ sampling
    def __len__(self) -> int:
        """Items in the store (the dataset's items that are not None)."""
        return self.num_items

    def num_batches(self, epoch: int = 0) -> int:
        return -(-self.samples_per_rank // self.batch_size)

    def batch_sizes(self, epoch: int = 0) -> List[int]:
        full, rest = divmod(self.samples_per_rank, self.batch_size)
        return [self.batch_size] * full + ([rest] if rest else [])

    def epoch_batches(self, epoch: int) -> List[List[int]]:
        """This rank's batches of `epoch` as indices into the non-None items (what the device kernels gather)."""
        return epoch_batches(self.num_items, self.world, self.rank, self.seed, epoch, self.batch_size)

    def begin_epoch(self, epoch: int) -> None:
        """Upload the epoch's index table (the only host-to-device transfer of an epoch) and rewind the batch cursor."""
        idx = torch.tensor([i for b in self.epoch_batches(epoch) for i in b], dtype=torch.int64)
        table = torch.full((self._table.numel(),), int(self._slots[0]), dtype=torch.int32)
        table[:idx.numel()] = self._slots[idx]
        self._table.copy_(table)
        self._state[2].zero_()
        self.epoch = epoch

    # ------------------------------------------------------------------ batch construction
    def next_batch_into(self, images: torch.Tensor, labels: torch.Tensor) -> None:
        """Draw the flips of the next batch of the current epoch and write it into `images` (n, C, H, W) and `labels`
        (n, 6, Sy, Sx), n = this batch's size.  Graph-capturable: nothing is read back to the host."""
        n = images.shape[0]
        C, H, W = self.image_shape
        Sy, Sx = self.grid
        if tuple(images.shape) != (n, C, H, W) or images.dtype != self.image_dtype or not images.is_contiguous() or \
                tuple(labels.shape) != (n, 6, Sy, Sx) or labels.dtype != torch.float32 or not labels.is_contiguous():
            raise ValueError("next_batch_into: output tensors do not match the store")
        lib, st = L.lib(), L.stream()
        L.check(lib.yg_dd_draw(self._state.data_ptr(), self._flags.data_ptr(), self.p_hflip, self.p_vflip, self.rank,
                                self.num_batches(), st))
        L.check(lib.yg_dd_gather_images(self._images.data_ptr(), images.data_ptr(), L.dtype_code(self.image_dtype),
                                        self._table.data_ptr(), self._flags.data_ptr(), self.batch_size, n, C, H, W, st))
        L.check(lib.yg_dd_build_labels(self._table.data_ptr(), self._flags.data_ptr(), self.batch_size,
                                       self._records.data_ptr(), self._rec_off.data_ptr(), n, Sy, Sx, labels.data_ptr(), st))

    def next_batch(self, n: int) -> Tuple[torch.Tensor, torch.Tensor]:
        images = torch.empty((n,) + self.image_shape, dtype=self.image_dtype, device=self.device)
        labels = torch.empty((n, 6) + self.grid, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            self.next_batch_into(images, labels)
        return images, labels

    def batches(self, epoch: int) -> Iterator[Tuple[torch.Tensor, torch.Tensor]]:
        """Eager generator of this rank's `(images, labels)` batches of `epoch` as device tensors."""
        with torch.cuda.device(self.device):
            self.begin_epoch(epoch)
        for n in self.batch_sizes(epoch):
            yield self.next_batch(n)

    def last_flips(self) -> Tuple[bool, bool]:
        """(hflip, vflip) of the batch drawn last (a device read)."""
        f = self._flags.cpu()
        return bool(f[0]), bool(f[1])

    def state(self) -> torch.Tensor:
        """Copy of the device state [seed, flip-draw counter, batch cursor], for `set_state`."""
        return self._state.clone()

    def set_state(self, state: torch.Tensor) -> None:
        self._state.copy_(state)
