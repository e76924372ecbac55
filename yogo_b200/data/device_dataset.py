"""Device-resident training data: the dataset is decoded once into HBM and every batch of every epoch is built on the GPU.

The reference's training loop reads, decodes and collates every image of every epoch on the host (yogo_dataloader.py,
utils.py:49-63); at the step rate of this project that host work, not the GPU, bounds training on real data.  YOGO trains
many epochs over the same images and its only augmentations are the two whole-batch flips, so
``DeviceResidentDataset`` decodes the dataset once (spread over the ranks of a process group, completed with
all-gathers so that every rank holds the full store) and afterwards builds each batch with three kernels
(csrc/input.cu): the flip draw, the image gather + flip and the label build.  They read the epoch's index table and their
own state from device memory, so they run inside the captured training step (``DataParallelTrainer.steps_from_device``)
and the host does no per-step data work.

A store too large for one GPU is sharded instead (``placement``): when the full store does not fit beside the training
reserve but a 1/W shard does, and all ranks run on one host, each rank keeps only the images it decoded, in a buffer of
its own that the other ranks map through CUDA IPC, and the gather kernel reads the other ranks' images over NVLink.  The
batches are bit-identical to the replicated store's.  A sharded store must be released with the collective ``close()``.

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

import socket
import warnings
from ctypes import byref, c_void_p, create_string_buffer
from typing import Callable, Iterator, List, Sequence, Tuple

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


def _rank_ranges(hosts: Sequence) -> str:
    """'ranks 0-3 on host a, 4-7 on host b' for the per-rank host names `hosts`."""
    parts, start = [], 0
    for r in range(1, len(hosts) + 1):
        if r == len(hosts) or hosts[r] != hosts[start]:
            span = f"{start}" if r - 1 == start else f"{start}-{r - 1}"
            parts.append(f"{span} on host {hosts[start]}")
            start = r
    return "ranks " + ", ".join(parts)


def placement(full_bytes: int, shard_bytes: int, free: Sequence[int], reserve: Sequence[int], hosts: Sequence) -> str:
    """Where the images of a store go, from what every rank observed (per rank: `free` device bytes, the `reserve` kept
    for training, `hosts` = (host name, boot id)): 'replicated' when `full_bytes` fit beside the reserve on every rank,
    'sharded' when only `shard_bytes` (a rank's 1/W of the image slots plus the replicated label and index tables) fit
    and every rank runs on one host.  ValueError otherwise, naming both byte counts, the free bytes and why sharding was
    not possible.  Every rank passes the same gathered lists, so every rank takes the same branch."""
    world = len(free)
    available = [f - r for f, r in zip(free, reserve)]
    worst = min(range(world), key=lambda r: available[r])
    if full_bytes <= available[worst]:
        return "replicated"
    if world == 1:
        check_capacity(full_bytes, free[0], reserve[0])
    need = (f"the device-resident dataset needs {full_bytes} bytes ({full_bytes / 2**30:.2f} GiB) but rank {worst} has "
            f"{free[worst]} bytes free ({free[worst] / 2**30:.2f} GiB), of which {reserve[worst]} are kept for training")
    if shard_bytes > available[worst]:
        raise ValueError(f"{need}; a shard over {world} ranks needs {shard_bytes} bytes ({shard_bytes / 2**30:.2f} GiB) "
                         f"per rank, which does not fit either")
    if len(set(hosts)) > 1:
        raise ValueError(f"{need}; a shard over {world} ranks ({shard_bytes} bytes per rank) would fit, but a sharded "
                         f"store needs every rank on one host and there are {_rank_ranges([h[0] for h in hosts])}")
    return "sharded"


def _host_id() -> Tuple[str, str]:
    """(host name, boot id): two processes can map each other's device memory only on the same running host."""
    try:
        with open("/proc/sys/kernel/random/boot_id") as f:
            boot = f.read().strip()
    except OSError:
        boot = ""
    return socket.gethostname(), boot


class _CudaBuffer:
    """`__cuda_array_interface__` of raw device bytes, so that torch.as_tensor gives a (non-owning) uint8 view."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class ShardMemory:
    """This rank's image shard of a sharded store and the peers' shards it has mapped.

    The own shard is its own cudaMalloc allocation (exportable by IPC handle).  Teardown is collective: `close()`
    synchronises, meets the other ranks in a barrier, closes every mapped peer shard, meets them again and only then frees
    the own shard, so no rank frees memory a peer can still read.  A ShardMemory collected without `close()` closes its
    mappings but never frees the own shard (its memory returns at process exit).  `lib`, `barrier` and `synchronize` are
    parameters so that the protocol can be checked with a fake library."""

    def __init__(self, lib, nbytes: int, barrier: Callable[[], None], synchronize: Callable[[], None]):
        self._lib, self._barrier, self._sync = lib, barrier, synchronize
        self.nbytes = int(nbytes)
        self.peers: List[int] = []     # opened peer pointers
        self.shared = False            # every rank exported its handle: peers may map the own shard
        self.closed = True             # nothing to release until the allocation succeeded
        p = c_void_p()
        L.check(lib.yg_dd_shard_alloc(self.nbytes, byref(p)))
        self.ptr = int(p.value)
        self.closed = False

    def export(self) -> bytes:
        buf = create_string_buffer(L.YG_IPC_HANDLE_BYTES)
        L.check(self._lib.yg_dd_shard_export(self.ptr, buf))
        return buf.raw

    def mark_shared(self) -> None:
        """Called on every rank once every rank has exported its handle (the handles are exchanged next): from here on
        the own shard is freed only through the collective `close()`.  Set on all ranks or on none, so the barriers of a
        failed build's cleanup always pair up."""
        self.shared = True

    def open(self, handle: bytes) -> int:
        p = c_void_p()
        L.check(self._lib.yg_dd_shard_open(handle, byref(p)))
        self.peers.append(int(p.value))
        return self.peers[-1]

    def _close_peers(self) -> None:
        while self.peers:
            L.check(self._lib.yg_dd_shard_close(self.peers.pop()))

    def close(self) -> None:
        """Collective: every rank of the store calls it."""
        if self.closed:
            return
        self.closed = True
        self._sync()
        self._barrier()          # no rank still reads a shard
        self._close_peers()
        self._barrier()          # no rank still maps a shard
        L.check(self._lib.yg_dd_shard_free(self.ptr))

    def release_after_failed_build(self) -> None:
        """Free after an exception of the build.  Once the shard is shared (every rank exported, handles exchanged), every
        rank raises together (the build gathers every rank's status), so the barriers of `close` pair up; before that no
        peer can have mapped the shard and it is freed at once."""
        if self.shared:
            self.close()
        else:
            self.closed = True
            L.check(self._lib.yg_dd_shard_free(self.ptr))

    def __del__(self):
        if self.closed:
            return
        self.closed = True
        try:
            self._sync()
            self._close_peers()
        except Exception:
            pass
        warnings.warn("DeviceResidentDataset: a sharded store was collected without close(); its shard "
                      f"({self.nbytes} bytes) stays allocated until the process exits, since a peer may still map it")


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
        self._mem: ShardMemory = None
        self._shard_ptrs = None
        self.sharded = False
        self._closed = False
        with torch.cuda.device(self.device):
            try:
                self._build(dataset, num_workers)
            except BaseException:
                self._images = self._records = self._rec_off = self._slots = self._table = None
                self._state = self._flags = self._shard_ptrs = None
                if self._mem is not None:
                    mem, self._mem = self._mem, None
                    mem.release_after_failed_build()
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
        # images and index tables are known now; label records are checked again once decoded.  The store is
        # replicated when it fits on every rank, else sharded (each rank keeps the `chunk` slots it decodes) if a shard
        # fits and the ranks can map each other's memory.
        full = store_bytes(n_slots, item_bytes, 0, samples, self.batch_size)
        shard = full - (n_slots - chunk) * item_bytes + world * 8
        seen = [(torch.cuda.mem_get_info(dev)[0], self.reserve_bytes, None)]
        if world > 1:
            seen = [None] * world
            dist.all_gather_object(seen, (torch.cuda.mem_get_info(dev)[0], self.reserve_bytes, _host_id()), group=self.pg)
        self.sharded = placement(full, shard, *zip(*seen)) == "sharded"
        if self.sharded:
            pg = self.pg
            self._mem = ShardMemory(L.lib(), chunk * item_bytes, lambda: dist.barrier(group=pg),
                                    lambda: torch.cuda.synchronize(dev))
            self._images = torch.as_tensor(_CudaBuffer(self._mem.ptr, chunk * item_bytes), device=dev).view(idt)
            self._images = self._images.view(chunk, C, H, W)
            self._images.zero_()
            slot0 = 0
        else:
            self._images = torch.zeros((n_slots, C, H, W), dtype=idt, device=dev)
            slot0 = rank * chunk

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
            s0 = slot0 + pos
            self._images[s0:s0 + len(batch)].copy_(imgs)
            pos += len(batch)
            batch = next(it, None)
        del it, loader
        recs = torch.cat(records) if records else torch.zeros((0, RECORD_WORDS), dtype=torch.int32)

        if world > 1:
            # images (replicated): in-place all-gather of the equal per-rank slot ranges; labels: variable-size, padded to
            # the largest
            if not self.sharded:
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
        if self.sharded:
            self._map_shards()
        self.shard_bytes = self._images.numel() * self._images.element_size()
        self.nbytes = (self.shard_bytes + self._records.numel() * 4 + self._rec_off.numel() * 8 + self._table.numel() * 4 +
                       (self._shard_ptrs.numel() * 8 if self.sharded else 0))
        self.epoch = None
        torch.cuda.synchronize(dev)

    def _on_every_rank(self, what: str, fn):
        """`fn()` on every rank; if it raises on any rank, every rank raises (naming each failure) instead of one rank
        raising while the others wait in the next collective.  The status gather is a barrier."""
        out, err = None, None
        try:
            out = fn()
        except Exception as e:
            err = f"{type(e).__name__}: {e}"
        errs = [None] * self.world
        dist.all_gather_object(errs, err, group=self.pg)
        bad = [f"rank {r}: {e}" for r, e in enumerate(errs) if e is not None]
        if bad:
            raise L.YogoB200Error(f"DeviceResidentDataset: {what} failed on " + "; ".join(bad))
        return out

    def _map_shards(self) -> None:
        """Exchange the shards' IPC handles, map every peer's shard and upload the W base pointers.  Each rank's shard is
        complete before its handle leaves (device synchronise), and the final status gather keeps every rank from
        reading before all are mapped."""
        dev, mem = self.device, self._mem

        def export():
            torch.cuda.synchronize(dev)
            return mem.export()

        handle = self._on_every_rank("exporting the shard", export)
        mem.mark_shared()        # every rank reported a handle: on all ranks or, after a raise above, on none
        handles = [None] * self.world
        dist.all_gather_object(handles, handle, group=self.pg)

        def open_peers():
            ptrs = [mem.ptr if r == self.rank else mem.open(h) for r, h in enumerate(handles)]
            self._shard_ptrs = torch.tensor(ptrs, dtype=torch.int64).to(dev)
            torch.cuda.synchronize(dev)

        self._on_every_rank("mapping the peers' shards (a sharded store needs CUDA IPC between the ranks of one host)",
                            open_peers)

    def close(self) -> None:
        """Release the store; afterwards `next_batch_into` and `begin_epoch` raise.  For a sharded store this is
        collective, every rank calls it (before destroy_process_group): device synchronise, barrier, unmap the peers'
        shards, barrier, free the own shard."""
        if self._closed:
            return
        self._closed = True
        self._images = self._records = self._rec_off = self._slots = self._table = None
        self._state = self._flags = self._shard_ptrs = None
        if self._mem is not None:
            mem, self._mem = self._mem, None
            with torch.cuda.device(self.device):
                mem.close()

    def _check_open(self) -> None:
        if self._closed:
            raise L.YogoB200Error("DeviceResidentDataset: the store was closed")

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
        self._check_open()
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
        self._check_open()
        n = images.shape[0]
        C, H, W = self.image_shape
        Sy, Sx = self.grid
        if tuple(images.shape) != (n, C, H, W) or images.dtype != self.image_dtype or not images.is_contiguous() or \
                tuple(labels.shape) != (n, 6, Sy, Sx) or labels.dtype != torch.float32 or not labels.is_contiguous():
            raise ValueError("next_batch_into: output tensors do not match the store")
        lib, st = L.lib(), L.stream()
        L.check(lib.yg_dd_draw(self._state.data_ptr(), self._flags.data_ptr(), self.p_hflip, self.p_vflip, self.rank,
                                self.num_batches(), st))
        if self.sharded:
            L.check(lib.yg_dd_gather_images_peers(self._shard_ptrs.data_ptr(), self._images.shape[0], images.data_ptr(),
                                                  L.dtype_code(self.image_dtype), self._table.data_ptr(),
                                                  self._flags.data_ptr(), self.batch_size, n, C, H, W, st))
        else:
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
