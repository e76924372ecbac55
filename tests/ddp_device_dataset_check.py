"""Multi-rank check of yogo_b200.data.DeviceResidentDataset (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29537 \
        tests/ddp_device_dataset_check.py

 (1) every item is decoded by exactly one rank (a wrapping dataset records what it decoded),
 (2) the stores are identical on every rank (checksums of the images and label records),
 (3) each rank's batches are those of its own DistributedSampler shard, built as collate + flip_batch would build them.
tests/test_device_dataset.py::test_multi_rank_store_and_shards launches this file when the box has >= 2 GPUs.
"""
import os
import sys

import torch
import torch.distributed as dist
from torch.utils.data import Dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from yogo_b200.data import (DeviceResidentDataset, MultiArgSequential, RandomHorizontalFlipWithBBs,  # noqa: E402
                            RandomVerticalFlipWithBBs, collate_batch_robust, flip_batch)


class Counting(Dataset):
    def __init__(self, n, C, H, W, Sy, Sx):
        self.n, self.shape, self.grid = n, (C, H, W), (Sy, Sx)
        self.decoded = []

    def __len__(self):
        return self.n

    def item(self, i):
        g = torch.Generator().manual_seed(1000 + i)
        img = torch.randint(0, 256, self.shape, dtype=torch.uint8, generator=g)
        lab = torch.zeros((6,) + self.grid)
        cells = torch.randperm(self.grid[0] * self.grid[1], generator=g)[:5]
        lab.view(6, -1)[:, cells] = torch.rand(6, 5, generator=g)
        return None if i == 7 else (img, lab)

    def __getitem__(self, i):
        self.decoded.append(int(i))
        return self.item(i)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    n = 53
    ds = Counting(n, 1, 40, 64, 5, 8)
    tr = MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5))
    dd = DeviceResidentDataset(ds, 4, tr, device=dev, seed=3, num_workers=0)

    decoded = [None] * world
    dist.all_gather_object(decoded, ds.decoded)
    flat = sorted(i for d in decoded for i in d)
    assert flat == list(range(n)), flat

    sums = torch.stack([dd._images.double().sum(), dd._records.double().sum(), (dd._images.view(-1)[::7].double() *
                        torch.arange(dd._images.numel() // 7 + (dd._images.numel() % 7 > 0), device=dev).double()).sum()])
    allsums = [torch.empty_like(sums) for _ in range(world)]
    dist.all_gather(allsums, sums)
    assert all(torch.equal(allsums[0], s) for s in allsums), allsums
    assert len(dd) == n - 1 and dd.num_dropped == 1

    valid = [i for i in range(n) if i != 7]
    for e in (0, 1):
        batches = dd.epoch_batches(e)
        for (img, lab), idx in zip(dd.batches(e), batches):
            h, v = dd.last_flips()
            x, y = collate_batch_robust([ds.item(valid[i]) for i in idx], device=dev)
            x, y = flip_batch(x, y, h, v)
            assert torch.equal(img, x) and torch.equal(lab.view(torch.int32), y.view(torch.int32)), (rank, e, idx)
    dist.barrier()
    if rank == 0:
        print("ddp_device_dataset_check ok")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
