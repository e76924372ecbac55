"""Multi-rank check of a sharded yogo_b200.data.DeviceResidentDataset (run under torchrun, one rank per GPU of one host):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 \
        tests/ddp_sharded_dataset_check.py

 (1) a reserve that leaves room for a shard but not for the full store gives a sharded store on every rank, holding 1/W
     of the replicated store's image bytes;
 (2) for two epochs every batch of the sharded store equals, bit for bit, the replicated store's batch (same dataset,
     seed and transforms) and collate_batch_robust + flip_batch of the sampler's items;
 (3) steps_from_device in graph mode: the static input slot holds the same bytes at every replay from either store, and
     losses and parameters agree within the spread of two runs from the replicated store;
 (4) close() on every rank returns the shard's device memory, then destroy_process_group.
tests/test_sharded_dataset.py launches this file on 2 GPUs and on all GPUs of the box (up to 8).
"""
import gc
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
from torch.utils.data import Dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import yogo_b200  # noqa: E402
from tools.synth import ANCHOR_H, ANCHOR_W  # noqa: E402
from yogo_b200.data import (DeviceResidentDataset, MultiArgSequential, RandomHorizontalFlipWithBBs,  # noqa: E402
                            RandomVerticalFlipWithBBs, collate_batch_robust, flip_batch)
from yogo_b200.data.device_dataset import store_bytes  # noqa: E402
from yogo_b200.train import DataParallelTrainer  # noqa: E402

H, W = 256, 384         # ~96 KB per image: the store (~250 MB) dwarfs the allocation granularity
N_ITEMS = 2603          # not a multiple of any world size up to 8
BS = 32
DROPPED = 7


class Synthetic(Dataset):
    def __init__(self, n, Sy, Sx):
        self.n, self.grid = n, (Sy, Sx)

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        if i == DROPPED:
            return None
        g = torch.Generator().manual_seed(1000 + i)
        img = torch.randint(0, 256, (1, H, W), dtype=torch.uint8, generator=g)
        lab = torch.zeros((6,) + self.grid)
        cells = torch.randperm(self.grid[0] * self.grid[1], generator=g)[:5]
        lo = torch.rand(2, 5, generator=g) * 0.8
        rows = torch.cat([torch.ones(1, 5), lo, lo + 0.05 + 0.1 * torch.rand(2, 5, generator=g),
                          torch.randint(0, 4, (1, 5), generator=g).float()])
        lab.view(6, -1)[:, cells] = rows
        return img, lab


def sharding_reserve(dev, world, n, item_bytes):
    """A reserve that leaves room for a shard plus 64 MiB, which is less than the full store."""
    chunk = -(-n // world)
    full = store_bytes(chunk * world, item_bytes, 0, chunk, BS)
    shard = full - (chunk * world - chunk) * item_bytes + world * 8
    assert shard + (64 << 20) < full, (shard, full)
    return torch.cuda.mem_get_info(dev)[0] - shard - (64 << 20)


def train(dd, sd, keeps, dev, epochs=2):
    net = yogo_b200.YOGO((H, W), ANCHOR_W, ANCHOR_H, 4)
    net.load_state_dict(sd)
    net = net.to(dev)
    net.compute_dtype = torch.bfloat16
    net.train()
    runner = net._get_runner()
    runner.drop_keep_override = keeps
    tr = DataParallelTrainer(net, yogo_b200.YOGOLoss().to(dev), total_steps=200)
    x0, y0 = next(dd.batches(0))
    tr.enable_cuda_graph(x0, y0)
    losses, slots = [], []
    for e in range(epochs):
        gen = tr.steps_from_device(dd, e)
        for n in dd.batch_sizes(e):
            runner.drop_keep_override = {i: k[:n] for i, k in keeps.items()}
            losses.append(next(gen).item())
            if n == dd.batch_size:
                slots.append([t.clone() for t in tr.static_inputs(0)])
        assert next(gen, None) is None
    p = tr.flat_p.cpu().numpy()
    del tr, net, runner
    return np.array(losses), p, slots


def train_and_compare(dd_s, dd_r, sd, dev):
    g = torch.Generator().manual_seed(5)
    keeps = {i: (torch.rand(BS, c, generator=g) > 0.1).float().to(dev) for i, c in ((1, 32), (2, 64), (3, 128))}
    # every run starts from the same flip-draw state, so the two replicated runs differ only by run-to-run noise
    state = dd_r.state()
    assert torch.equal(state, dd_s.state())
    dd_s.set_state(state)
    s_losses, s_p, s_slots = train(dd_s, sd, keeps, dev)
    dd_r.set_state(state)
    r1_losses, r1_p, r1_slots = train(dd_r, sd, keeps, dev)
    dd_r.set_state(state)
    r2_losses, r2_p, r2_slots = train(dd_r, sd, keeps, dev)
    assert len(s_slots) == len(r1_slots) > 0
    for a, b, c in zip(s_slots, r1_slots, r2_slots):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))
        assert torch.equal(b[0], c[0]) and torch.equal(b[1].view(torch.int32), c[1].view(torch.int32))
    assert np.isfinite(s_losses).all()
    spread_l, spread_p = np.abs(r1_losses - r2_losses).max(), np.abs(r1_p - r2_p).max()
    assert np.abs(s_losses - r1_losses).max() <= max(2 * spread_l, 1e-6 * np.abs(r1_losses).max()), (s_losses, r1_losses)
    assert np.abs(s_p - r1_p).max() <= max(2 * spread_p, 1e-6 * np.abs(r1_p).max()), (np.abs(s_p - r1_p).max(), spread_p)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    warm = torch.ones(1, device=dev)
    dist.all_reduce(warm)
    torch.manual_seed(0)
    net = yogo_b200.YOGO((H, W), ANCHOR_W, ANCHOR_H, 4)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.1)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    Sx, Sy = net.get_grid_size()
    ds = Synthetic(N_ITEMS, Sy, Sx)
    tr = MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5))
    item_bytes = H * W

    # (1) placement
    dd_r = DeviceResidentDataset(ds, BS, tr, device=dev, seed=3)
    dd_s = DeviceResidentDataset(ds, BS, tr, device=dev, seed=3, reserve_bytes=sharding_reserve(dev, world, N_ITEMS, item_bytes))
    assert not dd_r.sharded and dd_s.sharded, (dd_r.sharded, dd_s.sharded)
    chunk = -(-N_ITEMS // world)
    assert dd_s.shard_bytes == chunk * item_bytes and dd_r.shard_bytes == world * chunk * item_bytes
    assert len(dd_s) == len(dd_r) == N_ITEMS - 1 and dd_s.num_dropped == 1

    # (2) batches: sharded == replicated == collate + flip_batch
    valid = [i for i in range(N_ITEMS) if i != DROPPED]
    for e in (0, 1):
        batches = dd_s.epoch_batches(e)
        assert batches == dd_r.epoch_batches(e)
        for (xs, ys), (xr, yr), idx in zip(dd_s.batches(e), dd_r.batches(e), batches):
            h, v = dd_s.last_flips()
            assert (h, v) == dd_r.last_flips()
            x, y = collate_batch_robust([ds[valid[i]] for i in idx], device=dev)
            x, y = flip_batch(x, y, h, v)
            assert torch.equal(xs, xr) and torch.equal(xs, x), (rank, e, idx)
            assert torch.equal(ys.view(torch.int32), yr.view(torch.int32)) and torch.equal(ys.view(torch.int32), y.view(torch.int32))

    # (3) training in graph mode from either store
    train_and_compare(dd_s, dd_r, sd, dev)

    # (4) close: the shard's memory comes back
    dd_r.close()
    del dd_r
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free_before = torch.cuda.mem_get_info(dev)[0]
    dd_s.close()
    try:
        dd_s.next_batch(BS)
        raise AssertionError("next_batch after close did not raise")
    except yogo_b200._lib.YogoB200Error:
        pass
    del dd_s
    gc.collect()
    torch.cuda.empty_cache()
    freed = torch.cuda.mem_get_info(dev)[0] - free_before
    assert freed >= chunk * item_bytes, (rank, freed, chunk * item_bytes)
    # a new sharded store after the first was closed: build and close leave free memory where it was
    dist.barrier()
    free0 = torch.cuda.mem_get_info(dev)[0]
    dd = DeviceResidentDataset(ds, BS, tr, device=dev, seed=3, reserve_bytes=sharding_reserve(dev, world, N_ITEMS, item_bytes))
    assert dd.sharded
    assert free0 - torch.cuda.mem_get_info(dev)[0] >= dd.shard_bytes
    dd.close()
    del dd
    gc.collect()
    torch.cuda.empty_cache()
    dist.barrier()
    free1 = torch.cuda.mem_get_info(dev)[0]
    assert free1 >= free0 - (8 << 20), (rank, free0, free1)
    dist.barrier()
    if rank == 0:
        print("ddp_sharded_dataset_check ok")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
