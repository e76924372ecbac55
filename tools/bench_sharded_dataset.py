"""Sharded device-resident store (yogo_b200.data.DeviceResidentDataset over the ranks of one host) against the
replicated store.  Run under torchrun, one rank per GPU (2, 4 or 8 GPUs of one box):

    python -m torch.distributed.run --nproc-per-node 8 tools/bench_sharded_dataset.py

base_model, batch 64 per rank, bf16, 772x1032 uint8, a store larger than L2 (--items).  Rank 0 prints JSON lines (each
with the GPU's name, power limit and SM clocks) and appends them to --out:
  (a) the gather kernel alone, sharded (yg_dd_gather_images_peers over the peers' shards) against replicated
      (yg_dd_gather_images from the local store), alternated in one process: us per batch, bytes read from peers per rank
      (the batch's images that other ranks own) and GB/s of those bytes against NVLINK_GBPS;
  (b) steps_from_device step time from the sharded store against the replicated store of the same items, alternated
      epoch windows (as step_compare of tools/bench_device_dataset.py), medians and ranges;
  (c) build time and device bytes per rank of both placements.
With one process (no torchrun) it records only the local comparison the kernel choice rests on: the peer gather with
W = 8 pointers into ONE local store against yg_dd_gather_images on the same store."""
import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import yogo_b200  # noqa: E402
from tools import synth as O  # noqa: E402
from tools.bench_device_dataset import FLIPS, NC, H, W, make_dataset  # noqa: E402
from tools.bench_match import gpu_info  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402
from yogo_b200.data import DeviceResidentDataset  # noqa: E402
from yogo_b200.data.device_dataset import store_bytes  # noqa: E402
from yogo_b200.train import DataParallelTrainer  # noqa: E402

B = 64
# NVIDIA's HGX B200 data sheet: 1.8 TB/s of NVLink bandwidth per GPU, i.e. 900 GB/s per direction
NVLINK_GBPS = 900.0


def timed(fn, iters):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3   # us


def gather_fns(dd_r, dd_s, out, local_shards=None):
    """(draw, replicated gather, peer gather) launches; the peer gather reads `dd_s`'s shards, or `local_shards` =
    (pointer tensor, items per shard) into dd_r's store."""
    lib, st = L.lib(), L.stream()
    C, Hh, Ww = dd_r.image_shape
    code = L.dtype_code(dd_r.image_dtype)
    dd_r.begin_epoch(0)
    if dd_s is not None:
        dd_s.begin_epoch(0)
    ptrs, items = local_shards if local_shards is not None else (dd_s._shard_ptrs, dd_s._images.shape[0])
    src = dd_r if local_shards is not None else dd_s

    def draw(dd):
        L.check(lib.yg_dd_draw(dd._state.data_ptr(), dd._flags.data_ptr(), 0.5, 0.5, 0, dd.num_batches(), st))

    def rep():
        draw(dd_r)
        L.check(lib.yg_dd_gather_images(dd_r._images.data_ptr(), out.data_ptr(), code, dd_r._table.data_ptr(),
                                        dd_r._flags.data_ptr(), B, B, C, Hh, Ww, st))

    def peers():
        draw(src)
        L.check(lib.yg_dd_gather_images_peers(ptrs.data_ptr(), items, out.data_ptr(), code, src._table.data_ptr(),
                                              src._flags.data_ptr(), B, B, C, Hh, Ww, st))

    return (lambda: draw(dd_r)), rep, peers


def kernel_compare(dd_r, dd_s, rounds, iters, local_shards=None):
    out = torch.empty((B,) + dd_r.image_shape, dtype=dd_r.image_dtype, device=dd_r.device)
    draw, rep, peers = gather_fns(dd_r, dd_s, out, local_shards)
    d = timed(draw, iters)
    r_us, p_us = [], []
    for _ in range(rounds):
        r_us.append(timed(rep, iters) - d)
        p_us.append(timed(peers, iters) - d)
    return sorted(r_us), sorted(p_us)


def remote_bytes(dd_s, epoch=0):
    """Mean bytes per batch of this rank's batches that other ranks own."""
    chunk = dd_s._images.shape[0]
    item = dd_s.shard_bytes // chunk
    slots = dd_s._slots
    tot, nb = 0, 0
    for b in dd_s.epoch_batches(epoch):
        if len(b) == B:
            s = slots[torch.tensor(b)]
            tot += int(((s // chunk) != dd_s.rank).sum()) * item
            nb += 1
    return tot / max(nb, 1)


def step_compare(dd_a, dd_b, rounds):
    """Alternated epoch windows of steps_from_device from two stores of the same items (graph mode)."""
    dev = dd_a.device
    trs = []
    for dd in (dd_a, dd_b):
        torch.manual_seed(0)
        net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, NC).to(dev)
        net.compute_dtype = torch.bfloat16
        net.train()
        tr = DataParallelTrainer(net, yogo_b200.YOGOLoss().to(dev), total_steps=100000)
        x, y = next(dd.batches(0))
        tr.enable_cuda_graph(x, y)
        for _ in tr.steps_from_device(dd, 0):
            pass
        trs.append(tr)
    torch.cuda.synchronize()
    ms = ([], [])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for r in range(rounds):
        for k, (tr, dd) in enumerate(zip(trs, (dd_a, dd_b))):
            ev[0].record()
            for _ in tr.steps_from_device(dd, r + 1):
                pass
            ev[1].record()
            torch.cuda.synchronize()
            ms[k].append(ev[0].elapsed_time(ev[1]) / dd.num_batches(r + 1))
    return [sorted(m) for m in ms]


def build(ds, dev, reserve=None):
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    t0 = time.perf_counter()
    kw = {} if reserve is None else {"reserve_bytes": reserve}
    dd = DeviceResidentDataset(ds, B, FLIPS, device=dev, num_workers=8, **kw)
    torch.cuda.synchronize()
    return dd, time.perf_counter() - t0


def med(xs):
    return xs[len(xs) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sharded_dataset_bench.jsonl"))
    ap.add_argument("--items", type=int, default=2048, help="items of the store (1.6 GB at 772x1032 uint8)")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--step-rounds", type=int, default=6)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    rank = dist.get_rank() if world > 1 else 0
    info = gpu_info()
    ds = make_dataset(args.items)
    rows = []
    dd_r, t_r = build(ds, dev)
    common = {"world": world, "B": B, "shape": [1, H, W], "items": args.items}
    if world == 1:
        # local comparison: 8 "shards" that are slices of one local store
        k = 8
        items = -(-dd_r._images.shape[0] // k)
        ptrs = torch.tensor([dd_r._images[min(i * items, dd_r._images.shape[0] - 1)].data_ptr() for i in range(k)],
                            dtype=torch.int64, device=dev)
        r_us, p_us = kernel_compare(dd_r, None, args.rounds, args.iters, (ptrs, items))
        nbytes = 2 * B * H * W
        rows.append({**common, "case": "gather, local store: yg_dd_gather_images vs yg_dd_gather_images_peers (8 pointers)",
                     "replicated_us_median": med(r_us), "peers_us_median": med(p_us), "replicated_us": r_us,
                     "peers_us": p_us, "bytes": nbytes, "replicated_GBps": nbytes / med(r_us) / 1e3,
                     "peers_GBps": nbytes / med(p_us) / 1e3,
                     "note": "alternated rounds in one process, draw launch subtracted; bytes = read once + written once"})
    else:
        chunk = -(-args.items // world)
        full = store_bytes(chunk * world, H * W, 0, chunk, B)
        shard = full - (chunk * world - chunk) * H * W + world * 8
        reserve = torch.cuda.mem_get_info(dev)[0] - (full + shard) // 2   # room for a shard, not for the full store
        dd_s, t_s = build(ds, dev, reserve)
        assert dd_s.sharded and not dd_r.sharded
        r_us, p_us = kernel_compare(dd_r, dd_s, args.rounds, args.iters)
        rb = remote_bytes(dd_s)
        rows.append({**common, "case": "gather kernel alone: sharded (peers) vs replicated",
                     "replicated_us_median": med(r_us), "sharded_us_median": med(p_us),
                     "replicated_us": r_us, "sharded_us": p_us, "remote_bytes_per_rank": rb,
                     "remote_GBps": rb / med(p_us) / 1e3, "nvlink_GBps_per_direction_datasheet": NVLINK_GBPS,
                     "frac_of_nvlink": rb / med(p_us) / 1e3 / NVLINK_GBPS,
                     "note": "rank 0; every rank gathers at once; alternated rounds; draw launch subtracted"})
        s_ms, r_ms = step_compare(dd_s, dd_r, args.step_rounds)
        rows.append({**common, "case": "step base_model b64 bf16: steps_from_device sharded vs replicated",
                     "sharded_ms_median": med(s_ms), "replicated_ms_median": med(r_ms),
                     "sharded_ms_range": [s_ms[0], s_ms[-1]], "replicated_ms_range": [r_ms[0], r_ms[-1]],
                     "sharded_ms": s_ms, "replicated_ms": r_ms,
                     "note": "epoch windows alternate in one process; each includes the epoch's index-table upload"})
        rows.append({**common, "case": "build", "replicated_s": t_r, "sharded_s": t_s,
                     "replicated_nbytes_per_rank": dd_r.nbytes, "sharded_nbytes_per_rank": dd_s.nbytes,
                     "sharded_shard_bytes": dd_s.shard_bytes,
                     "note": "in-memory uint8 dataset, 300 labelled cells per image, DataLoader with 8 workers"})
        dd_s.close()
    dd_r.close()
    if rank == 0:
        with open(args.out, "a") as f:
            for r in rows:
                line = json.dumps({**info, **r})
                print(line)
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
