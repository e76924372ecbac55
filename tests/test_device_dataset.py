"""yogo_b200.data.DeviceResidentDataset and DataParallelTrainer.steps_from_device: the sampler contract and the argument
checks on the CPU; on a B200 the batches built on the device against collate + flip_batch of the same items, the flip
draws, training through the device path against training from host batches, guard bands and the error paths."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from torch.utils.data import Dataset, DistributedSampler

from yogo_b200.data import (DualInputId, ImageTransformLabelIdentity, MultiArgSequential, RandomHorizontalFlipWithBBs,
                            RandomVerticalFlipWithBBs)
from yogo_b200.data.device_dataset import (RECORD_WORDS, check_capacity, compact_labels, epoch_batches,
                                           flip_probabilities, store_bytes)

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------- CPU: sampling, transforms, capacity
class _Range(Dataset):
    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n

    def __getitem__(self, i):
        return i


@pytest.mark.parametrize("n,world,rank,seed,epoch,bs", [
    (100, 1, 0, 0, 0, 8), (100, 1, 0, 0, 3, 8), (100, 4, 2, 7, 1, 5), (37, 3, 0, 1, 2, 4), (37, 3, 2, 1, 2, 4),
    (2, 4, 3, 0, 0, 2),      # n < world: the sampler pads by repeating items
    (10, 3, 1, 5, 4, 64),    # n % world != 0 and n < batch_size
    (65, 1, 0, 0, 0, 64),    # ragged last batch of one item
])
def test_epoch_batches_are_the_distributed_sampler_in_batches(n, world, rank, seed, epoch, bs):
    ref = DistributedSampler(_Range(n), num_replicas=world, rank=rank, shuffle=True, seed=seed, drop_last=False)
    ref.set_epoch(epoch)
    idx = list(ref)
    got = epoch_batches(n, world, rank, seed, epoch, bs)
    assert got == [idx[i:i + bs] for i in range(0, len(idx), bs)]
    assert all(len(b) == bs for b in got[:-1]) and 0 < len(got[-1]) <= bs
    assert epoch_batches(n, world, rank, seed, epoch + 1, bs) != got or n <= 2


def test_transforms_read_the_flip_modules_and_reject_others():
    assert flip_probabilities(None) == (0.0, 0.0)
    assert flip_probabilities(MultiArgSequential()) == (0.0, 0.0)
    assert flip_probabilities(MultiArgSequential(RandomHorizontalFlipWithBBs(0.3), RandomVerticalFlipWithBBs(0.7))) == (0.3, 0.7)
    assert flip_probabilities(MultiArgSequential(RandomVerticalFlipWithBBs(0.25), DualInputId())) == (0.0, 0.25)
    assert flip_probabilities(RandomHorizontalFlipWithBBs(1.0)) == (1.0, 0.0)
    with pytest.raises(NotImplementedError, match="ImageTransformLabelIdentity"):
        flip_probabilities(MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), ImageTransformLabelIdentity(torch.nn.Identity())))
    with pytest.raises(NotImplementedError, match="RandomHorizontalFlipWithBBs"):
        flip_probabilities(MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomHorizontalFlipWithBBs(0.5)))


def test_capacity_check_names_the_byte_count():
    need = store_bytes(1000, 772 * 1032, 50_000, 1000, 64)
    assert need == 1000 * 772 * 1032 + 50_000 * RECORD_WORDS * 4 + 1001 * 8 + 1024 * 4
    check_capacity(need, need + 10, reserve=10)
    with pytest.raises(ValueError, match=str(need)):
        check_capacity(need, need + 9, reserve=10)
    with pytest.raises(ValueError, match=str(need)):
        check_capacity(need, 180 << 30, reserve=(180 << 30) - need + 1)


def test_compact_labels_keep_every_nonzero_cell():
    lab = torch.zeros(6, 3, 5)
    lab[:, 1, 2] = torch.tensor([1.0, 0.1, 0.2, 0.3, 0.4, 2.0])
    lab[3, 2, 4] = -0.0                     # a non-zero bit pattern is a labelled cell
    rec = compact_labels(lab)
    assert rec.shape == (2, RECORD_WORDS)
    assert rec[:, 0].tolist() == [1 * 5 + 2, 2 * 5 + 4]
    assert torch.equal(rec[0, 1:7], lab[:, 1, 2].view(torch.int32))
    assert rec[1, 4].item() == torch.tensor(-0.0).view(torch.int32).item()


# ----------------------------------------------------------------------------- GPU
class ListDataset(Dataset):
    def __init__(self, items):
        self.items = items

    def __len__(self):
        return len(self.items)

    def __getitem__(self, i):
        return self.items[i]


def _labels(n, Sy, Sx, seed, k=12, collide=False):
    from yogo_b200.data import format_labels_batch
    g = torch.Generator().manual_seed(seed)
    lists = []
    for _ in range(n):
        c = torch.rand(k, 2, generator=g) * 0.9 + 0.05
        wh = torch.rand(k, 2, generator=g) * 0.05 + 0.01
        rows = torch.cat([torch.randint(0, 4, (k, 1), generator=g).float(), c - wh / 2, c + wh / 2], 1)
        if collide:   # two boxes centred in the same cell: the later one wins, as in the reference's Python loop
            rows = torch.cat([rows, rows[:1] + torch.tensor([[1.0, 0.001, 0.001, 0.001, 0.001]])])
        lists.append(rows)
    return format_labels_batch(lists, Sx, Sy, device=DEV).cpu()


def _dataset(n, C, H, W, Sy, Sx, dtype=torch.uint8, seed=0, nones=(), collide=False):
    g = torch.Generator().manual_seed(seed)
    if dtype == torch.uint8:
        imgs = torch.randint(0, 256, (n, C, H, W), dtype=torch.uint8, generator=g)
    else:
        imgs = torch.rand((n, C, H, W), generator=g)
    labs = _labels(n, Sy, Sx, seed + 1, collide=collide)
    return ListDataset([None if i in nones else (imgs[i].clone(), labs[i].clone()) for i in range(n)])


def _expected(ds, valid, idx, h, v):
    from yogo_b200.data import collate_batch_robust, flip_batch
    x, y = collate_batch_robust([ds[valid[i]] for i in idx], device=DEV)
    return flip_batch(x, y, h, v)


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


def _check_batches(ds, bs, transforms, epochs=(0, 1), seed=0):
    from yogo_b200.data import DeviceResidentDataset
    dd = DeviceResidentDataset(ds, bs, transforms, device=DEV, seed=seed)
    valid = [i for i in range(len(ds)) if ds[i] is not None]
    assert len(dd) == len(valid) and dd.num_dropped == len(ds) - len(valid)
    seen = set()
    for e in epochs:
        batches = dd.epoch_batches(e)
        assert dd.num_batches(e) == len(batches)
        got = 0
        for (img, lab), idx in zip(dd.batches(e), batches):
            h, v = dd.last_flips()
            seen.add((h, v))
            ei, el = _expected(ds, valid, idx, h, v)
            assert _same(img, ei), (e, idx, h, v)
            assert _same(lab, el), (e, idx, h, v)
            got += 1
        assert got == len(batches)
    return dd, seen


@pytest.mark.gpu
def test_batches_bit_identical_grayscale_with_colliding_labels_and_dropped_items():
    ds = _dataset(45, 1, 64, 96, 6, 9, nones=(3, 17), collide=True)
    with pytest.warns(UserWarning, match="2 of 45"):
        _, seen = _check_batches(ds, 8, MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5)))
    assert len(seen) > 1
    _, seen = _check_batches(_dataset(20, 1, 64, 96, 6, 9, seed=5), 8,
                             MultiArgSequential(RandomHorizontalFlipWithBBs(1.0), RandomVerticalFlipWithBBs(1.0)))
    assert seen == {(True, True)}
    _, seen = _check_batches(_dataset(20, 1, 64, 96, 6, 9, seed=6), 8, None)
    assert seen == {(False, False)}


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,W,dtype", [(3, 40, 48, torch.uint8), (1, 33, 100, torch.uint8), (1, 31, 57, torch.uint8),
                                         (3, 24, 40, torch.float32), (1, 24, 37, torch.float32)])
def test_batches_bit_identical_rgb_odd_widths_fp32(C, H, W, dtype):
    ds = _dataset(23, C, H, W, 5, 7, dtype=dtype, seed=W)
    _check_batches(ds, 6, MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5)), seed=W)


@pytest.mark.gpu
def test_batches_bit_identical_full_size_images():
    ds = _dataset(5, 1, 772, 1032, 97, 129, seed=11)
    _check_batches(ds, 2, MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5)), seed=3)


def _draws(p_h, p_v, n, seed):
    from yogo_b200 import _lib as L
    st = torch.tensor([seed, 0, 0], dtype=torch.int64, device=DEV)
    hist = torch.zeros(n, 4, dtype=torch.int32, device=DEV)
    for i in range(n):
        L.check(L.lib().yg_dd_draw(st.data_ptr(), hist[i].data_ptr(), p_h, p_v, 0, 7, L.stream()))
    hist = hist.cpu()
    assert hist[:, 2].tolist() == [i % 7 for i in range(n)]
    return hist[:, 0].numpy(), hist[:, 1].numpy()


@pytest.mark.gpu
def test_flip_draws():
    n = 4000
    for p in (0.3, 0.5):
        h, v = _draws(p, p, n, seed=1)
        sigma = (p * (1 - p) / n) ** 0.5
        assert abs(h.mean() - p) < 5 * sigma and abs(v.mean() - p) < 5 * sigma, (p, h.mean(), v.mean())
        assert abs(np.corrcoef(h, v)[0, 1]) < 5 / n ** 0.5
    h, v = _draws(0.0, 1.0, 1000, seed=2)
    assert not h.any() and v.all()
    h2, v2 = _draws(0.5, 0.5, 200, seed=9)
    h3, v3 = _draws(0.5, 0.5, 200, seed=9)
    assert np.array_equal(h2, h3) and np.array_equal(v2, v3)
    h4, _ = _draws(0.5, 0.5, 200, seed=10)
    assert not np.array_equal(h2, h4)

    # graph replays draw fresh flips: the same sequence as the eager draws of the same seed
    from yogo_b200.data import DeviceResidentDataset
    ds = _dataset(8, 1, 16, 32, 3, 4, seed=2)
    tr = MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5))
    dd = DeviceResidentDataset(ds, 4, tr, device=DEV, seed=9)
    dd.begin_epoch(0)
    x = torch.empty((4, 1, 16, 32), dtype=torch.uint8, device=DEV)
    y = torch.empty((4, 6, 3, 4), dtype=torch.float32, device=DEV)
    dd.next_batch_into(x, y)
    torch.cuda.synchronize()
    dd.set_state(torch.tensor([9, 0, 0], dtype=torch.int64))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dd.next_batch_into(x, y)
    flips = []
    for _ in range(200):
        g.replay()
        flips.append(dd.last_flips())
    assert [f[0] for f in flips] == h2.astype(bool).tolist() and [f[1] for f in flips] == v2.astype(bool).tolist()


@pytest.mark.gpu
def test_guard_bands_of_the_new_kernels():
    from yogo_b200.data import DeviceResidentDataset
    for C, H, W, dt in ((1, 20, 64, torch.uint8), (3, 13, 21, torch.uint8), (1, 9, 12, torch.float32), (3, 7, 9, torch.float32)):
        ds = _dataset(11, C, H, W, 4, 5, dtype=dt, seed=H)
        dd = DeviceResidentDataset(ds, 4, MultiArgSequential(RandomHorizontalFlipWithBBs(1.0), RandomVerticalFlipWithBBs(1.0)),
                                   device=DEV)
        dd.begin_epoch(0)
        valid = list(range(11))
        for n, idx in zip(dd.batch_sizes(0), dd.epoch_batches(0)):
            pad = 64
            fill = 0xA5 if dt == torch.uint8 else float("nan")
            ibuf = torch.full((2 * pad + n * C * H * W,), fill, dtype=dt, device=DEV)
            lbuf = torch.full((2 * pad + n * 6 * 20,), float("nan"), dtype=torch.float32, device=DEV)
            x = ibuf[pad:pad + n * C * H * W].view(n, C, H, W)
            y = lbuf[pad:pad + n * 120].view(n, 6, 4, 5)
            dd.next_batch_into(x, y)
            ei, el = _expected(ds, valid, idx, True, True)
            assert _same(x, ei) and _same(y, el)
            for m in (ibuf[:pad], ibuf[-pad:]):
                assert (m == 0xA5).all() if dt == torch.uint8 else m.isnan().all()
            assert lbuf[:pad].isnan().all() and lbuf[-pad:].isnan().all()


@pytest.mark.gpu
def test_errors_raise_and_free_what_was_allocated():
    from yogo_b200.data import DeviceResidentDataset
    ds = _dataset(10, 1, 32, 48, 4, 6, seed=1)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    with pytest.raises(NotImplementedError, match="ImageTransformLabelIdentity"):
        DeviceResidentDataset(ds, 4, MultiArgSequential(ImageTransformLabelIdentity(torch.nn.Identity())), device=DEV)
    assert torch.cuda.memory_allocated(DEV) == base
    free = torch.cuda.mem_get_info(DEV)[0]
    with pytest.raises(ValueError, match=r"needs \d+ bytes"):
        DeviceResidentDataset(ds, 4, device=DEV, reserve_bytes=free)
    assert torch.cuda.memory_allocated(DEV) == base

    bad_img = ListDataset(list(ds.items[:6]) + [(torch.zeros(1, 32, 40, dtype=torch.uint8), ds.items[6][1])] + list(ds.items[7:]))
    bad_dt = ListDataset(list(ds.items[:5]) + [(ds.items[5][0].float(), ds.items[5][1])] + list(ds.items[6:]))
    bad_lab = ListDataset(list(ds.items[:8]) + [(ds.items[8][0], torch.zeros(6, 4, 5))] + list(ds.items[9:]))
    for bad, k in ((bad_img, 6), (bad_dt, 5), (bad_lab, 8)):
        with pytest.raises(ValueError, match=f"item {k} "):
            DeviceResidentDataset(bad, 4, device=DEV)
        torch.cuda.synchronize()
        assert torch.cuda.memory_allocated(DEV) == base, k
    with pytest.raises(ValueError, match=r"\(6, Sy, Sx\)"):
        DeviceResidentDataset(ListDataset([(ds.items[0][0], torch.zeros(5, 4, 6))]), 4, device=DEV)
    assert torch.cuda.memory_allocated(DEV) == base


# ----------------------------------------------------------------------------- training equivalence
def _train(mode, ds, dd_or_batches, sd, keeps, epochs, graph):
    import yogo_b200
    from tools.synth import ANCHOR_H, ANCHOR_W
    from yogo_b200.train import DataParallelTrainer
    net = yogo_b200.YOGO((64, 96), ANCHOR_W, ANCHOR_H, 4)
    net.load_state_dict(sd)
    net = net.to(DEV)
    net.compute_dtype = torch.bfloat16
    net.train()
    runner = net._get_runner()
    tr = DataParallelTrainer(net, yogo_b200.YOGOLoss().to(DEV), total_steps=50)
    losses, slots = [], []
    B = 8
    if graph:
        x0, y0 = ds.items[0]
        runner.drop_keep_override = keeps
        tr.enable_cuda_graph(x0.expand(B, -1, -1, -1).contiguous().to(DEV), y0.expand(B, -1, -1, -1).contiguous().to(DEV))
    for e in range(epochs):
        if mode == "device":
            gen = tr.steps_from_device(dd_or_batches, e)
            sizes = dd_or_batches.batch_sizes(e)
        else:
            gen = tr.steps_from_host(b for b in dd_or_batches[e])
            sizes = [b[0].shape[0] for b in dd_or_batches[e]]
        for n in sizes:
            runner.drop_keep_override = {i: k[:n] for i, k in keeps.items()}
            losses.append(next(gen).item())
            if mode == "device":
                slots.append((dd_or_batches.last_flips(), [t.clone() for t in tr.static_inputs(0)] if graph and n == B else None))
        assert next(gen, None) is None
    return np.array(losses), tr.flat_p.cpu().numpy(), slots


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [True, False])
def test_training_from_device_equals_training_from_host_batches(graph):
    import yogo_b200
    from tools.synth import ANCHOR_H, ANCHOR_W
    from yogo_b200.data import DeviceResidentDataset
    torch.manual_seed(0)
    net = yogo_b200.YOGO((64, 96), ANCHOR_W, ANCHOR_H, 4)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.1)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    Sx, Sy = net.get_grid_size()
    ds = _dataset(20, 1, 64, 96, Sy, Sx, seed=4)       # batches 8, 8, 4: the last one is ragged
    g = torch.Generator().manual_seed(5)
    keeps = {i: (torch.rand(8, c, generator=g) > 0.1).float().to(DEV) for i, c in ((1, 32), (2, 64), (3, 128))}
    dd = DeviceResidentDataset(ds, 8, MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5)),
                               device=DEV, seed=1)
    dev_losses, dev_p, slots = _train("device", ds, dd, sd, keeps, 2, graph)

    # the host runs get the batches the device run built, as pinned host tensors
    valid = list(range(20))
    host, k = [], 0
    for e in range(2):
        eb = []
        for idx in dd.epoch_batches(e):
            (h, v), static = slots[k]
            k += 1
            x, y = _expected(ds, valid, idx, h, v)
            if static is not None:   # the static input slot held exactly this batch at the replay
                assert _same(static[0], x) and _same(static[1], y)
            eb.append((x.cpu().pin_memory(), y.cpu().pin_memory()))
        host.append(eb)
    assert graph == any(s[1] is not None for s in slots)
    h1_losses, h1_p, _ = _train("host", ds, host, sd, keeps, 2, graph)
    h2_losses, h2_p, _ = _train("host", ds, host, sd, keeps, 2, graph)
    assert np.isfinite(dev_losses).all() and len(dev_losses) == 6
    spread_l = np.abs(h1_losses - h2_losses).max()
    spread_p = np.abs(h1_p - h2_p).max()
    assert np.abs(dev_losses - h1_losses).max() <= max(2 * spread_l, 1e-6 * np.abs(h1_losses).max()), (dev_losses, h1_losses)
    assert np.abs(dev_p - h1_p).max() <= max(2 * spread_p, 1e-6 * np.abs(h1_p).max()), (np.abs(dev_p - h1_p).max(), spread_p)


# ----------------------------------------------------------------------------- several GPUs
@pytest.mark.gpu
def test_multi_rank_store_and_shards():
    """tests/ddp_device_dataset_check.py under torchrun on 2 GPUs (skipped on single-GPU boxes)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29537", os.path.join(ROOT, "tests", "ddp_device_dataset_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ddp_device_dataset_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
