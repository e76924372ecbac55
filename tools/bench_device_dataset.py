"""Device-resident training data (yogo_b200.data.DeviceResidentDataset) on one GPU; prints JSON lines (each with the GPU's
name, power limit and SM clocks) and appends them to --out:
  (a) base_model, batch 64, 772x1032 uint8, bf16: the step replayed from static inputs (`step_static`, the number
      bench.py reports) against the step from the device store (`steps_from_device`: flip draw + gather + label build
      inside the graph), alternated epoch by epoch in one process, CUDA events;
  (b) the gather + flip kernel and the label kernel alone at batch 64 (store larger than L2, every batch other images),
      time and GB/s from the bytes they must move (computed from shapes) against 7.7 TB/s;
  (c) PNG decode rate of this host's CPUs (torchvision.io.decode_png) on seeded smooth synthetic 772x1032 grayscale PNGs
      written to a temporary directory, one process and one process per core;
  (d) build time and device bytes of a store of a few thousand images (in-memory dataset, no decoding)."""
import argparse
import json
import os
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import yogo_b200  # noqa: E402
from tools import synth as O  # noqa: E402
from tools.bench_match import gpu_info  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402
from yogo_b200.data import DeviceResidentDataset, MultiArgSequential, RandomHorizontalFlipWithBBs, RandomVerticalFlipWithBBs  # noqa: E402
from yogo_b200.train import DataParallelTrainer  # noqa: E402

DEV = "cuda:0"
H, W, NC = 772, 1032, 7
HBM_BYTES_PER_S = 7.7e12
FLIPS = MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), RandomVerticalFlipWithBBs(0.5))


class TensorDataset(torch.utils.data.Dataset):
    def __init__(self, imgs, labs):
        self.imgs, self.labs = imgs, labs

    def __len__(self):
        return self.imgs.shape[0]

    def __getitem__(self, i):
        return self.imgs[i], self.labs[i % self.labs.shape[0]]


def make_dataset(n, seed=0):
    imgs = torch.randint(0, 256, (n, 1, H, W), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))
    labs = O.synth_labels(64, 97, 129, NC, 300, seed=seed + 1)
    return TensorDataset(imgs, labs)


def step_compare(dd, rounds):
    torch.manual_seed(0)
    net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, NC).to(DEV)
    net.compute_dtype = torch.bfloat16
    net.train()
    tr = DataParallelTrainer(net, yogo_b200.YOGOLoss().to(DEV), total_steps=10000)
    x, y = next(dd.batches(0))
    tr.enable_cuda_graph(x, y)
    nb = dd.num_batches(0)
    for l in tr.steps_from_device(dd, 0):   # captures the device graph, warms both
        pass
    for _ in range(nb):
        tr.step_static(0)
    torch.cuda.synchronize()
    static_ms, device_ms = [], []
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for r in range(rounds):
        ev[0].record()
        for _ in range(nb):
            tr.step_static(0)
        ev[1].record()
        for l in tr.steps_from_device(dd, r + 1):
            pass
        ev[2].record()
        torch.cuda.synchronize()
        static_ms.append(ev[0].elapsed_time(ev[1]) / nb)
        device_ms.append(ev[1].elapsed_time(ev[2]) / nb)
    s, d = sorted(static_ms), sorted(device_ms)
    return {"case": "step base_model b64 bf16", "steps_per_window": nb, "rounds": rounds,
            "static_input_ms_median": s[len(s) // 2], "device_store_ms_median": d[len(d) // 2],
            "static_input_ms": static_ms, "device_store_ms": device_ms,
            "note": "windows alternate in one process; device_store windows include the epoch's index-table upload"}


def kernels_alone(dd, iters):
    lib, st = L.lib(), L.stream()
    B = dd.batch_size
    C, Hh, Ww = dd.image_shape
    Sy, Sx = dd.grid
    out_i = torch.empty((B, C, Hh, Ww), dtype=dd.image_dtype, device=DEV)
    out_l = torch.empty((B, 6, Sy, Sx), dtype=torch.float32, device=DEV)
    dd.begin_epoch(0)

    def draw():
        L.check(lib.yg_dd_draw(dd._state.data_ptr(), dd._flags.data_ptr(), 0.5, 0.5, 0, dd.num_batches(), st))

    def gather():
        draw()
        L.check(lib.yg_dd_gather_images(dd._images.data_ptr(), out_i.data_ptr(), L.dtype_code(dd.image_dtype),
                                        dd._table.data_ptr(), dd._flags.data_ptr(), B, B, C, Hh, Ww, st))

    def labels():
        draw()
        L.check(lib.yg_dd_build_labels(dd._table.data_ptr(), dd._flags.data_ptr(), B, dd._records.data_ptr(),
                                       dd._rec_off.data_ptr(), B, Sy, Sx, out_l.data_ptr(), st))

    def timed(fn):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    draw_ms = timed(draw)
    g_ms, l_ms = timed(gather) - draw_ms, timed(labels) - draw_ms
    g_bytes = 2 * out_i.numel() * out_i.element_size()
    nrec = int(dd._rec_off[-1].item()) * B // max(len(dd), 1)
    l_bytes = out_l.numel() * 4 + nrec * 32
    return [{"case": "yg_dd_draw", "us": draw_ms * 1e3},
            {"case": "yg_dd_gather_images", "B": B, "shape": [C, Hh, Ww], "us": g_ms * 1e3, "bytes": g_bytes,
             "GBps": g_bytes / g_ms / 1e6, "frac_of_hbm": g_bytes / g_ms * 1e3 / HBM_BYTES_PER_S,
             "note": "draw launch time subtracted; bytes = every image byte read once and written once"},
            {"case": "yg_dd_build_labels", "B": B, "grid": [Sy, Sx], "us": l_ms * 1e3, "bytes": l_bytes,
             "GBps": l_bytes / l_ms / 1e6, "frac_of_hbm": l_bytes / l_ms * 1e3 / HBM_BYTES_PER_S,
             "note": "draw launch time subtracted; bytes = label tensor written + mean records read per batch"}]


def _decode_files(paths):
    import torchvision.io as io
    t0 = time.perf_counter()
    for p in paths:
        io.decode_png(io.read_file(p))
    return len(paths), time.perf_counter() - t0


def png_decode(n_files, reps):
    import multiprocessing as mp

    import torchvision.io as io
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(0)
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    with tempfile.TemporaryDirectory() as d:
        paths, sizes = [], []
        for i in range(n_files):
            a, b, c = (torch.rand(3, generator=g) * 0.05).tolist()
            img = (128 + 60 * torch.sin(a * xx + b * yy + 10 * c) + 8 * torch.randn(H, W, generator=g)).clamp(0, 255)
            enc = io.encode_png(img.to(torch.uint8)[None])
            p = os.path.join(d, f"{i}.png")
            with open(p, "wb") as f:
                f.write(enc.numpy().tobytes())
            paths.append(p)
            sizes.append(enc.numel())
        _decode_files(paths[:2])
        n, s = _decode_files(paths * reps)
        cores = len(os.sched_getaffinity(0))
        work = [paths * reps] * cores
        with mp.get_context("fork").Pool(cores) as pool:
            t0 = time.perf_counter()
            res = pool.map(_decode_files, work)
            wall = time.perf_counter() - t0
    return {"case": "png decode (torchvision.io.decode_png, 772x1032x1 uint8)", "png_bytes_mean": sum(sizes) / len(sizes),
            "img_per_s_one_core": n / s, "cores": cores, "img_per_s_all_cores": sum(r[0] for r in res) / wall,
            "note": "smooth synthetic images with noise, seeded; one process per core"}


def build_cost(n):
    ds = make_dataset(n, seed=7)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dd = DeviceResidentDataset(ds, 64, FLIPS, device=DEV, num_workers=8)
    torch.cuda.synchronize()
    t = time.perf_counter() - t0
    out = {"case": "build", "items": n, "seconds": t, "img_per_s": n / t, "nbytes": dd.nbytes,
           "image_bytes": dd._images.numel(), "label_record_bytes": dd._records.numel() * 4,
           "note": "in-memory uint8 dataset with 300 labelled cells per image (no decoding), DataLoader with 8 workers"}
    del dd
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "device_dataset_bench.jsonl"))
    ap.add_argument("--items", type=int, default=640, help="store of the step and kernel measurements")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--build-items", type=int, default=3000)
    ap.add_argument("--png-files", type=int, default=16)
    ap.add_argument("--png-reps", type=int, default=4)
    args = ap.parse_args()
    info = gpu_info()
    rows = []
    dd = DeviceResidentDataset(make_dataset(args.items), 64, FLIPS, device=DEV, num_workers=4)
    rows.append(step_compare(dd, args.rounds))
    rows += kernels_alone(dd, args.iters)
    del dd
    torch.cuda.empty_cache()
    rows.append(build_cost(args.build_items))
    rows.append(png_decode(args.png_files, args.png_reps))
    with open(args.out, "a") as f:
        for r in rows:
            line = json.dumps({**info, **r})
            print(line)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
