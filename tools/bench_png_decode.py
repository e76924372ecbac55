"""PNG decoding on the GPU (yogo_b200.data.decode_png_batch) against torchvision.io.decode_png on the host, and predict()
over a folder of PNGs.  Writes profiles/png_decode_bench.jsonl (or --out); every line carries the GPU name, power limit
and SM clocks.

  (a) decode_png_batch on groups of 148 / 592 / 2048 seeded 772x1032 images at three noise levels (the generator of
      tools/bench_device_dataset.py::png_decode with sigma 8 and 2, and a flat background with sparse blobs): CUDA
      events after a warm-up, img/s, decoded GB/s, and the time of each kernel from torch.profiler in a separate pass;
  (b) torchvision.io.decode_png on one core and on all cores, same files;
  (c) predict(path_to_images=..., count_predictions=True, half=True, batch_size=64) over 4096 files in the page cache,
      next to predict(images=...) on the same images and the serial host decode of the files.

Groups larger than the number of distinct images repeat them; each group is 1.5-4.5 GB of input, output and scratch,
far more than the 126 MB L2, so the repeats are read from HBM."""
import argparse
import json
import multiprocessing as mp
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

H, W = 772, 1032
DEV = "cuda"


def image(kind: str, seed: int) -> np.ndarray:
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    if kind == "blobs":   # flat background, a few dozen dark cells
        img = torch.full((H, W), 200.0)
        for cy, cx, r in (torch.rand(40, 3, generator=g) * torch.tensor([H, W, 12.0])).tolist():
            img -= 120 * torch.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * (r + 3) ** 2))
        return img.clamp(0, 255).to(torch.uint8).numpy()
    sigma = {"sigma8": 8.0, "sigma2": 2.0}[kind]
    a, b, c = (torch.rand(3, generator=g) * 0.05).tolist()
    img = 128 + 60 * torch.sin(a * xx + b * yy + 10 * c) + sigma * torch.randn(H, W, generator=g)
    return img.clamp(0, 255).to(torch.uint8).numpy()


def encode(args):
    import torchvision.io as io

    torch.set_num_threads(1)
    kind, seed = args
    return io.encode_png(torch.from_numpy(image(kind, seed))[None]).numpy().tobytes()


def host_decode(files):
    import torchvision.io as io

    torch.set_num_threads(1)
    t = [torch.frombuffer(bytearray(f), dtype=torch.uint8) for f in files]
    t0 = time.perf_counter()
    for x in t:
        io.decode_png(x, io.ImageReadMode.GRAY)
    return len(t), time.perf_counter() - t0


def _decode_worker(files, barrier, q):
    import torchvision.io as io

    torch.set_num_threads(1)
    t = [torch.frombuffer(bytearray(f), dtype=torch.uint8) for f in files]
    io.decode_png(t[0], io.ImageReadMode.GRAY)
    barrier.wait()
    t0 = time.perf_counter()
    for x in t:
        io.decode_png(x, io.ImageReadMode.GRAY)
    q.put((len(t), t0, time.perf_counter()))


def host_decode_all_cores(files, cores):
    """torchvision decode on every core at once: images decoded, and seconds from the first start to the last end."""
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(cores), ctx.Queue()
    procs = [ctx.Process(target=_decode_worker, args=(files, barrier, q)) for _ in range(cores)]
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    return sum(r[0] for r in res), max(r[2] for r in res) - min(r[1] for r in res)


def kernel_times(files):
    from torch.profiler import ProfilerActivity, profile

    from yogo_b200.data import decode_png_batch

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        decode_png_batch(files, DEV)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "png_" in e.key:
            name = e.key.split("png_")[1].split("_kernel")[0]
            out[name] = out.get(name, 0.0) + e.device_time_total / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--distinct", type=int, default=256)
    ap.add_argument("--groups", default="148,592,2048")
    ap.add_argument("--predict-files", type=int, default=4096)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "png_decode_bench.jsonl"))
    a = ap.parse_args()
    from bench_match import gpu_info

    import yogo_b200
    from yogo_b200.data import decode_png_batch
    from yogo_b200.data.png import decode_entries
    from yogo_b200.infer import DECODE_IMAGES_PER_SM

    info = gpu_info()
    cores = len(os.sched_getaffinity(0))
    lines = []

    def emit(d):
        d = {**info, **d}
        print(json.dumps(d), flush=True)
        lines.append(d)

    with mp.get_context("fork").Pool(cores) as pool:
        files = {k: pool.map(encode, [(k, s) for s in range(a.distinct)]) for k in ("sigma8", "sigma2", "blobs")}
    for kind, fs in files.items():
        _, st = decode_entries(fs[:8], DEV)
        assert set(st.values()) == {0}, st
        ref = torch.stack([torch.from_numpy(image(kind, s))[None] for s in range(8)])
        assert torch.equal(decode_png_batch(fs[:8], DEV).cpu(), ref), kind
        for n in [int(g) for g in a.groups.split(",")]:
            group = (fs * (n // len(fs) + 1))[:n]
            decode_png_batch(group, DEV)
            torch.cuda.synchronize()
            reps = max(2, 4096 // n)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for _ in range(reps):
                decode_png_batch(group, DEV)
            e1.record()
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) / reps
            ms = e0.elapsed_time(e1) / reps
            k = kernel_times(group)
            kern = sum(k.values())
            emit({"case": "decode_png_batch", "images": kind, "png_bytes_mean": float(np.mean([len(f) for f in fs])), "group": n,
                  "ms_per_call": ms, "img_per_s": n / (ms / 1e3), "wall_ms_per_call": wall * 1e3,
                  "kernel_ms": k, "img_per_s_kernels_only": n / (kern / 1e3), "decoded_GBps_kernels": n * H * W / (kern / 1e3) / 1e9,
                  "note": "ms_per_call: CUDA events around whole calls (host chunk walk, staging, upload, kernels, status read)"})
        n1, s1 = host_decode(fs[:64])
        n_all, wall = host_decode_all_cores(fs[:64], cores)
        emit({"case": "torchvision.io.decode_png (host)", "images": kind, "img_per_s_one_core": n1 / s1, "cores": cores,
              "img_per_s_all_cores": n_all / wall,
              "note": "all cores: one forked process per core, the files inherited through fork; timed from a common "
                      "barrier to the last process's end, decode only"})

    # (c) predict over a folder
    torch.manual_seed(0)
    from oracle import yogo_oracle as O

    net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, 7, inference=True)
    with tempfile.TemporaryDirectory() as d:
        pth = os.path.join(d, "m.pth")
        torch.save({"step": 1, "model_state_dict": net.state_dict(), "model_version": "base_model",
                    "class_names": [str(i) for i in range(7)], "normalize_images": True}, pth)
        idir = os.path.join(d, "images")
        os.mkdir(idir)
        fs = files["sigma8"]
        for i in range(a.predict_files):
            with open(os.path.join(idir, f"{i:05d}.png"), "wb") as f:
                f.write(fs[i % len(fs)])
        distinct = torch.stack([torch.from_numpy(image("sigma8", s))[None] for s in range(len(fs))])
        imgs = distinct[torch.arange(a.predict_files) % len(fs)]
        kw = dict(count_predictions=True, half=True, batch_size=64)
        rates = {}
        import contextlib
        import io as _io

        for name, call in (("path_to_images", lambda: yogo_b200.predict(pth, path_to_images=idir, **kw)),
                           ("images", lambda: yogo_b200.predict(pth, images=imgs, **kw))) * 2:
            with contextlib.redirect_stdout(_io.StringIO()) as out:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                call()
                torch.cuda.synchronize()
                rates[name] = a.predict_files / (time.perf_counter() - t0)
            rates[name + "_counts"] = out.getvalue().strip()
        assert rates["path_to_images_counts"] == rates["images_counts"]
        n1, s1 = host_decode(fs[:64])
        emit({"case": "predict 772x1032 base_model bf16 batch 64", "files": a.predict_files,
              "img_per_s_path_to_images": rates["path_to_images"], "img_per_s_images_in_memory": rates["images"],
              "img_per_s_serial_host_decode": n1 / s1, "decode_images_per_sm": DECODE_IMAGES_PER_SM,
              "note": "second of two alternating runs each; files in the page cache; images= includes the upload of the stack"})
    with open(a.out, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
