#!/usr/bin/env python
"""Benchmark of the YOGO hot path (BASELINE.json metric: train img/s, 772x1032, fwd+bwd+loss; infer img/s incl. NMS).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU implementation on the host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + the last timed step's results as DIR/*.npy

A "step" is one data-parallel training step of `base_model` on a batch of 64 synthetic 772x1032 grayscale images per
GPU (BASELINE configs[1]): forward, YOGOLoss, backward, gradient all-reduce (N > 1, bucketed, overlapped with backward,
captured in the step's CUDA graph) and the fused AdamW update.  Rank 0 prints ONE JSON line.  Besides the contract keys
the line carries (N = 1 only) `infer` - the inference metric of BASELINE.json (forward + threshold + NMS + per-class
counts, batch 1 / 64 / 256, sparse and dense candidates, with the NMS kernel's own roofline) - and `ref_gpu` - the
UNMODIFIED reference (baseline/_ref) run by stock PyTorch on the same GPU: cuDNN under bf16 autocast with
`cudnn.benchmark` for training (yogo/train.py:37, 315-322), `torch.compile` + the per-image `format_preds` loop for
inference (yogo/infer.py:237, 374).  Nothing under oracle/ or the reference runs inside our arm's timed regions.
"""
from __future__ import annotations

import argparse
import json
import os

import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "train_img_per_s"
UNIT = "img/s"
H, W, NUM_CLASSES = 772, 1032, 7
SY, SX = 97, 129

# conv FLOPs and minimum HBM bytes per image of one training step, SURVEY.md 8(d) / Appendix A
TRAIN_GF = {"base_model": 66.483, "silu_model": 66.483, "double_filters": 265.472}
TRAIN_MB = {"base_model": 299.6, "silu_model": 299.6, "double_filters": 599.7}
FWD_GF = {"base_model": 22.180, "silu_model": 22.180, "double_filters": 88.529}
NMS_BYTES_PER_IMG = 12 * 4 * SY * SX          # 48 B/cell read once (SURVEY.md 8d)
LOSS_BYTES_PER_IMG = (72 + 48) * SY * SX      # 72 B/cell read + 48 B/cell dpred written


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md), polled through NVML
    every 5 ms from a thread (nvidia-smi -lms is too coarse for a sub-second timed region)."""

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons = [], set()
        self.sm_max = None
        self._stop = threading.Event()
        self.thread = None
        self.err = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(h))
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.005)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)
        out = {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
               "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if self.err:
            out["error"] = self.err
        return out


def cuda_timed(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (baseline/_ref) on the host cores; the oracle port when it is absent
# ------------------------------------------------------------------------------------------
def cpu_reference_step_time(model_name: str, batch: int, steps: int, warmup: int):
    """Train step (forward + YOGOLoss + backward) on all host cores.  -> (img/s, s/step, cores, kind)."""
    from tools import synth as S
    from tools.ref_import import import_reference

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    x = S.synth_images(batch).float()
    lab = S.synth_labels(batch)
    ref = None
    try:
        ref = import_reference()
    except Exception:
        ref = None
    if ref is not None:
        kind = "reference"
        net = ref["YOGO"](img_size=(H, W), anchor_w=S.ANCHOR_W, anchor_h=S.ANCHOR_H, num_classes=NUM_CLASSES,
                          model_func=ref["get_model_func"](model_name))
        net.train()
        loss_fn = ref["YOGOLoss"]()

        def step():
            net.zero_grad(set_to_none=True)
            loss, _ = loss_fn(net(x), lab)
            loss.backward()
    else:
        kind = "port"
        from oracle import yogo_oracle as O
        import yogo_b200

        net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, NUM_CLASSES, model_func=yogo_b200.get_model_func(model_name))
        blocks = O.blocks_from_state_dict(model_name, net.state_dict())
        leaves = []
        for b in blocks:
            for t in [b.weight, b.bias] + ([b.bn["weight"], b.bn["bias"]] if b.bn else []):
                if t is not None:
                    t.requires_grad_(True)
                    leaves.append(t)
        g = torch.Generator().manual_seed(5)
        keeps = [(torch.rand(batch, b.weight.shape[0], generator=g) >= b.p_drop).float() if b.p_drop > 0 else None
                 for b in blocks]

        def step():
            for t in leaves:
                t.grad = None
            tt = O.backbone_forward(x, blocks, train=True, drop_keep=keeps)
            out = O.head_transform(tt, O.ANCHOR_W, O.ANCHOR_H)
            _, _, dpred = O.yogo_loss_np(out.detach().numpy(), lab.numpy())
            out.backward(torch.from_numpy(dpred))

    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return batch / sec, sec, cores, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_batch = 8
    # bounded: the CPU step takes ~1 s per 8 images; cap the repetitions so the whole run ends within a few minutes
    steps, warmup = max(1, min(args.steps, 20)), max(1, min(args.warmup, 3))
    v, sec, cores, kind = cpu_reference_step_time(args.model, sample_batch, steps, warmup)
    what = ("the unmodified reference (baseline/_ref: yogo.model.YOGO + yogo.yogo_loss.YOGOLoss, torch CPU)" if kind == "reference"
            else "fp32 torch-CPU port of the reference path (oracle/)")
    sample = f"{sample_batch} images of the same 772x1032 workload per step, fp32, {what}, {cores} threads, {steps} timed steps"
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} train step (fwd+YOGOLoss+bwd), 772x1032x1, 7 classes", "batch_per_step": sample_batch},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# the reference's GPU path (stock PyTorch / cuDNN / torchvision) on this box: a comparator, not the product
# ------------------------------------------------------------------------------------------
def ref_gpu_record(args, dev, budget_s=150.0):
    from tools import synth as S
    from tools.ref_import import import_reference

    t_start = time.perf_counter()
    try:
        ref = import_reference()
    except Exception as e:
        return {"unavailable": "import failed: " + repr(e)[:200]}
    if ref is None:
        return {"unavailable": "no copy of the reference (baseline/_ref) on this box"}
    B = args.batch
    rec = {"what": "unmodified reference (baseline/_ref) on this GPU with stock torch %s / cuDNN %s" %
                   (torch.__version__, torch.backends.cudnn.version()), "batch": B}
    torch.backends.cudnn.benchmark = True            # yogo/train.py:37
    torch.manual_seed(0)
    net = ref["YOGO"](img_size=(H, W), anchor_w=S.ANCHOR_W, anchor_h=S.ANCHOR_H, num_classes=NUM_CLASSES,
                      model_func=ref["get_model_func"](args.model)).to(dev)
    loss_fn = ref["YOGOLoss"]().to(dev)
    x = S.synth_images(B).to(dev)
    lab = S.synth_labels(B).to(dev)
    opt = torch.optim.AdamW(net.parameters(), lr=3e-4, weight_decay=5e-2)

    def train_step(autocast):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            out = net(x)
            loss, _ = loss_fn(out, lab)          # includes the reference's three .item() syncs (yogo_loss.py:123-127)
        loss.backward()
        opt.step()

    try:
        net.train()
        ms = cuda_timed(lambda: train_step(True), 5, warmup=3)
        rec["train_step_bf16_autocast_ms"] = round(ms, 3)
        rec["train_img_s_bf16_autocast"] = round(B / ms * 1e3, 1)
        net.model.to(memory_format=torch.channels_last)      # a favour the reference does not do itself
        ms2 = cuda_timed(lambda: train_step(True), 5, warmup=3)
        rec["train_step_bf16_autocast_channels_last_ms"] = round(ms2, 3)
        rec["train_img_s_best"] = round(B / min(ms, ms2) * 1e3, 1)
        if time.perf_counter() - t_start < budget_s * 0.3:
            net.model.to(memory_format=torch.contiguous_format)
            ms3 = cuda_timed(lambda: train_step(False), 2, warmup=1)
            rec["train_step_fp32_default_ms"] = round(ms3, 3)      # the reference's default (no --half): TF32 off
    except Exception as e:
        rec["train_error"] = repr(e)[:300]
    # ---- inference as yogo/infer.py does it: inference=True, eval, torch.compile on CUDA (:237), then
    # get_prediction_class_counts(res.cpu(), ...) (:374-379): the per-image format_preds loop on the CPU copy
    try:
        del opt
        net_i = ref["YOGO"](img_size=(H, W), anchor_w=S.ANCHOR_W, anchor_h=S.ANCHOR_H, num_classes=NUM_CLASSES,
                            inference=True, model_func=ref["get_model_func"](args.model)).to(dev)
        net_i.eval()
        fwd = net_i
        compiled = False
        if time.perf_counter() - t_start < budget_s * 0.5:
            try:
                cand = torch.compile(net_i)
                with torch.no_grad():
                    cand(x[:1])
                fwd, compiled = cand, True
            except Exception as e:   # no working inductor toolchain on this box: eager forward
                rec["compile_error"] = repr(e)[:200]
        rec["infer_compiled"] = compiled
        sparse = S.synth_sparse_preds(B, K=300)
        with torch.no_grad():
            ms_f = cuda_timed(lambda: fwd(x), 5, warmup=3)
        rec["infer_fwd_ms"] = round(ms_f, 3)
        rec["infer_fwd_img_s"] = round(B / ms_f * 1e3, 1)
        sp_dev = sparse.to(dev)
        t0 = time.perf_counter()
        c_cpu = ref["get_prediction_class_counts"](sp_dev.cpu())     # stock: D2H + CPU loop
        rec["postproc_sparse_stock_cpu_ms"] = round((time.perf_counter() - t0) * 1e3, 3)
        best_post = rec["postproc_sparse_stock_cpu_ms"]
        try:
            # the same per-image loop with torch / torchvision CUDA ops (format_preds + argmax counts; the reference's
            # get_prediction_class_counts itself accumulates on the CPU and rejects CUDA tensors)
            def post_gpu():
                tot = torch.zeros(NUM_CLASSES, dtype=torch.long, device=dev)
                for pred in sp_dev:
                    rows = ref["format_preds"](pred)
                    if rows.numel():
                        vals, idx = rows[:, 5:].max(dim=1)
                        tot += torch.nn.functional.one_hot(idx[vals > 0], num_classes=NUM_CLASSES).sum(dim=0)
                return tot
            ms_p = cuda_timed(post_gpu, 2, warmup=1)
            rec["postproc_sparse_on_gpu_ms"] = round(ms_p, 3)
            assert post_gpu().cpu().tolist() == c_cpu.tolist()
            best_post = min(best_post, ms_p)
        except Exception as e:
            rec["postproc_gpu_error"] = repr(e)[:200]
        rec["infer_img_s_incl_nms_sparse"] = round(B / (ms_f + best_post) * 1e3, 1)
        rec["counts_sparse"] = [int(v) for v in c_cpu.tolist()]
    except Exception as e:
        rec["infer_error"] = repr(e)[:300]
    rec["seconds"] = round(time.perf_counter() - t_start, 1)
    return rec


# ------------------------------------------------------------------------------------------
# inference metric of our arm (BASELINE configs[4])
# ------------------------------------------------------------------------------------------
def infer_record(args, dev, peaks):
    import yogo_b200
    from tools import synth as S

    torch.manual_seed(0)
    net = yogo_b200.YOGO((H, W), S.ANCHOR_W, S.ANCHOR_H, NUM_CLASSES, inference=True,
                         model_func=yogo_b200.get_model_func(args.model)).to(dev)
    net.compute_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    net.eval()
    rows = []
    out_host = torch.empty(NUM_CLASSES, dtype=torch.int64).pin_memory()
    for B in (1, 64, 256):
        img = S.synth_images(B, seed=7).to(dev)
        img_host = S.synth_images(B, seed=7).pin_memory()
        sp = S.synth_sparse_preds(B, K=300).to(dev)
        with torch.no_grad():
            fwd_ms = cuda_timed(lambda: net(img), 5 if B > 1 else 20, warmup=2)
            pred = net(img)                                           # random-init output: ~96 % of the cells are candidates
        sparse_ms = cuda_timed(lambda: yogo_b200.format_preds_batch(sp), 10, warmup=2)
        dense_ms = cuda_timed(lambda: yogo_b200.format_preds_batch(pred), 2, warmup=1)
        _, kcs, _, counts = yogo_b200.format_preds_batch(sp)
        _, kcd, _, _ = yogo_b200.format_preds_batch(pred)

        def e2e():   # host images in, per-class counts out, through the public API
            with torch.no_grad():
                p = net(img_host.to(dev, non_blocking=True))
            out_host.copy_(yogo_b200.format_preds_batch(p)[3], non_blocking=True)

        e2e_ms = cuda_timed(e2e, 3, warmup=1)
        # the same pipeline (host images -> counts) replayed from one CUDA graph (yogo_b200.infer.GraphedInference)
        from yogo_b200.infer import GraphedInference
        gi = GraphedInference(net, img.shape)

        def e2e_graph():
            out_host.copy_(gi(img_host)[4], non_blocking=True)

        e2e_graph_ms = cuda_timed(e2e_graph, 5 if B > 1 else 20, warmup=2)
        # (sparse-realistic predictions cannot be produced by random weights: the graphed sparse figure is the graphed
        # forward plus the graphed NMS on the synthetic sparse prediction tensor)
        sp_static = sp.clone()
        g2 = torch.cuda.CUDAGraph()
        yogo_b200.format_preds_batch(sp_static)
        torch.cuda.synchronize()
        with torch.cuda.graph(g2):
            sp_out = yogo_b200.format_preds_batch(sp_static)
        nms_sparse_graph_ms = cuda_timed(g2.replay, 10, warmup=2)
        fwd_static = img.clone()
        g3 = torch.cuda.CUDAGraph()
        with torch.no_grad():
            net(fwd_static)
            torch.cuda.synchronize()
            with torch.cuda.graph(g3):
                fwd_out = net(fwd_static)
        fwd_graph_ms = cuda_timed(g3.replay, 5 if B > 1 else 20, warmup=2)
        del g2, g3, gi, sp_out, fwd_out
        rows.append({
            "batch": B, "fwd_ms": round(fwd_ms, 4), "fwd_img_s": round(B / fwd_ms * 1e3, 1),
            "nms_sparse_ms": round(sparse_ms, 4), "kept_sparse_per_img": round(float(kcs.float().mean()), 1),
            "infer_img_s_sparse": round(B / (fwd_ms + sparse_ms) * 1e3, 1),
            "nms_dense_ms": round(dense_ms, 4), "kept_dense_per_img": round(float(kcd.float().mean()), 1),
            "infer_img_s_dense": round(B / (fwd_ms + dense_ms) * 1e3, 1),
            "e2e_host_images_dense_img_s": round(B / e2e_ms * 1e3, 1),
            "graph": {"fwd_ms": round(fwd_graph_ms, 4), "nms_sparse_ms": round(nms_sparse_graph_ms, 4),
                      "infer_img_s_sparse": round(B / (fwd_graph_ms + nms_sparse_graph_ms) * 1e3, 1),
                      "e2e_host_images_dense_img_s": round(B / e2e_graph_ms * 1e3, 1)},
            "nms_roofline_sparse": {"bound": "hbm", "achieved": round(B * NMS_BYTES_PER_IMG / nms_sparse_graph_ms / 1e6, 1), "peak": peaks["hbm_gbs"],
                                    "unit": "GB/s", "frac": round(B * NMS_BYTES_PER_IMG / nms_sparse_graph_ms / 1e6 / peaks["hbm_gbs"], 4),
                                    "note": "whole threshold + NMS + counts pipeline (5 launches, graph replay) against the 48 B/cell it must read"},
            "fwd_tflops": round(B * FWD_GF.get(args.model, 0) / fwd_ms, 1),
            "counts_sparse": [int(v) for v in counts.tolist()],
        })
    return {"metric": "infer_img_per_s incl. threshold + NMS + per-class counts", "model": args.model, "dtype": args.dtype,
            "candidates": "sparse = 300 objects / image (SURVEY.md 8d); dense = random-init network output", "sweep": rows}


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import yogo_b200
    from yogo_b200 import _lib as L
    from yogo_b200.train import DataParallelTrainer
    from tools import synth as O  # seeded synthetic inputs (shared with the tests); the oracle is not imported on this arm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    B = args.batch
    torch.manual_seed(0)
    net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, NUM_CLASSES,
                         model_func=yogo_b200.get_model_func(args.model)).to(dev)
    net.compute_dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    if args.dtype == "fp32" and args.fp32_x3:
        yogo_b200.set_fp32_tensor_cores(True)   # split-bf16 convolutions of fp32 tensors on the tensor cores (csrc/x3.cu)
    if args.tc_or:   # experiment knob: extra option bits of the conv engine (include/yogo_b200.h, yg_set_tc_options) for A/B runs of the whole step
        from yogo_b200 import _lib as _L
        _L.check(_L.lib().yg_set_tc_options(_L.lib().yg_get_tc_options() | args.tc_or))
    net.train()
    loss_fn = yogo_b200.YOGOLoss().to(dev)
    trainer = DataParallelTrainer(net, loss_fn, total_steps=10000, overlap=bool(args.overlap))
    trainer.broadcast_state()
    initial = trainer.snapshot()   # seeded: the same on every run with the same arguments
    use_graph = bool(args.graph)

    nbuf = 2  # distinct host batches, alternated
    host_imgs = [O.synth_images(B, seed=10 * rank + i).pin_memory() for i in range(nbuf)]
    host_labs = [O.synth_labels(B, seed=100 + 10 * rank + i).pin_memory() for i in range(nbuf)]
    dev_imgs = [t.to(dev) for t in host_imgs]
    dev_labs = [t.to(dev) for t in host_labs]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value): inputs already in HBM (the two static slots of the step graph hold the two
    # batches; steps alternate between them), CUDA events on the launching stream, max over ranks
    if use_graph:
        trainer.step(dev_imgs[0], dev_labs[0])
        trainer.enable_cuda_graph(dev_imgs[0], dev_labs[0], slots=nbuf)
        for i in range(nbuf):
            xs, ys = trainer.static_inputs(i)
            xs.copy_(dev_imgs[i])
            ys.copy_(dev_labs[i])

    def resident_step(i):
        if use_graph:
            return trainer.step_static(i % nbuf)
        return trainer.step(dev_imgs[i % nbuf], dev_labs[i % nbuf])

    for i in range(args.warmup):
        resident_step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.load().yg_launch_count()
    e0, e1, e_pause, e_resume = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    e0.record()
    for i in range(args.steps - 1):
        resident_step(i)
    e_pause.record()
    # The last timed step starts again from the seeded initial state (the restore is not timed).  The reductions of the
    # kernels vary the last bits of a few gradients from run to run and AdamW spreads such differences over the steps
    # that follow; restarting makes the last step compute from the same parameters, optimizer state and BatchNorm
    # statistics on every run, so that its results (final_loss, --dump-outputs) are reproducible.
    trainer.restore(initial)
    e_resume.record()
    loss = resident_step(args.steps - 1)
    e1.record()
    barrier()
    launches = L.load().yg_launch_count() - launches0
    if use_graph:
        launches = trainer.graph_launches * args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, net)
    ms = e0.elapsed_time(e_pause) + e_resume.elapsed_time(e1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    final_loss = float(loss.item())

    # ---- end-to-end through the public API with HOST buffers: every step's images and labels cross PCIe from pinned
    # memory inside the timed region (copied straight into the idle static slot while the other slot's graph runs) and
    # every step's loss is read back.  3 x the device window, started from a drained device.
    out_host = torch.empty(1, dtype=torch.float32).pin_memory()
    e2e_steps = 3 * args.steps

    def e2e_run(nsteps):
        gen = ((host_imgs[i % nbuf], host_labs[i % nbuf]) for i in range(nsteps))
        for l in trainer.steps_from_host(gen):
            out_host.copy_(l.detach().reshape(1), non_blocking=True)

    e2e_run(max(2, args.warmup))
    barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / float(t.item())
    h2d = host_imgs[0].numel() * host_imgs[0].element_size() + host_labs[0].numel() * host_labs[0].element_size()

    # ---- per-kernel breakdown with CUDA events (instrumented eager pass, not part of `value`); every rank runs it
    # (the steps contain collectives), rank 0 reports it
    saved_graph, trainer._graph = trainer._graph, None
    breakdown, calls_per_step = kernel_breakdown(trainer, dev_imgs, dev_labs, args, L)
    trainer._graph = saved_graph
    barrier()

    line = None
    if rank == 0:
        roof = roofline_from_breakdown(breakdown, calls_per_step, args, B, peaks)
        gf, mb = TRAIN_GF.get(args.model), TRAIN_MB.get(args.model)
        step_roof = None
        if gf and mb:
            tf = gf * B / ms_step            # GF / ms = TFLOP/s
            gbs = mb * B / ms_step           # MB / ms = GB/s
            step_roof = {"conv_tflops": round(tf, 1), "frac_of_burst_bf16": round(tf / peaks["bf16_tflops"], 4),
                         "frac_of_sustained_bf16": round(tf / peaks["bf16_tflops_sustained"], 4),
                         "min_hbm_gbs": round(gbs, 1), "frac_of_hbm": round(gbs / peaks["hbm_gbs"], 4),
                         "note": "whole step: algorithmic conv FLOPs and minimum activation bytes per image (SURVEY.md 8d) x batch / step time"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {
                "workload": f"{args.model} training step: fwd + YOGOLoss + bwd + grad all-reduce + fused AdamW, "
                            f"772x1032x1 uint8 images, 7 classes, batch {B}/GPU "
                            + ("(BASELINE configs[1])" if args.model == "base_model" and B == 64 else
                               "(BASELINE configs[3])" if args.model in ("double_filters", "silu_model") and B == 128 else
                               "(parity / sweep configuration)"),
                "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                "l2_policy": "inputs+activations per step (>3 GB) far exceed the 126 MB L2; batches alternate",
                "conv_impl": L.get_conv_impl() + (" + fp32 x3" if yogo_b200.get_fp32_tensor_cores() else ""), "cuda_graph": bool(use_graph),
                "allreduce": "none (1 rank)" if world == 1 else
                             (f"{len(trainer.buckets)} NCCL bucket(s) on a side stream, overlapped with backward, captured in the step graph"
                              if args.overlap else f"{len(trainer.buckets)} NCCL bucket(s) on the main stream (no overlap), captured in the step graph"),
            },
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                    "how": "pinned host batches -> static graph slots (H2D on a copy stream, double-buffered) -> step -> loss read back"},
            "gpu_launches": int(launches),
            "roofline": roof,
            "step_roofline": step_roof,
            "cpu_baseline": None,
            "final_loss": final_loss,
            "kernel_breakdown_ms": breakdown,
        }
    if world > 1:
        # several ranks: nothing else to measure.  The step graphs hold captured NCCL work; tearing them (or the process
        # group) down can block in NCCL's cleanup, so the ranks leave through os._exit once the line is out.
        dist.barrier()
        if rank == 0:
            print(json.dumps(line), flush=True)
        sys.stdout.flush()
        sys.stderr.flush()
        dist.barrier()
        os._exit(0)
    # free the training state before the single-GPU extras
    if use_graph:
        trainer.disable_cuda_graph()
    if rank == 0 and world == 1:
        del trainer, net
        torch.cuda.empty_cache()
        if not args.no_infer:
            try:
                line["infer"] = infer_record(args, dev, peaks)
            except Exception as e:  # pragma: no cover
                line["infer"] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
        if not args.no_ref_gpu:
            try:
                line["ref_gpu"] = ref_gpu_record(args, dev)
            except Exception as e:  # pragma: no cover
                line["ref_gpu"] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            v, sec, cores, kind = cpu_reference_step_time(args.model, 8, 3, 1)
            what = "the unmodified reference (baseline/_ref) on torch CPU" if kind == "reference" else "fp32 torch-CPU port of the reference path (oracle/)"
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": f"8 images/step of the same workload, fp32, {what}, 3 timed steps"}
    if rank == 0:
        print(json.dumps(line), flush=True)


def dump_outputs(out_dir, loss, net):
    """What the last timed step hands its caller, as float32 .npy files: the loss, the updated parameters and the
    (clamped) gradients they were updated with, both concatenated in `net.named_parameters()` order, and the BatchNorm
    running statistics in `net.named_buffers()` order.  The step starts from the seeded initial state with seeded images,
    labels and dropout masks, so the same arguments give the same inputs on every run and two builds can be compared
    file by file."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    params = [p for _, p in net.named_parameters()]
    arrays = {
        "loss": loss.detach().float().reshape(1),
        "params": torch.cat([p.detach().reshape(-1) for p in params]),
        "grads": torch.cat([p.grad.reshape(-1) for p in params]),
        "bn_running_stats": torch.cat([b.reshape(-1) for n, b in net.named_buffers() if "running_" in n]),
    }
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def kernel_breakdown(trainer, dev_imgs, dev_labs, args, L):
    """Times every C-ABI call of a few steps with CUDA events on the launching stream."""
    lib = L.lib()
    names = [n for n in L.EXPORTED_SYMBOLS if n.startswith(("yg_conv", "yg_bn_act", "yg_bn_bwd", "yg_bn_stats", "yg_head", "yg_yogo", "yg_adamw"))
             and not n.endswith("workspace")]
    records = []

    def wrap(name, fn):
        def inner(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            records.append((name, a, e0, e1))
            return rc
        return inner

    class Proxy:
        def __getattr__(self, k):
            f = getattr(lib, k)
            return wrap(k, f) if k in names else f

    proxy = Proxy()
    orig_lib = L.lib
    L.lib = lambda: proxy
    try:
        steps = 2
        for i in range(steps):
            trainer.step(dev_imgs[i % len(dev_imgs)], dev_labs[i % len(dev_labs)])
        torch.cuda.synchronize()
    finally:
        L.lib = orig_lib
    agg = {}
    for name, a, e0, e1 in records:
        key = name
        if name in ("yg_conv_fwd", "yg_conv_dgrad", "yg_conv_wgrad"):
            # (.., dtype, N, H, W, Cin, Cout, k, s, ..): identify the layer by shape
            ints = [v for v in a if isinstance(v, int) and not isinstance(v, bool)]
            shape = [v for v in ints if 0 < v < 100000][:9]
            key = f"{name}[{'x'.join(str(v) for v in shape[-7:])}]"
        d = agg.setdefault(key, [0.0, 0])
        d[0] += e0.elapsed_time(e1) / steps
        d[1] += 1
    ordered = sorted(agg.items(), key=lambda kv: -kv[1][0])
    return ({k: round(v[0], 4) for k, v in ordered}, {k: v[1] / steps for k, v in ordered})


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/ncu_traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum), or None when that kernel has not been captured."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            ent = json.load(f).get(kernel)
        return float(ent["dram_bytes_per_launch"]) if ent else None
    except (OSError, ValueError, KeyError):
        return None


def roofline_from_breakdown(breakdown, calls_per_step, args, B, peaks):
    """roofline of the dominant kernel (largest share of the step).  Convolutions are judged against the roof that
    binds them: arithmetic intensity (FLOP per algorithmic byte) above the machine balance -> tensor, else HBM
    (SURVEY.md Appendix A: base_model layers 2, 3 are HBM-bound, 4-7 tensor-bound).  Per-kernel event timings are
    short bursts at the full SM clock, so the tensor peak is the measured BURST figure of MEASURED_PEAKS.json."""
    if not breakdown:
        return None
    top, ms = next(iter(breakdown.items()))
    ms = ms / max(calls_per_step.get(top, 1.0), 1.0)   # the breakdown sums same-shaped layers: per launch here
    traffic = measured_traffic(top)
    if top.startswith(("yg_conv_fwd[", "yg_conv_dgrad[", "yg_conv_wgrad[")):
        dims = [int(v) for v in top[top.index("[") + 1:-1].split("x")]
        N, Hh, Ww, Cin, Cout, k, s = dims
        pad = k // 2
        Ho, Wo = (Hh + 2 * pad - k) // s + 1, (Ww + 2 * pad - k) // s + 1
        flops = 2.0 * N * Ho * Wo * Cout * Cin * k * k
        # algorithmic bytes: every activation tensor the op must touch once (bf16); dgrad also reads what the fused
        # activation backward of the previous layer needs
        nbytes = 2.0 * (N * Hh * Ww * Cin + N * Ho * Wo * Cout)
        if top.startswith("yg_conv_dgrad["):
            nbytes += N * Hh * Ww * Cin / 8.0   # + the 1-bit-per-element activation sign mask of the previous layer
        balance = peaks["bf16_tflops"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
        if flops / nbytes >= balance:
            ach = flops / (ms * 1e-3) / 1e12
            return {"kernel": top, "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops"],
                    "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"], "traffic": traffic,
                    "peak_source": peaks["source"] + " (burst bf16: the kernel is timed alone with CUDA events)",
                    "frac_of_sustained": ach / peaks["bf16_tflops_sustained"],
                    "ms_per_launch": ms, "algorithmic_flops": flops}
        ach = nbytes / (ms * 1e-3) / 1e9
        return {"kernel": top, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peaks["source"] + " (copy bandwidth)",
                "ms_per_launch": ms, "algorithmic_bytes": nbytes, "flop_per_byte": flops / nbytes}
    # the other kernels of the step stream their operands once: algorithmic bytes per launch at the bench geometry
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    px1, px7 = B * Ho * Wo, B * 97 * 129
    stream_bytes = {
        "yg_conv_first_fwd": B * H * W + px1 * 16 * 2,              # uint8 image in, 16-channel bf16 out
        "yg_conv_first_bwd": B * H * W + px1 * 16 * 2,              # image + d(activation) in, 16x9 sums out
        "yg_conv_first_gram": B * H * W,
        "yg_bn_act_apply": 2 * px7 * 128 * 2 + px7 * 16,            # y_raw in, activation + sign mask out
        "yg_bn_bwd_apply": 3 * px7 * 128 * 2,                       # g, y_raw in, dz out
        "yg_bn_bwd_sums": 2 * px7 * 128 * 2,
        "yg_bn_stats": px7 * 128 * 2,
    }
    if top in stream_bytes:
        ach = stream_bytes[top] / (ms * 1e-3) / 1e9
        return {"kernel": top, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": ach / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peaks["source"] + " (copy bandwidth)",
                "ms_per_launch": ms, "algorithmic_bytes": float(stream_bytes[top])}
    return {"kernel": top, "bound": "hbm", "achieved": None, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": None,
            "traffic": traffic, "ms_per_launch": ms, "peak_source": peaks["source"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="base_model")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-infer", action="store_true", help="skip the inference sweep record (N = 1)")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip the reference-on-GPU comparator (N = 1)")
    ap.add_argument("--graph", type=int, default=1, help="replay the whole step from a CUDA graph")
    ap.add_argument("--fp32-x3", type=int, default=1, help="--dtype fp32: run the convolutions as split-bf16 x3 on the tensor cores")
    ap.add_argument("--tc-or", type=int, default=0, help="OR these bits into the conv engine's option word (A/B experiments)")
    ap.add_argument("--overlap", type=int, default=1, help="N > 1: all-reduce gradient buckets on a side stream while backward continues")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed training step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
