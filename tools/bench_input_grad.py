"""Image gradients on one GPU: yg_conv_first_dgrad alone (base_model's first layer at batch 64, 772x1032, bf16 da,
train-mode BatchNorm; inputs larger than L2) with its HBM floor, and a frozen eval-mode base_model at batch 64 in bf16:
forward + image-gradient backward against the same with parameter gradients on, and against the same torch.nn modules
under stock torch / cuDNN autograd (bf16 autocast, channels_last) as context.  CUDA events; prints one JSON line (with
the GPU's name, power limit and SM clocks) and appends it to --out."""
import argparse
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import yogo_b200  # noqa: E402
from oracle import yogo_oracle as O  # noqa: E402
from tools.bench_match import gpu_info  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402

DEV = "cuda:0"
HBM_BYTES_PER_S = 7.7e12


def event_ms(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def first_dgrad_case(N, H, W, iters):
    Cin, Cout, stride = 1, 16, 2
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = torch.rand(N, Cin, H, W, device=DEV)
    w = torch.randn(Cout, Cin, 3, 3, device=DEV) * 0.3
    da = torch.randn(N, Ho, Wo, Cout, device=DEV).to(torch.bfloat16)
    scale, shift = torch.rand(Cout, device=DEV) + 0.5, torch.randn(Cout, device=DEV) * 0.1
    mean, invstd = torch.randn(Cout, device=DEV) * 0.1, torch.rand(Cout, device=DEV) + 0.5
    m1, m2 = torch.randn(Cout, device=DEV) * 1e-3, torch.randn(Cout, device=DEV) * 1e-3
    dx = torch.empty_like(x)
    ep = L.BwdEpilogue(None, L.ACT_LRELU, None, scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), None)
    lib = L.lib()

    def call():
        L.check(lib.yg_conv_first_dgrad(x.data_ptr(), w.data_ptr(), da.data_ptr(), L.YG_BF16, N, H, W, Cin, Cout, stride,
                                        C.byref(ep), None, m1.data_ptr(), m2.data_ptr(), dx.data_ptr(), L.stream()))

    ms = event_ms(call, iters)
    nbytes = x.numel() * 4 + da.numel() * 2 + dx.numel() * 4
    return {"case": "yg_conv_first_dgrad", "N": N, "H": H, "W": W, "Cin": Cin, "Cout": Cout, "stride": stride,
            "da_dtype": "bf16", "bn": "batch", "ms": ms, "bytes": nbytes, "GBps": nbytes / ms / 1e6,
            "frac_of_7.7TBps": nbytes / (ms * 1e-3) / HBM_BYTES_PER_S}


def model_cases(N, H, W, iters):
    torch.manual_seed(0)
    net = yogo_b200.YOGO((H, W), O.ANCHOR_W, O.ANCHOR_H, 7)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.05)
    net = net.to(DEV)
    net.compute_dtype = torch.bfloat16
    net.eval()
    x = (O.synth_images(N, H, W).float() / 255.0).to(DEV)
    G = torch.randn((N, 12, net.Sy, net.Sx), device=DEV) * 0.1
    out = {}

    def step():
        xg = x.detach().requires_grad_(True)
        net(xg).backward(G)

    for p in net.parameters():
        p.requires_grad_(False)
    out["ours_frozen_image_grad_ms"] = event_ms(step, iters)
    for p in net.parameters():
        p.requires_grad_(True)
    net.zero_grad(set_to_none=True)
    out["ours_image_and_param_grads_ms"] = event_ms(step, iters)

    # stock torch / cuDNN autograd through the same modules, frozen, image gradient only
    backbone = net.model.to(memory_format=torch.channels_last)
    for p in backbone.parameters():
        p.requires_grad_(False)
    torch.backends.cudnn.benchmark = True
    hc = net._hc
    cxs, cys = net._Cxs, net._Cys

    def torch_step():   # model.py:277-313 with the module's grid offsets on the device
        xg = x.detach().to(memory_format=torch.channels_last).requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            t = backbone(xg)
        t = t.float()
        wh = torch.clamp(t[:, 2:4], max=80)
        o = torch.cat(((1 / net.Sx) * torch.sigmoid(t[:, 0:1]) + cxs, (1 / net.Sy) * torch.sigmoid(t[:, 1:2]) + cys,
                       hc["anchor_w"] * torch.exp(wh[:, 0:1]), hc["anchor_h"] * torch.exp(wh[:, 1:2]),
                       torch.sigmoid(t[:, 4:5]), t[:, 5:]), dim=1)
        o.backward(G)

    out["torch_cudnn_frozen_image_grad_ms"] = event_ms(torch_step, iters)
    out.update(model="base_model", N=N, H=H, W=W, compute="bf16", mode="eval, frozen")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "input_grad_bench.jsonl"))
    a = ap.parse_args()
    rec = {"bench": "input_grad", **gpu_info()}
    rec["first_dgrad"] = first_dgrad_case(a.batch, 772, 1032, a.iters)
    rec["model"] = model_cases(a.batch, 772, 1032, a.iters)
    line = json.dumps(rec)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
