"""Per-layer micro-benchmark of the convolution entry points (CUDA events, inputs > L2 rotate).

    python tools/bench_conv.py [--batch 64] [--only fwd,dgrad,wgrad] [--layers 2,3,4,5,6] [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402
if os.environ.get("YOGO_B200_LIB_ALT"):   # A/B runs of two builds on the same box
    L.LIB_PATH = os.environ["YOGO_B200_LIB_ALT"]

# base_model layers 2..7: (H, W, Cin, Cout, stride)
LAYERS = {2: (386, 516, 16, 32, 1), 3: (386, 516, 32, 64, 2), 4: (193, 258, 64, 128, 1), 5: (193, 258, 128, 128, 2),
          6: (97, 129, 128, 128, 1)}
DOUBLE = {12: (386, 516, 32, 64, 1), 13: (386, 516, 64, 128, 2), 14: (193, 258, 128, 256, 1), 15: (193, 258, 256, 256, 2),
          16: (97, 129, 256, 256, 1)}
LAYERS.update(DOUBLE)
# W-folded views of layer 2 (same bytes, 2x / 4x channels): tests the TMA row-rate hypothesis
LAYERS.update({22: (386, 258, 32, 64, 1), 23: (386, 129, 64, 128, 1), 32: (386, 258, 64, 64, 1)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--only", default="fwd,dgrad,wgrad")
    ap.add_argument("--layers", default="2,3,4,5,6")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--impl", default="auto")
    ap.add_argument("--stats", type=int, default=0)
    ap.add_argument("--tc-options", type=int, default=None, help="option word of include/yogo_b200.h (default: leave as is)")
    ap.add_argument("--no-saved", type=int, default=0)
    ap.add_argument("--mask", type=int, default=0)
    args = ap.parse_args()
    lib = L.lib()
    L.set_conv_impl(args.impl)
    if args.tc_options is not None:
        L.check(lib.yg_set_tc_options(args.tc_options))
    opt = lib.yg_get_tc_options()
    dev = "cuda:0"
    N = args.batch
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0}
    out = []
    for li in [int(v) for v in args.layers.split(",")]:
        H, W, Cin, Cout, s = LAYERS[li]
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        x = torch.randn(N, H, W, Cin, device=dev).bfloat16()
        dz = torch.randn(N, Ho, Wo, Cout, device=dev).bfloat16()
        w = torch.randn(Cout, Cin, 3, 3, device=dev) * 0.05
        b = torch.zeros(Cout, device=dev)
        y = torch.empty(N, Ho, Wo, Cout, device=dev, dtype=torch.bfloat16)
        dx = torch.empty_like(x)
        ymask = torch.empty(y.numel() // 8, dtype=torch.uint8, device=dev)
        mask = torch.randint(0, 255, (x.numel() // 8,), dtype=torch.uint8, device=dev)
        dw = torch.empty_like(w)
        stats = torch.zeros(2 * Cout, dtype=torch.float64, device=dev) if args.stats else None
        nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, 3, s)
        ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
        flops = 2.0 * N * Ho * Wo * Cout * Cin * 9
        st = L.stream()

        def fwd():
            ep = L.FwdEpilogue(None, b.data_ptr(), 1, None, L.ptr(stats), None, ymask.data_ptr() if args.mask else None)
            L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(ep), st))

        def dgrad():
            ep = L.BwdEpilogue(None if args.no_saved else x.data_ptr(), 1, None, None, None, None, None, None,
                               mask.data_ptr() if args.mask else None)
            L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(ep), st))

        def wgrad():
            L.check(lib.yg_conv_wgrad(x.data_ptr(), dz.data_ptr(), dw.data_ptr(), None, 1, N, H, W, Cin, Cout, 3, s, 1.0,
                                      ws.data_ptr(), nb, st))

        for name, fn in (("fwd", fwd), ("dgrad", dgrad), ("wgrad", wgrad)):
            if name not in args.only.split(","):
                continue
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / max(args.reps, 1)   # --reps 0: one launch per op (ncu captures)
            tf = flops / ms / 1e9
            act_bytes = (N * H * W * Cin + N * Ho * Wo * Cout) * 2
            rec = {"opt": opt, "layer": li, "op": name, "shape": [N, H, W, Cin, Cout, s], "ms": round(ms, 4), "TFLOPs": round(tf, 1),
                   "frac_bf16_peak": round(tf / peaks["bf16_tflops"], 3), "min_GBps": round(act_bytes / ms / 1e6, 1)}
            if (opt >> 11) & 1 and name != "wgrad":
                import numpy as np
                buf = np.zeros(148 * 16, dtype=np.uint64)
                L.check(lib.yg_tc_debug_read(buf.ctypes.data, buf.size))
                d = buf.reshape(148, 16).astype(np.float64)
                items = max(d[:, 5].mean(), 1.0)
                rec["mma_warp_cycles_per_item"] = {k: round(float(d[:, i].mean() / items), 1)
                                                   for i, k in enumerate(["wait_tempty", "wait_full", "issue", "commit", "rest"])}
                rec["items_per_cta"] = items
                rec["mma_warp_loop_entry_exit_cycles"] = [round(float(d[:, 6].mean())), round(float(d[:, 7].mean())), round(float(d[:, 7].max()))]
                tiles = max(d[:, 14].mean(), 1.0)
                rec["epi_warp_cycles_per_tile"] = {k: round(float(d[:, 8 + i].mean() / tiles), 1)
                                                   for i, k in enumerate(["wait_tfull", "ld_wait", "pre", "math", "store", "rest"])}
            print(json.dumps(rec), flush=True)
            out.append(rec)


if __name__ == "__main__":
    main()
