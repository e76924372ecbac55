"""Evaluation matching: the per-image loop (format_preds_and_labels_v2, scipy on the host) against the batched call
(format_preds_and_labels_batch, assignment on the device) and the assignment kernel alone, on sparse-realistic
97x129 inputs at B = 64 and 256 and on the dense output of a randomly initialised network.  Checks that the batched and
per-image results are bit-equal and prints one JSON line (with the GPU's name, power limit and SM clocks)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import yogo_b200  # noqa: E402
from oracle import yogo_oracle as O  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402
from yogo_b200.utils import PredictionLabelMatch, format_preds_and_labels_batch, format_preds_and_labels_v2, format_preds_batch  # noqa: E402
from yogo_b200.utils.prediction_formatting import _lsap_plan  # noqa: E402

DEV = "cuda:0"


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, pl, sm, smmax = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit_w": float(pl), "sm_clock_mhz": float(sm), "sm_clock_max_mhz": float(smmax)}


def sparse_inputs(B, distinct=64):
    """sparse-realistic predictions (tools/synth.py) with matching labels; images repeat every `distinct`."""
    p = O.synth_sparse_preds(distinct, 97, 129, 7, 300, seed=31)
    lab = torch.stack([O.synth_labels_for_preds(p[b], (0.05, 0.2, 0.4)[b % 3], (0, 5, 20)[b % 3], seed=b) for b in range(distinct)])
    reps = (B + distinct - 1) // distinct
    return p.repeat(reps, 1, 1, 1)[:B].contiguous(), lab.repeat(reps, 1, 1, 1)[:B].contiguous()


def dense_inputs(B):
    """output of a randomly initialised network (objectness near 0.5 everywhere: thousands of predictions per image)."""
    torch.manual_seed(0)
    net = yogo_b200.YOGO((772, 1032), O.ANCHOR_W, O.ANCHOR_H, 7).to(DEV).eval()
    x = (O.synth_images(B, 772, 1032).float() / 255.0).to(DEV)
    with torch.no_grad():
        out = net(x).float()
    return out.cpu(), O.synth_labels(B, 97, 129, 7, 300)


def same(a, b):
    pairs = ((a.preds, b.preds), (a.labels, b.labels), (a.missed_labels, b.missed_labels), (a.extra_predictions, b.extra_predictions))
    return all(x.shape == y.shape and torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in pairs)


def lsap_alone(p, l, reps):
    """the assignment kernel by itself on the pipeline's packed cost matrices, CUDA events over `reps` launches."""
    lib = L.lib()
    B, D, Sy, Sx = p.shape
    cells = Sy * Sx
    rows, kc, _, _ = format_preds_batch(p, 0.5, 0.5, "xyxy", 0.0)
    lrows = torch.empty((B, cells, 6), device=DEV)
    nl = torch.empty(B, dtype=torch.int32, device=DEV)
    L.check(lib.yg_compact_labels(l.float().contiguous().data_ptr(), B, Sy, Sx, lrows.data_ptr(), nl.data_ptr(), L.stream()))
    N, M = nl.cpu().numpy().astype(np.int64), kc.cpu().numpy().astype(np.int64)
    K = np.minimum(N, M)
    plan, words = _lsap_plan(N, M)
    table = torch.from_numpy(plan).to(DEV)
    Kt, Nt, Mt = int(K.sum()), int(N.sum()), int(M.sum())
    costs = torch.empty(max(int((N * M).sum()), 1), device=DEV)
    ws = torch.empty(max(words, 1), dtype=torch.float64, device=DEV)
    pr, pc = torch.empty(max(Kt, 1), dtype=torch.int64, device=DEV), torch.empty(max(Kt, 1), dtype=torch.int64, device=DEV)
    st = torch.empty(B, dtype=torch.int32, device=DEV)
    outs = [torch.empty((max(n, 1), w), device=DEV) for n, w in ((Kt, D), (Kt, 6), (Nt - Kt, 6), (Mt - Kt, D))]
    L.check(lib.yg_match_batch(lrows.data_ptr(), rows.data_ptr(), B, cells, D - 5, int(N.max()), int(M.max()), table.data_ptr(),
                               table[4 * B:].data_ptr(), costs.data_ptr(), ws.data_ptr(), pr.data_ptr(), pc.data_ptr(), st.data_ptr(),
                               *[o.data_ptr() for o in outs], L.stream()))

    def launch():
        L.check(lib.yg_lsap_batch(costs.data_ptr(), table.data_ptr(), B, ws.data_ptr(), pr.data_ptr(), pc.data_ptr(), st.data_ptr(),
                                  L.stream()))

    launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [0] * B
    return e0.elapsed_time(e1) / reps, {"labels_mean": float(N.mean()), "preds_mean": float(M.mean()), "labels_max": int(N.max()),
                                        "preds_max": int(M.max()), "cost_mb": float((N * M).sum() * 4 / 1e6)}


def run_case(name, p_cpu, l_cpu, loop_reps, reps):
    p, l = p_cpu.to(DEV), l_cpu.to(DEV)
    B = p.shape[0]

    def loop():
        return PredictionLabelMatch.concat([format_preds_and_labels_v2(p[b], l[b]) for b in range(B)])

    ref = loop()   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(loop_reps):
        loop()
    torch.cuda.synchronize()
    loop_ms = (time.perf_counter() - t0) * 1e3 / loop_reps
    got, _ = format_preds_and_labels_batch(p, l)
    got, _ = format_preds_and_labels_batch(p, l)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        format_preds_and_labels_batch(p, l)
    torch.cuda.synchronize()
    batch_ms = (time.perf_counter() - t0) * 1e3 / reps
    kern_ms, sizes = lsap_alone(p, l, reps)
    r = {"case": name, "B": B, "per_image_loop_ms": round(loop_ms, 3), "batched_ms": round(batch_ms, 3),
         "lsap_kernel_ms": round(kern_ms, 4), "speedup": round(loop_ms / batch_ms, 1), "bit_equal": same(got, ref)}
    r.update(sizes)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,256")
    ap.add_argument("--dense-batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop-reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    line = {"tool": "bench_match"}
    line.update(gpu_info())
    cases = []
    for B in [int(x) for x in a.batches.split(",") if x]:
        p, l = sparse_inputs(B)
        cases.append(run_case(f"sparse_realistic_97x129_b{B}", p, l, a.loop_reps, a.reps))
    if a.dense_batch > 0:
        p, l = dense_inputs(a.dense_batch)
        cases.append(run_case(f"dense_random_init_b{a.dense_batch}", p, l, 1, max(a.reps // 2, 1)))
    line["cases"] = cases
    line["timing"] = ("host clock around whole calls ending in a device synchronise (loop and batched call); CUDA events "
                      "around back-to-back launches of yg_lsap_batch alone; inputs resident in HBM, L2 not flushed")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")
    if not all(c["bit_equal"] for c in cases):
        raise SystemExit("batched and per-image results differ")


if __name__ == "__main__":
    main()
