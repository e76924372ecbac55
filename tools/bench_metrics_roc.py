"""ROC curves and calibration error of yogo_b200.metrics.Metrics: update() with include_roc and include_calibration against
update() without them (sparse-realistic 97x129 images in updates of 64), compute() with both flags at 2048 images and on
the dense output of a randomly initialised network, and the numpy restatement tools/roc_ece_np.py on the host fed the
same stored scores.  Checks that curves, AUC and bin counts are equal, prints one JSON line (with the GPU's name, power
limit and SM clocks) and appends it to --out.  tools/bench_metrics.py keeps timing the default metrics."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools import roc_ece_np as E  # noqa: E402
from tools.bench_match import DEV, dense_inputs, gpu_info, sparse_inputs  # noqa: E402
from yogo_b200 import Metrics  # noqa: E402

C = 7


def timed_updates(met, batches):
    met.reset()
    torch.cuda.synchronize()
    upd = []
    for p, l in batches:
        t0 = time.perf_counter()
        met.update(p, l)
        torch.cuda.synchronize()
        upd.append(time.perf_counter() - t0)
    return upd


def host_restatement(met, bins):
    scores = torch.cat(met._scores).cpu().numpy()
    targets = torch.cat(met._targets).cpu().numpy()
    t0 = time.perf_counter()
    curves, aucs = E.roc_all_np(scores, targets)
    count, correct, conf = E.calibration_bins_np(scores, targets, torch.linspace(0, 1, bins + 1).numpy())
    ece = E.calibration_error_np(count, correct, conf)[0]
    return curves, aucs, count, ece, time.perf_counter() - t0, scores.shape[0]


def run_case(name, p_cpu, l_cpu, batch, reps):
    batches = [(p_cpu[i:i + batch].to(DEV), l_cpu[i:i + batch].to(DEV)) for i in range(0, p_cpu.shape[0], batch)]
    names = [str(k) for k in range(C)]
    plain = Metrics(names)
    full = Metrics(names, include_roc=True, include_calibration=True)
    for met in (plain, full):   # warm-up
        met.update(*batches[0])
        met.compute()
    upd_plain, upd_full = [], []
    for _ in range(reps):   # alternate the two configurations
        upd_plain += timed_updates(plain, batches)
        upd_full += timed_updates(full, batches)
    comp = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = full.compute()
        comp.append(time.perf_counter() - t0)
    curves, aucs, count, ece, cpu_s, rows = host_restatement(full, full.calibration_bins)
    equal = (np.array_equal(res["roc_auc"].numpy(), aucs) and np.array_equal(res["calibration_bin_count"].numpy(), count)
             and all(np.array_equal(a.numpy(), b) for got, exp in zip(res["roc"], curves) for a, b in zip(got, exp))
             and abs(res["calibration_error"] - ece) <= 1e-12)
    return {"case": name, "images": int(p_cpu.shape[0]), "update_batch": batch, "updates": len(batches), "score_rows": rows,
            "update_ms_mean_without_flags": round(1e3 * float(np.mean(upd_plain)), 3),
            "update_ms_mean_with_roc_and_calibration": round(1e3 * float(np.mean(upd_full)), 3),
            "update_ms_median_without_flags": round(1e3 * float(np.median(upd_plain)), 3),
            "update_ms_median_with_roc_and_calibration": round(1e3 * float(np.median(upd_full)), 3),
            "update_ms_max_without_flags": round(1e3 * float(np.max(upd_plain)), 3),
            "update_ms_max_with_roc_and_calibration": round(1e3 * float(np.max(upd_full)), 3),
            "compute_ms_with_roc_and_calibration": round(1e3 * float(np.min(comp)), 3),
            "cpu_restatement_roc_ece_s": round(cpu_s, 3), "calibration_error": res["calibration_error"],
            "roc_auc": [round(float(x), 6) for x in res["roc_auc"]], "results_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=2048)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--dense-images", type=int, default=64)
    ap.add_argument("--reps", type=int, default=2, help="alternating passes over the updates of each configuration")
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    line = {"tool": "bench_metrics_roc"}
    line.update(gpu_info())
    cases = []
    p, l = sparse_inputs(a.images, distinct=128)
    cases.append(run_case(f"sparse_realistic_97x129_{a.images}_images", p, l, a.batch, a.reps))
    if a.dense_images > 0:
        p, l = dense_inputs(a.dense_images)
        cases.append(run_case(f"dense_random_init_{a.dense_images}_images", p, l, min(a.batch, a.dense_images), a.reps))
    line["cases"] = cases
    line["timing"] = ("host clock around each update() and around compute(), each ending in a device synchronise, after a "
                      "warm-up; the two configurations alternate pass by pass; compute_ms is the best of 3 calls; "
                      "cpu_restatement_roc_ece_s is tools/roc_ece_np.py on the host from the same stored scores")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")
    if not all(c["results_equal"] for c in cases):
        raise SystemExit("device and host ROC / calibration differ")


if __name__ == "__main__":
    main()
