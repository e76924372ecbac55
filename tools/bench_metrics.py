"""Evaluation metrics: yogo_b200.metrics.Metrics (matching, confusion and COCO matching per update on the device,
COCO accumulation in compute()) against the same evaluation through the numpy restatement tools/coco_eval_np.py on the
host (the CPU restatement: torchmetrics and pycocotools are not the baseline here).  Workloads: sparse-realistic 97x129
images in updates of 64, and the dense output of a randomly initialised network.  Checks that both give the same
confusion matrix and COCO arrays, prints one JSON line (with the GPU's name, power limit and SM clocks) and appends it to
--out."""
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

from tools import coco_eval_np as E  # noqa: E402
from tools.bench_match import DEV, dense_inputs, gpu_info, sparse_inputs  # noqa: E402
from yogo_b200 import Metrics  # noqa: E402
from yogo_b200.utils import format_preds_and_labels_batch, format_preds_batch  # noqa: E402

C = 7


def host_eval(batches):
    """The same evaluation on the host: the batched matching's rows, then the numpy restatement."""
    conf = np.zeros((C + 1, C + 1), np.int64)
    images = []
    for p, l in batches:
        m, _ = format_preds_and_labels_batch(p, l)
        cb = m.convert_background_errors(C + 1)
        conf += E.confusion_from_converted(cb.preds.cpu().numpy(), cb.labels.cpu().numpy(), C + 1)
        rows, kc, _, _ = format_preds_batch(p, 0.5, 0.5, "xyxy", 0.0)
        rows, kc, lab = rows.cpu().numpy(), kc.cpu().numpy(), l.cpu().numpy()
        for b in range(p.shape[0]):
            lr = lab[b].reshape(6, -1).T
            images.append(E.image_inputs(rows[b, :kc[b]], lr[lr[:, 0] != 0]))
    t0 = time.perf_counter()
    prec, rec, summ = E.coco_eval_np(images, C)
    return conf, prec, rec, summ, time.perf_counter() - t0


def run_case(name, p_cpu, l_cpu, batch):
    batches = [(p_cpu[i:i + batch].to(DEV), l_cpu[i:i + batch].to(DEV)) for i in range(0, p_cpu.shape[0], batch)]
    met = Metrics([str(k) for k in range(C)])
    met.update(*batches[0])   # warm-up
    met.compute()
    met.reset()
    torch.cuda.synchronize()
    upd = []
    for p, l in batches:
        t0 = time.perf_counter()
        met.update(p, l)
        torch.cuda.synchronize()
        upd.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    res = met.compute()
    compute_s = time.perf_counter() - t0
    conf, prec, rec, summ, cpu_s = host_eval(batches)
    equal = (np.array_equal(res["confusion"].numpy(), conf) and np.array_equal(res["coco_precision"].numpy(), prec)
             and np.array_equal(res["coco_recall"].numpy(), rec)
             and all(abs(res[k] - summ[k]) <= 1e-12 * abs(summ[k]) for k in ("map", "map_50", "map_75", "mar_1", "mar_10", "mar_100")))
    return {"case": name, "images": int(p_cpu.shape[0]), "update_batch": batch, "updates": len(batches),
            "update_ms_mean": round(1e3 * float(np.mean(upd)), 3), "update_ms_max": round(1e3 * float(np.max(upd)), 3),
            "compute_ms": round(1e3 * compute_s, 3), "cpu_restatement_coco_s": round(cpu_s, 2),
            "kept_predictions": int(sum(int((format_preds_batch(p)[1]).sum()) for p, _ in batches)),
            "map": res["map"], "map_50": res["map_50"], "mar_100": res["mar_100"], "results_equal": bool(equal)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=2048)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--dense-images", type=int, default=64)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    line = {"tool": "bench_metrics"}
    line.update(gpu_info())
    cases = []
    p, l = sparse_inputs(a.images, distinct=128)
    cases.append(run_case(f"sparse_realistic_97x129_{a.images}_images", p, l, a.batch))
    if a.dense_images > 0:
        p, l = dense_inputs(a.dense_images)
        cases.append(run_case(f"dense_random_init_{a.dense_images}_images", p, l, min(a.batch, a.dense_images)))
    line["cases"] = cases
    line["timing"] = ("host clock around each update() and around compute(), each ending in a device synchronise, after a "
                      "warm-up update; cpu_restatement_coco_s is tools/coco_eval_np.py's COCO evaluation on the host alone "
                      "(from the same matched rows), not the reference's torchmetrics")
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(s + "\n")
    if not all(c["results_equal"] for c in cases):
        raise SystemExit("device and host metrics differ")


if __name__ == "__main__":
    main()
