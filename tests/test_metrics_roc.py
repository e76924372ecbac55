"""ROC curves and calibration error of yogo_b200.metrics.Metrics: the numpy restatement (tools/roc_ece_np.py) against
known answers and sklearn on the CPU; on the GPU the stored score rows against the matched rows, curves, AUC and bins bit
for bit against the restatement fed the stored scores, invariance to how images are split into updates, the unchanged
outputs of the other metrics, errors, recovery and the buffers of the new C-ABI entry points."""
import numpy as np
import pytest
import torch

from oracle import yogo_oracle as O
from tools import roc_ece_np as E

DEV = "cuda:0"
C = 7


# ----------------------------------------------------------------------------------------------------- CPU: restatement
def test_roc_known_answer():
    fpr, tpr, thr, auc = E.roc_np([0.9, 0.8, 0.8, 0.3], [1, 0, 1, 0])
    assert fpr.dtype == tpr.dtype == np.float64 and thr.dtype == np.float32
    assert fpr.tolist() == [0, 0, 0.5, 1] and tpr.tolist() == [0, 0.5, 1, 1]
    assert np.array_equal(thr, np.float32([1, 0.9, 0.8, 0.3])) and auc == 0.875


def test_roc_degenerate_classes():
    fpr, tpr, thr, auc = E.roc_np([0.2, 0.7, 0.7], [1, 1, 1])   # no negatives
    assert fpr.tolist() == [0, 0, 0] and tpr.tolist() == [0, 2 / 3, 1] and auc == -1
    fpr, tpr, _, auc = E.roc_np([0.2, 0.7], [0, 0])             # no positives
    assert fpr.tolist() == [0, 0.5, 1] and tpr.tolist() == [0, 0, 0] and auc == -1
    fpr, tpr, thr, auc = E.roc_np([], [])
    assert fpr.tolist() == [0] and tpr.tolist() == [0] and thr.tolist() == [1] and auc == -1


def test_calibration_bin_edges():
    bounds = torch.linspace(0, 1, 16).numpy()
    scores = np.float32([[1.0, 0.0], [bounds[1], 0.0], [0.0, 0.0], [np.nextafter(bounds[1], np.float32(0)), 0.0]])
    count, correct, conf = E.calibration_bins_np(scores, [0, 1, 0, 0], bounds)
    assert count.size == 16 and count[15] == 1 and count[1] == 1 and count[0] == 2 and count.sum() == 4
    assert correct[15] == 1 and correct[1] == 0 and correct[0] == 2   # the first maximum of [0, 0] is class 0
    assert conf[15] == 1.0 and conf[1] == np.float64(bounds[1])
    ece, bconf, bacc = E.calibration_error_np(count, correct, conf)
    assert bconf[15] == 1 and bacc[15] == 1 and bacc[1] == 0 and bconf[2] == 0 and bacc[2] == 0
    assert ece == pytest.approx(0.25 * bounds[1] + 0.5 * (1 - np.float64(np.nextafter(bounds[1], np.float32(0))) / 2), abs=1e-12)
    assert E.calibration_error_np(np.zeros(16, np.int64), np.zeros(16, np.int64), np.zeros(16))[0] == -1


def test_missed_labels_have_confidence_one():
    scores, targets = E.score_rows_np(np.zeros((0, 5 + C)), np.zeros((0, 6)), [[1, 0, 0, .1, .1, 3]], np.zeros((0, 5 + C)), C)
    assert scores.tolist() == [[0] * C + [1]] and targets.tolist() == [3]
    count, correct, _ = E.calibration_bins_np(scores, targets, torch.linspace(0, 1, 16).numpy())
    assert count[15] == 1 and correct[15] == 0


@pytest.mark.parametrize("kind", ["random", "tie_heavy", "single_class", "all_positive"])
def test_roc_restatement_matches_sklearn(kind):
    skm = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(7)
    for n in (1, 2, 5, 50, 3000):
        s = rng.random(n).astype(np.float32)
        y = rng.random(n) < 0.3
        if kind == "tie_heavy":
            s = np.ceil(s * 8).astype(np.float32) / 8
        elif kind == "single_class":
            y[:] = False
            y[0] = True
        elif kind == "all_positive":
            y[:] = True
            y[0] = n == 1
        fpr, tpr, thr, auc = E.roc_np(s, y)
        if y.all() or not y.any():
            continue   # sklearn warns and returns NaN rates where torchmetrics and the restatement return zeros
        f, t, th = skm.roc_curve(y, s, drop_intermediate=False)
        assert np.array_equal(fpr, f) and np.array_equal(tpr, t) and np.array_equal(thr[1:], th[1:].astype(np.float32))
        assert abs(auc - skm.auc(f, t)) <= 1e-12


def test_format_rule():
    p = np.float32([[0.2, 0.8], [0.0, 1.0]])
    s, soft = E.apply_format_rule(p)
    assert not soft and s is not None and np.array_equal(s, p)
    s, soft = E.apply_format_rule(np.float32([[0.2, 1.5], [0.0, 1.0]]))
    x = np.float64([[0.2, 1.5], [0.0, 1.0]])
    assert soft and np.allclose(s, np.exp(x) / np.exp(x).sum(1, keepdims=True), rtol=1e-7, atol=0)


# ----------------------------------------------------------------------------------------------------- GPU helpers
def _sparse_batch(B, seed):
    """Sparse-realistic 97x129 predictions with labels; image 1 has more labels than predictions (missed labels)."""
    preds = O.synth_sparse_preds(B, 97, 129, C, 300, seed=seed)
    labels = torch.stack([O.synth_labels_for_preds(preds[b], (0.05, 0.2, 0.5)[b % 3], (0, 5, 40)[b % 3], seed=seed * 100 + b)
                          for b in range(B)])
    if B > 1:
        labels[1] = O.synth_labels_for_preds(preds[1], 0.0, 30, seed=5)
        preds[1] = O.synth_sparse_preds(1, 97, 129, C, 20, seed=seed + 1)[0]
    return preds, labels


def _expected_rows(p, l, with_bg=True):
    """The update's raw score rows and targets in the kernel's order: image by image, matched / missed / extra."""
    from yogo_b200.utils import format_preds_and_labels_batch
    m, counts = format_preds_and_labels_batch(p, l)
    mp, ml, mm, me = (x.cpu().numpy() for x in (m.preds, m.labels, m.missed_labels, m.extra_predictions))
    off = np.zeros(3, np.int64)
    rows, targets = [], []
    for k, n, e in counts.numpy():
        s, t = E.score_rows_np(mp[off[0]:off[0] + k], ml[off[0]:off[0] + k], mm[off[1]:off[1] + n], me[off[2]:off[2] + e], C,
                               with_bg)
        rows.append(s)
        targets.append(t)
        off += (k, n, e)
    return np.concatenate(rows), np.concatenate(targets)


def _stored(met):
    return (torch.cat(met._scores).cpu().numpy() if met._scores else np.zeros((0, met._side), np.float32),
            torch.cat(met._targets).cpu().numpy())


def _assert_matches_restatement(met, res, bins=15):
    """Curves, AUC and bin counts bit-identical to the restatement fed the stored scores; confidence sums to 1e-12."""
    skm = pytest.importorskip("sklearn.metrics")
    scores, targets = _stored(met)
    curves, aucs = E.roc_all_np(scores, targets)
    assert len(res["roc"]) == met._side and np.array_equal(res["roc_auc"].numpy(), aucs)
    for k, ((fpr, tpr, thr), (f, t, th)) in enumerate(zip(res["roc"], curves)):
        assert fpr.dtype == tpr.dtype == torch.float64 and thr.dtype == torch.float32
        assert np.array_equal(fpr.numpy(), f) and np.array_equal(tpr.numpy(), t), k
        assert np.array_equal(thr.numpy().view(np.uint32), th.view(np.uint32)), k
        pos = targets == k
        if pos.any() and not pos.all():
            sf, st, _ = skm.roc_curve(pos, scores[:, k], drop_intermediate=False)
            assert np.array_equal(fpr.numpy(), sf) and np.array_equal(tpr.numpy(), st), k
    count, correct, conf = E.calibration_bins_np(scores, targets, torch.linspace(0, 1, bins + 1).numpy())
    assert np.array_equal(res["calibration_bin_count"].numpy(), count)
    ece, bconf, bacc = E.calibration_error_np(count, correct, conf)
    assert np.array_equal(res["calibration_bin_accuracy"].numpy(), bacc)
    assert np.allclose(res["calibration_bin_confidence"].numpy(), bconf, rtol=1e-12, atol=0)
    assert res["calibration_error"] == pytest.approx(ece, rel=1e-12, abs=1e-15)
    return scores, targets


def _metrics(**kw):
    from yogo_b200 import Metrics
    return Metrics([str(k) for k in range(C)], include_roc=True, include_calibration=True, **kw)


# ----------------------------------------------------------------------------------------------------- GPU: scores
@pytest.mark.gpu
def test_stored_scores_follow_the_per_update_format_rule():
    met = _metrics(include_mAP=False)
    exp_rows, soft = [], []
    for i, seed in enumerate((81, 82, 83)):
        p, l = _sparse_batch(12, seed)
        if i == 1:
            p[:, 5:] = torch.log(p[:, 5:]) * 1.7   # logits: this update alone is softmaxed
        p, l = p.to(DEV), l.to(DEV)
        met.update(p, l)
        raw, _ = _expected_rows(p, l)
        exp_rows.append(raw)
        soft.append(E.apply_format_rule(raw)[1])
    assert soft == [False, True, False]
    for i, (st, raw) in enumerate(zip(met._scores, exp_rows)):
        st = st.cpu().numpy()
        if i == 1:
            ref = torch.softmax(torch.from_numpy(raw).double(), 1).numpy()
            ulp = np.spacing(ref.astype(np.float32))
            assert np.all(np.abs(st - ref) <= 2 * ulp)
        else:
            assert np.array_equal(st.view(np.uint32), raw.view(np.uint32))
    _assert_matches_restatement(met, met.compute())


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["sparse", "sparse_no_background", "tie_heavy", "degenerate_classes", "dense_random_init"])
def test_roc_and_calibration_match_the_restatement(case):
    with_bg = case not in ("sparse_no_background", "degenerate_classes")
    met = _metrics(include_background=with_bg, calibration_bins=10 if case == "tie_heavy" else 15)
    if case == "dense_random_init":
        import yogo_b200
        torch.manual_seed(0)
        net = yogo_b200.YOGO((772, 1032), O.ANCHOR_W, O.ANCHOR_H, C).to(DEV).eval()
        with torch.no_grad():
            p = net((O.synth_images(4, 772, 1032).float() / 255.0).to(DEV)).float()
        batches = [(p, O.synth_labels(4, 97, 129, C, 300).to(DEV))]
    else:
        batches = []
        for seed in (91, 92, 93):
            p, l = _sparse_batch(16, seed)
            if case == "tie_heavy":
                p[:, 5:] = torch.ceil(p[:, 5:] * 8) / 8
            if case == "degenerate_classes":
                l[:, 5] = 0   # class 0: no negatives (every matched pair is class 0); classes 1..6: no positives
            batches.append((p.to(DEV), l.to(DEV)))
    for p, l in batches:
        met.update(p, l)
        raw, tgt = _expected_rows(p, l, with_bg)
        assert np.array_equal(E.apply_format_rule(raw)[0], met._scores[-1].cpu().numpy()) or case == "dense_random_init"
        assert np.array_equal(tgt, met._targets[-1].cpu().numpy())
    res = met.compute()
    scores, targets = _assert_matches_restatement(met, res, 10 if case == "tie_heavy" else 15)
    assert res["calibration_bin_count"].numel() == (11 if case == "tie_heavy" else 16)
    if case != "dense_random_init":   # missed labels (image 1) and extra predictions
        assert (targets == C).any() == with_bg and (res["calibration_bin_count"][-1] > 0) == with_bg
    if case == "tie_heavy":
        assert np.unique(scores).size <= 9 and all(len(c[0]) <= 10 for c in res["roc"])
    if case == "degenerate_classes":
        auc = res["roc_auc"].numpy()
        assert np.all(auc == -1) and np.all(res["roc"][0][0].numpy() == 0) and np.all(res["roc"][1][1].numpy() == 0)
    else:
        assert np.all((res["roc_auc"].numpy() > 0.3) & (res["roc_auc"].numpy() <= 1))


@pytest.mark.gpu
def test_splitting_updates_and_repeating_runs_give_the_same_outputs():
    p, l = _sparse_batch(48, 95)
    p, l = p.to(DEV), l.to(DEV)

    def run(splits):
        met = _metrics()
        o = 0
        for n in splits:
            met.update(p[o:o + n], l[o:o + n])
            o += n
        return met.compute()

    a, b, c = run([48]), run([5, 30, 13]), run([5, 30, 13])
    for x in (b, c):
        assert np.array_equal(a["roc_auc"].numpy(), x["roc_auc"].numpy())
        for ca, cx in zip(a["roc"], x["roc"]):
            assert all(torch.equal(u, v) for u, v in zip(ca, cx))
        assert torch.equal(a["calibration_bin_count"], x["calibration_bin_count"])
        assert torch.equal(a["calibration_bin_accuracy"], x["calibration_bin_accuracy"])
        assert np.allclose(a["calibration_bin_confidence"].numpy(), x["calibration_bin_confidence"].numpy(), rtol=1e-12, atol=0)
    assert torch.equal(b["calibration_bin_confidence"], c["calibration_bin_confidence"])
    assert b["calibration_error"] == c["calibration_error"]


@pytest.mark.gpu
@pytest.mark.parametrize("with_bg", [True, False])
def test_flags_leave_the_other_outputs_unchanged(with_bg):
    from yogo_b200 import Metrics
    on = _metrics(include_background=with_bg, min_class_confidence_threshold=0.1)
    off = Metrics([str(k) for k in range(C)], include_background=with_bg, min_class_confidence_threshold=0.1)
    for seed in (97, 98):
        p, l = _sparse_batch(8, seed)
        p, l = p.to(DEV), l.to(DEV)
        on.update(p, l)
        off.update(p, l)
    a, b = on.compute(), off.compute()
    assert set(b) == {"confusion", "precision", "recall", "num_images", "map", "map_50", "map_75", "mar_1", "mar_10", "mar_100",
                      "map_per_class", "mar_100_per_class", "coco_precision", "coco_recall"}
    assert set(a) == set(b) | {"roc", "roc_auc", "calibration_error", "calibration_bin_count", "calibration_bin_confidence",
                               "calibration_bin_accuracy"}
    for k, v in b.items():
        assert (torch.equal(v, a[k]) if isinstance(v, torch.Tensor) else v == a[k]), k
    only_roc = Metrics([str(k) for k in range(C)], include_mAP=False, include_roc=True)
    only_roc.update(p, l)
    assert set(only_roc.compute()) == {"confusion", "precision", "recall", "num_images", "roc", "roc_auc"}


# ----------------------------------------------------------------------------------------------------- GPU: errors
@pytest.mark.gpu
def test_errors_raise_and_the_new_state_recovers():
    met = _metrics()
    p, l = _sparse_batch(4, 99)
    p, l = p.to(DEV), l.to(DEV)
    met.update(p, l)
    before = met.compute()
    n_scores = sum(s.shape[0] for s in met._scores)

    def unchanged():
        res = met.compute()
        assert sum(s.shape[0] for s in met._scores) == n_scores and res["num_images"] == 4
        assert torch.equal(res["calibration_bin_count"], before["calibration_bin_count"])
        assert torch.equal(res["calibration_bin_confidence"], before["calibration_bin_confidence"])
        assert all(torch.equal(u, v) for cu, cv in zip(res["roc"], before["roc"]) for u, v in zip(cu, cv))

    lb = l.clone()
    cells = torch.nonzero(lb[1, 0].reshape(-1)).flatten()
    lb[1, 5].view(-1)[cells[len(cells) // 2]] = float(C)
    with pytest.raises(ValueError, match=r"label class outside \[0, 7\) \(image 1\)"):
        met.update(p, lb)
    unchanged()
    for value in (float("nan"), float("inf")):   # an infinite class value becomes NaN under the softmax, as in torch
        pb = p.clone()
        kept = torch.nonzero(pb[2, 4].reshape(-1) > 0.5).flatten()
        pb[2, 6].view(-1)[kept[0]] = value
        with pytest.raises(ValueError, match=r"NaN class score \(image 2\)"):
            met.update(pb, l)
        unchanged()
    met.update(p, l)   # the next update succeeds
    res = met.compute()
    assert torch.equal(res["calibration_bin_count"], 2 * before["calibration_bin_count"]) and res["num_images"] == 8
    _assert_matches_restatement(met, res)
    met.reset()
    assert met._scores == [] and met._targets == [] and met._bins is None
    with pytest.raises(RuntimeError):
        met.compute()
    met.update(p, l)
    res = met.compute()
    assert torch.equal(res["calibration_bin_count"], before["calibration_bin_count"])
    assert all(torch.equal(u, v) for cu, cv in zip(res["roc"], before["roc"]) for u, v in zip(cu, cv))
    with pytest.raises(ValueError, match="calibration_bins"):
        _metrics(calibration_bins=0)


# ----------------------------------------------------------------------------------------------------- GPU: buffers
@pytest.mark.gpu
def test_outputs_of_the_roc_and_calibration_kernels_stay_inside_their_buffers():
    """Guard regions around every output of yg_score_rows_batch, yg_roc_keys and yg_roc_curves."""
    import ctypes

    from yogo_b200 import _lib as L
    from yogo_b200.utils.prediction_formatting import _match_batch
    lib = L.lib()
    GUARD = 4096

    def guarded(shape, dtype, fill):
        numel = int(np.prod(shape))
        buf = torch.full((numel + 2 * GUARD,), fill, dtype=dtype, device=DEV)
        return buf, buf[GUARD:GUARD + numel].view(*shape)

    def intact(buf, view, fill):
        n = view.numel()
        return bool((buf[:GUARD] == fill).all()) and bool((buf[GUARD + n:] == fill).all())

    B, Sy, Sx, bins = 3, 13, 17, 15
    preds = O.synth_sparse_preds(B, Sy, Sx, C, 25, seed=8)
    labels = torch.stack([O.synth_labels_for_preds(preds[b], 0.3, (0, 3, 30)[b], seed=b) for b in range(B)])
    r = _match_batch(preds.to(DEV), labels.to(DEV), 0.5, 0.0)
    m = r.match
    nk, ne = m.preds.shape[0], m.extra_predictions.shape[0]
    R, nb, nbin = nk + m.missed_labels.shape[0] + ne, C + 1, bins + 1
    bounds = torch.linspace(0, 1, nbin).numpy()
    outs = [guarded((1,), torch.int32, 77), guarded((R, nb), torch.float32, 7.0), guarded((R,), torch.int32, 77),
            guarded((B,), torch.int32, 77), guarded((B * nbin * 16,), torch.uint8, 77), guarded((nbin,), torch.int64, 77),
            guarded((nbin,), torch.int64, 77), guarded((nbin,), torch.float64, 7.0)]
    flag, scores, targets, nan_status, partials, count, correct, conf = (v for _, v in outs)
    L.check(lib.yg_score_rows_batch(m.preds.data_ptr(), m.labels.data_ptr(), m.missed_labels.data_ptr(),
                                    m.extra_predictions.data_ptr(), nk, ne, B, C, 1, r.table.data_ptr(), r.table[4 * B:].data_ptr(),
                                    r.status.data_ptr(), (ctypes.c_float * nbin)(*bounds.tolist()), bins, flag.data_ptr(),
                                    scores.data_ptr(), targets.data_ptr(), nan_status.data_ptr(), partials.data_ptr(),
                                    count.data_ptr(), correct.data_ptr(), conf.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert r.status.cpu().tolist() == [0] * B and nan_status.cpu().tolist() == [0] * B and flag.item() == 0
    assert int(count.sum()) == R and bool((scores != 7.0).all()) and bool((targets != 77).all())
    for (buf, view), fill in zip(outs, (77, 7.0, 77, 77, 77, 77, 77, 7.0)):
        assert intact(buf, view, fill)
    kbuf, keys = guarded((nb * R,), torch.int64, 77)
    L.check(lib.yg_roc_keys(scores.data_ptr(), R, nb, keys.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert intact(kbuf, keys, 77) and bool((keys != 77).all())
    sk, perm = torch.sort(keys)
    curve = [guarded((nb, R + 1), torch.float64, 7.0), guarded((nb, R + 1), torch.float64, 7.0),
             guarded((nb, R + 1), torch.float32, 7.0), guarded((nb,), torch.int64, 77), guarded((nb,), torch.float64, 7.0)]
    fpr, tpr, thr, lengths, auc = (v for _, v in curve)
    L.check(lib.yg_roc_curves(sk.data_ptr(), perm.data_ptr(), targets.data_ptr(), R, nb, fpr.data_ptr(), tpr.data_ptr(),
                              thr.data_ptr(), lengths.data_ptr(), auc.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    for (buf, view), fill in zip(curve, (7.0, 7.0, 7.0, 77, 7.0)):
        assert intact(buf, view, fill)
    n = lengths.cpu().tolist()
    assert all(2 <= x <= R + 1 for x in n) and bool((auc != 7.0).all())
    curves, aucs = E.roc_all_np(scores.cpu().numpy(), targets.cpu().numpy())
    for k in range(nb):
        assert np.array_equal(fpr[k, :n[k]].cpu().numpy(), curves[k][0]) and np.array_equal(thr[k, :n[k]].cpu().numpy(), curves[k][2])
    assert np.array_equal(auc.cpu().numpy(), aucs)
