"""Evaluation metrics (yogo_b200.metrics.Metrics): the numpy restatement (tools/coco_eval_np.py) against known answers and
sklearn on the CPU; on the GPU the confusion matrix against the reference goldens and the host path, COCO mAP bit for
bit against the restatement, errors, recovery and the buffers of the new C-ABI entry points."""
import numpy as np
import pytest
import torch

from _golden import load as _load
from oracle import yogo_oracle as O
from tools import coco_eval_np as E

DEV = "cuda:0"
C = 7


def _single(dts, scores, gts, dcls=None, gcls=None, num_classes=1):
    dts, gts = np.float32(dts).reshape(-1, 4), np.float32(gts).reshape(-1, 4)
    dcls = np.zeros(len(dts), np.int64) if dcls is None else np.array(dcls)
    gcls = np.zeros(len(gts), np.int64) if gcls is None else np.array(gcls)
    return E.coco_eval_np([(dts, np.float32(scores), dcls, gts, gcls)], num_classes)


# ----------------------------------------------------------------------------------------------------- CPU: restatement
def test_coco_restatement_known_answers():
    close = lambda a, b: abs(a - b) <= 1e-12   # noqa: E731 - the spacing(1) term keeps precision just below 1
    # (a) one detection at IoU ~ .62
    p, _, s = _single([[0, 0, .1, .062]], [.9], [[0, 0, .1, .1]])
    assert close(s["map"], 0.3) and close(s["map_50"], 1) and s["map_75"] == 0 and close(s["mar_100"], 0.3)
    assert np.all(p[:3, :, 0, 2] == 1 - 2.0 ** -52) and np.all(p[3:, :, 0, 2] == 0)
    # (b) the top-scored detection hits nothing, the next two hit the two labels exactly
    _, _, s = _single([[.5, .5, .6, .6], [0, 0, .1, .1], [.2, .2, .3, .3]], [.9, .8, .7], [[0, 0, .1, .1], [.2, .2, .3, .3]])
    assert close(s["map"], 2 / 3) and s["mar_1"] == 0 and s["mar_10"] == 1
    # (c) 150 exact detections with distinct scores: 100 are kept
    g = np.float32([[i * .006, 0, i * .006 + .005, .005] for i in range(150)])
    _, _, s = _single(g, (150 - np.arange(150)) / 200, g)
    assert close(s["map"], 67 / 101) and close(s["mar_100"], 2 / 3) and close(s["mar_10"], 1 / 15) and close(s["mar_1"], 1 / 150)
    # (d) class 0 perfect, class 1 a label and no detection, class 2 a detection and no label
    _, _, s = _single([[0, 0, .1, .1], [.5, .5, .6, .6]], [.9, .8], [[0, 0, .1, .1], [.3, .3, .4, .4]], [0, 2], [0, 1], 3)
    assert close(s["map"], 0.5) and np.allclose(s["map_per_class"], [1, 0, -1], rtol=0, atol=1e-12)
    # (e) d0 has equal IoU with g0 and g1: the later ground truth wins, so d1 is a false positive
    iou = E.box_iou_np([[0, 0, .4, .1], [.2, 0, .6, .1]], [[.1, 0, .5, .1]])
    assert iou[0, 0] == iou[1, 0]
    _, _, s = _single([[.1, 0, .5, .1], [.22, 0, .62, .1]], [.9, .8], [[0, 0, .4, .1], [.2, 0, .6, .1]])
    assert close(s["map_50"], 51 / 101)
    _, _, s = _single([[.1, 0, .5, .1], [.22, 0, .62, .1]], [.9, .8], [[.2, 0, .6, .1], [0, 0, .4, .1]])
    assert close(s["map_50"], 1)


def test_coco_restatement_without_labels_is_minus_one():
    _, _, s = _single([[0, 0, .1, .1]], [.9], np.zeros((0, 4)))
    assert s["map"] == s["map_50"] == s["mar_100"] == -1 and list(s["map_per_class"]) == [-1]


def test_confusion_restatement_matches_sklearn():
    skm = pytest.importorskip("sklearn.metrics")
    rng = np.random.default_rng(3)
    for n in (1, 2, 5, 8):
        for size in (0, 1, 7, 300):
            t, p = rng.integers(0, n, size), rng.integers(0, n, size)
            p[t == n - 1] = 0   # some classes never predicted: zero denominators
            m = E.confusion_matrix_np(t, p, n)
            assert np.array_equal(m, skm.confusion_matrix(t, p, labels=np.arange(n)) if size else np.zeros((n, n)))
            if size:
                prec, rec = E.precision_recall_np(m)
                kw = dict(labels=np.arange(n), average=None, zero_division=0)
                assert np.array_equal(prec, skm.precision_score(t, p, **kw)) and np.array_equal(rec, skm.recall_score(t, p, **kw))


def _golden_confusion(z, case):
    D = z[case + "_pred"].shape[0]
    return E.confusion_from_converted(z[case + "_bg_preds"], z[case + "_bg_labels"], D - 5 + 1)


@pytest.mark.parametrize("case", ["m0", "m1", "m2", "m3", "m4"])
def test_golden_confusion_equals_the_direct_rule(golden_dir, case):
    """The kernel's rule - matched (label class, argmax of the classes and a 0), missed (label class, background), extra
    (background, argmax of the classes and a 0) - on the reference's unconverted rows gives the confusion matrix of its
    convert_background_errors rows, which the GPU test expects."""
    z = _load(golden_dir, "match.npz")
    nc = z[case + "_pred"].shape[0] - 5
    am = lambda rows: np.argmax(np.concatenate([rows[:, 5:], np.zeros((len(rows), 1))], 1), 1)   # noqa: E731
    t = np.concatenate([z[case + "_labels"][:, 5], z[case + "_missed"][:, 5], np.full(len(z[case + "_extra"]), nc)])
    p = np.concatenate([am(z[case + "_preds"]), np.full(len(z[case + "_missed"]), nc), am(z[case + "_extra"])])
    exp = _golden_confusion(z, case)
    assert np.array_equal(E.confusion_matrix_np(t.astype(np.int64), p, nc + 1), exp)
    assert exp.sum() == len(z[case + "_bg_labels"])


# ----------------------------------------------------------------------------------------------------- GPU helpers
def _sparse_batch(B, seed):
    """Sparse-realistic 97x129 predictions with labels; image 1 has more labels than predictions, image 2 no labels,
    image 3 no prediction above the threshold."""
    preds = O.synth_sparse_preds(B, 97, 129, C, 300, seed=seed)
    labels = torch.stack([O.synth_labels_for_preds(preds[b], (0.05, 0.2, 0.5)[b % 3], (0, 5, 40)[b % 3], seed=seed * 100 + b)
                          for b in range(B)])
    if B > 3:
        few = O.synth_sparse_preds(1, 97, 129, C, 20, seed=seed + 1)[0]
        labels[1] = O.synth_labels_for_preds(preds[1], 0.0, 30, seed=5)
        preds[1] = few
        labels[2] = 0
        preds[3, 4] = 0.25
    return preds, labels


def _host_confusion(p, l, nc, mincls=0.0, with_bg=True):
    from yogo_b200.utils import format_preds_and_labels_batch
    m, _ = format_preds_and_labels_batch(p, l, 0.5, mincls)
    if not with_bg:
        return E.confusion_matrix_np(m.labels[:, 5].long().cpu().numpy(), m.preds[:, 5:].argmax(1).cpu().numpy(), nc)
    cb = m.convert_background_errors(nc + 1)
    return E.confusion_from_converted(cb.preds.cpu().numpy(), cb.labels.cpu().numpy(), nc + 1)


def _host_coco_images(p, l, mincls=0.0):
    from yogo_b200.utils import format_preds_batch
    rows, kc, _, _ = format_preds_batch(p, 0.5, 0.5, "xyxy", mincls)
    rows, kc, lab = rows.cpu().numpy(), kc.cpu().numpy(), l.cpu().numpy()
    out = []
    for b in range(p.shape[0]):
        lr = lab[b].reshape(6, -1).T
        out.append(E.image_inputs(rows[b, :kc[b]], lr[lr[:, 0] != 0]))
    return out


def _assert_coco_equal(res, images, nc):
    prec, rec, summ = E.coco_eval_np(images, nc)
    assert np.array_equal(res["coco_precision"].numpy(), prec)
    assert np.array_equal(res["coco_recall"].numpy(), rec)
    for k in ("map", "map_50", "map_75", "mar_1", "mar_10", "mar_100"):
        assert res[k] == pytest.approx(summ[k], rel=1e-12, abs=0), k
    for k in ("map_per_class", "mar_100_per_class"):
        assert np.allclose(res[k].numpy(), summ[k], rtol=1e-12, atol=0), k
    return summ


# ----------------------------------------------------------------------------------------------------- GPU: confusion
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["m0", "m1", "m2", "m3", "m4"])
def test_confusion_matches_reference_golden(golden_dir, case):
    from yogo_b200 import Metrics
    z = _load(golden_dir, "match.npz")
    obj, mincls = z[case + "_cfg"]
    pred = torch.from_numpy(z[case + "_pred"]).clone()
    # Metrics thresholds objectness at 0.5; cells at or below the golden's threshold are dropped first, so the candidate
    # set (objectness > threshold) and everything after it are the golden's
    pred[4][pred[4] <= np.float32(obj)] = 0
    nc = pred.shape[0] - 5
    met = Metrics([str(k) for k in range(nc)], min_class_confidence_threshold=float(mincls))
    met.update(pred[None].to(DEV), torch.from_numpy(z[case + "_label"])[None].to(DEV))
    res = met.compute()
    exp = _golden_confusion(z, case)
    assert res["confusion"].dtype == torch.int64 and res["confusion"].device.type == "cpu"
    assert np.array_equal(res["confusion"].numpy(), exp)
    prec, rec = E.precision_recall_np(exp)
    assert np.array_equal(res["precision"].numpy(), prec) and np.array_equal(res["recall"].numpy(), rec)
    assert res["num_images"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["probabilities", "raw_logits", "no_background"])
def test_confusion_matches_host_path_over_updates(mode):
    from yogo_b200 import Metrics
    met = Metrics([str(k) for k in range(C)], include_mAP=False, include_background=mode != "no_background")
    side = C + (mode != "no_background")
    exp = np.zeros((side, side), np.int64)
    for B, seed in ((12, 41), (1, 42), (5, 43)):
        p, l = _sparse_batch(B, seed)
        if mode == "raw_logits":
            p[:, 5:] -= torch.where(torch.arange(p.shape[-1]) % 2 == 0, 2.0, 0.0)   # every other column: background wins
        p, l = p.to(DEV), l.to(DEV)
        met.update(p, l)
        exp += _host_confusion(p, l, C, with_bg=mode != "no_background")
    res = met.compute()
    if mode == "raw_logits":
        assert exp[:, C].sum() > exp[C, C] + 10 and exp[C, :C].sum() > 0
    assert np.array_equal(res["confusion"].numpy(), exp) and res["num_images"] == 18
    prec, rec = E.precision_recall_np(exp)
    assert np.array_equal(res["precision"].numpy(), prec) and np.array_equal(res["recall"].numpy(), rec)
    assert "map" not in res
    met.reset()
    p, l = _sparse_batch(4, 44)
    p, l = p.to(DEV), l.to(DEV)
    met.update(p, l)
    assert np.array_equal(met.compute()["confusion"].numpy(), _host_confusion(p, l, C, with_bg=mode != "no_background"))


# ----------------------------------------------------------------------------------------------------- GPU: mAP
@pytest.mark.gpu
def test_map_sparse_realistic_three_updates():
    from yogo_b200 import Metrics
    met = Metrics([str(k) for k in range(C)], min_class_confidence_threshold=0.1)
    images = []
    for seed in (51, 52, 53):
        p, l = _sparse_batch(32, seed)
        p, l = p.to(DEV), l.to(DEV)
        met.update(p, l)
        images += _host_coco_images(p, l, 0.1)
    res = met.compute()
    summ = _assert_coco_equal(res, images, C)
    assert 0.3 < summ["map"] < 1 and res["num_images"] == 96
    # compute() again after more state, and the confusion alongside
    p, l = _sparse_batch(6, 54)
    p, l = p.to(DEV), l.to(DEV)
    met.update(p, l)
    _assert_coco_equal(met.compute(), images + _host_coco_images(p, l, 0.1), C)


@pytest.mark.gpu
def test_map_dense_random_init_output_cuts_to_100_per_class():
    import yogo_b200
    from yogo_b200 import Metrics
    torch.manual_seed(0)
    B = 4
    net = yogo_b200.YOGO((772, 1032), O.ANCHOR_W, O.ANCHOR_H, C).to(DEV).eval()
    with torch.no_grad():
        p = net((O.synth_images(B, 772, 1032).float() / 255.0).to(DEV)).float()
    l = O.synth_labels(B, 97, 129, C, 300).to(DEV)
    met = Metrics([str(k) for k in range(C)])
    met.update(p, l)
    images = _host_coco_images(p, l)
    assert max(np.bincount(im[2], minlength=C).max() for im in images) > 100
    _assert_coco_equal(met.compute(), images, C)


@pytest.mark.gpu
def test_map_tie_heavy_scores():
    from yogo_b200 import Metrics
    met = Metrics([str(k) for k in range(C)])
    images = []
    for seed in (61, 62):
        p, l = _sparse_batch(16, seed)
        p[:, 4] = torch.ceil(p[:, 4] * 8) / 8   # objectness in multiples of 1/8: ties within and across images
        p, l = p.to(DEV), l.to(DEV)
        met.update(p, l)
        images += _host_coco_images(p, l)
    scores = np.concatenate([im[1] for im in images])
    assert np.unique(scores).size <= 4 < scores.size
    _assert_coco_equal(met.compute(), images, C)


def _case_e_grid(swap):
    """Case (e) on a 4x8 grid, one class: labels g0 [0, 0, .5, .125], g1 [.25, 0, .75, .125] (in grid order, or swapped);
    d0 [.125, 0, .625, .125] (objectness .9) has IoU .6 with both, d1 [.375, 0, .875, .125] (.8) overlaps g1 only."""
    pred = torch.zeros(1, 6, 4, 8)
    pred[0, 5] = 1.0
    for cell, (cx, score) in zip((9, 20), ((.375, .9), (.625, .8))):
        j, i = divmod(cell, 8)
        pred[0, :5, j, i] = torch.tensor([cx, .0625, .5, .125, score])
    label = torch.zeros(1, 6, 4, 8)
    boxes = [[0, 0, .5, .125], [.25, 0, .75, .125]]
    for cell, box in zip((3, 17), boxes[::-1] if swap else boxes):
        j, i = divmod(cell, 8)
        label[0, :, j, i] = torch.tensor([1.0] + box + [0.0])
    return pred, label


@pytest.mark.gpu
@pytest.mark.parametrize("swap,expected", [(False, 51 / 101), (True, 1.0)])
def test_map_equal_iou_tie_takes_the_later_ground_truth(swap, expected):
    from yogo_b200 import Metrics
    p, l = _case_e_grid(swap)
    p, l = p.to(DEV), l.to(DEV)
    images = _host_coco_images(p, l)
    iou = E.box_iou_np(images[0][3], images[0][0])
    assert images[0][0].shape[0] == 2 and iou[0, 0] == iou[1, 0] == np.float32(0.6)
    met = Metrics(["cell"])
    met.update(p, l)
    res = met.compute()
    _assert_coco_equal(res, images, 1)
    assert abs(res["map_50"] - expected) <= 1e-12


# ----------------------------------------------------------------------------------------------------- GPU: errors
@pytest.mark.gpu
def test_errors_raise_and_the_state_recovers():
    from yogo_b200 import Metrics
    met = Metrics([str(k) for k in range(C)])
    p, l = _sparse_batch(4, 71)
    p, l = p.to(DEV), l.to(DEV)
    met.update(p, l)
    exp = _host_confusion(p, l, C)
    images = _host_coco_images(p, l)

    def ok():
        nonlocal exp, images
        met.update(p, l)
        exp = exp + _host_confusion(p, l, C)
        images = images + _host_coco_images(p, l)
        res = met.compute()
        assert np.array_equal(res["confusion"].numpy(), exp)
        _assert_coco_equal(res, images, C)

    for bad_class in (float(C), -1.0, float("nan")):
        lb = l.clone()
        cells = torch.nonzero(lb[1, 0].reshape(-1)).flatten()
        lb[1, 5].view(-1)[cells[len(cells) // 2]] = bad_class
        with pytest.raises(ValueError, match=r"label class outside \[0, 7\) \(image 1\)"):
            met.update(p, lb)
        ok()
    with pytest.raises(ValueError, match="one device"):
        met.update(p, l.cpu())
    ok()
    with pytest.raises(ValueError, match="metric state is on"):
        met.update(p.cpu(), l.cpu())
    ok()
    with pytest.raises(ValueError, match="classes"):
        met.update(p[:, :-1], l)
    ok()
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="metric state is on"):
            met.update(p.to("cuda:1"), l.to("cuda:1"))
        ok()
    with pytest.raises(RuntimeError):
        Metrics(["a"]).compute()


# ----------------------------------------------------------------------------------------------------- GPU: buffers
@pytest.mark.gpu
def test_outputs_of_the_metric_kernels_stay_inside_their_buffers():
    """Guard regions around every output of yg_confusion_batch, yg_coco_match_batch and yg_coco_accumulate."""
    from yogo_b200 import _lib as L
    from yogo_b200.metrics import IOU_THRESHOLDS, RECALL_POINTS, _doubles
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

    B, Sy, Sx = 3, 13, 17
    preds = O.synth_sparse_preds(B, Sy, Sx, C, 25, seed=8)
    labels = torch.stack([O.synth_labels_for_preds(preds[b], 0.3, (0, 3, 30)[b], seed=b) for b in range(B)])
    r = _match_batch(preds.to(DEV), labels.to(DEV), 0.5, 0.0)
    m, desc, goff = r.match, r.table, r.table[4 * B:]
    assert r.n_host[2] > r.m_host[2] and r.n_host[0] < r.m_host[0]
    nb = C + 1
    cbuf, conf = guarded((nb * nb,), torch.int64, 0)
    sbuf, lst = guarded((B,), torch.int32, 77)
    L.check(lib.yg_confusion_batch(m.preds.data_ptr(), m.labels.data_ptr(), m.missed_labels.data_ptr(), m.extra_predictions.data_ptr(),
                                   B, C, 1, desc.data_ptr(), goff.data_ptr(), r.status.data_ptr(), lst.data_ptr(), conf.data_ptr(),
                                   L.stream()))
    n = int(r.m_host.sum())
    rbuf, rec = guarded((n, 4), torch.int32, 77)
    kbuf, keys = guarded((n,), torch.int64, 77)
    gbuf, gt = guarded((C,), torch.int64, 0)
    L.check(lib.yg_coco_match_batch(r.rows.data_ptr(), r.label_rows.data_ptr(), B, Sy * Sx, C, int(r.n_host.max()), int(r.m_host.max()),
                                    desc.data_ptr(), goff.data_ptr(), 5, _doubles(IOU_THRESHOLDS), rec.data_ptr(), keys.data_ptr(),
                                    gt.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert r.status.cpu().tolist() == [0] * B and lst.cpu().tolist() == [0] * B
    assert int(conf.sum()) == int(r.n_host.sum() + r.m_host.sum() - np.minimum(r.n_host, r.m_host).sum())
    assert int(gt.sum()) == int(r.n_host.sum()) and sorted(set(rec[:, 2].tolist())) == [5, 6, 7]
    for buf, view, fill in ((cbuf, conf, 0), (sbuf, lst, 77), (rbuf, rec, 77), (kbuf, keys, 77), (gbuf, gt, 0)):
        assert intact(buf, view, fill)
    sk, perm = torch.sort(keys, stable=True)
    T, R = len(IOU_THRESHOLDS), len(RECALL_POINTS)
    pbuf, prec = guarded((T * R * C * 3,), torch.float64, 7.0)
    qbuf, rcl = guarded((T * C * 3,), torch.float64, 7.0)
    L.check(lib.yg_coco_accumulate(rec.data_ptr(), sk.data_ptr(), perm.data_ptr(), n, gt.data_ptr(), C, _doubles(RECALL_POINTS),
                                   prec.data_ptr(), rcl.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert bool((prec != 7.0).all()) and bool((rcl != 7.0).all())
    for buf, view, fill in ((pbuf, prec, 7.0), (qbuf, rcl, 7.0)):
        assert intact(buf, view, fill)
