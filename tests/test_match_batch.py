"""Batched evaluation matching: format_preds_and_labels_batch against the reference goldens and the per-image path, the
device assignment solver (linear_sum_assignment_batch) against scipy, and the buffers of the new C-ABI entry points.
The CPU test pins the plain restatement of scipy's algorithm that the device solver mirrors (tools/lsap_np.py)."""
import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

from _golden import load as _load
from oracle import yogo_oracle as O
from tools.lsap_np import linear_sum_assignment_np

DEV = "cuda:0"
C = 7


def _tie_heavy(rng, r, c, kind):
    if kind == 0:
        return rng.integers(0, 3, (r, c)).astype(np.float32)
    if kind == 1:
        return np.full((r, c), float(rng.integers(0, 3)), np.float32)
    if kind == 2:
        return np.where(rng.random((r, c)) < 0.8, 1.0, rng.random((r, c))).astype(np.float32)
    return rng.random((r, c)).astype(np.float32)


def _iou_cost(rng, n, m):
    def boxes(k):
        cxy = rng.random((k, 2), dtype=np.float32)
        wh = (0.02 + 0.04 * rng.random((k, 2), dtype=np.float32)).astype(np.float32)
        return np.concatenate([cxy - wh / 2, cxy + wh / 2], 1).astype(np.float32)
    a = boxes(n)
    b = np.concatenate([a[: min(n, m)] + np.float32(0.003) * rng.standard_normal((min(n, m), 4)).astype(np.float32),
                        boxes(max(m - n, 0))]).astype(np.float32)
    return O.box_iou_cost_np(a, b[rng.permutation(m)])


def test_lsap_restatement_matches_scipy_on_tie_heavy_matrices():
    rng = np.random.default_rng(11)
    for t in range(1200):
        r, c = (int(x) for x in rng.integers(0, 9, 2))
        m = _tie_heavy(rng, r, c, t % 4)
        exp, got = linear_sum_assignment(m), linear_sum_assignment_np(m)
        assert np.array_equal(exp[0], got[0]) and np.array_equal(exp[1], got[1]), m
    m = rng.random((40, 120)).astype(np.float32)
    for x in (m, m.T):
        assert all(np.array_equal(a, b) for a, b in zip(linear_sum_assignment(x), linear_sum_assignment_np(x)))
    with pytest.raises(ValueError, match="cost matrix is infeasible"):
        linear_sum_assignment_np(np.array([[np.inf, np.inf], [1.0, 2.0]]))
    with pytest.raises(ValueError, match="matrix contains invalid numeric entries"):
        linear_sum_assignment_np(np.array([[0.0, -np.inf]]))


# ----------------------------------------------------------------------------------------------------- GPU: the pipeline
def _bits(t):
    return t.detach().cpu().numpy().view(np.uint32)


def _assert_same(got, exp):
    for a, b in ((got.preds, exp.preds), (got.labels, exp.labels), (got.missed_labels, exp.missed_labels),
                 (got.extra_predictions, exp.extra_predictions)):
        assert tuple(a.shape) == tuple(b.shape)
        assert a.dtype == b.dtype and a.device == b.device
        assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["m0", "m1", "m2", "m3", "m4"])
def test_batch_of_one_bit_exact_vs_reference_golden(golden_dir, case):
    from yogo_b200.utils import format_preds_and_labels_batch
    z = _load(golden_dir, "match.npz")
    obj, mincls = z[case + "_cfg"]
    pred = torch.from_numpy(z[case + "_pred"]).to(DEV)[None]
    label = torch.from_numpy(z[case + "_label"]).to(DEV)[None]
    m, counts = format_preds_and_labels_batch(pred, label, objectness_thresh=float(obj), min_class_confidence_threshold=float(mincls))
    for got, key in ((m.preds, "_preds"), (m.labels, "_labels"), (m.missed_labels, "_missed"), (m.extra_predictions, "_extra")):
        exp = z[case + key].astype(np.float32)
        assert tuple(got.shape) == exp.shape, key
        assert np.array_equal(_bits(got), exp.view(np.uint32)), key
    assert counts.device.type == "cpu" and counts.dtype == torch.int64
    assert counts.tolist() == [[z[case + "_preds"].shape[0], z[case + "_missed"].shape[0], z[case + "_extra"].shape[0]]]
    cb = m.convert_background_errors(pred.shape[1] - 5 + 1)
    assert np.array_equal(cb.preds.cpu().numpy(), z[case + "_bg_preds"].astype(np.float32))
    assert np.array_equal(cb.labels.cpu().numpy(), z[case + "_bg_labels"].astype(np.float32))


@pytest.mark.gpu
def test_two_golden_images_in_one_batch(golden_dir):
    from yogo_b200.utils import format_preds_and_labels_batch
    z = _load(golden_dir, "match.npz")
    assert np.array_equal(z["m3_cfg"], z["m4_cfg"])
    obj, mincls = z["m3_cfg"]
    pred = torch.from_numpy(np.stack([z["m3_pred"], z["m4_pred"]])).to(DEV)
    label = torch.from_numpy(np.stack([z["m3_label"], z["m4_label"]])).to(DEV)
    m, counts = format_preds_and_labels_batch(pred, label, float(obj), float(mincls))
    for got, key in ((m.preds, "_preds"), (m.labels, "_labels"), (m.missed_labels, "_missed"), (m.extra_predictions, "_extra")):
        exp = np.concatenate([z["m3" + key], z["m4" + key]]).astype(np.float32)
        assert tuple(got.shape) == exp.shape, key
        assert np.array_equal(_bits(got), exp.view(np.uint32)), key
    assert counts[:, 0].tolist() == [z["m3_preds"].shape[0], z["m4_preds"].shape[0]]


def _realistic_batch(B, seed, obj_thresh):
    """Sparse-realistic 97x129 predictions with labels of varying drop / extra, plus the corner cases: more labels than
    predictions (transposed problem), no labels, no prediction above the threshold, an empty image."""
    preds = O.synth_sparse_preds(B, 97, 129, C, 300, seed=seed)
    labels = torch.zeros(B, 6, 97, 129)
    for b in range(B):
        labels[b] = O.synth_labels_for_preds(preds[b], drop=(0.05, 0.2, 0.5)[b % 3], extra=(0, 5, 40)[b % 3], seed=seed * 100 + b)
    few = O.synth_sparse_preds(1, 97, 129, C, 20, seed=seed + 1)[0]
    preds[1] = few                                           # 20 objects ...
    labels[1] = O.synth_labels_for_preds(preds[2], 0.0, 30, seed=5)   # ... against ~300 labels
    labels[3] = 0                                            # no labels
    preds[4, 4] = 0.5 * obj_thresh                           # nothing above the threshold
    preds[5, 4] = 0.5 * obj_thresh
    labels[5] = 0                                            # neither
    return preds, labels


@pytest.mark.gpu
@pytest.mark.parametrize("obj,mincls,seed", [(0.5, 0.0, 21), (0.6, 0.5, 22), (0.5, 0.0, 23)])
def test_batch_matches_per_image_path(obj, mincls, seed):
    from yogo_b200.utils import PredictionLabelMatch, format_preds_and_labels_batch, format_preds_and_labels_v2
    B = 18
    preds, labels = _realistic_batch(B, seed, obj)
    p, l = preds.to(DEV), labels.to(DEV)
    per = [format_preds_and_labels_v2(p[b], l[b], obj, mincls) for b in range(B)]
    exp = PredictionLabelMatch.concat(per)
    got, counts = format_preds_and_labels_batch(p, l, obj, mincls)
    _assert_same(got, exp)
    assert counts.tolist() == [[r.preds.shape[0], r.missed_labels.shape[0], r.extra_predictions.shape[0]] for r in per]
    n_lab = [int((labels[b, 0] != 0).sum()) for b in range(B)]
    n_pred = [r.preds.shape[0] + r.extra_predictions.shape[0] for r in per]
    assert n_lab[1] > n_pred[1] > 0 and n_lab[3] == 0 and n_pred[4] == 0 and n_lab[4] > 0 and n_lab[5] == n_pred[5] == 0
    # per-image pieces by torch.split on the counts
    parts = torch.split(got.preds, counts[:, 0].tolist())
    assert all(np.array_equal(_bits(a), _bits(r.preds)) for a, r in zip(parts, per))


@pytest.mark.gpu
def test_nan_cost_from_zero_area_boxes_raises_like_the_per_image_path():
    from yogo_b200.utils import format_preds_and_labels_batch, format_preds_and_labels_v2
    pred = torch.zeros(2, 5 + C, 12, 16)
    pred[:, 5] = 1.0
    pred[:, 0, 3, 4], pred[:, 1, 3, 4] = 0.3, 0.3     # zero-area prediction box (w = h = 0) at (0.3, 0.3)
    pred[:, 4, 3, 4] = 0.9
    label = torch.zeros(2, 6, 12, 16)
    label[:, 0, 8, 8] = 1.0
    label[:, 1:5, 8, 8] = 0.7                          # zero-area label at (0.7, 0.7): 0 / 0 in the IoU
    pred[0, 4, 3, 4] = 0.1                            # image 0 has no prediction: no cost matrix
    p, l = pred.to(DEV), label.to(DEV)
    format_preds_and_labels_v2(p[0], l[0])
    with pytest.raises(ValueError, match="matrix contains invalid numeric entries"):
        format_preds_and_labels_v2(p[1], l[1])
    with pytest.raises(ValueError, match=r"matrix contains invalid numeric entries \(image 1\)"):
        format_preds_and_labels_batch(p, l)


@pytest.mark.gpu
def test_bad_arguments_raise():
    from yogo_b200 import _lib as L
    from yogo_b200.utils import format_preds_and_labels_batch, linear_sum_assignment_batch
    p = torch.zeros(2, 12, 8, 8, device=DEV)
    with pytest.raises(ValueError):
        format_preds_and_labels_batch(p[0], torch.zeros(6, 8, 8, device=DEV))
    with pytest.raises(ValueError):
        format_preds_and_labels_batch(p, torch.zeros(2, 6, 8, 9, device=DEV))
    with pytest.raises(L.YogoB200Error):
        format_preds_and_labels_batch(p, torch.zeros(2, 6, 8, 8))
    with pytest.raises(L.YogoB200Error):
        linear_sum_assignment_batch([torch.zeros(2, 2)])
    with pytest.raises(ValueError, match="2-D"):
        linear_sum_assignment_batch([torch.zeros(2, 2, device=DEV), torch.zeros(3, device=DEV)])
    with pytest.raises(ValueError, match="float32"):
        linear_sum_assignment_batch([torch.zeros(2, 2, device=DEV, dtype=torch.float64)])
    assert linear_sum_assignment_batch([]) == []


# ----------------------------------------------------------------------------------------------------- GPU: the solver
def _check_against_scipy(mats):
    from yogo_b200.utils import linear_sum_assignment_batch
    res = linear_sum_assignment_batch([torch.from_numpy(np.ascontiguousarray(m)).to(DEV) for m in mats])
    assert len(res) == len(mats)
    for m, (r, c) in zip(mats, res):
        er, ec = linear_sum_assignment(m)
        assert r.dtype == torch.int64 and c.dtype == torch.int64 and r.device == c.device == torch.device(DEV)
        assert np.array_equal(r.cpu().numpy(), er) and np.array_equal(c.cpu().numpy(), ec), m.shape


@pytest.mark.gpu
def test_solver_matches_scipy_on_small_tie_heavy_matrices():
    rng = np.random.default_rng(12)
    mats = [np.zeros((0, 3), np.float32), np.zeros((4, 0), np.float32), np.zeros((0, 0), np.float32), np.float32([[2.5]])]
    for t in range(2400):
        r, c = (int(x) for x in rng.integers(1, 10, 2))
        mats.append(_tie_heavy(rng, r, c, t % 4))
    _check_against_scipy(mats)


@pytest.mark.gpu
def test_solver_matches_scipy_on_wide_tall_and_line_shapes():
    rng = np.random.default_rng(13)
    mats = []
    for t in range(400):
        n = int(rng.integers(1, 70))
        k = int(rng.integers(1, 6))
        shape = [(1, n), (n, 1), (n, n), (k, n), (n, k)][t % 5]
        mats.append(_tie_heavy(rng, *shape, kind=t % 4))
    _check_against_scipy(mats)


@pytest.mark.gpu
def test_solver_matches_scipy_on_iou_structured_matrices():
    rng = np.random.default_rng(14)
    mats = [_iou_cost(rng, 300, 300), _iou_cost(rng, 300, 300), _iou_cost(rng, 300, 5000), _iou_cost(rng, 5000, 300),
            _iou_cost(rng, 270, 280), _iou_cost(rng, 666, 288)]
    _check_against_scipy(mats)


@pytest.mark.gpu
def test_solver_inf_entries_and_errors_like_scipy():
    from yogo_b200.utils import linear_sum_assignment_batch
    rng = np.random.default_rng(15)
    feasible, infeasible = [], []
    for t in range(600):
        r, c = (int(x) for x in rng.integers(1, 8, 2))
        m = np.where(rng.random((r, c)) < 0.45, np.inf, rng.integers(0, 3, (r, c))).astype(np.float32)
        try:
            linear_sum_assignment(m)
            feasible.append(m)
        except ValueError as e:
            assert "infeasible" in str(e)
            infeasible.append(m)
    assert len(feasible) > 100 and len(infeasible) > 20
    _check_against_scipy(feasible)
    ok = [torch.from_numpy(m).to(DEV) for m in feasible[:5]]
    for bad in infeasible[:10]:
        with pytest.raises(ValueError, match=r"cost matrix is infeasible \(cost matrix 5\)"):
            linear_sum_assignment_batch(ok + [torch.from_numpy(bad).to(DEV)])
    nan = np.ones((3, 4), np.float32)
    nan[1, 2] = np.nan
    neginf = np.ones((5, 2), np.float32)
    neginf[4, 0] = -np.inf
    for bad in (nan, neginf):
        with pytest.raises(ValueError, match="matrix contains invalid numeric entries"):
            linear_sum_assignment(bad)
        with pytest.raises(ValueError, match=r"matrix contains invalid numeric entries \(cost matrix 2\)"):
            linear_sum_assignment_batch(ok[:2] + [torch.from_numpy(bad).to(DEV)] + ok[2:])
    # a failed call leaves nothing behind
    _check_against_scipy(feasible[:50] + [_tie_heavy(rng, 6, 9, 0), _tie_heavy(rng, 9, 6, 2)])


# ----------------------------------------------------------------------------------------------------- GPU: buffers
@pytest.mark.gpu
def test_outputs_of_the_matching_kernels_stay_inside_their_buffers():
    """Guard regions around every output of yg_compact_labels, yg_lsap_batch and yg_match_batch, ragged sizes."""
    from yogo_b200 import _lib as L
    from yogo_b200.utils import format_preds_batch
    from yogo_b200.utils.prediction_formatting import _lsap_plan
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
    cells, D = Sy * Sx, 5 + C
    preds = O.synth_sparse_preds(B, Sy, Sx, C, 25, seed=8)
    labels = torch.stack([O.synth_labels_for_preds(preds[b], 0.3, (0, 3, 30)[b], seed=b) for b in range(B)])
    lab = labels.to(DEV)
    lrbuf, lrows = guarded((B, cells, 6), torch.float32, 7.0)
    nlbuf, nl = guarded((B,), torch.int32, 77)
    L.check(lib.yg_compact_labels(lab.data_ptr(), B, Sy, Sx, lrows.data_ptr(), nl.data_ptr(), L.stream()))
    rows, kc, _, _ = format_preds_batch(preds.to(DEV), 0.5, 0.5, "xyxy", 0.0)
    torch.cuda.synchronize()
    assert intact(lrbuf, lrows, 7.0) and intact(nlbuf, nl, 77)
    N, M = nl.cpu().numpy().astype(np.int64), kc.cpu().numpy().astype(np.int64)
    K = np.minimum(N, M)
    assert N.tolist() == [int((labels[b, 0] != 0).sum()) for b in range(B)] and N[2] > M[2] and N[0] < M[0]
    plan, words = _lsap_plan(N, M)
    table = torch.from_numpy(plan).to(DEV)
    Kt, Nt, Mt = int(K.sum()), int(N.sum()), int(M.sum())
    cbuf, costs = guarded((int((N * M).sum()),), torch.float32, 7.0)
    wbuf, ws = guarded((words,), torch.float64, 7.0)
    prbuf, pr = guarded((Kt,), torch.int64, 77)
    pcbuf, pc = guarded((Kt,), torch.int64, 77)
    sbuf, st = guarded((B,), torch.int32, 77)
    opbuf, op = guarded((Kt, D), torch.float32, 7.0)
    olbuf, ol = guarded((Kt, 6), torch.float32, 7.0)
    mbuf, mi = guarded((Nt - Kt, 6), torch.float32, 7.0)
    ebuf, ex = guarded((Mt - Kt, D), torch.float32, 7.0)
    L.check(lib.yg_match_batch(lrows.data_ptr(), rows.data_ptr(), B, cells, C, int(N.max()), int(M.max()), table.data_ptr(),
                               table[4 * B:].data_ptr(), costs.data_ptr(), ws.data_ptr(), pr.data_ptr(), pc.data_ptr(),
                               st.data_ptr(), op.data_ptr(), ol.data_ptr(), mi.data_ptr(), ex.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [0] * B
    for buf, view, fill in ((cbuf, costs, 7.0), (wbuf, ws, 7.0), (prbuf, pr, 77), (pcbuf, pc, 77), (sbuf, st, 77), (opbuf, op, 7.0),
                            (olbuf, ol, 7.0), (mbuf, mi, 7.0), (ebuf, ex, 7.0)):
        assert intact(buf, view, fill)
    # the solver alone on the packed cost matrices
    s2buf, st2 = guarded((B,), torch.int32, 77)
    pr.fill_(-5)
    L.check(lib.yg_lsap_batch(costs.data_ptr(), table.data_ptr(), B, ws.data_ptr(), pr.data_ptr(), pc.data_ptr(), st2.data_ptr(),
                              L.stream()))
    torch.cuda.synchronize()
    assert st2.cpu().tolist() == [0] * B and bool((pr >= 0).all())
    for buf, view, fill in ((wbuf, ws, 7.0), (prbuf, pr, 77), (pcbuf, pc, 77), (s2buf, st2, 77)):
        assert intact(buf, view, fill)
