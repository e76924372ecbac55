"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI by the
Python mirror of the reference API, against (a) the golden vectors produced by the real
reference and (b) the CPU oracle on seeded inputs.  Nothing here reads /root/reference.

Tolerances: fp32 storage path - 1e-3 relative (north star); bf16 storage path - per-tensor
bounds calibrated from the reference's own bf16-autocast error (SURVEY.md Appendix E)."""
import os

import numpy as np
import pytest
import torch

import yogo_b200
from _golden import load as _load
from yogo_b200 import _lib as L
from oracle import yogo_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rel(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ----------------------------------------------------------------------------- loss
@pytest.mark.parametrize("case", ["loss0", "loss1", "loss2", "loss3", "lossw"])
def test_loss_matches_reference_golden(golden_dir, case):
    z = _load(golden_dir, "loss.npz")
    kw = dict(no_obj_weight=0.3, iou_weight=2.5, classify_weight=0.7, label_smoothing=0.1) if case == "lossw" else {}
    pred = torch.from_numpy(z[f"{case}_pred"]).to(DEV).requires_grad_(True)
    label = torch.from_numpy(z[f"{case}_label"]).to(DEV)
    loss_fn = yogo_b200.YOGOLoss(**kw).to(DEV)
    loss, comps = loss_fn(pred, label)
    loss.backward()
    ref = z[f"{case}_loss"]
    got = [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]]
    np.testing.assert_allclose(got, ref, rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(pred.grad.cpu().numpy(), z[f"{case}_dpred"], rtol=1e-3, atol=2e-6)


def test_loss_and_grad_equals_the_autograd_route(golden_dir):
    # the trainer's direct route: same kernel launch, gradient handed over without the autograd `grad_out * dpred` pass
    z = _load(golden_dir, "loss.npz")
    pred = torch.from_numpy(z["loss1_pred"]).to(DEV).requires_grad_(True)
    label = torch.from_numpy(z["loss1_label"]).to(DEV)
    loss_fn = yogo_b200.YOGOLoss().to(DEV)
    loss, comps = loss_fn(pred, label)
    loss.backward()
    loss2, comps2, dpred = loss_fn.loss_and_grad(pred.detach(), label)
    assert loss2.item() == loss.item()
    assert dict(comps2) == dict(comps)
    assert torch.equal(dpred, pred.grad)


def test_loss_full_size_vs_oracle_and_scaling_property():
    # BASELINE size: 12,513 cells per image, 300 labels per image
    N = 8
    lab = O.synth_labels(N)
    g = torch.Generator().manual_seed(3)
    pred = torch.rand(N, 12, 97, 129, generator=g)
    pred[:, 2:4] = 0.02 + 0.08 * pred[:, 2:4]
    pred[:, 5:] = 3 * torch.randn(N, 7, 97, 129, generator=g)
    ref_loss, ref_comps, ref_d = O.yogo_loss_np(pred.numpy(), lab.numpy())
    p = pred.to(DEV).requires_grad_(True)
    loss, comps = yogo_b200.YOGOLoss().to(DEV)(p, lab.to(DEV))
    (3.0 * loss).backward()  # upstream gradient scaling must pass through linearly
    assert abs(loss.item() - ref_loss) <= 2e-5 * abs(ref_loss)
    for k in ref_comps:
        assert abs(comps[k] - ref_comps[k]) <= 2e-5 * abs(ref_comps[k]) + 1e-6
    np.testing.assert_allclose(p.grad.cpu().numpy() / 3.0, ref_d, rtol=1e-3, atol=2e-6)
    # batch-replication property: duplicating the batch leaves the loss unchanged (sum / N)
    loss2, _ = yogo_b200.YOGOLoss().to(DEV)(torch.cat([p.detach(), p.detach()]), torch.cat([lab, lab]).to(DEV))
    assert abs(loss2.item() - loss.item()) <= 1e-5 * abs(loss.item())


# ----------------------------------------------------------------------------- format_preds / NMS
@pytest.mark.parametrize("case", ["nms0", "nms1", "nms2", "nms3", "nms4", "nms5", "nmsD"])
def test_format_preds_bit_exact_vs_reference_golden(golden_dir, case):
    z = _load(golden_dir, "nms.npz")
    obj, iou, xyxy, mincls = z[f"{case}_cfg"]
    pred = torch.from_numpy(z[f"{case}_pred"]).to(DEV)
    offs, rows = z[f"{case}_offsets"], z[f"{case}_rows"]
    fmt = "xyxy" if xyxy else "cxcywh"
    out_rows, keep_count, keep_index, counts = yogo_b200.format_preds_batch(pred, obj, iou, fmt, mincls)
    kc = keep_count.cpu().numpy()
    for b in range(pred.shape[0]):
        exp = rows[offs[b]: offs[b + 1]]
        assert kc[b] == exp.shape[0]
        got = out_rows[b, : kc[b]].cpu().numpy()
        assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))
        single = yogo_b200.format_preds(pred[b], obj, iou, fmt, mincls).cpu().numpy()
        assert np.array_equal(single.view(np.uint32), exp.view(np.uint32))
    assert np.array_equal(counts.cpu().numpy(), z[f"{case}_counts"])
    cc = yogo_b200.get_prediction_class_counts(pred, obj, iou, mincls)
    assert cc.device.type == "cpu" and np.array_equal(cc.numpy(), z[f"{case}_counts"])


def test_format_preds_reference_known_answers():
    # /root/reference/tests/test_utils_tensor_formatting.py:9-68 through the CUDA path
    none = torch.zeros(12, 4, 4, device=DEV)
    assert tuple(yogo_b200.format_preds(none).shape) == (0, 12)
    single = torch.zeros(12, 4, 4, device=DEV)
    single[4, 0, 0] = 1.0
    single[5] = 1.0
    torch.testing.assert_close(yogo_b200.format_preds(single), single[:, 0, 0].unsqueeze(0))
    box = torch.zeros(12, 4, 4, device=DEV)
    box[5] = 1.0
    box[4, 1, 1] = 1.0
    box[0:2, 1, 1] = 0.5
    box[2:4, 1, 1] = 0.1
    torch.testing.assert_close(yogo_b200.format_preds(box), box[:, 1, 1].unsqueeze(0))
    actual = box[:, 1, 1].unsqueeze(0).clone()
    actual[:, 0] = actual[:, 0] - actual[:, 2] / 2
    actual[:, 1] = actual[:, 1] - actual[:, 3] / 2
    actual[:, 2] = actual[:, 0] + actual[:, 2]
    actual[:, 3] = actual[:, 1] + actual[:, 3]
    torch.testing.assert_close(yogo_b200.format_preds(box, box_format="xyxy"), actual)
    # two identical zero-area boxes: 0/0 = NaN never suppresses (SURVEY.md Appendix C)
    two = torch.zeros(12, 4, 4, device=DEV)
    two[4, 0, 0] = two[4, 0, 1] = 0.9
    two[5] = 1.0
    assert yogo_b200.format_preds(two).shape[0] == 2


@pytest.mark.parametrize("thr", [0.5, 1.0 / 3.0, 0.3, 0.25])
def test_nms_pairs_sitting_on_the_iou_threshold(thr):
    """The suppression masks decide most pairs without the IEEE division (two fp32 products against thresholds a hair
    below / above); pairs inside that sliver take the exact quotient path.  Boxes on a lattice - equal sizes, shifts of
    1/3, 1/2, 3/5 of the width - put hundreds of pairs at IoU = 1/2, 1/3, 1/4 up to rounding noise, where the fp32 quotient
    lands on either side of the threshold: results must still equal the oracle (torchvision CPU semantics) bit for bit."""
    g = torch.Generator().manual_seed(int(thr * 1000))
    B, C, Sy, Sx = 3, 7, 24, 32
    p = torch.zeros(B, 5 + C, Sy, Sx)
    jj, ii = torch.meshgrid(torch.arange(Sy), torch.arange(Sx), indexing="ij")
    w = 0.06
    for b in range(B):
        frac = [1.0 / 3.0, 0.5, 0.6][b]
        # neighbouring cells hold the same box shifted by `frac` of its width: IoU = (1 - frac) / (1 + frac) = 1/2, 1/3, 1/4
        p[b, 0] = 0.1 + (ii.float() * frac * w) % 0.8
        p[b, 1] = 0.1 + 0.03 * (jj % 3).float() + 0.2 * (jj // 3).float() / 8
        p[b, 2] = w
        p[b, 3] = 0.05
        p[b, 4] = 0.55 + 0.4 * torch.rand(Sy, Sx, generator=g)
        p[b, 5:] = torch.softmax(3 * torch.randn(C, Sy, Sx, generator=g), dim=0)
    import torchvision.ops as ops
    rows, kc, kidx, counts = yogo_b200.format_preds_batch(p.to(DEV), 0.5, thr)
    tot = np.zeros(C, np.int64)
    near = 0
    for b in range(B):
        exp = O.format_preds_np(p[b].numpy(), 0.5, thr)
        assert int(kc[b]) == exp.shape[0], (b, int(kc[b]), exp.shape[0])
        assert np.array_equal(rows[b, : exp.shape[0]].cpu().numpy().view(np.uint32), exp.view(np.uint32))
        tot += O.count_cells_np(exp[:, 5:])
        # the installed torchvision CPU kernel itself, on the same candidates
        pb = p[b].reshape(5 + C, -1).T
        m = pb[:, 4] > 0.5
        c = pb[m]
        boxes = ops.box_convert(c[:, :4], "cxcywh", "xyxy")
        keep = ops.nms(boxes, c[:, 5:].max(1).values * c[:, 4], thr)
        assert np.array_equal(kidx[b, : int(kc[b])].cpu().numpy(), torch.nonzero(m)[:, 0][keep].numpy())
        near += int(((ops.box_iou(boxes, boxes) - thr).abs() < 1e-6).sum())
    assert np.array_equal(counts.cpu().numpy(), tot)
    assert near > 100 or thr == 0.3   # the fixture really has pairs on the threshold (1/2, 1/3, 1/4)


@pytest.mark.parametrize("K,B", [(50, 8), (300, 8), (1000, 4)])
def test_format_preds_full_size_sparse_vs_oracle(K, B):
    p = O.synth_sparse_preds(B, K=K, seed=100 + K)
    rows, kc, kidx, counts = yogo_b200.format_preds_batch(p.to(DEV))
    kc = kc.cpu().numpy()
    tot = np.zeros(7, np.int64)
    for b in range(B):
        exp, idx = O.format_preds_np(p[b].numpy(), return_index=True)
        assert kc[b] == exp.shape[0]
        assert np.array_equal(rows[b, : kc[b]].cpu().numpy().view(np.uint32), exp.view(np.uint32))
        assert np.array_equal(kidx[b, : kc[b]].cpu().numpy(), idx)
        tot += O.count_cells_np(exp[:, 5:])
    assert np.array_equal(counts.cpu().numpy(), tot)


def test_format_preds_dense_full_size_and_idempotence():
    # dense-adversarial case: ~all 12,513 cells are candidates (SURVEY.md 8d)
    g = torch.Generator().manual_seed(7)
    p = torch.rand(2, 12, 97, 129, generator=g)
    p[:, 2:4] = 0.01 + 0.05 * p[:, 2:4]
    p[:, 4] = 0.5 + 0.5 * p[:, 4]
    p[:, 5:] = torch.softmax(4 * p[:, 5:], dim=1)
    rows, kc, kidx, counts = yogo_b200.format_preds_batch(p.to(DEV))
    kc = kc.cpu().numpy()
    for b in range(2):
        exp = O.format_preds_np(p[b].numpy())
        assert kc[b] == exp.shape[0]
        assert np.array_equal(rows[b, : kc[b]].cpu().numpy().view(np.uint32), exp.view(np.uint32))
    # torchvision (installed library on the GPU box, CPU kernel) agrees on keep indices
    import torchvision.ops as ops
    pb = p[0].reshape(12, -1).T
    m = pb[:, 4] > 0.5
    c = pb[m]
    keep = ops.nms(ops.box_convert(c[:, :4], "cxcywh", "xyxy"), c[:, 5:].max(1).values * c[:, 4], 0.5)
    cells = torch.nonzero(m)[:, 0][keep]
    assert np.array_equal(kidx[0, : kc[0]].cpu().numpy(), cells.numpy())
    # idempotence: the kept boxes, scattered back on an empty grid, all survive a second pass
    q = torch.zeros_like(p[0])
    q[:, :, :] = 0
    flat = q.reshape(12, -1)
    flat[:, kidx[0, : kc[0]].cpu().long()] = rows[0, : kc[0]].cpu().T
    rows2, kc2, _, _ = yogo_b200.format_preds_batch(q.unsqueeze(0).to(DEV))
    assert int(kc2[0]) == int(kc[0])
    assert np.array_equal(rows2[0, : kc[0]].cpu().numpy().view(np.uint32), rows[0, : kc[0]].cpu().numpy().view(np.uint32))


# ----------------------------------------------------------------------------- evaluation matching (SURVEY.md 8f N2)
@pytest.mark.parametrize("case", ["m0", "m1", "m2", "m3", "m4"])
def test_format_preds_and_labels_v2_bit_exact_vs_reference_golden(golden_dir, case):
    """prediction_formatting.py:254-330 (+ :96-156, :206-251) of the real reference vs the CUDA path: threshold + NMS kernel,
    pairwise-IoU cost kernel, scipy assignment on the bit-identical matrix."""
    from yogo_b200.utils import format_preds_and_labels_v2, format_to_numpy
    z = _load(golden_dir, "match.npz")
    obj, mincls = z[case + "_cfg"]
    pred = torch.from_numpy(z[case + "_pred"]).to(DEV)
    label = torch.from_numpy(z[case + "_label"]).to(DEV)
    m = format_preds_and_labels_v2(pred, label, objectness_thresh=float(obj), min_class_confidence_threshold=float(mincls))
    for got, key in ((m.preds, "_preds"), (m.labels, "_labels"), (m.missed_labels, "_missed"), (m.extra_predictions, "_extra")):
        exp = z[case + key].astype(np.float32)
        assert tuple(got.shape) == exp.shape, key
        assert np.array_equal(got.cpu().numpy().view(np.uint32), exp.view(np.uint32)), key
    C = pred.shape[0] - 5
    cb = m.convert_background_errors(C + 1)
    assert cb.missed_labels is None and cb.extra_predictions is None
    assert np.array_equal(cb.preds.cpu().numpy(), z[case + "_bg_preds"].astype(np.float32))
    assert np.array_equal(cb.labels.cpu().numpy(), z[case + "_bg_labels"].astype(np.float32))
    npy = format_to_numpy(7, z[case + "_pred"], 772, 1032)
    assert npy.dtype == z[case + "_npy"].dtype and np.array_equal(npy, z[case + "_npy"])


def test_box_iou_cost_full_size_vs_oracle_and_torchvision():
    from yogo_b200.utils import box_iou_cost
    import torchvision.ops as ops
    g = torch.Generator().manual_seed(5)
    n, m = 700, 2347
    def boxes(k):
        c = torch.rand(k, 2, generator=g)
        wh = torch.rand(k, 2, generator=g) * 0.08
        return torch.cat([c - wh / 2, c + wh / 2], 1)
    a, b = boxes(n), boxes(m)
    a[3] = a[4]                      # duplicates
    b[10, 2:] = b[10, :2]            # zero-area prediction
    lab = torch.cat([torch.ones(n, 1), a, torch.zeros(n, 1)], 1).to(DEV)
    rows = torch.cat([b, torch.rand(m, 8, generator=g)], 1).to(DEV)
    cost = box_iou_cost(lab[:, 1:5], rows[:, :4]).cpu().numpy()
    assert np.array_equal(cost.view(np.uint32), O.box_iou_cost_np(a.numpy(), b.numpy()).view(np.uint32))
    assert np.array_equal(cost.view(np.uint32), (1 - ops.box_iou(a, b).numpy()).view(np.uint32))
    assert box_iou_cost(lab[:0, 1:5], rows[:, :4]).shape == (0, m)


def test_predict_loop_matches_direct_forward_and_writes_reference_format(tmp_path):
    """infer.py:140-421 / :39-57: checkpoint -> predict() over a folder of PNGs == model forward + format_preds per image."""
    from torchvision.io import write_png
    torch.manual_seed(3)
    H, W, C = 96, 128, 4
    net = yogo_b200.YOGO((H, W), 0.1, 0.1, C, inference=True)
    with torch.no_grad():
        net.model[-1].bias[4] = 1.0   # objectness logits above threshold on part of the grid
    pth = tmp_path / "m.pth"
    torch.save({"step": 5, "model_state_dict": net.state_dict(), "model_version": "base_model", "class_names": list("abcd"),
                "normalize_images": False}, pth)
    imgs = torch.randint(0, 256, (5, 1, H, W), dtype=torch.uint8)
    idir = tmp_path / "images"
    idir.mkdir()
    for i, im in enumerate(imgs):
        write_png(im, str(idir / f"img_{i:03d}.png"))
    odir = tmp_path / "out"
    res = yogo_b200.predict(str(pth), path_to_images=idir, output_dir=str(odir), save_preds=True, count_predictions=True,
                            batch_size=2, return_full_predictions=True, class_names=list("abcd"))
    net = net.to(DEV).eval()
    net.compute_dtype = torch.float32
    with torch.no_grad():
        direct = net(imgs.to(DEV)).cpu()
    assert res.shape == direct.shape and _rel(res.numpy(), direct.numpy()) < 1e-5
    # in-memory images give the same tensor
    res2 = yogo_b200.predict(str(pth), images=imgs, batch_size=3, return_full_predictions=True)
    assert torch.equal(res2, res)
    for i in range(5):
        rows = O.format_preds_np(res[i].numpy())
        exp = "\n".join(f"{int(np.argmax(r[5:]))} {torch.tensor(r[0])} {torch.tensor(r[1])} {torch.tensor(r[2])} {torch.tensor(r[3])}"
                        for r in rows)
        assert (odir / f"img_{i:03d}.txt").read_text() == exp
    with pytest.raises(ValueError):
        yogo_b200.predict(str(pth), path_to_images=idir, save_preds=True)
    with pytest.raises(ValueError):
        yogo_b200.predict(str(pth), images=imgs, class_names=["a"])
    # vertical crop: centre rows of the image through a resized model
    res3 = yogo_b200.predict(str(pth), images=imgs, vertical_crop_height=0.5, return_full_predictions=True)
    assert res3.shape[0] == 5 and res3.shape[2] < res.shape[2]


# ----------------------------------------------------------------------------- input side (SURVEY.md 8f N3)
def test_flips_and_label_rasterisation_bit_exact_vs_reference_golden(golden_dir):
    """RandomHorizontal/VerticalFlipWithBBs (data_transforms.py:51-98) and format_labels_tensor (yogo_dataset.py:24-46)
    of the real reference vs csrc/input.cu."""
    from yogo_b200.data import flip_batch, format_labels_batch, format_labels_tensor
    z = _load(golden_dir, "input.npz")
    for ci in range(3):
        img, lab = torch.from_numpy(z[f"f{ci}_img"]).to(DEV), torch.from_numpy(z[f"f{ci}_lab"]).to(DEV)
        for tag, h, v in (("h", True, False), ("v", False, True), ("hv", True, True)):
            a, b = flip_batch(img, lab, h, v)
            assert np.array_equal(a.cpu().numpy(), z[f"f{ci}_{tag}_img"]), (ci, tag)
            assert np.array_equal(b.cpu().numpy().view(np.uint32), z[f"f{ci}_{tag}_lab"].view(np.uint32)), (ci, tag)
        # the inputs are untouched (out of place) and two flips are the identity on the image
        assert np.array_equal(img.cpu().numpy(), z[f"f{ci}_img"])
        a2, _ = flip_batch(*flip_batch(img, lab, True, True), True, True)
        assert torch.equal(a2, img)
    for ci in range(3):
        B, Sx, Sy = (int(v) for v in z[f"l{ci}_cfg"])
        offs = np.concatenate([[0], np.cumsum(z[f"l{ci}_counts"])])
        lists = [torch.from_numpy(z[f"l{ci}_labels"][offs[b]:offs[b + 1]]) for b in range(B)]
        out = format_labels_batch(lists, Sx, Sy)
        assert np.array_equal(out.cpu().numpy().view(np.uint32), z[f"l{ci}_out"].view(np.uint32)), ci
        assert torch.equal(format_labels_tensor(lists[0].to(DEV), Sx, Sy), out[0])
    with pytest.raises(IndexError):
        format_labels_tensor(torch.tensor([[0, 0.9, 0.9, 1.2, 1.2]]), 8, 6)


def test_flip_modules_follow_the_host_rng_like_the_reference():
    from yogo_b200.data import MultiArgSequential, RandomHorizontalFlipWithBBs, RandomVerticalFlipWithBBs, DualInputId
    img = O.synth_images(4, 772, 1032).to(DEV)
    lab = O.synth_labels(4).to(DEV)
    tf = MultiArgSequential(RandomHorizontalFlipWithBBs(0.5), DualInputId(), RandomVerticalFlipWithBBs(0.5))
    assert len(tf) == 2
    for seed in range(4):
        torch.manual_seed(seed)
        h, v = bool(torch.rand(1) < 0.5), bool(torch.rand(1) < 0.5)
        torch.manual_seed(seed)
        a, b = tf(img, lab)
        ea, eb = O.flip_batch_np(img.cpu().numpy(), lab.cpu().numpy(), h, v)
        assert np.array_equal(a.cpu().numpy(), ea) and np.array_equal(b.cpu().numpy().view(np.uint32), eb.view(np.uint32))


# ----------------------------------------------------------------------------- conv kernels vs oracle
def _conv_case(N, H, W, Cin, Cout, k, s, dtype, act, with_stats, seed=0):
    import ctypes as C
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, Cin, H, W, generator=g)
    w = torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5
    b = torch.randn(Cout, generator=g) * 0.1
    keep = (torch.rand(N, Cout, generator=g) > 0.2).float() / 0.8
    xd = x.permute(0, 2, 3, 1).contiguous().to(DEV).to(dtype)
    x_ref = xd.float().permute(0, 3, 1, 2).cpu()
    y_ref = torch.nn.functional.conv2d(x_ref, w, b, stride=s, padding=k // 2)
    Ho, Wo = y_ref.shape[-2:]
    lib = L.lib()
    y = torch.empty(N, Ho, Wo, Cout, device=DEV, dtype=dtype)
    stats = torch.zeros(2 * Cout, dtype=torch.float64, device=DEV) if with_stats else None
    wd, bd, kd = w.to(DEV), b.to(DEV), keep.to(DEV).contiguous()
    ep = L.FwdEpilogue(None, bd.data_ptr(), act, kd.data_ptr(), L.ptr(stats), None)
    L.check(lib.yg_conv_fwd(xd.data_ptr(), wd.data_ptr(), y.data_ptr(), L.dtype_code(dtype), N, H, W, Cin, Cout, k, s,
                            C.byref(ep), L.stream()))
    a_ref = O._act(y_ref, {0: None, 1: "lrelu", 2: "silu"}[act]) * keep[:, :, None, None]
    tol = 2e-5 if dtype == torch.float32 else 6e-3
    got = y.float().permute(0, 3, 1, 2).cpu()
    assert _rel(got, a_ref) < tol, ("fwd", _rel(got, a_ref))
    if with_stats:
        s_ref = torch.stack([y_ref.double().sum((0, 2, 3)), (y_ref.double() ** 2).sum((0, 2, 3))]).reshape(-1)
        # (fp32 tensors run as split-bf16 "x3" convolutions on the tensor cores under impl = auto: ~2^-16 per product)
        assert _rel(stats.cpu(), s_ref) < (3e-5 if dtype == torch.float32 else 5e-3)
    # dgrad + wgrad against autograd of the CPU conv
    dz = torch.randn(N, Cout, Ho, Wo, generator=g)
    dzd = dz.permute(0, 2, 3, 1).contiguous().to(DEV).to(dtype)
    dz_ref = dzd.float().permute(0, 3, 1, 2).cpu()
    xr = x_ref.clone().requires_grad_(True)
    wr = w.clone().requires_grad_(True)
    br = b.clone().requires_grad_(True)
    torch.nn.functional.conv2d(xr, wr, br, stride=s, padding=k // 2).backward(dz_ref)
    dx = torch.empty(N, H, W, Cin, device=DEV, dtype=dtype)
    L.check(lib.yg_conv_dgrad(dzd.data_ptr(), wd.data_ptr(), dx.data_ptr(), L.dtype_code(dtype), N, H, W, Cin, Cout, k, s,
                              None, L.stream()))
    assert _rel(dx.float().permute(0, 3, 1, 2).cpu(), xr.grad) < tol, "dgrad"
    dw = torch.empty_like(wd)
    db = torch.empty_like(bd)
    nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, k, s)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_conv_wgrad(xd.data_ptr(), dzd.data_ptr(), dw.data_ptr(), db.data_ptr(), L.dtype_code(dtype), N, H, W,
                              Cin, Cout, k, s, 0.0, ws.data_ptr(), nb, L.stream()))
    assert _rel(dw.cpu(), wr.grad) < (5e-5 if dtype == torch.float32 else 3e-3), ("wgrad", _rel(dw.cpu(), wr.grad))
    assert _rel(db.cpu(), br.grad) < (5e-5 if dtype == torch.float32 else 3e-3), "dbias"


SHAPES = [
    # N, H, W, Cin, Cout, k, s
    (2, 13, 17, 5, 12, 3, 1),
    (2, 13, 17, 5, 12, 3, 2),
    (1, 26, 34, 16, 32, 3, 1),
    (3, 26, 35, 32, 64, 3, 2),
    (2, 9, 11, 64, 128, 3, 1),
    (2, 20, 28, 128, 128, 3, 2),
    (1, 10, 14, 128, 128, 3, 1),
    (2, 10, 14, 48, 96, 3, 1),
    (2, 10, 14, 24, 12, 1, 1),
    # double_filters / triple_filters widths (model_defns.py:130-227): N = 256 MMAs, non-resident weights
    (2, 9, 11, 128, 256, 3, 1),
    (1, 10, 14, 256, 256, 3, 1),
    (2, 20, 28, 256, 256, 3, 2),
    (2, 11, 14, 96, 192, 3, 2),
    (1, 10, 14, 192, 384, 3, 1),
    (1, 9, 13, 384, 384, 3, 2),
    (2, 10, 14, 256, 12, 1, 1),
]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_conv_kernels_vs_oracle(shape, dtype, impl):
    L.set_conv_impl(impl)
    try:
        _conv_case(*shape, dtype=dtype, act=(shape[3] % 3), with_stats=True, seed=sum(shape))
    finally:
        L.set_conv_impl("auto")


@pytest.mark.parametrize("shape", [s for s in SHAPES if s[5] == 3 and s[3] % 16 == 0 and s[4] % 16 == 0])
def test_fp32_convs_on_tensor_cores_x3(shape):
    """csrc/x3.cu: fp32 tensors as split-bf16 convolutions on the tcgen05 kernels ([hi, lo, hi] x [hi, hi, lo], fp32
    accumulation, fp32 I/O epilogue) - forward with the fused epilogue, dgrad, wgrad and bias gradient against the CPU fp32
    convolution at the same 2e-5 / 5e-5 tolerances as the exact SIMT kernels (incl. K = 3 x 256 and 3 x 384 > 512 channels)."""
    yogo_b200.set_fp32_tensor_cores(True)
    try:
        assert yogo_b200.get_fp32_tensor_cores()
        n0 = L.load().yg_launch_count()
        _conv_case(*shape, dtype=torch.float32, act=(shape[3] % 3), with_stats=True, seed=sum(shape))
        assert L.load().yg_launch_count() - n0 >= 12   # split / concat / pack / tcgen05 launches, not three SIMT kernels
    finally:
        yogo_b200.set_fp32_tensor_cores(False)
    assert not yogo_b200.get_fp32_tensor_cores()


@pytest.mark.parametrize("name,prefix", [("silu_model", "silu_train."), ("base_model", "base_train.")])
def test_train_step_fp32_on_tensor_cores_x3(golden_dir, name, prefix):
    """Whole train step with compute_dtype = float32 on the x3 path vs the real reference's fp32 step.  silu_model (smooth):
    outputs, loss and every gradient within the fp32 tolerance.  base_model (LeakyReLU): forward and loss within 1e-3; the
    gradients differ wherever a pre-activation lies within the 2^-16 rounding of the kink (each such element moves a small
    fixture's gradient by ~0.5 %), so they are held to 5e-2 with a median <= 1e-2 - the reference's own default on the GPU
    (TF32 convolutions, 2^-11) sits 30x further from its fp32 result."""
    z = _load(golden_dir, "model_base.npz")
    yogo_b200.set_fp32_tensor_cores(True)
    try:
        net, sd = _build_from_golden(z, name)
        net.train()
        net._get_runner().drop_keep_override = {
            int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")}
        x = (torch.from_numpy(z["img"]).float() / 255.0).to(DEV)
        out = net(x)
        loss, comps = yogo_b200.YOGOLoss().to(DEV)(out, torch.from_numpy(z["label"]).to(DEV))
        loss.backward()
    finally:
        yogo_b200.set_fp32_tensor_cores(False)
    assert _rel(out.detach().cpu().numpy(), z[prefix + "out"]) < 1e-3
    assert abs(loss.item() - z[prefix + "loss"][0]) < 1e-3 * abs(z[prefix + "loss"][0])
    errs = {}
    for k, p in net.named_parameters():
        g = p.grad.detach().cpu().numpy().reshape(-1)
        exp = z[prefix + "grad." + k]
        if g.size > 16384:
            g = g[::5]
        errs[k] = float(np.linalg.norm(g - exp)) / max(float(np.linalg.norm(exp)), 1e-2)
    if name == "silu_model":
        bad = {k: v for k, v in errs.items() if v > 2e-3}
    else:
        bad = {k: v for k, v in errs.items() if v > 5e-2}
        assert float(np.median(list(errs.values()))) <= 1e-2, errs
    assert not bad, bad


@pytest.mark.parametrize("shape", [(2, 20, 36, 32, 64, 3, 2), (2, 19, 36, 32, 64, 3, 1), (2, 12, 20, 64, 128, 3, 1),
                                   (1, 21, 37, 128, 128, 3, 2)])
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_leaky_relu_sign_mask_equals_saved_activation_path(shape, impl):
    """yg_fwd_epilogue.actmask / yg_bwd_epilogue.actmask: the 1-bit-per-element LeakyReLU record must give the
    same dgrad result, bit for bit, as reading the saved activation (yogo/model.py's autograd keeps the tensor)."""
    import ctypes as C
    N, H, W, Cin, Cout, k, s = shape
    g = torch.Generator().manual_seed(sum(shape))
    dt = torch.bfloat16
    lib = L.lib()
    L.set_conv_impl(impl)
    try:
        # producer: conv (Cin_p -> Cin) + bias + LeakyReLU + Dropout2d writes y and its sign mask
        Cp = 16
        xp = torch.randn(N, H, W, Cp, generator=g).to(DEV).to(dt)
        wp = (torch.randn(Cin, Cp, 3, 3, generator=g) / 12).to(DEV)
        bp = (torch.randn(Cin, generator=g) * 0.1).to(DEV)
        keep = ((torch.rand(N, Cin, generator=g) > 0.2).float() / 0.8).to(DEV).contiguous()
        y = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
        pre = torch.empty_like(y)
        mask = torch.zeros(N * H * W * Cin // 8, dtype=torch.uint8, device=DEV)
        ep = L.FwdEpilogue(None, bp.data_ptr(), L.ACT_LRELU, keep.data_ptr(), None, pre.data_ptr(), mask.data_ptr())
        L.check(lib.yg_conv_fwd(xp.data_ptr(), wp.data_ptr(), y.data_ptr(), 1, N, H, W, Cp, Cin, 3, 1, C.byref(ep), L.stream()))
        bits = torch.from_numpy(np.unpackbits(mask.cpu().numpy(), bitorder="little")).reshape(N, H, W, Cin).bool()
        kept = (keep > 0)[:, None, None, :].expand(N, H, W, Cin).cpu()
        # wherever the channel was not dropped the bit is the sign of the activation input
        assert torch.equal(bits[kept], (pre.float().cpu() > 0)[kept])
        # the straight-line epilogue (taken when no pre-activation copy is requested): same output, bits = sign of it
        y2 = torch.empty_like(y)
        mask2 = torch.zeros_like(mask)
        ep2 = L.FwdEpilogue(None, bp.data_ptr(), L.ACT_LRELU, keep.data_ptr(), None, None, mask2.data_ptr())
        L.check(lib.yg_conv_fwd(xp.data_ptr(), wp.data_ptr(), y2.data_ptr(), 1, N, H, W, Cp, Cin, 3, 1, C.byref(ep2), L.stream()))
        # (with a pre-activation copy the value is rounded to bf16 before the activation, without it after: <= 1 ulp apart)
        torch.testing.assert_close(y2.float(), y.float(), rtol=2e-2, atol=1e-3)
        bits2 = torch.from_numpy(np.unpackbits(mask2.cpu().numpy(), bitorder="little")).reshape(N, H, W, Cin).bool()
        assert torch.equal(bits2[kept], (y2.float().cpu() > 0)[kept])
        # consumer: dgrad of the next conv with the activation backward fused, mask vs saved tensor
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        dz = torch.randn(N, Ho, Wo, Cout, generator=g).to(DEV).to(dt)
        w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(DEV)
        outs = []
        for use_mask in (False, True):
            dx = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
            sums = torch.zeros(2 * Cin, dtype=torch.float64, device=DEV)
            be = L.BwdEpilogue(y.data_ptr(), L.ACT_LRELU, keep.data_ptr(), None, None, None, None, sums.data_ptr(),
                               mask.data_ptr() if use_mask else None)
            L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, k, s, C.byref(be), L.stream()))
            outs.append((dx.float().cpu(), sums.cpu()))
        assert torch.equal(outs[0][0], outs[1][0])
        assert torch.allclose(outs[0][1], outs[1][1], rtol=1e-4, atol=1e-3)   # fp32 smem + fp64 global atomics: order varies
    finally:
        L.set_conv_impl("auto")


@pytest.mark.parametrize("shape", [(2, 20, 36, 32, 64, 3, 2), (2, 19, 37, 32, 64, 3, 1), (2, 12, 20, 64, 128, 3, 1),
                                   (1, 21, 37, 128, 128, 3, 2), (2, 13, 18, 128, 128, 3, 1)])
@pytest.mark.parametrize("with_bn", [False, True])
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_silu_epilogues_vs_torch(shape, with_bn, impl):
    """silu_model blocks (model_defns.py:80-127): forward = conv + bias + SiLU + Dropout2d with the bf16 pre-activation kept,
    backward = the next conv's dgrad with SiLU' (through the BatchNorm affine when the block has one) fused into its epilogue."""
    import ctypes as C
    N, H, W, Cin, Cout, k, s = shape
    g = torch.Generator().manual_seed(sum(shape) + int(with_bn))
    dt = torch.bfloat16
    lib = L.lib()
    L.set_conv_impl(impl)
    try:
        Cp = 16
        xp = torch.randn(N, H, W, Cp, generator=g).to(DEV).to(dt)
        wp = (torch.randn(Cin, Cp, 3, 3, generator=g) / 12)
        bp = (torch.randn(Cin, generator=g) * 0.1)
        keep = ((torch.rand(N, Cin, generator=g) > 0.2).float() / 0.8)
        y = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
        pre = torch.empty_like(y)
        wpd, bpd, kd = wp.to(DEV), bp.to(DEV), keep.to(DEV).contiguous()
        ep = L.FwdEpilogue(None, bpd.data_ptr(), L.ACT_SILU, kd.data_ptr(), None, pre.data_ptr(), None)
        L.check(lib.yg_conv_fwd(xp.data_ptr(), wpd.data_ptr(), y.data_ptr(), 1, N, H, W, Cp, Cin, 3, 1, C.byref(ep), L.stream()))
        pre_ref = torch.nn.functional.conv2d(xp.float().cpu().permute(0, 3, 1, 2), wp, bp, padding=1).permute(0, 2, 3, 1)
        assert _rel(pre.float().cpu(), pre_ref) < 6e-3
        # the activation is taken from the rounded pre-activation: compare with torch on exactly that tensor
        pr = pre.float().cpu()
        y_ref = torch.nn.functional.silu(pr) * keep[:, None, None, :]
        torch.testing.assert_close(y.float().cpu(), y_ref, rtol=1e-2, atol=1e-3)
        # consumer: dx = dgrad(dz) * SiLU'(pre or scale * saved + shift) * dropscale
        Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
        dz = torch.randn(N, Ho, Wo, Cout, generator=g).to(DEV).to(dt)
        w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5)
        wd = w.to(DEV)
        sc = (torch.rand(Cin, generator=g) + 0.5)
        sh = torch.randn(Cin, generator=g) * 0.2
        mean = torch.randn(Cin, generator=g) * 0.1
        istd = torch.rand(Cin, generator=g) + 0.5
        scd, shd, md, isd = sc.to(DEV), sh.to(DEV), mean.to(DEV), istd.to(DEV)
        dx = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
        if with_bn:
            be = L.BwdEpilogue(pre.data_ptr(), L.ACT_SILU, kd.data_ptr(), scd.data_ptr(), shd.data_ptr(), md.data_ptr(),
                               isd.data_ptr(), None, None)
        else:
            be = L.BwdEpilogue(pre.data_ptr(), L.ACT_SILU, kd.data_ptr(), None, None, None, None, None, None)
        L.check(lib.yg_conv_dgrad(dz.data_ptr(), wd.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, k, s, C.byref(be), L.stream()))
        a = (pr * sc + sh) if with_bn else pr
        a = a.clone().requires_grad_(True)
        xin = torch.nn.functional.silu(a) * keep[:, None, None, :]
        torch.nn.functional.conv2d(xin.permute(0, 3, 1, 2), w, None, stride=s, padding=k // 2).backward(
            dz.float().cpu().permute(0, 3, 1, 2))
        assert _rel(dx.float().cpu(), a.grad) < 6e-3, _rel(dx.float().cpu(), a.grad)
        # with the BN sums requested (generic epilogue) the result is the same up to bf16 rounding of the last factor
        if with_bn:
            sums = torch.zeros(2 * Cin, dtype=torch.float64, device=DEV)
            dx2 = torch.empty_like(dx)
            be2 = L.BwdEpilogue(pre.data_ptr(), L.ACT_SILU, kd.data_ptr(), scd.data_ptr(), shd.data_ptr(), md.data_ptr(),
                                isd.data_ptr(), sums.data_ptr(), None)
            L.check(lib.yg_conv_dgrad(dz.data_ptr(), wd.data_ptr(), dx2.data_ptr(), 1, N, H, W, Cin, Cout, k, s, C.byref(be2), L.stream()))
            torch.testing.assert_close(dx2.float(), dx.float(), rtol=2e-2, atol=2e-3)
            gsum = a.grad.double().sum((0, 1, 2))
            assert _rel(sums[:Cin].cpu(), gsum) < 2e-2
    finally:
        L.set_conv_impl("auto")


@pytest.mark.parametrize("Cout", [16, 32, 48])
@pytest.mark.parametrize("act", [1, 2])
@pytest.mark.parametrize("HW", [(70, 90), (71, 91), (64, 129)])
def test_first_layer_tensor_core_kernels_vs_torch(Cout, act, HW):
    """1 -> 16 / 32 / 48 channels, stride 2, uint8 image (base / double_filters / triple_filters, model_defns.py:39, 139, 189):
    forward = conv * scale + shift -> activation -> Dropout2d scale; backward = raw sums P[c][t] = sum g x_t and sum g with
    g = da * act'(pre) * dropscale, both on mma.sync with split-bf16 weights (first_layer.cu)."""
    import ctypes as C
    # (even widths take the aligned 16-bit tap loads, odd widths the per-lane byte loads; 129 leaves a one-pixel row segment)
    N, (H, W) = 3, HW
    g = torch.Generator().manual_seed(Cout + act)
    lib = L.lib()
    img = torch.randint(0, 256, (N, 1, H, W), dtype=torch.uint8, generator=g)
    w = torch.randn(Cout, 1, 3, 3, generator=g) / 300.0
    sc = torch.rand(Cout, generator=g) + 0.5
    sh = torch.randn(Cout, generator=g) * 0.3
    keep = ((torch.rand(N, Cout, generator=g) > 0.2).float() / 0.8)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    xd, wd, scd, shd, kd = img.to(DEV), w.to(DEV), sc.to(DEV), sh.to(DEV), keep.to(DEV).contiguous()
    y = torch.empty(N, Ho, Wo, Cout, device=DEV, dtype=torch.bfloat16)
    ep = L.FwdEpilogue(scd.data_ptr(), shd.data_ptr(), act, kd.data_ptr(), None, None)
    L.check(lib.yg_conv_first_fwd(xd.data_ptr(), L.YG_U8, wd.data_ptr(), y.data_ptr(), 1, N, H, W, 1, Cout, 2, C.byref(ep), L.stream()))
    z = torch.nn.functional.conv2d(img.float(), w, None, stride=2, padding=1)
    pre = (z * sc[None, :, None, None] + sh[None, :, None, None]).requires_grad_(True)
    a = O._act(pre, {1: "lrelu", 2: "silu"}[act]) * keep[:, :, None, None]
    assert _rel(y.float().cpu().permute(0, 3, 1, 2), a.detach()) < 4e-3
    da = torch.randn(N, Ho, Wo, Cout, generator=g).to(DEV).bfloat16()
    a.backward(da.float().cpu().permute(0, 3, 1, 2))
    gpre = pre.grad
    dw_ref = torch.nn.grad.conv2d_weight(img.float(), (Cout, 1, 3, 3), gpre, stride=2, padding=1)
    ds_ref = gpre.sum((0, 2, 3))
    dw = torch.empty(Cout, 1, 3, 3, device=DEV)
    dsh = torch.empty(Cout, device=DEV)
    nb = lib.yg_conv_first_bwd_workspace(1, Cout)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    be = L.BwdEpilogue(None, act, kd.data_ptr(), scd.data_ptr(), shd.data_ptr(), None, None, None, None)
    L.check(lib.yg_conv_first_bwd(xd.data_ptr(), L.YG_U8, wd.data_ptr(), da.data_ptr(), 1, N, H, W, 1, Cout, 2, C.byref(be),
                                  None, None, None, dw.data_ptr(), dsh.data_ptr(), 0.0, ws.data_ptr(), nb, L.stream()))
    # g is rounded to bf16 before the P = g . X product (2^-9 relative per term, random sign)
    assert _rel(dw.cpu(), dw_ref) < 4e-3, _rel(dw.cpu(), dw_ref)
    assert _rel(dsh.cpu(), ds_ref) < 4e-3
    # the SIMT kernels (any channel count) agree
    L.set_conv_impl("simt")
    try:
        y2 = torch.empty_like(y)
        L.check(lib.yg_conv_first_fwd(xd.data_ptr(), L.YG_U8, wd.data_ptr(), y2.data_ptr(), 1, N, H, W, 1, Cout, 2, C.byref(ep), L.stream()))
        dw2 = torch.empty_like(dw)
        dsh2 = torch.empty_like(dsh)
        L.check(lib.yg_conv_first_bwd(xd.data_ptr(), L.YG_U8, wd.data_ptr(), da.data_ptr(), 1, N, H, W, 1, Cout, 2, C.byref(be),
                                      None, None, None, dw2.data_ptr(), dsh2.data_ptr(), 0.0, ws.data_ptr(), nb, L.stream()))
    finally:
        L.set_conv_impl("auto")
    assert _rel(y2.float().cpu(), y.float().cpu()) < 4e-3
    assert _rel(dw2.cpu(), dw_ref) < 4e-3 and _rel(dsh2.cpu(), ds_ref) < 4e-3


def test_tensors_that_are_only_16_byte_aligned_take_the_generic_path():
    """The tensor-core epilogues use 32-byte stores; a 16-byte aligned view must not fault and must give the same result."""
    import ctypes as C
    N, H, W, Cin, Cout = 2, 12, 20, 64, 128
    g = torch.Generator().manual_seed(9)
    lib = L.lib()
    x = torch.randn(N, H, W, Cin, generator=g).to(DEV).bfloat16()
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / 24).to(DEV)
    b = torch.zeros(Cout, device=DEV)
    y = torch.empty(N, H, W, Cout, device=DEV, dtype=torch.bfloat16)
    ep = L.FwdEpilogue(None, b.data_ptr(), L.ACT_LRELU, None, None, None)
    L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, C.byref(ep), L.stream()))
    buf = torch.empty(y.numel() + 8, device=DEV, dtype=torch.bfloat16)
    y2 = buf[8:].view(N, H, W, Cout)
    assert y2.data_ptr() % 32 == 16
    L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y2.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, C.byref(ep), L.stream()))
    torch.cuda.synchronize()
    assert _rel(y2.float().cpu(), y.float().cpu()) < 6e-3
    dx = torch.empty_like(x)
    dxb = torch.empty(x.numel() + 8, device=DEV, dtype=torch.bfloat16)
    dx2 = dxb[8:].view(N, H, W, Cin)
    L.check(lib.yg_conv_dgrad(y.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, None, L.stream()))
    L.check(lib.yg_conv_dgrad(y.data_ptr(), w.data_ptr(), dx2.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, None, L.stream()))
    torch.cuda.synchronize()
    assert _rel(dx2.float().cpu(), dx.float().cpu()) < 6e-3


# ----------------------------------------------------------------------------- whole model vs golden
def _build_from_golden(z, name, sdprefix="sd.", dtype=torch.float32, inference=False):
    sd = {k[len(sdprefix):]: torch.from_numpy(z[k]) for k in z.files if k.startswith(sdprefix)}
    H, W = z["img"].shape[-2:]
    net = yogo_b200.YOGO((H, W), float(sd["anchor_w"]), float(sd["anchor_h"]), 7,
                         model_func=yogo_b200.get_model_func(name), inference=inference)
    net.load_state_dict(sd)
    net.compute_dtype = dtype
    return net.to(DEV), sd


def _grad_check(z, prefix, net, tol_rel, tol_floor):
    worst = {}
    for k, p in net.named_parameters():
        g = p.grad.detach().cpu().numpy().reshape(-1)
        exp = z[prefix + "grad." + k]
        if g.size > 16384:
            g = g[::5]
        denom = max(float(np.linalg.norm(exp)), tol_floor)
        worst[k] = float(np.linalg.norm(g - exp)) / denom
    bad = {k: v for k, v in worst.items() if v > tol_rel}
    assert not bad, bad


@pytest.mark.parametrize(
    "fname,prefix,name",
    [
        ("model_base.npz", "base_train.", "base_model"),
        ("model_base.npz", "silu_train.", "silu_model"),
        ("model_quarter_filters.npz", "train.", "quarter_filters"),
        ("model_depth_ver_0.npz", "train.", "depth_ver_0"),
    ],
)
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_train_step_fp32_matches_reference_golden(golden_dir, fname, prefix, name, impl):
    L.set_conv_impl(impl)
    try:
        z = _load(golden_dir, fname)
        net, sd = _build_from_golden(z, name)
        net.train()
        runner = net._get_runner()
        runner.drop_keep_override = {
            int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")
        }
        x = (torch.from_numpy(z["img"]).float() / 255.0).to(DEV)
        out = net(x)
        loss, comps = yogo_b200.YOGOLoss().to(DEV)(out, torch.from_numpy(z["label"]).to(DEV))
        loss.backward()
        assert _rel(out.detach().cpu().numpy(), z[prefix + "out"]) < 1e-3
        ref = z[prefix + "loss"]
        np.testing.assert_allclose(
            [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]], ref, rtol=1e-3)
        # conv bias in front of BatchNorm has a ~0 gradient: absolute floor (SURVEY.md 7)
        _grad_check(z, prefix, net, tol_rel=2e-3, tol_floor=1e-3)
        for k, v in net.state_dict().items():
            if "running_" in k:
                np.testing.assert_allclose(v.cpu().numpy(), z[f"{prefix}after.{k}"], rtol=1e-3, atol=1e-6)
    finally:
        L.set_conv_impl("auto")


@pytest.mark.parametrize("name,prefix", [("base_model", "base_train."), ("silu_model", "silu_train.")])
def test_train_step_bf16_within_calibrated_tolerance(golden_dir, name, prefix):
    """bf16 storage path, tolerance calibrated per tensor from the reference (SURVEY.md Appendix E)."""
    z = _load(golden_dir, "model_base.npz")
    net, sd = _build_from_golden(z, name, dtype=torch.bfloat16)
    net.train()
    net._get_runner().drop_keep_override = {
        int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")
    }
    x = (torch.from_numpy(z["img"]).float() / 255.0).to(DEV)
    out = net(x)
    loss, comps = yogo_b200.YOGOLoss().to(DEV)(out, torch.from_numpy(z["label"]).to(DEV))
    loss.backward()
    # acceptance: error vs the fp32 reference <= 1.5 x the reference's OWN bf16-autocast error on the
    # same inputs/weights/masks (recorded by tests/golden/make_golden.py), with small floors
    def bound(key, floor):
        return max(1.5 * float(z[prefix + "bf16err." + key][0]), floor)

    assert _rel(out.detach().cpu().numpy(), z[prefix + "out"]) < bound("out", 1e-2)
    assert abs(loss.item() - z[prefix + "loss"][0]) < bound("loss", 1e-3) * abs(z[prefix + "loss"][0])
    report = {}
    for k, p in net.named_parameters():
        g = p.grad.detach().cpu().numpy().reshape(-1)
        exp = z[prefix + "grad." + k]
        if g.size > 16384:
            g = g[::5]
        denom = max(float(np.linalg.norm(exp)), 1e-3)
        err = float(np.linalg.norm(g - exp)) / denom
        report[k] = (err, bound("grad." + k, 2e-2))
    bad = {k: v for k, v in report.items() if v[0] >= v[1]}
    assert not bad, bad


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-3), (torch.bfloat16, 3e-2)])
def test_eval_and_inference_forward_match_reference_golden(golden_dir, dtype, tol):
    z = _load(golden_dir, "model_base.npz")
    x = (torch.from_numpy(z["img"]).float() / 255.0).to(DEV)
    for name, key, inf in (("base_model", "base_eval.out", False), ("base_model", "base_infer.out", True),
                           ("silu_model", "silu_eval.out", False)):
        net, _ = _build_from_golden(z, name, dtype=dtype, inference=inf)
        net.eval()
        with torch.no_grad():
            out = net(x)
        assert out.dtype == torch.float32 and out.is_contiguous()
        assert _rel(out.cpu().numpy(), z[key]) < tol, (name, key)
        # uint8 input path == float input path (x.float(), model.py:272-273)
        with torch.no_grad():
            a = net(torch.from_numpy(z["img"]).to(DEV))
            b = net(torch.from_numpy(z["img"]).float().to(DEV))
        if dtype == torch.float32:
            assert torch.equal(a, b)
        else:
            # bf16: the uint8 path runs the first layer on the tensor cores with split-bf16 weights (2^-17 relative), the
            # float path on the FMA pipe; both round to the same bf16 activations except at rounding boundaries
            assert _rel(a.cpu().numpy(), b.cpu().numpy()) < 1e-2


def test_full_size_train_step_vs_oracle_fp32():
    """BASELINE geometry (772x1032 -> 97x129 grid), small batch, fp32 path vs the CPU oracle."""
    torch.manual_seed(0)
    net = yogo_b200.YOGO((772, 1032), O.ANCHOR_W, O.ANCHOR_H, 7)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.05)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.to(DEV)
    net.compute_dtype = torch.float32
    net.train()
    N = 2
    img = O.synth_images(N)
    lab = O.synth_labels(N)
    keeps = {1: (torch.rand(N, 32) > 0.05).float(), 2: (torch.rand(N, 64) > 0.1).float(),
             3: (torch.rand(N, 128) > 0.15).float()}
    net._get_runner().drop_keep_override = keeps
    out = net(img.to(DEV))  # raw uint8, un-normalised (reference default)
    x = img.float() / 255.0
    out = net(x.to(DEV))
    loss, comps = yogo_b200.YOGOLoss().to(DEV)(out, lab.to(DEV))
    loss.backward()
    blocks = O.blocks_from_state_dict("base_model", sd)
    for b in blocks:
        b.weight.requires_grad_(True)
    t = O.backbone_forward(x, blocks, train=True, drop_keep=[keeps.get(i) for i in range(len(blocks))])
    ref_out = O.head_transform(t, O.ANCHOR_W, O.ANCHOR_H)
    ref_loss, ref_comps, dpred = O.yogo_loss_np(ref_out.detach().numpy(), lab.numpy())
    ref_out.backward(torch.from_numpy(dpred))
    assert _rel(out.detach().cpu().numpy(), ref_out.detach().numpy()) < 1e-3
    assert abs(loss.item() - ref_loss) < 1e-3 * abs(ref_loss)
    for i, b in enumerate(blocks):
        key = f"model.{i}.weight" if i == len(blocks) - 1 else f"model.{i}.0.weight"
        g = dict(net.named_parameters())[key].grad.cpu()
        r = b.weight.grad.clamp(-1, 1)
        assert _rel(g.numpy(), r.numpy()) < 3e-3, (key, _rel(g.numpy(), r.numpy()))


# ----------------------------------------------------------------------------- every definition, RGB, BASELINE geometry
from _zoo_cases import ZOO_CASES, grad_sample, zoo_inputs  # noqa: E402

FULL_CASES = ["full_base_model", "full_silu_model", "full_double_filters"]


def _zoo_step(z, case, dtype, impl="auto"):
    name, net, img, lab, ostride = zoo_inputs(z, case)
    prefix = case + ".train."
    net = net.to(DEV)
    net.compute_dtype = dtype
    net.train()
    net._get_runner().drop_keep_override = {
        int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")}
    out = net((img.float() / 255.0).to(DEV))
    loss, comps = yogo_b200.YOGOLoss().to(DEV)(out, lab.to(DEV))
    loss.backward()
    o = out.detach().cpu().numpy()[:, :, ::ostride, ::ostride]
    # a conv bias in front of BatchNorm has a mathematically zero gradient (the batch mean removes it): what is left is
    # rounding noise of a cancelling sum, compared against the scale of the BatchNorm bias gradient of the same block
    zero_keys = {f"model.{i}.0.bias": f"model.{i}.1.bias" for i, blk in enumerate(net.model)
                 if isinstance(blk, torch.nn.Sequential) and len(blk) > 1 and isinstance(blk[1], torch.nn.BatchNorm2d)
                 and blk[0].bias is not None}
    errs = {}
    for k, p in net.named_parameters():
        g = p.grad.detach().cpu().numpy().reshape(-1)
        exp = z[prefix + "grad." + k]
        g = grad_sample(g, exp.size)
        scale = float(np.linalg.norm(exp))
        if k in zero_keys:
            scale = max(scale, float(z[prefix + "gradnorm." + zero_keys[k]][0]))
        errs[k] = float(np.linalg.norm(g - exp)) / max(scale, 1e-3)
    return net, o, loss, comps, errs


@pytest.mark.parametrize("case", ZOO_CASES)
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_zoo_train_step_fp32_matches_reference_golden(golden_dir, case, impl):
    """double/triple/half_filters, depth_ver_1..4 (model_defns.py:130-277, 358-529) and RGB input (:32): one fp32
    train step vs the real reference, 1e-3 relative."""
    z = _load(golden_dir, "model_zoo.npz")
    L.set_conv_impl(impl)
    try:
        net, o, loss, comps, errs = _zoo_step(z, case, torch.float32)
    finally:
        L.set_conv_impl("auto")
    prefix = case + ".train."
    assert _rel(o, z[prefix + "out"]) < 1e-3
    np.testing.assert_allclose(
        [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]], z[prefix + "loss"], rtol=1e-3)
    bad = {k: v for k, v in errs.items() if v > 2e-3}
    assert not bad, bad
    for k, v in net.state_dict().items():
        if "running_" in k:
            np.testing.assert_allclose(v.cpu().numpy(), z[f"{prefix}after.{k}"], rtol=1e-3, atol=1e-6)


def _bf16_bounds_ok(z, case, o, loss, errs, factor=2.0):
    """Yardstick = the reference's OWN bf16-autocast error against its fp32 run on the same inputs, weights and masks,
    recorded per tensor by make_golden.py (SURVEY.md Appendix E).  Measured over the 12 cases x ~20 tensors of
    model_zoo.npz / model_full.npz, our error / the reference's error has a median of 0.8 (the engine is a little more
    accurate than autocast), but a single tensor is a single draw of a rounding error: on 7x9 grids the weight gradient of
    the last 3x3 conv is dominated by the two dozen labelled cells and reaches 1.4 - 2.4 x.  Acceptance: every tensor
    <= `factor` x the yardstick (floors for near-zero tensors) AND the median ratio over the tensors <= 1.25."""
    pre = case + "."

    def bound(key, floor):
        return max(factor * float(z[pre + "bf16err." + key][0]), floor)

    report = {}
    e = _rel(o, z[pre + "train.out"])
    if e >= bound("out", 1e-2):
        report["out"] = (e, bound("out", 1e-2))
    ref_loss = z[pre + "train.loss"][0]
    e = abs(loss.item() - ref_loss) / abs(ref_loss)
    if e >= bound("loss", 1e-3):
        report["loss"] = (e, bound("loss", 1e-3))
    for k, v in errs.items():
        if v >= bound("grad." + k, 2e-2):
            report[k] = (v, bound("grad." + k, 2e-2))
    ratios = [v / max(float(z[pre + "bf16err.grad." + k][0]), 1e-2) for k, v in errs.items()]
    if float(np.median(ratios)) > 1.25:
        report["median ratio"] = float(np.median(ratios))
    return report


@pytest.mark.parametrize("case", ZOO_CASES)
def test_zoo_train_step_bf16_within_calibrated_tolerance(golden_dir, case):
    z = _load(golden_dir, "model_zoo.npz")
    net, o, loss, comps, errs = _zoo_step(z, case, torch.bfloat16)
    report = _bf16_bounds_ok(z, case, o, loss, errs, factor=3.0)   # tiny grids: see _bf16_bounds_ok
    assert not report, report


@pytest.mark.parametrize("case", FULL_CASES)
def test_full_geometry_train_step_bf16_vs_reference_golden(golden_dir, case):
    """BASELINE configs[1] / configs[3] geometry (772x1032 -> 97x129; many tiles per CTA, TMEM accumulators in rotation,
    W-fold, CTA pairs, parity classes with 97x129 tails, N = 256 MMAs) on the bf16 tcgen05 path that bench.py times,
    against the real reference's fp32 step with its own bf16-autocast error as the yardstick."""
    z = _load(golden_dir, "model_full.npz")
    net, o, loss, comps, errs = _zoo_step(z, case, torch.bfloat16)
    report = _bf16_bounds_ok(z, case, o, loss, errs)
    assert not report, report
    name, net, img, _, ostride = zoo_inputs(z, case)   # fresh buffers: the golden eval output uses the initial running stats
    net = net.to(DEV)
    net.compute_dtype = torch.bfloat16
    net.eval()
    with torch.no_grad():
        ev = net((img.float() / 255.0).to(DEV)).cpu().numpy()[:, :, ::ostride, ::ostride]
    assert _rel(ev, z[case + ".eval.out"]) < 3e-2


@pytest.mark.parametrize("case", ["full_base_model", "full_silu_model"])
def test_full_geometry_train_step_fp32_vs_reference_golden(golden_dir, case):
    """fp32 storage path at the BASELINE geometry.  With 1e8 LeakyReLU inputs some always sit within rounding noise of
    the kink, and taking the other slope there is a legitimate fp32 result: the reference's own fp32 gradients differ from
    its float64 gradients by up to 1.5e-2 on this fixture (fp32err.*, make_golden.py).  Bound per tensor: max(1e-3 (north
    star), 3 x that error).  silu_model has no kink: its bounds stay at 1e-3 for every tensor."""
    z = _load(golden_dir, "model_full.npz")
    net, o, loss, comps, errs = _zoo_step(z, case, torch.float32)
    assert _rel(o, z[case + ".train.out"]) < 1e-3
    assert abs(loss.item() - z[case + ".train.loss"][0]) < 1e-3 * abs(z[case + ".train.loss"][0])
    bound = {k: max(1e-3, 3.0 * float(z[f"{case}.fp32err.grad.{k}"][0])) for k in errs}
    if case == "full_silu_model":
        bound = {k: 1e-3 for k in errs}
    bad = {k: (v, bound[k]) for k, v in errs.items() if v > bound[k]}
    assert not bad, bad


def test_variable_batch_and_3d_input():
    net = yogo_b200.YOGO((64, 96), 0.05, 0.05, 7).to(DEV)
    net.eval()
    with torch.no_grad():
        o1 = net(torch.rand(1, 64, 96, device=DEV))       # 3-D input is unsqueezed (model.py:269-270)
        o5 = net(torch.rand(5, 1, 64, 96, device=DEV))    # ragged last batch (drop_last=False)
    assert tuple(o1.shape) == (1, 12, 8, 12) and tuple(o5.shape) == (5, 12, 8, 12)
    assert torch.isfinite(o5).all()


# ----------------------------------------------------------------------------- trainer
def _make_trainer(seed=0, dtype=torch.float32):
    from yogo_b200.train import DataParallelTrainer
    torch.manual_seed(seed)
    net = yogo_b200.YOGO((96, 128), O.ANCHOR_W, O.ANCHOR_H, 7).to(DEV)
    net.compute_dtype = dtype
    net.train()
    for m in net.model.modules():
        if isinstance(m, torch.nn.Dropout2d):
            m.p = 0.0  # deterministic comparison between eager and graph replay
    net._runner = None
    return net, DataParallelTrainer(net, yogo_b200.YOGOLoss().to(DEV), total_steps=50)


def test_trainer_step_matches_torch_adamw_and_graph_replay():
    """fused flat AdamW + cosine schedule == torch.optim.AdamW + CosineAnnealingLR on the same gradients
    (train.py:213-223); CUDA-graph replay of the whole step == eager execution."""
    img = O.synth_images(4, 96, 128).to(DEV)
    lab = O.synth_labels(4, 12, 16, 7, 10).to(DEV)
    net_a, tr_a = _make_trainer()
    net_b, tr_b = _make_trainer()
    ref_params = [p.detach().clone().requires_grad_(True) for p in net_a.parameters()]
    opt = torch.optim.AdamW(ref_params, lr=3e-4, weight_decay=5e-2)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=50, eta_min=3e-4 / 10)
    tr_b.enable_cuda_graph(img, lab)
    for step in range(3):
        la = tr_a.step(img, lab)
        lb = tr_b.step(img, lab)
        # step 0 starts from identical parameters: loss and gradients agree up to the fp32 summation order of
        # the BN statistics (atomics).  Adam's first steps turn a sign flip of a ~0 gradient into a +-lr
        # difference, which then propagates, so later steps are compared statistically.
        if step == 0:
            assert abs(la.item() - lb.item()) <= 1e-5 * abs(la.item())
            assert float((tr_a.flat_g - tr_b.flat_g).norm() / tr_a.flat_g.norm()) < 1e-4
            # BN buffers advanced identically in both modes
            for (ka, va), (kb, vb) in zip(net_a.state_dict().items(), net_b.state_dict().items()):
                if "running_" in ka or "num_batches" in ka:
                    torch.testing.assert_close(va.float(), vb.float(), rtol=1e-4, atol=1e-6)
        else:
            assert abs(la.item() - lb.item()) <= 1e-2 * abs(la.item())
        bad = ((tr_a.flat_p - tr_b.flat_p).abs() > 1e-6 + 1e-5 * tr_a.flat_p.abs()).float().mean().item()
        assert bad < 0.05, bad
        for rp, p in zip(ref_params, net_a.parameters()):
            rp.grad = p.grad.detach().clone()
        opt.step()
        sched.step()
        for rp, p in zip(ref_params, net_a.parameters()):
            torch.testing.assert_close(p.detach(), rp.detach(), rtol=2e-5, atol=2e-7)
    assert tr_b.graph_launches > 20
    assert int(net_a.model[0][1].num_batches_tracked) == int(net_b.model[0][1].num_batches_tracked) == 3


def test_device_prefetcher_yields_batches_in_order():
    """DevicePrefetcher (the pin_memory + non_blocking loader pattern of train.py:288-291): every batch arrives, in
    order, bit-identical, while the next copy is already in flight."""
    from yogo_b200.train import DevicePrefetcher
    g = torch.Generator().manual_seed(3)
    host = [(torch.randint(0, 255, (2, 1, 32, 48), generator=g, dtype=torch.uint8).pin_memory(),
             torch.rand(2, 6, 4, 6, generator=g).pin_memory()) for _ in range(5)]
    got = [(x.cpu(), y.cpu()) for x, y in DevicePrefetcher(iter(host), DEV)]
    assert len(got) == len(host)
    for (hx, hy), (dx, dy) in zip(host, got):
        assert torch.equal(hx, dx) and torch.equal(hy, dy)


@pytest.mark.parametrize("shape", [(3, 33, 20, 128, 128, 3, 1), (1, 17, 9, 128, 128, 3, 1), (2, 21, 37, 128, 128, 3, 2),
                                   (2, 19, 36, 64, 128, 3, 1), (3, 20, 36, 32, 64, 3, 2), (2, 19, 36, 16, 32, 3, 1)])
def test_conv_outputs_stay_inside_their_buffers(shape):
    """Guard regions around every output of the tensor-core paths (CTA pairs with a padding tile, 2-D halo boxes, parity
    classes, W-folded views, sign masks): nothing outside the tensors may be written."""
    import ctypes as C
    N, H, W, Cin, Cout, k, s = shape
    g = torch.Generator().manual_seed(sum(shape))
    dt = torch.bfloat16
    lib = L.lib()
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    GUARD = 4096

    def guarded(numel, dtype, fill):
        buf = torch.full((numel + 2 * GUARD,), fill, dtype=dtype, device=DEV)
        return buf, buf[GUARD:GUARD + numel]

    def intact(buf, numel, fill):
        return bool((buf[:GUARD] == fill).all()) and bool((buf[GUARD + numel:] == fill).all())

    x = torch.randn(N, H, W, Cin, generator=g).to(DEV).to(dt)
    w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(DEV)
    b = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    ybuf, y = guarded(N * Ho * Wo * Cout, dt, 7.0)
    mbuf, m = guarded(N * Ho * Wo * Cout // 8, torch.uint8, 0xA5)
    ep = L.FwdEpilogue(None, b.data_ptr(), L.ACT_LRELU, None, None, None, m.data_ptr())
    L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, k, s, C.byref(ep), L.stream()))
    torch.cuda.synchronize()
    assert intact(ybuf, y.numel(), 7.0) and intact(mbuf, m.numel(), 0xA5)
    ref = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2).cpu(), w.cpu(), b.cpu(), stride=s, padding=1), 0.01)
    assert _rel(y.float().reshape(N, Ho, Wo, Cout).permute(0, 3, 1, 2).cpu(), ref) < 6e-3
    dz = torch.randn(N, Ho, Wo, Cout, generator=g).to(DEV).to(dt)
    dxbuf, dx = guarded(N * H * W * Cin, dt, 7.0)
    xmask = torch.randint(0, 255, (N * H * W * Cin // 8,), dtype=torch.uint8, device=DEV)
    be = L.BwdEpilogue(x.data_ptr(), L.ACT_LRELU, None, None, None, None, None, None, xmask.data_ptr())
    L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, k, s, C.byref(be), L.stream()))
    dwbuf, dw = guarded(w.numel(), torch.float32, 7.0)
    dbbuf, db = guarded(Cout, torch.float32, 7.0)
    nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, k, s)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_conv_wgrad(x.data_ptr(), dz.data_ptr(), dw.data_ptr(), db.data_ptr(), 1, N, H, W, Cin, Cout, k, s, 0.0,
                              ws.data_ptr(), nb, L.stream()))
    torch.cuda.synchronize()
    assert intact(dxbuf, dx.numel(), 7.0) and intact(dwbuf, dw.numel(), 7.0) and intact(dbbuf, db.numel(), 7.0)
    assert bool(torch.isfinite(dx.float()).all()) and bool(torch.isfinite(dw).all())


@pytest.mark.parametrize("shape", [(2, 40, 64, 16, 32, 1), (2, 39, 36, 64, 128, 1), (2, 41, 38, 32, 64, 2), (2, 37, 36, 128, 128, 2),
                                   (2, 33, 24, 128, 128, 1), (1, 38, 40, 48, 96, 1)])
def test_flat_mma_issue_list_is_bit_identical_to_the_table_walk(shape):
    """The MMA warp issues from a flat host-built list (one word per MMA, structurally zero K steps of W-folded layers left out);
    option bit 22 restores the per-tap table walk.  Same MMAs in the same order: forward and dgrad outputs must be bit-identical
    (W-folded, CTA-pair, stride-2 parity-class and streamed-weight configurations)."""
    import ctypes as C
    N, H, W, Cin, Cout, s = shape
    lib = L.lib()
    g = torch.Generator().manual_seed(sum(shape))
    dt = torch.bfloat16
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    x = torch.randn(N, H, W, Cin, generator=g).to(DEV).to(dt)
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (Cin * 9) ** 0.5).to(DEV)
    b = (torch.randn(Cout, generator=g) * 0.1).to(DEV)
    dz = torch.randn(N, Ho, Wo, Cout, generator=g).to(DEV).to(dt)
    xmask = torch.randint(0, 255, (N * H * W * Cin // 8,), generator=g, dtype=torch.uint8).to(DEV)
    outs = []
    base = lib.yg_get_tc_options()
    try:
        for bit in (0, 1 << 22):
            L.check(lib.yg_set_tc_options(base | bit))
            y = torch.zeros(N, Ho, Wo, Cout, dtype=dt, device=DEV)
            m = torch.zeros(y.numel() // 8, dtype=torch.uint8, device=DEV)
            ep = L.FwdEpilogue(None, b.data_ptr(), L.ACT_LRELU, None, None, None, m.data_ptr())
            L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(ep), L.stream()))
            dx = torch.zeros(N, H, W, Cin, dtype=dt, device=DEV)
            be = L.BwdEpilogue(x.data_ptr(), L.ACT_LRELU, None, None, None, None, None, None, xmask.data_ptr())
            L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(be), L.stream()))
            torch.cuda.synchronize()
            outs.append((y, m, dx))
    finally:
        L.check(lib.yg_set_tc_options(base))
    assert bool(outs[0][0].float().abs().sum() > 0) and bool(outs[0][2].float().abs().sum() > 0)
    for a, b_ in zip(outs[0], outs[1]):
        assert torch.equal(a, b_)


FULL_LAYERS = [
    # (N, H, W, Cin, Cout, stride): every 3x3 layer of base_model / double_filters at the 772x1032 geometry
    (3, 386, 516, 16, 32, 1), (3, 386, 516, 32, 64, 2), (3, 193, 258, 64, 128, 1), (3, 193, 258, 128, 128, 2),
    (5, 97, 129, 128, 128, 1),
    (2, 386, 516, 32, 64, 1), (2, 386, 516, 64, 128, 2), (2, 193, 258, 128, 256, 1), (2, 193, 258, 256, 256, 2),
    (3, 97, 129, 256, 256, 1),
]


@pytest.mark.parametrize("shape", FULL_LAYERS)
def test_full_geometry_layers_tcgen05_equals_simt(shape):
    """The tcgen05 kernels at the benchmark geometry (many tiles per CTA, accumulators in rotation, W-fold, CTA pairs,
    parity classes with 97x129 / 193x258 tails, N = 256) against the straightforward SIMT kernels on the same bf16
    inputs: both accumulate in fp32, so outputs agree up to the accumulation order (one bf16 ulp on a few elements)."""
    import ctypes as C
    N, H, W, Cin, Cout, s = shape
    lib = L.lib()
    g = torch.Generator(device=DEV).manual_seed(sum(shape))
    dt = torch.bfloat16
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    x = torch.randn(N, H, W, Cin, device=DEV, generator=g).to(dt)
    # weights representable in bf16: the tcgen05 path packs them to bf16 (as autocast does), the SIMT path reads fp32
    w = (torch.randn(Cout, Cin, 3, 3, device=DEV, generator=g) / (Cin * 9) ** 0.5).bfloat16().float()
    b = torch.randn(Cout, device=DEV, generator=g) * 0.1
    keep = ((torch.rand(N, Cout, device=DEV, generator=g) > 0.15).float() / 0.85).contiguous()
    keep_in = ((torch.rand(N, Cin, device=DEV, generator=g) > 0.15).float() / 0.85).contiguous()
    dz = torch.randn(N, Ho, Wo, Cout, device=DEV, generator=g).to(dt)
    res = {}
    for impl in ("simt", "auto"):
        L.set_conv_impl(impl)
        try:
            y = torch.empty(N, Ho, Wo, Cout, device=DEV, dtype=dt)
            mask = torch.zeros(N * Ho * Wo * Cout // 8, dtype=torch.uint8, device=DEV)
            ep = L.FwdEpilogue(None, b.data_ptr(), L.ACT_LRELU, keep.data_ptr(), None, None, mask.data_ptr())
            L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(ep), L.stream()))
            dx = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
            be = L.BwdEpilogue(x.data_ptr(), L.ACT_LRELU, keep_in.data_ptr(), None, None, None, None, None, None)
            L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, C.byref(be), L.stream()))
            dw = torch.empty_like(w)
            db = torch.empty_like(b)
            nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, 3, s)
            ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
            L.check(lib.yg_conv_wgrad(x.data_ptr(), dz.data_ptr(), dw.data_ptr(), db.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, 0.0,
                                      ws.data_ptr(), nb, L.stream()))
            torch.cuda.synchronize()
            res[impl] = (y.float(), dx.float(), dw, db, mask)
        finally:
            L.set_conv_impl("auto")
    (y0, dx0, dw0, db0, m0), (y1, dx1, dw1, db1, m1) = res["simt"], res["auto"]

    def close(a, b_, what):
        # bf16 outputs: every element within one bf16 ulp (2^-7 relative at worst) of the SIMT result - the fp32 accumulation
        # order and the order of the epilogue's roundings differ - plus the fp32 noise of cancelling sums near zero
        d = (a - b_).abs()
        rms = float(b_.pow(2).mean().sqrt())
        viol = d > (2.0 ** -7) * torch.maximum(a.abs(), b_.abs()) + 1e-5 * rms
        assert int(viol.sum()) == 0, (what, int(viol.sum()), float(d.max()))
        assert float(torch.linalg.vector_norm(d) / torch.linalg.vector_norm(b_)) < 2e-3, what

    close(y1, y0, "fwd")
    close(dx1, dx0, "dgrad")
    assert float((dw1 - dw0).norm() / dw0.norm()) < 2e-5 and float((db1 - db0).norm() / db0.norm()) < 2e-5
    # sign masks may differ only where the activation input is within rounding of zero
    assert float((m0 != m1).float().mean()) < 1e-3


def test_conv_tensors_larger_than_4GiB():
    """Index arithmetic beyond 2^32 bytes (double_filters at batch >= 168, base_model at batch 256 x 2 maps): a 32 -> 64
    stride-1 conv whose bf16 output is 4.4 GB.  Forward and dgrad are compared at sampled pixels (the last image sits
    above the 4 GiB line) with F.conv2d on the surrounding patches; wgrad by additivity over the batch."""
    import ctypes as C
    lib = L.lib()
    N, H, W, Cin, Cout = 172, 386, 516, 32, 64
    assert N * H * W * Cout * 2 > (1 << 32) + (1 << 26)
    g = torch.Generator(device=DEV).manual_seed(5)
    dt = torch.bfloat16
    x = torch.randn(N, H, W, Cin, device=DEV, generator=g, dtype=torch.float32).to(dt)
    w = torch.randn(Cout, Cin, 3, 3, device=DEV, generator=g) / (Cin * 9) ** 0.5
    b = torch.randn(Cout, device=DEV, generator=g) * 0.1
    y = torch.empty(N, H, W, Cout, device=DEV, dtype=dt)
    ep = L.FwdEpilogue(None, b.data_ptr(), L.ACT_NONE, None, None, None, None)
    L.check(lib.yg_conv_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, C.byref(ep), L.stream()))
    dz = torch.randn(N, H, W, Cout, device=DEV, generator=g, dtype=torch.float32).to(dt)
    dx = torch.empty(N, H, W, Cin, device=DEV, dtype=dt)
    L.check(lib.yg_conv_dgrad(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), 1, N, H, W, Cin, Cout, 3, 1, None, L.stream()))
    rs = np.random.RandomState(0)
    pts = [(n, int(rs.randint(0, H)), int(rs.randint(0, W))) for n in (0, 1, 85, 86, 167, 168, 169, 170, 171) for _ in range(24)]
    pts += [(171, H - 1, W - 1), (171, 0, 0), (171, H - 1, 0), (168, H - 1, W - 1), (0, 0, 0)]
    wc, bc = w.cpu(), b.cpu()
    for (n, h, ww) in pts:
        h0, h1, w0, w1 = max(h - 1, 0), min(h + 2, H), max(ww - 1, 0), min(ww + 2, W)
        patch = torch.zeros(1, Cin, 3, 3)
        patch[0, :, h0 - h + 1:h1 - h + 1, w0 - ww + 1:w1 - ww + 1] = x[n, h0:h1, w0:w1].float().cpu().permute(2, 0, 1)
        ref = torch.nn.functional.conv2d(patch, wc, bc)[0, :, 0, 0]
        assert _rel(y[n, h, ww].float().cpu(), ref) < 6e-3, ("fwd", n, h, ww)
        gp = torch.zeros(1, Cout, 3, 3)
        gp[0, :, h0 - h + 1:h1 - h + 1, w0 - ww + 1:w1 - ww + 1] = dz[n, h0:h1, w0:w1].float().cpu().permute(2, 0, 1)
        # dx[ci] = sum_{co,r,s} dz[h+1-r, w+1-s, co] w[co,ci,r,s]  == conv of the dz patch with the flipped, transposed filter
        refd = torch.nn.functional.conv2d(gp, wc.flip(2, 3).permute(1, 0, 2, 3))[0, :, 0, 0]
        assert _rel(dx[n, h, ww].float().cpu(), refd) < 6e-3, ("dgrad", n, h, ww)
    # wgrad is additive over images: whole batch == first 160 + last 12 (the last chunk starts beyond 4 GiB of dz)
    nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, 3, 1)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)

    def wgrad(xs, dzs):
        n = xs.shape[0]
        dw = torch.empty_like(w)
        db = torch.empty_like(b)
        L.check(lib.yg_conv_wgrad(xs.data_ptr(), dzs.data_ptr(), dw.data_ptr(), db.data_ptr(), 1, n, H, W, Cin, Cout, 3, 1, 0.0,
                                  ws.data_ptr(), nb, L.stream()))
        return dw.double().cpu(), db.double().cpu()

    dw_all, db_all = wgrad(x, dz)
    dw_a, db_a = wgrad(x[:160], dz[:160])
    dw_b, db_b = wgrad(x[160:], dz[160:])
    assert _rel(dw_all, dw_a + dw_b) < 1e-4 and _rel(db_all, db_a + db_b) < 1e-4
    # and the tail chunk against autograd on the CPU
    xr = x[160:].float().cpu().permute(0, 3, 1, 2)
    wr = wc.clone().requires_grad_(True)
    torch.nn.functional.conv2d(xr, wr, None, padding=1).backward(dz[160:].float().cpu().permute(0, 3, 1, 2))
    assert _rel(dw_b, wr.grad.double()) < 3e-3


@pytest.mark.parametrize("shape", [(2, 19, 35, 16, 32, 1), (1, 8, 32, 16, 32, 1), (3, 21, 37, 32, 64, 2), (2, 40, 70, 16, 32, 1)])
def test_small_channel_wgrad_on_mma_sync_matches_autograd(shape):
    """wgrad_hmma.cu (16->32 by default, 32->64 stride 2 with option bit 16) against autograd of the CPU convolution."""
    N, H, W, Cin, Cout, s = shape
    g = torch.Generator().manual_seed(sum(shape))
    lib = L.lib()
    x = torch.randn(N, Cin, H, W, generator=g)
    w = torch.randn(Cout, Cin, 3, 3, generator=g) / (Cin * 9) ** 0.5
    b = torch.zeros(Cout)
    xd = x.permute(0, 2, 3, 1).contiguous().to(DEV).bfloat16()
    xr = xd.float().permute(0, 3, 1, 2).cpu()
    wr = w.clone().requires_grad_(True)
    br = b.clone().requires_grad_(True)
    y = torch.nn.functional.conv2d(xr, wr, br, stride=s, padding=1)
    dz = torch.randn(y.shape, generator=g)
    dzd = dz.permute(0, 2, 3, 1).contiguous().to(DEV).bfloat16()
    y.backward(dzd.float().permute(0, 3, 1, 2).cpu())
    lib.yg_set_tc_options(25 + 8192 + 16384 + 65536)
    try:
        dw = torch.empty(Cout, Cin, 3, 3, device=DEV)
        db = torch.empty(Cout, device=DEV)
        nb = lib.yg_conv_wgrad_workspace(N, H, W, Cin, Cout, 3, s)
        ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
        L.check(lib.yg_conv_wgrad(xd.data_ptr(), dzd.data_ptr(), dw.data_ptr(), db.data_ptr(), 1, N, H, W, Cin, Cout, 3, s, 0.0,
                                  ws.data_ptr(), nb, L.stream()))
        assert _rel(dw.cpu(), wr.grad) < 1e-4 and _rel(db.cpu(), br.grad) < 1e-4
    finally:
        lib.yg_set_tc_options(25 + 8192 + 16384)


def test_multi_rank_equivalence(tmp_path):
    """tests/ddp_gpu_check.py under torchrun on 2 GPUs (skipped on single-GPU boxes; its log from a 2-GPU gpurun is kept
    under profiles/)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29533", os.path.join(root, "tests", "ddp_gpu_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ddp_gpu_check ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_graphed_inference_equals_eager():
    """yogo_b200.infer.GraphedInference: forward + threshold + NMS + counts replayed from one CUDA graph gives exactly
    the eager results, for successive different batches."""
    from yogo_b200.infer import GraphedInference
    torch.manual_seed(0)
    net = yogo_b200.YOGO((196, 260), O.ANCHOR_W, O.ANCHOR_H, 7, inference=True).to(DEV)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.3)
    net.eval()
    gi = GraphedInference(net, (3, 1, 196, 260))
    for seed in (1, 2, 3):
        img = O.synth_images(3, 196, 260, seed=seed).to(DEV)
        pred, rows, kc, kidx, counts = gi(img)
        with torch.no_grad():
            ref = net(img)
        r2, kc2, kidx2, counts2 = yogo_b200.format_preds_batch(ref)
        assert torch.equal(pred, ref) and torch.equal(kc, kc2) and torch.equal(counts, counts2)
        for b in range(3):
            n = int(kc[b])
            assert torch.equal(rows[b, :n], r2[b, :n]) and torch.equal(kidx[b, :n], kidx2[b, :n])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fused_input_normalisation_equals_divide_by_255(golden_dir, dtype):
    """N3 (yogo_dataset.py:280-283, image_path_dataset.py:71-73): uint8 images with the /255 folded into the first layer
    give the same train step as feeding `x.float() / 255` - outputs, loss, every gradient (incl. the clamped first-layer
    weight gradient) and the BatchNorm running statistics - and therefore match the reference golden as well."""
    z = _load(golden_dir, "model_base.npz")
    prefix = "base_train."
    keeps = {int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")}
    img = torch.from_numpy(z["img"])
    res = []
    for fused in (False, True):
        net, _ = _build_from_golden(z, "base_model", dtype=dtype)
        net.train()
        net._get_runner().drop_keep_override = keeps
        if fused:
            net.set_fused_input_scale(1.0 / 255.0)
            x = img.to(DEV)
            assert x.dtype == torch.uint8
        else:
            x = (img.float() / 255.0).to(DEV)
        out = net(x)
        loss, _ = yogo_b200.YOGOLoss().to(DEV)(out, torch.from_numpy(z["label"]).to(DEV))
        loss.backward()
        res.append((out.detach(), loss.detach(), {k: p.grad.clone() for k, p in net.named_parameters()},
                    {k: v.clone() for k, v in net.state_dict().items() if "running_" in k}))
    tol = 1e-4 if dtype == torch.float32 else 3e-2
    assert _rel(res[1][0].cpu().numpy(), res[0][0].cpu().numpy()) < tol
    assert abs(float(res[1][1]) - float(res[0][1])) < tol * abs(float(res[0][1]))
    for k in res[0][2]:
        a, b = res[1][2][k].cpu().numpy(), res[0][2][k].cpu().numpy()
        # (floor 1e-2: the conv bias in front of BatchNorm has a ~0 gradient that is pure rounding noise)
        assert np.linalg.norm(a - b) <= (2e-3 if dtype == torch.float32 else 0.35) * max(np.linalg.norm(b), 1e-2), k
        assert np.abs(a).max() <= 1.0 + 1e-6   # clamp(+-clip_value) still holds after the rescaling
    for k in res[0][3]:
        # (a running mean of ~1e-4 is a cancelling sum of bf16-rounded activations: absolute floor 1e-4 in bf16)
        torch.testing.assert_close(res[1][3][k], res[0][3][k], rtol=1e-3 if dtype == torch.float32 else 2e-2,
                                   atol=1e-5 if dtype == torch.float32 else 1e-4)
    if dtype == torch.float32:
        assert _rel(res[1][0].cpu().numpy(), z[prefix + "out"]) < 1e-3


def test_nan_gradient_propagates_like_torch_clamp():
    """The reference's gradient hook is torch.clamp (model.py:76-77), which keeps NaN; the fused reduce kernels must not turn
    a NaN gradient into a finite -clip."""
    net = yogo_b200.YOGO((64, 96), O.ANCHOR_W, O.ANCHOR_H, 7).to(DEV)
    net.train()
    x = torch.rand(2, 1, 64, 96, device=DEV)
    out = net(x)
    g = torch.zeros_like(out)
    g[0, 5, 3, 3] = float("nan")
    out.backward(g)
    assert torch.isnan(net.model[-1].weight.grad).any() and torch.isnan(net.model[-1].bias.grad).any()
    assert torch.isnan(net.model[3][0].weight.grad).any()


def test_collate_batch_robust_on_device():
    """yogo/data/utils.py:49-63: None items are dropped, the rest stacked, batch transforms applied (here on the GPU)."""
    from yogo_b200.data import MultiArgSequential, RandomHorizontalFlipWithBBs, collate_batch_robust
    imgs = O.synth_images(3, 32, 48)
    labs = O.synth_labels(3, 4, 6, 7, 5)
    batch = [(imgs[0], labs[0]), None, (imgs[1], labs[1]), (imgs[2], labs[2]), None]
    a, b = collate_batch_robust(batch, MultiArgSequential(RandomHorizontalFlipWithBBs(1.0)), device=DEV)
    ea, eb = O.flip_batch_np(imgs.numpy(), labs.numpy(), True, False)
    assert a.is_cuda and np.array_equal(a.cpu().numpy(), ea) and np.array_equal(b.cpu().numpy().view(np.uint32), eb.view(np.uint32))
    with pytest.raises(ValueError):
        collate_batch_robust([None, None])


def test_model_on_second_gpu_while_first_is_current():
    """Every entry point switches to the device of its tensors (ATen does this for every op of the reference): a model, loss
    and post-processing on cuda:1 while cuda:0 is current give the same results as on cuda:0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    torch.manual_seed(0)
    net0 = yogo_b200.YOGO((96, 128), O.ANCHOR_W, O.ANCHOR_H, 7)
    sd = {k: v.clone() for k, v in net0.state_dict().items()}
    img, lab = O.synth_images(2, 96, 128), O.synth_labels(2, 12, 16, 7, 10)
    res = []
    for dev in ("cuda:0", "cuda:1"):
        assert torch.cuda.current_device() == 0
        net = yogo_b200.YOGO((96, 128), O.ANCHOR_W, O.ANCHOR_H, 7)
        net.load_state_dict(sd)
        net = net.to(dev)
        net.train()
        for m in net.model.modules():
            if isinstance(m, torch.nn.Dropout2d):
                m.p = 0.0
        out = net(img.to(dev))
        loss, _ = yogo_b200.YOGOLoss().to(dev)(out, lab.to(dev))
        loss.backward()
        rows, kc, _, counts = yogo_b200.format_preds_batch(out.detach())
        torch.cuda.synchronize(dev)
        res.append((out.detach().cpu(), float(loss), net.model[-1].weight.grad.cpu(), kc.cpu(), counts.cpu()))
    assert torch.cuda.current_device() == 0
    torch.testing.assert_close(res[1][0], res[0][0], rtol=1e-3, atol=1e-4)
    assert abs(res[1][1] - res[0][1]) < 1e-3 * abs(res[0][1])
    torch.testing.assert_close(res[1][2], res[0][2], rtol=2e-2, atol=1e-3)


def test_outputs_of_the_other_kernels_stay_inside_their_buffers():
    """Guard regions around the outputs of the first-layer, BatchNorm, head, loss and NMS kernels (the convolution engine has
    its own test): nothing outside the tensors may be written, at sizes with ragged tails."""
    import ctypes as C
    lib = L.lib()
    GUARD = 4096

    def guarded(shape, dtype, fill):
        numel = int(np.prod(shape))
        buf = torch.full((numel + 2 * GUARD,), fill, dtype=dtype, device=DEV)
        return buf, buf[GUARD:GUARD + numel].view(*shape)

    def intact(buf, view, fill):
        n = view.numel()
        return bool((buf[:GUARD] == fill).all()) and bool((buf[GUARD + n:] == fill).all())

    g = torch.Generator().manual_seed(4)
    N, H, W, C1 = 3, 70, 90, 16
    Ho, Wo = 35, 45
    img = torch.randint(0, 256, (N, 1, H, W), dtype=torch.uint8, generator=g).to(DEV)
    w1 = (torch.randn(C1, 1, 3, 3, generator=g) / 300).to(DEV)
    sc, sh = (torch.rand(C1, generator=g) + 0.5).to(DEV), (torch.randn(C1, generator=g) * 0.1).to(DEV)
    # first layer forward (tensor-core and generic kernels)
    for impl in ("auto", "simt"):
        L.set_conv_impl(impl)
        try:
            ybuf, y = guarded((N, Ho, Wo, C1), torch.bfloat16, 7.0)
            ep = L.FwdEpilogue(sc.data_ptr(), sh.data_ptr(), L.ACT_LRELU, None, None, None, None)
            L.check(lib.yg_conv_first_fwd(img.data_ptr(), L.YG_U8, w1.data_ptr(), y.data_ptr(), 1, N, H, W, 1, C1, 2, C.byref(ep), L.stream()))
            torch.cuda.synchronize()
            assert intact(ybuf, y, 7.0) and bool(torch.isfinite(y.float()).all()) and float(y.float().abs().sum()) > 0
        finally:
            L.set_conv_impl("auto")
    # BatchNorm apply (+ sign mask) and backward apply, ragged pixel count
    Cb, HW = 128, 97 * 13 + 5
    yraw = torch.randn(N, HW, Cb, generator=g).to(DEV).bfloat16()
    bsc, bsh = (torch.rand(Cb, generator=g) + 0.5).to(DEV), torch.randn(Cb, generator=g).to(DEV)
    abuf, a = guarded((N, HW, Cb), torch.bfloat16, 7.0)
    mbuf, m = guarded((N * HW * Cb // 8,), torch.uint8, 0xA5)
    L.check(lib.yg_bn_act_apply(yraw.data_ptr(), a.data_ptr(), 1, N, HW, Cb, bsc.data_ptr(), bsh.data_ptr(), L.ACT_LRELU, None,
                                m.data_ptr(), L.stream()))
    gbuf, gg = guarded((N, HW, Cb), torch.bfloat16, 7.0)
    gg.copy_(torch.randn(N, HW, Cb, generator=g).to(DEV).bfloat16())
    sums = torch.zeros(2 * Cb, dtype=torch.float64, device=DEV)
    mean, istd = torch.zeros(Cb, device=DEV), torch.ones(Cb, device=DEV)
    L.check(lib.yg_bn_bwd_sums(gg.data_ptr(), yraw.data_ptr(), 1, N, HW, Cb, mean.data_ptr(), istd.data_ptr(), sums.data_ptr(), L.stream()))
    dgb, dg = guarded((Cb,), torch.float32, 7.0)
    dbb, db = guarded((Cb,), torch.float32, 7.0)
    L.check(lib.yg_bn_bwd_apply(gg.data_ptr(), yraw.data_ptr(), 1, N, HW, Cb, sums.data_ptr(), bsc.data_ptr(), mean.data_ptr(),
                                istd.data_ptr(), dg.data_ptr(), db.data_ptr(), 1.0, 1, L.stream()))
    torch.cuda.synchronize()
    assert intact(abuf, a, 7.0) and intact(mbuf, m, 0xA5) and intact(gbuf, gg, 7.0) and intact(dgb, dg, 7.0) and intact(dbb, db, 7.0)
    # head forward + backward on an odd grid
    Sy, Sx, Cl, nc = 13, 17, 128, 7
    D = 5 + nc
    xh = torch.randn(N, Sy, Sx, Cl, generator=g).to(DEV).bfloat16()
    wh, bh = (torch.randn(D, Cl, 1, 1, generator=g) * 0.05).to(DEV), torch.zeros(D, device=DEV)
    obuf, o = guarded((N, D, Sy, Sx), torch.float32, 7.0)
    tbuf, t = guarded((N, Sy, Sx, D), torch.float32, 7.0)
    L.check(lib.yg_head_fwd(xh.data_ptr(), 1, wh.data_ptr(), bh.data_ptr(), o.data_ptr(), t.data_ptr(), N, Sy, Sx, Cl, nc,
                            0.04, 0.05, 1.0, 1.0, 0, None, None, L.stream()))
    dpred = torch.randn(N, D, Sy, Sx, generator=g).to(DEV)
    dxbuf, dx = guarded((N, Sy, Sx, Cl), torch.bfloat16, 7.0)
    dwbuf, dw = guarded((D, Cl, 1, 1), torch.float32, 7.0)
    dbbuf, dbh = guarded((D,), torch.float32, 7.0)
    nb = lib.yg_head_bwd_workspace(N, Sy, Sx, Cl, nc)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_head_bwd(dpred.data_ptr(), t.data_ptr(), xh.data_ptr(), wh.data_ptr(), dx.data_ptr(), 1, dw.data_ptr(), dbh.data_ptr(),
                            N, Sy, Sx, Cl, nc, 0.04, 0.05, 1.0, 1.0, None, 1.0, ws.data_ptr(), nb, L.stream()))
    torch.cuda.synchronize()
    assert intact(obuf, o, 7.0) and intact(tbuf, t, 7.0) and intact(dxbuf, dx, 7.0) and intact(dwbuf, dw, 7.0) and intact(dbbuf, dbh, 7.0)
    # loss
    lab = O.synth_labels(N, Sy, Sx, nc, 20).to(DEV)
    pbuf, dp = guarded((N, D, Sy, Sx), torch.float32, 7.0)
    o4buf, o4 = guarded((4,), torch.float32, 7.0)
    nbl = lib.yg_yogo_loss_workspace(N, Sy, Sx)
    wsl = torch.empty(max(nbl, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_yogo_loss_fwd_bwd(o.data_ptr(), lab.data_ptr(), o4.data_ptr(), dp.data_ptr(), N, nc, Sy, Sx, 0.5, 5.0, 1.0, 0.01,
                                     wsl.data_ptr(), nbl, L.stream()))
    torch.cuda.synchronize()
    assert intact(pbuf, dp, 7.0) and intact(o4buf, o4, 7.0) and bool(torch.isfinite(o4).all())
    # threshold + NMS + counts
    p = O.synth_sparse_preds(N, Sy, Sx, nc, 30).to(DEV)
    cells = Sy * Sx
    rbuf, rows = guarded((N, cells, D), torch.float32, 7.0)
    kbuf, kc = guarded((N,), torch.int32, 77)
    ibuf, ki = guarded((N, cells), torch.int32, 77)
    cbuf, cnt = guarded((nc,), torch.int64, 77)
    nbn = lib.yg_format_preds_workspace(N, nc, Sy, Sx)
    wsn = torch.empty(max(nbn, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_format_preds_batch(p.data_ptr(), N, nc, Sy, Sx, 0.5, 0.5, 0, 0.0, kc.data_ptr(), rows.data_ptr(), ki.data_ptr(),
                                      cnt.data_ptr(), wsn.data_ptr(), nbn, L.stream()))
    torch.cuda.synchronize()
    assert intact(rbuf, rows, 7.0) and intact(kbuf, kc, 77) and intact(ibuf, ki, 77) and intact(cbuf, cnt, 77)
    assert int(cnt.sum()) == int(kc.sum()) > 0


def test_dropout_scales_kernel_statistics_and_counters():
    """yg_dropout_scales: Bernoulli(1 - p) keep decisions per (n, c) plane scaled by 1 / (1 - p) (nn.Dropout2d), fresh on every
    call (also when replayed from a CUDA graph), and `num_batches_tracked += 1` for every training-mode BatchNorm."""
    torch.manual_seed(0)
    net = yogo_b200.YOGO((96, 128), O.ANCHOR_W, O.ANCHOR_H, 7).to(DEV)
    net.train()
    r = net._get_runner()
    N = 512
    a = {i: t.clone() for i, t in r._step_randoms(N, torch.device(DEV), True).items()}
    b = {i: t.clone() for i, t in r._step_randoms(N, torch.device(DEV), True).items()}
    ps = {i: blk.p_drop for i, blk in enumerate(r.plan.blocks) if blk.p_drop > 0}
    assert set(a) == set(ps) == {1, 2, 3}
    for i, p in ps.items():
        assert tuple(a[i].shape) == (N, r.plan.blocks[i].cout)
        vals = torch.unique(a[i])
        assert len(vals) == 2 and float(vals[0]) == 0.0 and abs(float(vals[1]) - 1.0 / (1.0 - p)) < 1e-6
        frac = float((a[i] == 0).float().mean())
        assert abs(frac - p) < 4 * (p * (1 - p) / a[i].numel()) ** 0.5 + 1e-3, (i, frac, p)
        assert not torch.equal(a[i], b[i])                          # a new draw per call
    assert int(net.model[0][1].num_batches_tracked) == 2 and int(net.model[4][1].num_batches_tracked) == 2
    # graph replay: masks change between replays, counters advance
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        r._step_randoms(N, torch.device(DEV), True)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        out = r._step_randoms(N, torch.device(DEV), True)
    g.replay(); torch.cuda.synchronize(); m1 = out[2].clone()
    g.replay(); torch.cuda.synchronize(); m2 = out[2].clone()
    assert not torch.equal(m1, m2)
    assert int(net.model[0][1].num_batches_tracked) == 5
    # eval mode: nothing is drawn or counted
    net.eval()
    assert r._step_randoms(4, torch.device(DEV), False) == {}
    assert int(net.model[0][1].num_batches_tracked) == 5


def test_steps_from_host_equals_step_and_handles_a_ragged_last_batch():
    """DataParallelTrainer.steps_from_host: pinned host batches copied straight into the graph's two input slots give the same
    parameters as feeding device batches to `step`, including a last batch of another size (eager fallback)."""
    imgs = [O.synth_images(4, 96, 128, seed=s) for s in range(4)] + [O.synth_images(2, 96, 128, seed=9)]
    labs = [O.synth_labels(4, 12, 16, 7, 10, seed=s) for s in range(4)] + [O.synth_labels(2, 12, 16, 7, 10, seed=9)]
    net_a, tr_a = _make_trainer()
    net_b, tr_b = _make_trainer()
    tr_a.enable_cuda_graph(imgs[0].to(DEV), labs[0].to(DEV), slots=2)
    tr_b.enable_cuda_graph(imgs[0].to(DEV), labs[0].to(DEV))
    host = [(x.pin_memory(), y.pin_memory()) for x, y in zip(imgs, labs)]
    la = [float(l.detach()) for l in tr_a.steps_from_host(iter(host))]
    lb = [float(tr_b.step(x.to(DEV), y.to(DEV)).detach()) for x, y in zip(imgs, labs)]
    assert len(la) == len(lb) == 5 and tr_a.step_count == tr_b.step_count == 5
    for a, b in zip(la, lb):
        assert abs(a - b) <= 1e-2 * abs(b), (la, lb)
    assert abs(la[0] - lb[0]) <= 1e-5 * abs(lb[0])
    # (after five Adam steps sign flips of ~0 gradients have spread: compared by norm, as in the multi-rank check)
    drift = float((tr_a.flat_p - tr_b.flat_p).norm() / tr_b.flat_p.norm())
    assert drift < 2e-3, drift
