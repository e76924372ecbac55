"""Pins the CPU oracle (oracle/yogo_oracle.py) against vectors produced by the real reference
(tests/golden/make_golden.py) and against the reference's own known-answer tests
(/root/reference/tests/test_utils_tensor_formatting.py, test_count_predictions.py)."""
import os

import numpy as np
import pytest
import torch

from _golden import load as _load
from oracle import yogo_oracle as O


@pytest.mark.parametrize("case", ["loss0", "loss1", "loss2", "loss3", "lossw"])
def test_loss_oracle_matches_reference(golden_dir, case):
    z = _load(golden_dir, "loss.npz")
    kw = {}
    if case == "lossw":
        kw = dict(no_obj_weight=0.3, iou_weight=2.5, classify_weight=0.7, label_smoothing=0.1)
    loss, comps, dpred = O.yogo_loss_np(z[f"{case}_pred"], z[f"{case}_label"], **kw)
    ref = z[f"{case}_loss"]
    got = np.array([loss, comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]])
    np.testing.assert_allclose(got, ref, rtol=2e-5, atol=1e-6)
    np.testing.assert_allclose(dpred, z[f"{case}_dpred"], rtol=2e-4, atol=2e-6)


@pytest.mark.parametrize("case", ["nms0", "nms1", "nms2", "nms3", "nms4", "nms5", "nmsD"])
def test_format_preds_oracle_bit_exact(golden_dir, case):
    z = _load(golden_dir, "nms.npz")
    obj, iou, xyxy, mincls = z[f"{case}_cfg"]
    pred = z[f"{case}_pred"]
    offs = z[f"{case}_offsets"]
    rows = z[f"{case}_rows"]
    for b in range(pred.shape[0]):
        got = O.format_preds_np(pred[b], obj, iou, "xyxy" if xyxy else "cxcywh", mincls)
        exp = rows[offs[b] : offs[b + 1]]
        assert got.shape == exp.shape
        assert np.array_equal(got.view(np.uint32), exp.view(np.uint32))  # bit-exact, same order
    counts = O.prediction_class_counts_np(pred, obj, iou, mincls)
    assert np.array_equal(counts, z[f"{case}_counts"])


@pytest.mark.parametrize("case", ["m0", "m1", "m2", "m3", "m4"])
def test_matching_oracle_bit_exact(golden_dir, case):
    """format_preds_and_labels_v2 of the real reference (prediction_formatting.py:254-330) vs the numpy restatement."""
    z = np.load(os.path.join(golden_dir, "match.npz"))
    obj, mincls = z[case + "_cfg"]
    mp, ml, missed, extra = O.match_preds_and_labels_np(z[case + "_pred"], z[case + "_label"], float(obj), float(mincls))
    for got, key in ((mp, "_preds"), (ml, "_labels"), (missed, "_missed"), (extra, "_extra")):
        exp = z[case + key]
        assert got.shape == exp.shape, key
        assert np.array_equal(got.view(np.uint32), exp.astype(np.float32).view(np.uint32)), key


def test_input_side_oracle_bit_exact(golden_dir):
    """data_transforms.py:51-98 and yogo_dataset.py:24-46 of the real reference vs the numpy restatement."""
    z = np.load(os.path.join(golden_dir, "input.npz"))
    for ci in range(3):
        img, lab = z[f"f{ci}_img"], z[f"f{ci}_lab"]
        for tag, h, v in (("h", True, False), ("v", False, True), ("hv", True, True)):
            a, b = O.flip_batch_np(img, lab, h, v)
            assert np.array_equal(a, z[f"f{ci}_{tag}_img"]), (ci, tag)
            assert np.array_equal(b.view(np.uint32), z[f"f{ci}_{tag}_lab"].view(np.uint32)), (ci, tag)
    for ci in range(3):
        B, Sx, Sy = (int(v) for v in z[f"l{ci}_cfg"])
        offs = np.concatenate([[0], np.cumsum(z[f"l{ci}_counts"])])
        for b in range(B):
            got = O.format_labels_tensor_np(z[f"l{ci}_labels"][offs[b]:offs[b + 1]], Sx, Sy)
            assert np.array_equal(got.view(np.uint32), z[f"l{ci}_out"][b].view(np.uint32)), (ci, b)
    with pytest.raises(IndexError):
        O.format_labels_tensor_np(np.array([[0, 0.9, 0.9, 1.2, 1.2]], np.float32), 8, 6)


def test_reference_known_answers_format_preds():
    # /root/reference/tests/test_utils_tensor_formatting.py:9-68
    none = np.zeros((12, 4, 4), np.float32)
    assert O.format_preds_np(none).shape == (0, 12)
    single = np.zeros((12, 4, 4), np.float32)
    single[4, 0, 0] = 1.0
    single[5] = 1.0
    np.testing.assert_array_equal(O.format_preds_np(single), single[:, 0, 0][None])
    box = np.zeros((12, 4, 4), np.float32)
    box[5] = 1.0
    box[4, 1, 1] = 1.0
    box[0:2, 1, 1] = 0.5
    box[2:4, 1, 1] = 0.1
    np.testing.assert_array_equal(O.format_preds_np(box), box[:, 1, 1][None])
    exp = box[:, 1, 1][None].copy()
    exp[:, 0] = exp[:, 0] - exp[:, 2] / 2
    exp[:, 1] = exp[:, 1] - exp[:, 3] / 2
    exp[:, 2] = exp[:, 0] + exp[:, 2]
    exp[:, 3] = exp[:, 1] + exp[:, 3]
    np.testing.assert_allclose(O.format_preds_np(box, box_format="xyxy"), exp, rtol=1.3e-6, atol=1e-5)
    with pytest.raises(ValueError):
        O.format_preds_np(np.zeros((1, 12, 4, 4), np.float32))
    with pytest.raises(ValueError):
        O.format_preds_np(none, box_format="bogus")


def test_reference_known_answers_counts():
    # /root/reference/tests/test_count_predictions.py:8-42
    inp = np.zeros((3, 5), np.float32)
    inp[:, 0] = 1
    assert O.count_cells_np(inp).tolist() == [3, 0, 0, 0, 0]
    row = np.array([0.1, 0.2, 0.3, 0.4], np.float32)
    assert O.count_cells_np(np.stack([row] * 3)).tolist() == [0, 0, 0, 3]
    inp = np.array([[0.2, 0.4, 0.2, 0.2]] * 3, np.float32)
    assert O.count_cells_np(inp, 0.6).tolist() == [0, 0, 0, 0]
    inp = np.array([[0.2, 0.7, 0.2, 0.2], [0.2, 0.4, 0.2, 0.2], [0.2, 0.4, 0.9, 0.2]], np.float32)
    assert O.count_cells_np(inp, 0.6).tolist() == [0, 1, 1, 0]


def _oracle_train(z, prefix, name, sdprefix="sd."):
    sd = {k[len(sdprefix) :]: torch.from_numpy(z[k]) for k in z.files if k.startswith(sdprefix)}
    blocks = O.blocks_from_state_dict(name, sd)
    for b in blocks:
        b.weight.requires_grad_(True)
        if b.bias is not None:
            b.bias.requires_grad_(True)
        if b.bn is not None:
            b.bn["weight"].requires_grad_(True)
            b.bn["bias"].requires_grad_(True)
    keeps = [
        torch.from_numpy(z[f"{prefix}keep.{i}"]) if f"{prefix}keep.{i}" in z.files else None
        for i in range(len(blocks))
    ]
    x = torch.from_numpy(z["img"]).float() / 255.0
    t = O.backbone_forward(x, blocks, train=True, drop_keep=keeps, update_running=True)
    out = O.head_transform(t, float(sd["anchor_w"]), float(sd["anchor_h"]))
    out.retain_grad()
    loss, comps, dpred = O.yogo_loss_np(out.detach().numpy(), z["label"])
    out.backward(torch.from_numpy(dpred))
    return sd, blocks, out, loss, comps


@pytest.mark.parametrize(
    "fname,prefix,name",
    [
        ("model_base.npz", "base_train.", "base_model"),
        ("model_base.npz", "silu_train.", "silu_model"),
        ("model_quarter_filters.npz", "train.", "quarter_filters"),
        ("model_depth_ver_0.npz", "train.", "depth_ver_0"),
    ],
)
def test_model_oracle_train_step_matches_reference(golden_dir, fname, prefix, name):
    z = _load(golden_dir, fname)
    sd, blocks, out, loss, comps = _oracle_train(z, prefix, name)
    np.testing.assert_allclose(out.detach().numpy(), z[prefix + "out"], rtol=2e-4, atol=2e-5)
    ref = z[prefix + "loss"]
    np.testing.assert_allclose(
        [loss, comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]], ref, rtol=2e-4
    )
    clip = 1.0  # YOGO registers clamp(grad, +-clip_value) on every parameter (model.py:76-77)
    for i, b in enumerate(blocks):
        last = i == len(blocks) - 1
        pre = f"model.{i}." if last else f"model.{i}.0."
        pairs = [(pre + "weight", b.weight)] + ([(pre + "bias", b.bias)] if b.bias is not None else [])
        if b.bn is not None:
            pairs += [(f"model.{i}.1.weight", b.bn["weight"]), (f"model.{i}.1.bias", b.bn["bias"])]
        for key, p in pairs:
            g = p.grad.clamp(-clip, clip).numpy().reshape(-1)
            exp = z[prefix + "grad." + key]
            if g.size > 16384:
                g = g[::5]
            scale = max(1e-6, float(np.abs(exp).max()))
            assert np.abs(g - exp).max() <= 5e-4 * scale + 2e-6, key
        if b.bn is not None:
            for kk in ("running_mean", "running_var"):
                np.testing.assert_allclose(
                    b.bn[kk].detach().numpy(), z[f"{prefix}after.model.{i}.1.{kk}"], rtol=1e-4, atol=1e-6
                )


def test_model_oracle_eval_and_inference(golden_dir):
    z = _load(golden_dir, "model_base.npz")
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    x = torch.from_numpy(z["img"]).float() / 255.0
    for name, key, inf in (("base_model", "base_eval.out", False), ("base_model", "base_infer.out", True),
                           ("silu_model", "silu_eval.out", False)):
        blocks = O.blocks_from_state_dict(name, sd)
        with torch.no_grad():
            t = O.backbone_forward(x, blocks, train=False)
            out = O.head_transform(t, float(sd["anchor_w"]), float(sd["anchor_h"]), inference=inf)
        np.testing.assert_allclose(out.numpy(), z[key], rtol=2e-4, atol=2e-5)


from _zoo_cases import ZOO_CASES, grad_sample, zoo_inputs  # noqa: E402


@pytest.mark.parametrize("case", ZOO_CASES)
def test_zoo_oracle_train_step_matches_reference(golden_dir, case):
    """Every registered definition (model_defns.py:130-529) and RGB input (:32) through the oracle vs the real reference."""
    z = _load(golden_dir, "model_zoo.npz")
    name, net, img, lab, _ = zoo_inputs(z, case)
    prefix = case + ".train."
    sd = net.state_dict()
    blocks = O.blocks_from_state_dict(name, sd)
    for b in blocks:
        b.weight.requires_grad_(True)
    keeps = [torch.from_numpy(z[f"{prefix}keep.{i}"]) if f"{prefix}keep.{i}" in z.files else None
             for i in range(len(blocks))]
    t = O.backbone_forward(img.float() / 255.0, blocks, train=True, drop_keep=keeps, update_running=True)
    out = O.head_transform(t, 0.0425, 0.0555)
    loss, comps, dpred = O.yogo_loss_np(out.detach().numpy(), lab.numpy())
    out.backward(torch.from_numpy(dpred))
    np.testing.assert_allclose(out.detach().numpy(), z[prefix + "out"], rtol=5e-4, atol=5e-5)
    np.testing.assert_allclose(loss, z[prefix + "loss"][0], rtol=2e-4)
    for i, b in enumerate(blocks):
        key = f"model.{i}.weight" if i == len(blocks) - 1 else f"model.{i}.0.weight"
        g = b.weight.grad.clamp(-1, 1).numpy().reshape(-1)
        exp = z[prefix + "grad." + key]
        g = grad_sample(g, exp.size)
        scale = max(1e-6, float(np.abs(exp).max()))
        assert np.abs(g - exp).max() <= 1e-3 * scale + 2e-6, key
