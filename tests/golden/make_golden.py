"""Generate tests/golden/*.npz by running the REAL reference (/root/reference) on seeded inputs.

Run in the build container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference is imported unmodified with the stubs of SURVEY.md 8c for modules that are
off the hot path and absent here (matplotlib, zarr, ruamel.yaml; np.unicode_).
Outputs are small .npz files committed next to this script; `shrink` keeps each under 1 MB.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def import_reference():
    for name in ("matplotlib", "matplotlib.pyplot", "zarr", "ruamel", "ruamel.yaml"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["ruamel.yaml"].YAML = object
    sys.modules["ruamel"].yaml = sys.modules["ruamel.yaml"]
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    if not hasattr(np, "unicode_"):
        np.unicode_ = np.str_
    sys.path.insert(0, "/root/reference")
    import yogo  # noqa: F401
    from yogo.model import YOGO
    from yogo.model_defns import get_model_func
    from yogo.yogo_loss import YOGOLoss
    from yogo.utils import format_preds
    from yogo.utils.prediction_formatting import format_preds_and_labels_v2, format_to_numpy, PredictionLabelMatch
    from yogo.infer import get_prediction_class_counts, count_cells_for_formatted_preds

    return dict(
        YOGO=YOGO,
        get_model_func=get_model_func,
        YOGOLoss=YOGOLoss,
        format_preds=format_preds,
        format_preds_and_labels_v2=format_preds_and_labels_v2,
        format_to_numpy=format_to_numpy,
        PredictionLabelMatch=PredictionLabelMatch,
        get_prediction_class_counts=get_prediction_class_counts,
        count_cells_for_formatted_preds=count_cells_for_formatted_preds,
    )


def golden_loss(ref, out):
    from oracle.yogo_oracle import synth_labels

    cases = {}
    for ci, (N, C, Sy, Sx, K, seed) in enumerate(
        [(2, 7, 10, 14, 30, 11), (3, 4, 13, 9, 40, 12), (1, 7, 97, 129, 300, 13), (2, 7, 6, 5, 0, 14)]
    ):
        g = torch.Generator().manual_seed(seed)
        lab = synth_labels(N, Sy, Sx, C, K, seed=seed)
        # predictions in head-output space: centres/sizes near the labels for some cells,
        # arbitrary elsewhere; logits random
        pred = torch.zeros(N, 5 + C, Sy, Sx)
        pred[:, 0] = torch.rand(N, Sy, Sx, generator=g)
        pred[:, 1] = torch.rand(N, Sy, Sx, generator=g)
        pred[:, 2] = 0.02 + 0.1 * torch.rand(N, Sy, Sx, generator=g)
        pred[:, 3] = 0.02 + 0.1 * torch.rand(N, Sy, Sx, generator=g)
        near = torch.rand(N, Sy, Sx, generator=g) < 0.6
        cxl = (lab[:, 1] + lab[:, 3]) / 2
        cyl = (lab[:, 2] + lab[:, 4]) / 2
        pred[:, 0] = torch.where(near, cxl + 0.01 * torch.randn(N, Sy, Sx, generator=g), pred[:, 0])
        pred[:, 1] = torch.where(near, cyl + 0.01 * torch.randn(N, Sy, Sx, generator=g), pred[:, 1])
        pred[:, 4] = torch.rand(N, Sy, Sx, generator=g)
        pred[:, 5:] = 2 * torch.randn(N, C, Sy, Sx, generator=g)
        if ci == 1:
            # edge cases: boxes leaving the image (clamp), a degenerate zero-width box
            pred[0, 0, 0, 0] = 0.001
            pred[0, 2, 0, 0] = 0.2
            lab[0, :, 0, 0] = torch.tensor([1.0, 0.0, 0.0, 0.05, 0.06, 1.0])
            pred[1, 2, 3, 3] = 0.0  # x1 == x2 -> dropped from the box term
            lab[1, :, 3, 3] = torch.tensor([1.0, 0.3, 0.3, 0.35, 0.36, 2.0])
            pred[2, 0, 5, 5] = 0.999
            pred[2, 1, 5, 5] = 0.999
            pred[2, 2, 5, 5] = 0.3
            pred[2, 3, 5, 5] = 0.3
            lab[2, :, 5, 5] = torch.tensor([1.0, 0.9, 0.9, 0.97, 0.99, 3.0])
        pred.requires_grad_(True)
        loss_fn = ref["YOGOLoss"]()
        loss, comps = loss_fn(pred, lab)
        loss.backward()
        cases[f"loss{ci}_pred"] = pred.detach().numpy()
        cases[f"loss{ci}_label"] = lab.numpy()
        cases[f"loss{ci}_loss"] = np.array(
            [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]],
            dtype=np.float64,
        )
        cases[f"loss{ci}_dpred"] = pred.grad.numpy()
    # non-default weights
    g = torch.Generator().manual_seed(99)
    lab = synth_labels(2, 8, 8, 5, 20, seed=99)
    pred = torch.rand(2, 10, 8, 8, generator=g)
    pred[:, 2:4] = 0.03 + 0.05 * pred[:, 2:4]
    pred.requires_grad_(True)
    loss_fn = ref["YOGOLoss"](no_obj_weight=0.3, iou_weight=2.5, classify_weight=0.7, label_smoothing=0.1)
    loss, comps = loss_fn(pred, lab)
    loss.backward()
    cases["lossw_pred"] = pred.detach().numpy()
    cases["lossw_label"] = lab.numpy()
    cases["lossw_loss"] = np.array(
        [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]], dtype=np.float64
    )
    cases["lossw_dpred"] = pred.grad.numpy()
    np.savez_compressed(os.path.join(out, "loss.npz"), **cases)


def golden_nms(ref, out):
    from oracle.yogo_oracle import synth_sparse_preds

    cases = {}
    configs = [
        # (B, Sy, Sx, C, K, seed, obj, iou, fmt, mincls)
        (3, 20, 28, 7, 40, 21, 0.5, 0.5, "cxcywh", 0.0),
        (2, 20, 28, 7, 60, 22, 0.5, 0.3, "xyxy", 0.0),
        (2, 97, 129, 7, 300, 23, 0.5, 0.5, "cxcywh", 0.0),
        (2, 12, 12, 4, 30, 24, 0.6, 0.0, "cxcywh", 0.0),  # iou_thresh 0 = NMS disabled
        (2, 16, 16, 7, 50, 25, 0.5, 0.5, "xyxy", 0.6),  # class-confidence filter
        (1, 8, 8, 7, 0, 26, 0.5, 0.5, "cxcywh", 0.0),  # nothing above threshold
    ]
    for ci, (B, Sy, Sx, C, K, seed, obj, iou, fmt, mincls) in enumerate(configs):
        p = synth_sparse_preds(B, Sy, Sx, C, K, seed=seed)
        if ci == 0:
            # tie-heavy + degenerate: duplicate boxes with equal scores, zero-area boxes
            p[0, :, 3, 3] = p[0, :, 3, 4]
            p[0, :, 3, 5] = p[0, :, 3, 4]
            p[0, 4, 7, 7] = 0.9
            p[0, 2:4, 7, 7] = 0.0
            p[0, :, 7, 8] = p[0, :, 7, 7]
        cases[f"nms{ci}_pred"] = p.numpy()
        cases[f"nms{ci}_cfg"] = np.array([obj, iou, 1.0 if fmt == "xyxy" else 0.0, mincls], dtype=np.float64)
        offs = [0]
        rows = []
        for b in range(B):
            r = ref["format_preds"](
                p[b].clone(), obj_thresh=obj, iou_thresh=iou, box_format=fmt, min_class_confidence_threshold=mincls
            )
            rows.append(r.numpy())
            offs.append(offs[-1] + r.shape[0])
        cases[f"nms{ci}_rows"] = np.concatenate(rows, axis=0)
        cases[f"nms{ci}_offsets"] = np.array(offs, dtype=np.int64)
        cases[f"nms{ci}_counts"] = (
            ref["get_prediction_class_counts"](p.clone(), obj_thresh=obj, iou_thresh=iou, min_class_confidence_threshold=mincls)
            .numpy()
            .astype(np.int64)
        )
    # dense-adversarial: many overlapping boxes on a small grid
    g = torch.Generator().manual_seed(31)
    B, C, Sy, Sx = 2, 7, 24, 32
    p = torch.rand(B, 5 + C, Sy, Sx, generator=g)
    p[:, 2:4] = 0.05 + 0.2 * p[:, 2:4]
    p[:, 5:] = torch.softmax(4 * p[:, 5:], dim=1)
    cases["nmsD_pred"] = p.numpy()
    cases["nmsD_cfg"] = np.array([0.5, 0.5, 0.0, 0.0])
    offs, rows = [0], []
    for b in range(B):
        r = ref["format_preds"](p[b].clone())
        rows.append(r.numpy())
        offs.append(offs[-1] + r.shape[0])
    cases["nmsD_rows"] = np.concatenate(rows, axis=0)
    cases["nmsD_offsets"] = np.array(offs, dtype=np.int64)
    cases["nmsD_counts"] = ref["get_prediction_class_counts"](p.clone()).numpy().astype(np.int64)
    np.savez_compressed(os.path.join(out, "nms.npz"), **cases)


def golden_match(ref, out):
    """format_preds_and_labels_v2 / convert_background_errors / format_to_numpy of the real reference."""
    from oracle.yogo_oracle import synth_sparse_preds, synth_labels_for_preds

    cases = {}
    configs = [
        # (Sy, Sx, C, K, seed, obj, mincls, drop, extra)
        (20, 28, 7, 40, 41, 0.5, 0.0, 0.2, 5),
        (97, 129, 7, 300, 42, 0.5, 0.0, 0.1, 12),
        (16, 16, 4, 30, 43, 0.6, 0.5, 0.3, 3),
        (12, 12, 7, 20, 44, 0.5, 0.0, 1.0, 4),   # labels only at empty cells: every match has cost 1 (ties)
        (12, 12, 7, 6, 45, 0.5, 0.0, 0.0, 40),   # more labels than predictions: missed labels
    ]
    for ci, (Sy, Sx, C, K, seed, obj, mincls, drop, extra) in enumerate(configs):
        p = synth_sparse_preds(1, Sy, Sx, C, K, seed=seed)[0]
        lab = synth_labels_for_preds(p, drop=drop, extra=extra, seed=seed)
        m = ref["format_preds_and_labels_v2"](p.clone(), lab.clone(), objectness_thresh=obj,
                                              min_class_confidence_threshold=mincls)
        cases[f"m{ci}_pred"] = p.numpy()
        cases[f"m{ci}_label"] = lab.numpy()
        cases[f"m{ci}_cfg"] = np.array([obj, mincls], dtype=np.float64)
        cases[f"m{ci}_preds"] = m.preds.numpy()
        cases[f"m{ci}_labels"] = m.labels.numpy()
        cases[f"m{ci}_missed"] = m.missed_labels.numpy()
        cases[f"m{ci}_extra"] = m.extra_predictions.numpy()
        cb = m.convert_background_errors(C + 1)
        cases[f"m{ci}_bg_preds"] = cb.preds.numpy()
        cases[f"m{ci}_bg_labels"] = cb.labels.numpy()
        cases[f"m{ci}_npy"] = ref["format_to_numpy"](7, p.numpy().copy(), 772, 1032)
    np.savez_compressed(os.path.join(out, "match.npz"), **cases)


def synth_label_lists(B, Sx, Sy, C, K, seed):
    """ragged [class, x1, y1, x2, y2] lists; image 0 repeats a cell (last label wins) and has a box touching the border."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for b in range(B):
        n = int(torch.randint(K // 2, K + 1, (), generator=g)) if K else 0
        cx, cy = torch.rand(n, generator=g), torch.rand(n, generator=g)
        w, h = 0.04 * (0.75 + 0.5 * torch.rand(n, generator=g)), 0.05 * (0.75 + 0.5 * torch.rand(n, generator=g))
        cls = torch.randint(0, C, (n,), generator=g).float()
        t = torch.stack([cls, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1)
        if b == 0 and n >= 4:
            t[3, 1:] = t[1, 1:] + 1e-4
            t[2, 1:] = torch.tensor([0.0, 0.0, 0.03, 0.04])
        out.append(t)
    return out


def golden_input(ref, out):
    """RandomHorizontal/VerticalFlipWithBBs (p = 1) and format_labels_tensor of the real reference."""
    from yogo.data.data_transforms import RandomHorizontalFlipWithBBs, RandomVerticalFlipWithBBs
    from yogo.data.yogo_dataset import format_labels_tensor
    from tools.synth import synth_images, synth_labels

    cases = {}
    hf, vf = RandomHorizontalFlipWithBBs(1.0), RandomVerticalFlipWithBBs(1.0)
    for ci, (N, H, W, Sy, Sx, K, seed, as_float) in enumerate(
        [(2, 16, 24, 6, 8, 10, 51, False), (3, 772 // 8, 1032 // 8, 13, 17, 40, 52, False), (2, 15, 21, 5, 7, 8, 53, True)]
    ):
        img = synth_images(N, H, W, seed=seed)
        if as_float:
            img = img.float() / 255.0
        lab = synth_labels(N, Sy, Sx, 7, K, seed=seed)
        cases[f"f{ci}_img"], cases[f"f{ci}_lab"] = img.numpy(), lab.numpy()
        a, b = hf(img.clone(), lab.clone())
        cases[f"f{ci}_h_img"], cases[f"f{ci}_h_lab"] = a.numpy(), b.numpy()
        a, b = vf(img.clone(), lab.clone())
        cases[f"f{ci}_v_img"], cases[f"f{ci}_v_lab"] = a.numpy(), b.numpy()
        a, b = vf(*hf(img.clone(), lab.clone()))
        cases[f"f{ci}_hv_img"], cases[f"f{ci}_hv_lab"] = a.numpy(), b.numpy()
    for ci, (B, Sx, Sy, C, K, seed) in enumerate([(3, 8, 6, 7, 10, 61), (2, 129, 97, 7, 300, 62), (2, 5, 4, 3, 0, 63)]):
        lists = synth_label_lists(B, Sx, Sy, C, K, seed)
        cases[f"l{ci}_cfg"] = np.array([B, Sx, Sy], dtype=np.int64)
        cases[f"l{ci}_counts"] = np.array([t.shape[0] for t in lists], dtype=np.int64)
        cases[f"l{ci}_labels"] = torch.cat(lists).numpy() if sum(t.shape[0] for t in lists) else np.zeros((0, 5), np.float32)
        cases[f"l{ci}_out"] = torch.stack([format_labels_tensor(t, Sx, Sy) for t in lists]).numpy()
    np.savez_compressed(os.path.join(out, "input.npz"), **cases)


GRAD_STRIDE = 5


def grad_sample_stride(size, cap):
    """fixtures keep at most ~cap samples of a gradient tensor (plus its norm)"""
    return max(1, -(-size // cap))


def _run_model(ref, name, sd_from, img, lab, train, inference=False, normalize=True, autocast=False, fill_seed=None,
               grad_cap=None, double=False, margins=None):
    torch.manual_seed(0)
    H, W = img.shape[-2:]
    net = ref["YOGO"](
        img_size=(H, W),
        anchor_w=0.0425,
        anchor_h=0.0555,
        num_classes=7,
        is_rgb=img.shape[1] == 3,
        model_func=ref["get_model_func"](name),
        inference=inference,
        clip_value=1.0,
    )
    if sd_from is not None:
        net.load_state_dict(sd_from)
    elif fill_seed is not None:
        from tools.synth import synth_fill_model

        synth_fill_model(net, fill_seed)
    else:
        # tame the head so w/h stay O(anchor) (SURVEY.md 8d) and give BN non-trivial affine
        with torch.no_grad():
            head = list(net.model.children())[-1]
            head.weight.mul_(0.05)
            for m in net.model.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.weight.uniform_(0.5, 1.5)
                    m.bias.uniform_(-0.2, 0.2)
                if isinstance(m, torch.nn.Conv2d) and m.bias is not None:
                    m.bias.uniform_(-0.1, 0.1)
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    keeps = {}

    def mk_hook(idx):
        def hook(mod, inp, outp):
            x = inp[0]
            keeps[idx] = ((outp.abs().sum(dim=(2, 3)) > 0) | (x.abs().sum(dim=(2, 3)) == 0)).float()

        return hook

    for i, blk in enumerate(net.model.children()):
        for m in blk.modules():
            if isinstance(m, torch.nn.Dropout2d):
                m.register_forward_hook(mk_hook(i))
    net.train(train)
    x = img.float() / 255.0 if normalize else img.float()
    if double:
        # the reference in float64 = "truth" for calibrating what fp32 rounding alone does to the gradients (LeakyReLU kinks)
        net = net.double()
        x = x.double()
        net.forward = lambda xx, _f=net.forward.__func__, _n=net: _f(_n, xx)  # unchanged forward; input stays float64
    if margins is not None:
        # distance of every LeakyReLU input from the kink, relative to the tensor's rms
        def kink_hook(mod, inp):
            v = inp[0].detach()
            margins.append(float(v.abs().min() / v.pow(2).mean().sqrt()))

        for m in net.model.modules():
            if isinstance(m, torch.nn.LeakyReLU):
                m.register_forward_pre_hook(kink_hook)
    res = {}
    if train:
        if autocast:
            # Dropout2d must draw the same masks as the fp32 run: same seed, same call order
            torch.manual_seed(1234)
            with torch.autocast("cpu", dtype=torch.bfloat16):
                out = net(x)
            out = out.float()
        else:
            torch.manual_seed(1234)
            out = net(x)
        if double:
            out = out.float()
        loss, comps = ref["YOGOLoss"]()(out, lab)
        loss.backward()
        res["loss"] = np.array(
            [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]], dtype=np.float64
        )
        for k, p in net.named_parameters():
            gflat = p.grad.float().numpy().reshape(-1)
            res["gradnorm." + k] = np.array([np.linalg.norm(gflat.astype(np.float64))])
            # big tensors: keep every GRAD_STRIDE-th element (plus the norm) to keep fixtures small
            if grad_cap is not None:
                res["grad." + k] = gflat[:: grad_sample_stride(gflat.size, grad_cap)].copy()
            else:
                res["grad." + k] = gflat[::GRAD_STRIDE].copy() if gflat.size > 16384 else gflat.copy()
        for k, v in net.state_dict().items():
            if "running_" in k:
                res["after." + k] = v.float().numpy().copy()
    else:
        with torch.no_grad():
            out = net(x)
    res["out"] = out.detach().float().numpy().copy()
    for i, kk in keeps.items():
        res[f"keep.{i}"] = kk.numpy()
    return sd0, res


def golden_model(ref, out):
    from oracle.yogo_oracle import synth_images, synth_labels

    img = synth_images(2, 80, 112, seed=5)
    lab = synth_labels(2, 10, 14, 7, 25, seed=6)
    cases = {"img": img.numpy(), "label": lab.numpy()}
    sd_base, res = _run_model(ref, "base_model", None, img, lab, train=True)
    for k, v in sd_base.items():
        cases["sd." + k] = v.numpy()
    for k, v in res.items():
        cases["base_train." + k] = v
    # calibration of the bf16 tolerance: the reference's OWN bf16-autocast error against its fp32
    # run on the same inputs, weights and dropout masks (SURVEY.md Appendix E)
    for nm, pre in (("base_model", "base_train."), ("silu_model", "silu_train.")):
        _, r32 = _run_model(ref, nm, sd_base, img, lab, train=True)
        _, r16 = _run_model(ref, nm, sd_base, img, lab, train=True, autocast=True)
        same_masks = all(np.array_equal(r32[k], r16[k]) for k in r32 if k.startswith("keep."))
        assert same_masks, "dropout masks differ between fp32 and autocast runs"
        def rel(a, b):
            return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-3))
        cases[pre + "bf16err.out"] = np.array([rel(r16["out"], r32["out"])])
        cases[pre + "bf16err.loss"] = np.array([abs(r16["loss"][0] - r32["loss"][0]) / abs(r32["loss"][0])])
        for k in r32:
            if k.startswith("grad."):
                cases[pre + "bf16err." + k] = np.array([rel(r16[k], r32[k])])
    _, res = _run_model(ref, "base_model", sd_base, img, lab, train=False)
    cases["base_eval.out"] = res["out"]
    _, res = _run_model(ref, "base_model", sd_base, img, lab, train=False, inference=True)
    cases["base_infer.out"] = res["out"]
    _, res = _run_model(ref, "silu_model", sd_base, img, lab, train=True)
    for k, v in res.items():
        cases["silu_train." + k] = v
    _, res = _run_model(ref, "silu_model", sd_base, img, lab, train=False)
    cases["silu_eval.out"] = res["out"]
    np.savez_compressed(os.path.join(out, "model_base.npz"), **cases)

    # small-width and odd-topology definitions: weights are small enough to commit
    for name in ("quarter_filters", "depth_ver_0"):
        img = synth_images(3, 52, 68, seed=7)  # odd intermediate sizes: 26x34 -> 13x17 -> 7x9
        sd, res = _run_model(ref, name, None, img, None, train=False)
        Sy, Sx = res["out"].shape[-2:]
        lab = synth_labels(3, Sy, Sx, 7, 12, seed=8)
        sd, res = _run_model(ref, name, sd, img, lab, train=True)
        cases = {"img": img.numpy(), "label": lab.numpy()}
        for k, v in sd.items():
            cases["sd." + k] = v.numpy()
        for k, v in res.items():
            cases["train." + k] = v
        _, res = _run_model(ref, name, sd, img, lab, train=False)
        cases["eval.out"] = res["out"]
        np.savez_compressed(os.path.join(out, f"model_{name}.npz"), **cases)


# every registered definition that the round-1 fixtures do not cover, RGB input, and the BASELINE geometry.
# Weights are NOT stored: tools/synth.py::synth_fill_model regenerates them bit for bit from the seed.
ZOO = [
    # (case, model name, channels, N, H, W, labels per image, seed)
    ("double_filters", "double_filters", 1, 2, 80, 112, 25, 71),
    ("triple_filters", "triple_filters", 1, 2, 52, 68, 12, 72),
    ("half_filters", "half_filters", 1, 3, 52, 68, 12, 73),
    ("depth_ver_1", "depth_ver_1", 1, 2, 52, 68, 12, 74),
    ("depth_ver_2", "depth_ver_2", 1, 2, 52, 68, 12, 75),
    ("depth_ver_3", "depth_ver_3", 1, 2, 52, 68, 12, 76),
    ("depth_ver_4", "depth_ver_4", 1, 2, 52, 68, 12, 77),
    ("rgb_base_model", "base_model", 3, 2, 52, 68, 12, 78),
    ("rgb_silu_model", "silu_model", 3, 2, 48, 64, 12, 79),
]
FULL = [
    # BASELINE geometry 772x1032 -> 97x129 (configs[1] and configs[3]), 300 labels per image
    ("full_base_model", "base_model", 1, 4, 772, 1032, 300, 81),
    ("full_silu_model", "silu_model", 1, 2, 772, 1032, 300, 82),
    ("full_double_filters", "double_filters", 1, 2, 772, 1032, 300, 83),
]
ZOO_GRAD_CAP = 4096


def _rel64(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / max(np.linalg.norm(b.astype(np.float64)), 1e-3))


KINK_MARGIN = 3e-6   # ~10x the fp32 rounding noise of a pre-activation relative to its rms


def golden_zoo(ref, out, table, fname, out_stride=1, pick_seed=False):
    """pick_seed: small fixtures have ~2e5 LeakyReLU inputs, so about every second seed puts one of them within fp32
    rounding noise of the kink; an implementation that rounds differently then legitimately takes the other slope for
    that element, which alone is a 0.5 % gradient error at this size (observed on the GPU).  Such seeds are skipped: the
    first seed (seed, seed + 1000, ...) whose closest pre-activation is > KINK_MARGIN x rms away from zero is used and
    recorded in the cfg row.  At the BASELINE geometry (1e8 activations) kinks cannot be avoided; there the fixtures
    record the reference's OWN fp32 error against its float64 run per tensor (fp32err.*) as the yardstick."""
    from tools.synth import synth_images, synth_labels

    cases = {}
    for case, name, ch, N, H, W, K, seed0 in table:
        seed = seed0
        while True:
            img = synth_images(N, H, W, seed=seed, channels=ch)
            sd, res = _run_model(ref, name, None, img, None, train=False, fill_seed=seed)
            Sy, Sx = res["out"].shape[-2:]
            lab = synth_labels(N, Sy, Sx, 7, K, seed=seed + 100)
            margins = []
            _, r32 = _run_model(ref, name, sd, img, lab, train=True, grad_cap=ZOO_GRAD_CAP, margins=margins)
            if not pick_seed or not margins or min(margins) > KINK_MARGIN:
                break
            print(case, "seed", seed, "skipped: kink margin", min(margins), flush=True)
            seed += 1000
        _, r16 = _run_model(ref, name, sd, img, lab, train=True, grad_cap=ZOO_GRAD_CAP, autocast=True)
        _, r64 = _run_model(ref, name, sd, img, lab, train=True, grad_cap=ZOO_GRAD_CAP, double=True)
        assert all(np.array_equal(r32[k], r16[k]) for k in r32 if k.startswith("keep."))
        assert all(np.array_equal(r32[k], r64[k]) for k in r32 if k.startswith("keep."))
        pre = case + "."
        cases[pre + "cfg"] = np.array([ch, N, H, W, K, seed, out_stride], dtype=np.int64)
        for k, v in r32.items():
            cases[pre + "train." + k] = v[:, :, ::out_stride, ::out_stride].copy() if k == "out" else v
        cases[pre + "bf16err.out"] = np.array([_rel64(r16["out"], r32["out"])])
        cases[pre + "bf16err.loss"] = np.array([abs(r16["loss"][0] - r32["loss"][0]) / abs(r32["loss"][0])])
        cases[pre + "fp32err.out"] = np.array([_rel64(r32["out"], r64["out"])])
        for k in r32:
            if k.startswith("grad."):
                cases[pre + "bf16err." + k] = np.array([_rel64(r16[k], r32[k])])
                cases[pre + "fp32err." + k] = np.array([_rel64(r32[k], r64[k])])
        _, res = _run_model(ref, name, sd, img, lab, train=False)
        cases[pre + "eval.out"] = res["out"][:, :, ::out_stride, ::out_stride].copy()
        worst32 = max(float(cases[pre + "fp32err." + k][0]) for k in r32 if k.startswith("grad.") and r32["gradnorm." + k[5:]][0] > 1e-2)
        print(case, "seed", seed, "loss", r32["loss"][0], "bf16 out err", cases[pre + "bf16err.out"][0],
              "worst fp32-vs-fp64 grad err", worst32, "kink margin", min(margins) if margins else None, flush=True)
    np.savez_compressed(os.path.join(out, fname), **cases)


FULL_OUT_STRIDE = 4
ZOO_GRAD_KEEP = 2048


def shrink(out):
    """Keeps every fixture under 1 MB without changing a result of the reference.  Applying it again changes nothing.
      - model_base.npz: the weights are replaced by their SHA-256 digest; tests/_golden.py regenerates them from the
        seed of `_run_model` and checks the digest.
      - nms.npz, nms2: the class probabilities of the cells at or below the objectness threshold are zeroed.  format_preds
        drops those cells before it reads anything else, so no row or count can change; the oracle re-checks it here.
      - model_full.npz: outputs on every FULL_OUT_STRIDE-th grid row and column (recorded in the cfg row).
      - model_zoo.npz: gradient samples of more than ZOO_GRAD_KEEP elements keep every second one
        (tests/_zoo_cases.py::grad_sample)."""
    sys.path.insert(0, os.path.dirname(HERE))
    from _golden import digest
    from oracle.yogo_oracle import format_preds_np, prediction_class_counts_np

    def rewrite(fname, edit):
        path = os.path.join(out, fname)
        with np.load(path) as npz:
            z = dict(npz.items())
        if edit(z):
            np.savez_compressed(path, **z)

    def base(z):
        sd = {k: z.pop(k) for k in list(z) if k.startswith("sd.")}
        if sd:
            z["digest.sd"] = np.array(digest(sd))
        return bool(sd)

    def nms(z):
        p = z["nms2_pred"].copy()
        obj, iou, xyxy, mincls = z["nms2_cfg"]
        p[:, 5:] *= (p[:, 4:5] > np.float32(obj))
        for b in range(p.shape[0]):
            rows = format_preds_np(p[b], obj, iou, "xyxy" if xyxy else "cxcywh", mincls)
            exp = z["nms2_rows"][z["nms2_offsets"][b]:z["nms2_offsets"][b + 1]]
            assert rows.shape == exp.shape and np.array_equal(rows.view(np.uint32), exp.view(np.uint32))
        assert np.array_equal(prediction_class_counts_np(p, obj, iou, mincls), z["nms2_counts"])
        changed = not np.array_equal(p, z["nms2_pred"])
        z["nms2_pred"] = p
        return changed

    def full(z):
        changed = False
        for k in [k for k in z if k.endswith(".cfg")]:
            case, step = k[:-4], FULL_OUT_STRIDE // int(z[k][6])
            if step > 1:
                for o in (case + ".train.out", case + ".eval.out"):
                    z[o] = z[o][:, :, ::step, ::step].copy()
                z[k][6] = FULL_OUT_STRIDE
                changed = True
        return changed

    def zoo(z):
        big = [k for k in z if ".train.grad." in k and z[k].size > ZOO_GRAD_KEEP]
        for k in big:
            z[k] = z[k][::2].copy()
        return bool(big)

    rewrite("model_base.npz", base)
    rewrite("nms.npz", nms)
    rewrite("model_full.npz", full)
    rewrite("model_zoo.npz", zoo)


if __name__ == "__main__":
    torch.set_num_threads(1)
    torch.use_deterministic_algorithms(True)
    if "--only-shrink" in sys.argv:  # shrink the committed fixtures alone (no reference needed)
        shrink(HERE)
        sys.exit(0)
    ref = import_reference()
    if "--only-match" in sys.argv:   # regenerate match.npz alone
        golden_match(ref, HERE)
        sys.exit(0)
    if "--only-input" in sys.argv:   # regenerate input.npz alone
        golden_input(ref, HERE)
        sys.exit(0)
    if "--only-zoo" in sys.argv:     # regenerate model_zoo.npz / model_full.npz alone
        golden_zoo(ref, HERE, ZOO, "model_zoo.npz", pick_seed=True)
        torch.set_num_threads(16)
        golden_zoo(ref, HERE, FULL, "model_full.npz", out_stride=2)
        shrink(HERE)
        sys.exit(0)
    golden_loss(ref, HERE)
    golden_nms(ref, HERE)
    golden_match(ref, HERE)
    golden_input(ref, HERE)
    golden_model(ref, HERE)
    golden_zoo(ref, HERE, ZOO, "model_zoo.npz", pick_seed=True)
    torch.set_num_threads(16)
    golden_zoo(ref, HERE, FULL, "model_full.npz", out_stride=2)
    shrink(HERE)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
