"""Gradients with respect to the input image (saliency maps, sensitivity checks) through yogo_b200.YOGO, against float64
autograd of the oracle on the same state_dict: the direct first-layer input gradient (yg_conv_first_dgrad), the softmax
backward of the inference head (yg_head_softmax_bwd), the backward of a frozen model, and the other first blocks."""
import os

import numpy as np
import pytest
import torch
from torch import nn

import yogo_b200
from _golden import load as _load
from _zoo_cases import ZOO_CASES, zoo_inputs
from oracle import yogo_oracle as O
from yogo_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def _oracle_blocks(net):
    """oracle Blocks (float64, CPU) of the net's backbone, any registered definition"""
    blocks = []
    for child in list(net.model.children())[:-1]:
        mods = list(child.children()) if isinstance(child, nn.Sequential) else [child]
        conv, bn, act, p = mods[0], None, None, 0.0
        for m in mods[1:]:
            if isinstance(m, nn.BatchNorm2d):
                bn = {k: getattr(m, k).detach().cpu().double().clone() for k in ("weight", "bias", "running_mean", "running_var")}
            elif isinstance(m, nn.LeakyReLU):
                act = "lrelu"
            elif isinstance(m, nn.SiLU):
                act = "silu"
            elif isinstance(m, nn.Dropout2d):
                p = float(m.p)
        bias = conv.bias.detach().cpu().double().clone() if conv.bias is not None else None
        blocks.append(O.Block(conv.weight.detach().cpu().double().clone(), bias, conv.stride[0], conv.padding[0], bn, act, p))
    head = net.model[-1]
    blocks.append(O.Block(head.weight.detach().cpu().double().clone(), head.bias.detach().cpu().double().clone(), 1, 0,
                          None, None, 0.0))
    return blocks


def _reference(net, x, G, train, keeps, inference=False, dtype=torch.float64, autocast=False):
    """d(sum(out * G))/dx and the oracle blocks (whose .weight.grad etc. hold the parameter gradients)"""
    blocks = _oracle_blocks(net)
    params = []
    for b in blocks:
        params += [b.weight] + ([b.bias] if b.bias is not None else []) + ([b.bn["weight"], b.bn["bias"]] if b.bn else [])
    for p in params:
        p.requires_grad_(True)
    xr = x.detach().cpu().to(dtype if not autocast else torch.float32).requires_grad_(True)
    drop = [keeps.get(i) for i in range(len(blocks))] if (keeps and train) else None
    hc = net._hc
    if autocast:
        with torch.autocast("cpu", dtype=torch.bfloat16):
            t = O.backbone_forward(xr, blocks, train=train, drop_keep=drop, dtype=torch.float32)
        t = t.float()
    else:
        t = O.backbone_forward(xr, blocks, train=train, drop_keep=drop, dtype=dtype)
    out = O.head_transform(t, hc["anchor_w"], hc["anchor_h"], hc["width_multiplier"], hc["height_multiplier"],
                           inference=inference)
    out.backward(G.detach().cpu().to(out.dtype))
    return xr.grad.double(), blocks


def _engine(net, x, G, train, keeps, dtype):
    net.compute_dtype = dtype
    net.train(train)
    net._get_runner().drop_keep_override = keeps if train else None
    xg = x.detach().to(DEV).requires_grad_(True)
    out = net(xg)
    out.backward(G.to(DEV))
    return xg.grad, out


def _zoo(case):
    z = _load(GOLDEN, "model_zoo.npz")
    name, net, img, _, _ = zoo_inputs(z, case)
    prefix = case + ".train."
    keeps = {int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith(prefix + "keep.")}
    x = img.float() / 255.0
    return net.to(DEV), x, keeps


def _grad_out(net, N, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((N, net.model[-1].out_channels, net.Sy, net.Sx), generator=g) * 0.1


# ----------------------------------------------------------------------------- 1: fp32 image gradient, every definition
@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("case", ZOO_CASES)
@pytest.mark.parametrize("impl", ["simt", "auto"])
def test_image_gradient_fp32_every_definition(case, impl, train):
    """Zoo seeds keep every LeakyReLU input of the train step > 3e-6 x rms from the kink (DESIGN.md §1): 1e-4.  Eval mode
    normalises with the running statistics, which moves the pre-activations off those margins: the fp32 bound of the
    parameter gradients, 2e-3."""
    net, x, keeps = _zoo(case)
    G = _grad_out(net, x.shape[0])
    L.set_conv_impl(impl)
    try:
        dx, _ = _engine(net, x, G, train, keeps, torch.float32)
    finally:
        L.set_conv_impl("auto")
    ref, _ = _reference(net, x, G, train, keeps)
    assert dx.dtype == torch.float32 and tuple(dx.shape) == tuple(x.shape)
    err = _rel(dx.cpu(), ref)
    assert err < (1e-4 if train else 2e-3), err


# ----------------------------------------------------------------------------- 2: bf16 path vs torch bf16 autocast
def test_image_gradient_bf16_within_autocast_error():
    ratios, report = [], {}
    for case in ZOO_CASES:
        net, x, keeps = _zoo(case)
        G = _grad_out(net, x.shape[0])
        dx, _ = _engine(net, x, G, True, keeps, torch.bfloat16)
        ref, _ = _reference(net, x, G, True, keeps)
        ac, _ = _reference(net, x, G, True, keeps, autocast=True)
        ours, theirs = _rel(dx.cpu(), ref), _rel(ac, ref)
        ratios.append(ours / max(theirs, 1e-2))
        if ours > max(2.0 * theirs, 2e-2):
            report[case] = (ours, theirs)
    assert not report, report
    assert float(np.median(ratios)) <= 1.25, ratios


# ----------------------------------------------------------------------------- 3: inference head (softmax)
def test_inference_model_gradients_through_the_softmax():
    z = _load(GOLDEN, "model_base.npz")
    sd = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}
    H, W = z["img"].shape[-2:]
    net = yogo_b200.YOGO((H, W), float(sd["anchor_w"]), float(sd["anchor_h"]), 7, inference=True)
    net.load_state_dict(sd)
    net = net.to(DEV)
    keeps = {int(k.split(".")[-1]): torch.from_numpy(z[k]) for k in z.files if k.startswith("base_train.keep.")}
    x = torch.from_numpy(z["img"]).float() / 255.0
    G = _grad_out(net, x.shape[0], seed=1)
    dx, out = _engine(net, x, G, True, keeps, torch.float32)
    ref, blocks = _reference(net, x, G, True, keeps, inference=True)
    assert _rel(dx.cpu(), ref) < 2e-3
    # parameter gradients (plan order = block by block: conv weight, conv bias, BN weight, BN bias; then the head), clamped
    # by the module's hook like the reference's
    refs = []
    for b in blocks:
        refs += [b.weight.grad] + ([b.bias.grad] if b.bias is not None else []) + \
                ([b.bn["weight"].grad, b.bn["bias"].grad] if b.bn else [])
    names = {id(p): k for k, p in net.named_parameters()}
    plan = net._get_runner().plan.params
    assert len(plan) == len(refs)
    bad = {}
    for p, r in zip(plan, refs):
        r = r.clamp(-1, 1)
        e = float((p.grad.cpu().double() - r).norm()) / max(float(r.norm()), 1e-3)
        if e > 2e-3:
            bad[names[id(p)]] = e
    assert not bad, bad


# ----------------------------------------------------------------------------- 4: frozen model
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_frozen_model_image_gradient_runs_no_weight_gradient_kernel(dtype):
    net, x, keeps = _zoo("double_filters")
    for p in net.parameters():
        p.requires_grad_(False)
    G = _grad_out(net, x.shape[0])
    net.compute_dtype = dtype
    net.eval()
    xg = x.to(DEV).requires_grad_(True)
    out = net(xg)
    assert out.requires_grad
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out.backward(G.to(DEV))
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "yg::" in e.name]
    assert names, "no library kernel in the trace"
    banned = [n for n in names if any(s in n for s in ("wgrad", "reduce", "param_grad", "finalize"))]
    assert not banned, sorted(set(banned))
    assert all(p.grad is None for p in net.parameters())
    ref, _ = _reference(net, x, G, False, None)
    err = _rel(xg.grad.cpu(), ref)
    if dtype == torch.float32:
        assert err < 2e-3, err
    else:   # the bf16 yardstick of the parameter tests: 2 x torch's own CPU bf16-autocast error on the same modules
        ac, _ = _reference(net, x, G, False, None, autocast=True)
        assert err <= max(2.0 * _rel(ac, ref), 2e-2), (err, _rel(ac, ref))


# ----------------------------------------------------------------------------- 5: parameter gradients unchanged
@pytest.mark.parametrize("case", ["rgb_base_model", "depth_ver_1"])
def test_parameter_gradients_identical_with_and_without_image_gradient(case):
    """Every parameter gradient is the same with and without the image gradient, up to the last bits: BatchNorm sums,
    bias sums and first-layer weight-gradient partials are reduced with atomics in a run-dependent order, so two runs of
    the same step already differ by an ulp here and there (measured on a B200: the head bias by 2e-9 between two identical
    runs)."""
    net, x, keeps = _zoo(case)
    G = _grad_out(net, x.shape[0])
    net.compute_dtype = torch.float32
    net.train()
    net._get_runner().drop_keep_override = keeps
    grads = []
    for need_x in (False, True):
        net.zero_grad(set_to_none=True)
        out = net(x.to(DEV).requires_grad_(need_x))
        out.backward(G.to(DEV))
        grads.append([p.grad.clone() for p in net.parameters()])
    for (k, _), a, b in zip(net.named_parameters(), *grads):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6 * float(a.abs().max())), (k, float((a - b).abs().max()))


# ----------------------------------------------------------------------------- 6: other first blocks
def _defn(name, first, rest_cin):
    def f(num_classes, rgb_input=False):
        return nn.Sequential(first(), nn.Sequential(nn.Conv2d(rest_cin, 32, 3, 2, 1, bias=False), nn.BatchNorm2d(32),
                                                    nn.LeakyReLU(), nn.Dropout2d(0.1)),
                             nn.Sequential(nn.Conv2d(32, 32, 3, 2, 1), nn.SiLU()), nn.Conv2d(32, 5 + num_classes, 1))
    f.__name__ = name
    return yogo_b200.model_defns.register_model(f)


FIRST_BLOCKS = {
    # not a direct block: a 1x1 first conv and a first conv on four channels take yg_conv_dgrad
    "t_first_1x1": (1, lambda: nn.Sequential(nn.Conv2d(1, 16, 1), nn.BatchNorm2d(16), nn.LeakyReLU()), 16),
    "t_first_4ch": (4, lambda: nn.Sequential(nn.Conv2d(4, 16, 3, 2, 1, bias=False), nn.BatchNorm2d(16), nn.LeakyReLU()), 16),
    # direct blocks outside the registered definitions: stride 1, conv bias, no BatchNorm, Dropout2d, Cout < 16
    "t_first_s1_bias": (1, lambda: nn.Sequential(nn.Conv2d(1, 8, 3, 1, 1, bias=True), nn.LeakyReLU(), nn.Dropout2d(0.2)), 8),
    "t_first_rgb_s1_bn": (3, lambda: nn.Sequential(nn.Conv2d(3, 24, 3, 1, 1, bias=True), nn.BatchNorm2d(24), nn.SiLU()), 24),
    "t_first_s2_silu": (1, lambda: nn.Sequential(nn.Conv2d(1, 4, 3, 2, 1, bias=True), nn.SiLU()), 4),
}


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("name", sorted(FIRST_BLOCKS))
def test_image_gradient_of_other_first_blocks(name, train):
    cin, first, rest = FIRST_BLOCKS[name]
    defn = _defn(name, first, rest)
    torch.manual_seed(3)
    net = yogo_b200.YOGO((40, 56), 0.05, 0.05, 7, model_func=defn)
    with torch.no_grad():
        for m in net.model.modules():
            if isinstance(m, nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.2, 0.2)
                m.running_mean.uniform_(-0.1, 0.1)
                m.running_var.uniform_(0.5, 1.5)
        net.model[-1].weight.mul_(0.1)
    net = net.to(DEV)
    x = torch.rand(3, cin, 40, 56)
    keeps = {i: (torch.rand(3, blk[0].out_channels) > 0.3).float() for i, blk in enumerate(net.model[:-1])
             if any(isinstance(m, nn.Dropout2d) for m in blk)}
    G = _grad_out(net, 3)
    dx, _ = _engine(net, x, G, train, keeps, torch.float32)
    ref, _ = _reference(net, x, G, train, keeps)
    assert tuple(dx.shape) == (3, cin, 40, 56)
    assert _rel(dx.cpu(), ref) < 2e-3


# ----------------------------------------------------------------------------- 7: input shapes and dtypes
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64, torch.float32])
def test_image_gradient_follows_the_input_shape_and_dtype(dtype):
    net = yogo_b200.YOGO((64, 96), 0.05, 0.05, 7).to(DEV)
    net.eval()
    for p in net.parameters():
        p.requires_grad_(False)
    x = torch.rand(1, 64, 96, device=DEV).to(dtype).requires_grad_(True)   # (C, H, W), unsqueezed by the module
    out = net(x)
    out.sum().backward()
    assert x.grad is not None and x.grad.dtype == dtype and tuple(x.grad.shape) == (1, 64, 96)
    x4 = x.detach().float().unsqueeze(0).requires_grad_(True)
    net(x4).sum().backward()
    tol = {torch.float16: 1e-3, torch.bfloat16: 1e-2}.get(dtype, 0.0)
    assert _rel(x.grad.float().cpu(), x4.grad[0].cpu()) <= max(tol, 1e-6)


# ----------------------------------------------------------------------------- 8: BASELINE geometry
def test_image_gradient_full_geometry_fp32():
    """772x1032, batch 2: 2e8 LeakyReLU inputs, some within rounding of the kink, where a different fp32 summation order
    legitimately takes the other slope.  Bound = max(3e-3 (the bound of test_full_size_train_step_vs_oracle_fp32), 3 x the
    error of the reference's own fp32 gradient against float64)."""
    torch.manual_seed(0)
    net = yogo_b200.YOGO((772, 1032), O.ANCHOR_W, O.ANCHOR_H, 7)
    with torch.no_grad():
        net.model[-1].weight.mul_(0.05)
    net = net.to(DEV)
    N = 2
    x = O.synth_images(N).float() / 255.0
    keeps = {1: (torch.rand(N, 32) > 0.05).float(), 2: (torch.rand(N, 64) > 0.1).float(),
             3: (torch.rand(N, 128) > 0.15).float()}
    G = _grad_out(net, N)
    dx, _ = _engine(net, x, G, True, keeps, torch.float32)
    ref, _ = _reference(net, x, G, True, keeps)
    ref32, _ = _reference(net, x, G, True, keeps, dtype=torch.float32)
    err, err32 = _rel(dx.cpu(), ref), _rel(ref32, ref)
    assert err < max(3e-3, 3 * err32), (err, err32)


# ----------------------------------------------------------------------------- kernels alone: vs torch, guard bands
def _guarded(shape, dtype, fill, pad=4096):
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * pad,), fill, dtype=dtype, device=DEV)
    return buf, buf[pad:pad + n].view(shape)


def _untouched(buf, n, fill, pad=4096):
    return bool((buf[:pad] == fill).all()) and bool((buf[pad + n:] == fill).all())


@pytest.mark.parametrize("Cin,Cout,stride,H,W", [(1, 16, 2, 37, 71), (3, 24, 1, 20, 33), (1, 48, 2, 64, 130),
                                                 (3, 4, 2, 9, 70), (1, 8, 1, 17, 31)])
@pytest.mark.parametrize("mode", ["bn_batch", "bn_running", "plain"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_first_dgrad_kernel_vs_autograd_and_guard_bands(Cin, Cout, stride, H, W, mode, dtype):
    """Dyadic inputs and weights keep every pre-activation exact in fp32 and off the LeakyReLU kink, so the slope taken is
    the same as float64 autograd's; the rest is fp32 rounding."""
    g = torch.Generator().manual_seed(Cin * 100 + Cout + stride)
    N = 2
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    x = torch.randint(-8, 9, (N, Cin, H, W), generator=g).double() / 8
    w = torch.randint(-8, 9, (Cout, Cin, 3, 3), generator=g).double() / 16
    fsh = (torch.randint(-8, 9, (Cout,), generator=g).double() * 2 + 1) / 256   # odd multiples of 1/256: y != 0
    scl = torch.tensor([0.5, 1.0, 2.0, 1.5] * 12)[:Cout].double()
    sft = (torch.randint(-8, 9, (Cout,), generator=g).double() * 2 + 1) / 1024
    mean, istd = torch.rand(Cout, generator=g).double() - 0.5, torch.rand(Cout, generator=g).double() + 0.5
    m1, m2 = torch.randn(Cout, generator=g).double() * 0.1, torch.randn(Cout, generator=g).double() * 0.1
    ds = (torch.rand(N, Cout, generator=g) > 0.2).double() / 0.8
    da = torch.randn(N, Ho, Wo, Cout, generator=g).to(dtype).double()
    act = L.ACT_LRELU
    # reference
    xr = x.clone().requires_grad_(True)
    y = torch.nn.functional.conv2d(xr, w, stride=stride, padding=1) + fsh[None, :, None, None]
    yv = y.detach().permute(0, 2, 3, 1)
    pre = yv * scl + sft if mode != "plain" else yv
    gp = da * ds[:, None, None, :] * torch.where(pre > 0, 1.0, 0.01)
    if mode == "bn_batch":
        dz = scl * (gp - m1 - (yv - mean) * istd * m2)
    elif mode == "bn_running":
        dz = scl * gp
    else:
        dz = gp
    y.backward(dz.permute(0, 3, 1, 2))
    # kernel
    f = lambda t: t.float().to(DEV).contiguous()
    xs, ws_, fs, sc, sh, mu, isd, a1, a2, dsd = (f(t) for t in (x, w, fsh, scl, sft, mean, istd, m1, m2, ds))
    dad = da.to(dtype).to(DEV).contiguous()
    bn = mode != "plain"
    ep = L.BwdEpilogue(None, act, dsd.data_ptr(), sc.data_ptr() if bn else None, sh.data_ptr() if bn else None,
                       mu.data_ptr() if bn else None, isd.data_ptr() if bn else None, None)
    buf, dx = _guarded((N, Cin, H, W), torch.float32, 7.0)
    lib = L.lib()
    L.check(lib.yg_conv_first_dgrad(xs.data_ptr(), ws_.data_ptr(), dad.data_ptr(), L.dtype_code(dtype), N, H, W, Cin, Cout,
                                    stride, ep, fs.data_ptr(), a1.data_ptr() if mode == "bn_batch" else None,
                                    a2.data_ptr() if mode == "bn_batch" else None, dx.data_ptr(), L.stream()))
    torch.cuda.synchronize()
    assert _untouched(buf, dx.numel(), 7.0)
    assert _rel(dx.cpu(), xr.grad) < 1e-5


@pytest.mark.parametrize("nc", [1, 7, 11, 27])
def test_head_softmax_bwd_vs_autograd_and_guard_bands(nc):
    g = torch.Generator().manual_seed(nc)
    N, Sy, Sx, D = 3, 13, 17, 5 + nc
    t = torch.randn(N, Sy, Sx, D, generator=g) * 3
    dp = torch.randn(N, D, Sy, Sx, generator=g)
    tr = t.double().permute(0, 3, 1, 2).requires_grad_(True)
    p = torch.softmax(tr[:, 5:], dim=1)
    p.backward(dp[:, 5:].double())
    exp = dp.double().clone()
    exp[:, 5:] = tr.grad[:, 5:]
    buf, out = _guarded((N, D, Sy, Sx), torch.float32, 7.0)
    dpd, td = dp.to(DEV), t.to(DEV).contiguous()
    L.check(L.lib().yg_head_softmax_bwd(dpd.data_ptr(), td.data_ptr(), out.data_ptr(), N, Sy, Sx, nc, L.stream()))
    torch.cuda.synchronize()
    assert _untouched(buf, out.numel(), 7.0)
    assert torch.equal(out[:, :5].cpu(), dp[:, :5])
    assert _rel(out.cpu(), exp) < 1e-6
