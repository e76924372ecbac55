"""The prediction head, YOGOLoss and format_preds kernels at every class-count code path, against float64 references.

The kernels after the backbone pick their code path from D = 5 + num_classes and their persistent loops behave differently
with the batch size.  The class counts NCS cross every boundary: the loss kernel's MAXC = 4 / 8 / 16 / 27, the head's
D <= 16 tcgen05 forward and kmask = 1 backward against the D > 16 SIMT kernels and kmask = 3, and the
head_bwd_warp_kernel / head_bwd_kernel split.  Batch 64 at the 97 x 129 grid makes every grid-stride, run and chunk loop
take more than one sweep.

Bounds.  Each reference rounds exactly the operands the path rounds (bf16 W and bf16 d(logits) on the tensor cores, fp32
W on the SIMT kernels), so what remains is fp32 arithmetic.  Sums of n terms are bounded with the probabilistic bound
LAM * sqrt(n) * u * sum|terms| (u = 2^-24; rounding errors as independent zero-mean variables, Higham & Mary 2019:
with LAM = 8 it fails with probability < 1e-13 per sum); elementwise functions add a few u per operation.  Every
comparison also builds the reference once more with one deliberate change and asserts that the kernel's distance from
the reference is at most a tenth of that change (`_margin`), so each bound is shown to catch a subtle error.

Tests without the gpu mark pin the references themselves on the CPU.  `python tests/test_head_loss_classes.py` runs the GPU
tests and prints, per test, path and output, the largest error as a fraction of its bound and the kernel's distance as a
fraction of the nearest changed reference's."""
import copy
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

if __name__ == "__main__":   # run as a script (see above): the repository root on the path, as conftest.py puts it
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import yogo_b200  # noqa: E402
from oracle import yogo_oracle as O  # noqa: E402
from yogo_b200 import _lib as L  # noqa: E402

DEV = "cuda:0"
U = 2.0 ** -24
LAM = 8.0
NCS = [1, 4, 5, 8, 9, 11, 12, 16, 17, 27]
CINS = [32, 64, 128, 256, 384]   # heads of quarter / half / base / double / triple_filters
AW, AH, WM, HM = O.ANCHOR_W, O.ANCHOR_H, 1.25, 0.8
PATHS = ["bf16-auto", "bf16-simt", "fp32"]
GUARD = 4096
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------- helpers
def guarded(shape, dtype, fill):
    numel = int(np.prod(shape))
    buf = torch.full((numel + 2 * GUARD,), fill, dtype=dtype, device=DEV)
    return buf, buf[GUARD:GUARD + numel].view(*shape)


def intact(buf, view, fill):
    n = view.numel()
    return bool((buf[:GUARD] == fill).all()) and bool((buf[GUARD + n:] == fill).all())


def _bf16(a):
    """float64 values rounded as the kernels round them (fp32, then bf16), back in float64."""
    return torch.as_tensor(a).float().bfloat16().double()


def _f32(a):
    return torch.as_tensor(a).float().double()


def _ulp_bf16(v):
    """spacing of the bf16 numbers at |v| (8 significant bits)."""
    e = torch.frexp(v.abs().clamp_min(2.0 ** -126))[1]
    return torch.ldexp(torch.ones_like(v), e - 8)


def _near_tie_bf16(v, err):
    """where a value within err of v may round to another bf16 number than v does."""
    return _bf16(v - err) != _bf16(v + err)


def _cpu64(t):
    return t.detach().cpu().double()


def _dist(a, r, dim=None):
    """Frobenius-relative distance; with dim, the largest one over the slices along dim (per output plane)."""
    a, r = torch.as_tensor(a).double(), torch.as_tensor(r).double()
    if dim is None:
        return float((a - r).norm() / r.norm().clamp_min(1e-300))
    a, r = a.movedim(dim, 0).flatten(1), r.movedim(dim, 0).flatten(1)
    return float(((a - r).norm(dim=1) / r.norm(dim=1).clamp_min(1e-300)).max())


def _worst(got, ref, bound):
    """largest |got - ref| / bound, elementwise (<= 1 passes)."""
    return float(((torch.as_tensor(got).double() - ref).abs() / bound).max())


def _margin(name, got, ref, alts, dim=None, rnd=_f32):
    """the kernel is at most 1/10 as far from the reference as each deliberately changed reference is.  Distances are
    taken between the stored values, with the references rounded to the storage type (rnd).  Returns the largest
    kernel / changed-reference distance ratio."""
    dk = _dist(got, rnd(ref), dim)
    worst = 0.0
    for what, alt in alts.items():
        da = _dist(rnd(alt), rnd(ref), dim)
        assert dk <= 0.1 * da, (name, what, dk, da)
        worst = max(worst, dk / da)
    return worst


MEASURED = {}   # (test, path, output) -> [largest error / bound, largest margin ratio], printed by running this file


def _record(path, output, ratio, margin):
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split("::")[-1].split("[")[0].split(" ")[0]
    r = MEASURED.setdefault((test, path, output), [0.0, 0.0])
    r[0], r[1] = max(r[0], ratio), max(r[1], margin)


@pytest.fixture
def impl_guard():
    """restores the global kernel choices whatever the test does."""
    try:
        yield
    finally:
        L.set_conv_impl("auto")
        L.set_fp32_tensor_cores(False)


def _set_path(path):
    L.set_conv_impl("simt" if path == "bf16-simt" else "auto")
    L.set_fp32_tensor_cores(False)
    return torch.float32 if path == "fp32" else torch.bfloat16


def _tc_fwd(path, D, Cin):
    """the bf16 forward runs on the tensor cores (pack_head_weights_fwd_kernel rounds W to bf16) when D <= 16 and Cin is
    a multiple of 16 up to 512; every Cin of CINS qualifies."""
    return path == "bf16-auto" and D <= 16


def _tc_bwd(path):
    """the bf16 backward runs on the tensor cores for every D <= 32 and every Cin of CINS."""
    return path == "bf16-auto"


# ----------------------------------------------------------------------------- head forward: reference and bound
def _head_fwd_ref(x, w, b, inference, cxs=None, cys=None):
    """x (N,Sy,Sx,Cin), w (D,Cin), b (D), all float64 holding the values the path multiplies -> out (N,D,Sy,Sx), t (N,Sy,Sx,D)."""
    Sy, Sx = x.shape[1:3]
    t = torch.einsum("nyxc,dc->nyxd", x, w) + b
    out = O.head_transform(t.permute(0, 3, 1, 2), AW, AH, WM, HM, inference=inference).clone()
    if cxs is not None:   # head_transform uses the default offsets
        out[:, 0] += cxs.double() - torch.linspace(0, 1 - 1 / Sx, Sx, dtype=torch.float32).double()
        out[:, 1] += cys.double() - torch.linspace(0, 1 - 1 / Sy, Sy, dtype=torch.float32).double()[:, None]
    return out, t


def _head_fwd_bound(x, w, b, out, t, inference):
    """elementwise bounds of (out, t_raw).  t: Cin + 1 products and the bias summed in fp32 -> LAM sqrt(Cin + 1) u sum|x w|
    (+ u |t| for the store).  out: the transform propagates the error of t by its derivative, and its own fp32 evaluation
    (sigmoid / expf, a multiply and an add; expf and 1/x within 2 ulp) adds 16 u |out|."""
    Cin = x.shape[-1]
    c = torch.einsum("nyxc,dc->nyxd", x.abs(), w.abs()) + b.abs()
    et = LAM * math.sqrt(Cin + 1) * U * c + U * t.abs()
    etn = et.permute(0, 3, 1, 2)
    tn = t.permute(0, 3, 1, 2)
    Sy, Sx = x.shape[1:3]
    eo = torch.empty_like(out)
    s = torch.sigmoid(tn[:, [0, 1, 4]])
    ds = s * (1 - s)
    eo[:, 0] = ds[:, 0] / Sx * etn[:, 0]
    eo[:, 1] = ds[:, 1] / Sy * etn[:, 1]
    eo[:, 4] = ds[:, 2] * etn[:, 4]
    # exp(min(t, 80)): relative error = absolute error of t below the clamp, none above it
    eo[:, 2:4] = out[:, 2:4] * torch.where(tn[:, 2:4] < 80 + etn[:, 2:4], etn[:, 2:4], torch.zeros_like(etn[:, 2:4]))
    if inference:   # d softmax_d = p_d (dt_d - sum_j p_j dt_j)
        p = out[:, 5:]
        eo[:, 5:] = p * (etn[:, 5:] + (p * etn[:, 5:]).sum(1, keepdim=True))
    else:
        eo[:, 5:] = etn[:, 5:]
    eo += 16 * U * out.abs() + 2.0 ** -140   # (results below 2^-126 are subnormal: absolute error of a few 2^-149)
    return eo, et + 1e-300


def _head_fwd_case(N, Sy, Sx, Cin, nc, path, seed, with_offsets=False):
    """inputs of one forward case: t[2], t[3] spread to ~40 so that some cells pass the clamp at 80."""
    D = 5 + nc
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, Sy, Sx, Cin, generator=g)
    w = torch.randn(D, Cin, generator=g) / math.sqrt(Cin)
    w[2:4] *= 40.0
    b = 0.1 * torch.randn(D, generator=g)
    if path != "fp32":
        x = x.bfloat16()
    cxs = cys = None
    if with_offsets:   # the module's _Cxs / _Cys buffers, moved off the default grid so that they must be read
        cxs = (torch.linspace(0, 1 - 1 / Sx, Sx).expand(Sy, -1) + 0.01 * torch.rand(Sy, Sx, generator=g)).contiguous()
        cys = (torch.linspace(0, 1 - 1 / Sy, Sy)[:, None].expand(Sy, Sx) + 0.01 * torch.rand(Sy, Sx, generator=g)).contiguous()
    return x, w, b, cxs, cys


def _run_head_fwd(x, w, b, nc, inference, cxs=None, cys=None):
    N, Sy, Sx, Cin = x.shape
    D = 5 + nc
    xd = x.to(DEV)
    wd, bd = w.to(DEV), b.to(DEV)
    out = torch.empty(N, D, Sy, Sx, device=DEV)
    t = torch.empty(N, Sy, Sx, D, device=DEV)
    cd = cxs.to(DEV) if cxs is not None else None
    yd = cys.to(DEV) if cys is not None else None
    L.check(L.lib().yg_head_fwd(xd.data_ptr(), L.dtype_code(x.dtype), wd.data_ptr(), bd.data_ptr(), out.data_ptr(), t.data_ptr(),
                                N, Sy, Sx, Cin, nc, AW, AH, WM, HM, int(inference), L.ptr(cd), L.ptr(yd), L.stream()))
    return _cpu64(out), _cpu64(t)


def _check_head_fwd(x, w, b, nc, path, inference, cxs=None, cys=None):
    D = 5 + nc
    tc = _tc_fwd(path, D, x.shape[-1])
    out, t = _run_head_fwd(x, w, b, nc, inference, cxs, cys)
    x64, b64 = x.double(), b.double()
    wp = _bf16(w) if tc else w.double()
    ref_o, ref_t = _head_fwd_ref(x64, wp, b64, inference, cxs, cys)
    eo, et = _head_fwd_bound(x64, wp, b64, ref_o, ref_t, inference)
    worst = (_worst(out, ref_o, eo), _worst(t, ref_t, et))
    assert worst[0] <= 1 and worst[1] <= 1, worst
    # deliberate changes: the other rounding of W, and the last class plane of W zeroed
    w_other = w.double() if tc else _bf16(w)
    w_zero = wp.clone()
    w_zero[D - 1] = 0
    variants = [("W rounding", w_other)]
    if not (inference and nc == 1):   # the softmax of a single class is 1 whatever its logit
        variants.append(("last class zeroed", w_zero))
    alts = {k: _head_fwd_ref(x64, wa, b64, inference, cxs, cys) for k, wa in variants}
    _record(path, "out", worst[0], _margin("out", out, ref_o, {k: v[0] for k, v in alts.items()}, dim=1))
    _record(path, "t_raw", worst[1], _margin("t_raw", t, ref_t, {k: v[1] for k, v in alts.items()}, dim=3))
    return worst


# ----------------------------------------------------------------------------- head backward: reference and bound
EPILOGUES = ["none", "lrelu", "silu_drop", "lrelu_mask_drop", "bn_silu_sums", "bn_lrelu_sums"]


def _epilogue_inputs(kind, N, Sy, Sx, Cin, dtype, g):
    """the backward epilogues engine.py builds for the last conv block: none; activation through the saved
    pre-activation; LeakyReLU through the sign mask (saved = the block output); BatchNorm + activation with the two BN sums."""
    if kind == "none":
        return {}
    e = {"act": L.ACT_SILU if "silu" in kind else L.ACT_LRELU}
    sv = torch.randn(N, Sy, Sx, Cin, generator=g).to(dtype)
    if "drop" in kind:
        e["drop"] = (torch.rand(N, Cin, generator=g) > 0.15).float() / 0.85
    if kind.startswith("bn"):
        e["bn"] = (torch.rand(Cin, generator=g) + 0.5, 0.3 * torch.randn(Cin, generator=g),
                   0.2 * torch.randn(Cin, generator=g), torch.rand(Cin, generator=g) + 0.5)
        e["sums"] = True
    if "mask" in kind:
        sv = torch.where(sv > 0, sv, 0.01 * sv).to(dtype)   # the LeakyReLU output
        bits = np.packbits((sv.float() > 0).numpy().reshape(-1), bitorder="little")
        e["mask"] = torch.from_numpy(bits)
    e["saved"] = sv
    return e


def _head_bwd_ref(dpred, traw, x, w, epi, tc, dtype, P_zero=False):
    """float64 yg_head_bwd.  dpred (N,D,Sy,Sx), traw (N,Sy,Sx,D), x (N,Sy,Sx,Cin), w (D,Cin): float64 of the stored values.
    On the tensor cores d(logits) is rounded to bf16 before dx and dW, W is bf16, and d(bias) is summed from the fp32
    d(logits).  Returns dict(dt, dtm, g (dx before its storage rounding), dw, db, sums) and the pieces of the bounds."""
    D = dpred.shape[1]
    if P_zero:
        dpred = dpred.clone()
        dpred[:, D - 1] = 0
    t = traw.permute(0, 3, 1, 2).clone().requires_grad_(True)
    O.head_transform(t, AW, AH, WM, HM).backward(dpred)
    dt = t.grad.permute(0, 2, 3, 1)
    dtm = _bf16(dt) if tc else dt
    wm_ = _bf16(w) if tc else w
    g0 = dtm @ wm_
    ds = epi["drop"].double()[:, None, None, :] if "drop" in epi else 1.0
    a = torch.ones_like(g0)
    pre = xhat = dpre = None
    if "saved" in epi:
        sv = epi["saved"].double()
        if "bn" in epi:
            sc, sh, mu, istd = (v.double() for v in epi["bn"])
            pre = sv * sc + sh
            dpre = 2 * U * ((sv * sc).abs() + sh.abs())   # fp32 (fused) multiply-add
            xhat = (sv - mu) * istd
        else:
            pre, dpre = sv, torch.zeros_like(sv)
        if epi["act"] == L.ACT_SILU:
            s = torch.sigmoid(pre)
            a = s * (1 + pre * (1 - s))
        else:
            a = torch.where(pre > 0, torch.ones_like(pre), torch.full_like(pre, 0.01))
    g = g0 * ds * a
    r = dict(dt=dt, dtm=dtm, g=g, dw=torch.einsum("nyxd,nyxc->dc", dtm, x), db=dt.sum((0, 1, 2)))
    if epi.get("sums"):
        gr = _bf16(g) if dtype == torch.bfloat16 else g
        r["sums"] = torch.cat([gr.sum((0, 1, 2)), (gr * xhat).sum((0, 1, 2))])
    return r, (g0, ds, a, pre, dpre, xhat, wm_)


def _head_bwd_bounds(ref, parts, x, epi, tc, dtype):
    """elementwise bound of dx and Frobenius bounds of dW, d(bias) and the BN sums (see the module docstring).
    d(logits): a few fp32 operations (sigmoid, expf, products) -> 16 u |dt|; where it sits that close to a bf16 rounding
    boundary the tensor-core operand may be the neighbouring bf16 number (amb).  dx: D products summed, then the
    epilogue factor a (SiLU derivative: 32 u (1 + |pre|); BN pre-activation error dpre moves it by <= 1.1 dpre; where
    |pre| <= dpre the LeakyReLU slope may be either), then one rounding to the storage type (one bf16 ulp)."""
    g0, ds, a, pre, dpre, xhat, wm_ = parts
    dt, dtm = ref["dt"], ref["dtm"]
    D = dt.shape[-1]
    P = dt.shape[0] * dt.shape[1] * dt.shape[2]
    edt = 16 * U * dt.abs()
    amb = (_near_tie_bf16(dt, edt) * _ulp_bf16(dt)) if tc else edt
    absdt = dtm.abs() + amb
    eg0 = LAM * math.sqrt(D + 1) * U * (dtm.abs() @ wm_.abs()) + amb @ wm_.abs()
    ea = torch.zeros_like(g0)
    if pre is not None:
        if epi["act"] == L.ACT_SILU:
            ea = 32 * U * (1 + pre.abs()) + 1.1 * dpre
        else:
            ea = torch.where(pre.abs() <= dpre, 0.99, 0.0).double()   # (fp32 0.01f of the kernels: 2e-8 relative)
    dsa = ds.abs() if torch.is_tensor(ds) else 1.0
    eg = dsa * (a.abs() * eg0 + (g0.abs() + eg0) * ea) + 4 * U * ref["g"].abs()
    ulp = _ulp_bf16(ref["g"]) if dtype == torch.bfloat16 else U * ref["g"].abs()
    b = dict(dx=eg + ulp + 1e-300)
    b["dw"] = float(LAM * math.sqrt(P) * U * torch.einsum("nyxd,nyxc->dc", absdt, x.abs()).norm()
                    + torch.einsum("nyxd,nyxc->dc", amb, x.abs()).norm())
    b["db"] = float((LAM * math.sqrt(P) + 16) * U * dt.abs().sum((0, 1, 2)).norm())
    if "sums" in ref:
        # each summand is the kernel's rounded dx: within eg of the reference before rounding, equal after it unless that
        # close to a rounding boundary
        gr = ref["g"]
        esum = eg + (_near_tie_bf16(gr, eg) * _ulp_bf16(gr) if dtype == torch.bfloat16 else U * gr.abs())
        s1 = LAM * math.sqrt(P) * U * gr.abs().sum((0, 1, 2)) + esum.sum((0, 1, 2))
        s2 = LAM * math.sqrt(P) * U * (gr * xhat).abs().sum((0, 1, 2)) + (esum * xhat.abs()).sum((0, 1, 2)) \
            + 4 * U * (gr * xhat).abs().sum((0, 1, 2))
        b["sums"] = float(torch.cat([s1, s2]).norm())
    return b


def _head_bwd_case(N, Sy, Sx, Cin, nc, dtype, epi_kind, seed):
    D = 5 + nc
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, Sy, Sx, Cin, generator=g).abs().to(dtype)   # the last block's output is mostly positive
    w = torch.randn(D, Cin, generator=g) / math.sqrt(Cin)
    traw = torch.randn(N, Sy, Sx, D, generator=g)
    traw[..., 2:4] -= 2.0
    hot = torch.rand(N, Sy, Sx, 2, generator=g) < 0.03   # past the clamp at 80: no gradient
    traw[..., 2:4] = torch.where(hot, 81 + 9 * torch.rand(N, Sy, Sx, 2, generator=g), traw[..., 2:4])
    dpred = torch.randn(N, D, Sy, Sx, generator=g) + 0.3
    epi = _epilogue_inputs(epi_kind, N, Sy, Sx, Cin, dtype, g)
    return x, w, traw, dpred, epi


def _run_head_bwd(x, w, traw, dpred, epi, nc, clip, want_params=True):
    N, Sy, Sx, Cin = x.shape
    D = 5 + nc
    lib = L.lib()
    xd, wd, td, pd = x.to(DEV), w.to(DEV), traw.to(DEV), dpred.to(DEV)
    dx = torch.empty(N, Sy, Sx, Cin, dtype=x.dtype, device=DEV)
    dw = torch.empty(D, Cin, device=DEV) if want_params else None
    db = torch.empty(D, device=DEV) if want_params else None
    dev = {k: (v.to(DEV) if torch.is_tensor(v) else tuple(t.to(DEV) for t in v)) for k, v in epi.items() if k not in ("act", "sums")}
    sums = torch.zeros(2 * Cin, dtype=torch.float64, device=DEV) if epi.get("sums") else None
    ep = None
    if epi:
        bn = dev.get("bn", (None,) * 4)
        ep = L.BwdEpilogue(dev["saved"].data_ptr(), epi["act"], L.ptr(dev.get("drop")), L.ptr(bn[0]), L.ptr(bn[1]),
                           L.ptr(bn[2]), L.ptr(bn[3]), L.ptr(sums), L.ptr(dev.get("mask")))
    nb = lib.yg_head_bwd_workspace(N, Sy, Sx, Cin, nc)
    ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_head_bwd(pd.data_ptr(), td.data_ptr(), xd.data_ptr(), wd.data_ptr(), dx.data_ptr(), L.dtype_code(x.dtype),
                            L.ptr(dw), L.ptr(db), N, Sy, Sx, Cin, nc, AW, AH, WM, HM, C.byref(ep) if ep is not None else None,
                            float(clip), ws.data_ptr(), nb, L.stream()))
    res = dict(dx=_cpu64(dx))
    if want_params:
        res.update(dw=_cpu64(dw), db=_cpu64(db))
    if sums is not None:
        res["sums"] = _cpu64(sums)
    return res


def _check_head_bwd(x, w, traw, dpred, epi, nc, path, want_params=True):
    D = 5 + nc
    dtype = x.dtype
    tc = _tc_bwd(path)
    x64, w64, t64, p64 = x.double(), w.double(), traw.double(), dpred.double()
    ref, parts = _head_bwd_ref(p64, t64, x64, w64, epi, tc, dtype)
    # a clip that clamps about a tenth of the weight and bias gradients (clamping is 1-Lipschitz: the bounds stand)
    clip = float(torch.cat([ref["dw"].flatten(), ref["db"]]).abs().quantile(0.9))
    got = _run_head_bwd(x, w, traw, dpred, epi, nc, clip, want_params)
    bnd = _head_bwd_bounds(ref, parts, x64, epi, tc, dtype)
    rnd = _bf16 if dtype == torch.bfloat16 else _f32
    res = {"dx": _worst(got["dx"], ref["g"], bnd["dx"])}
    alt_round = _head_bwd_ref(p64, t64, x64, w64, epi, not tc if path != "fp32" else True, dtype)[0]
    alt_zero = _head_bwd_ref(p64, t64, x64, w64, epi, tc, dtype, P_zero=True)[0]
    mar = {"dx": _margin("dx", got["dx"], ref["g"], {"roundings of the other path": alt_round["g"],
                                                     "last class zeroed": alt_zero["g"]}, rnd=rnd)}
    if want_params:
        for k in ("dw", "db"):
            r = ref[k].clamp(-clip, clip)
            res[k] = _dist(got[k], r) / (bnd[k] / float(r.norm()))
            mar[k] = _margin(k, got[k], r, {"last class zeroed": alt_zero[k].clamp(-clip, clip)})
        assert int((ref["dw"].abs() > clip).sum()) > 0
    if "sums" in ref:
        res["sums"] = _dist(got["sums"], ref["sums"]) / (bnd["sums"] / float(ref["sums"].norm()))
        mar["sums"] = _margin("sums", got["sums"], ref["sums"], {"roundings of the other path": alt_round["sums"],
                                                                 "last class zeroed": alt_zero["sums"]},
                              rnd=lambda v: torch.as_tensor(v).double())
    for k in res:
        _record(path, k, res[k], mar[k])
    assert all(v <= 1 for v in res.values()), res
    return res


# ----------------------------------------------------------------------------- loss: inputs, reference, bounds
def _loss_case(N, Sy, Sx, nc, K, seed):
    lab = O.synth_labels(N, Sy, Sx, nc, K, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    pred = torch.rand(N, 5 + nc, Sy, Sx, generator=g)
    pred[:, 2:4] = 0.02 + 0.08 * pred[:, 2:4]
    pred[:, 5:] = 3 * torch.randn(N, nc, Sy, Sx, generator=g)
    return pred, lab


LOSS_W = dict(no_obj_weight=0.5, iou_weight=5.0, classify_weight=1.0, label_smoothing=0.01)
LOSS_W_ALT = dict(no_obj_weight=0.3, iou_weight=2.5, classify_weight=0.7, label_smoothing=0.1)   # the `lossw` golden case


def _loss_ref(pred, lab, w):
    loss, comps, d = O.yogo_loss_np(pred.numpy(), lab.numpy(), dtype=np.float64, **w)
    return np.array([loss, comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]]), torch.from_numpy(d)


def _loss_bounds(pred, lab, ref4, w):
    """bounds of the four outputs (absolute) and of dpred (classes and objectness elementwise, boxes Frobenius).
    Every per-cell term is non-negative and summed in fp64, so the error of a component is the sum of the cells' errors:
    objectness 3 fp32 operations (4 u relative); cross-entropy lse - logit: 8 u (|max| + |target logit| + mean |logit|),
    __logf 2^-21 absolute, and the __expf terms (2 + 1.17 |arg|) ulp each, whose se-weighted sum is <= (2 + 0.44 C) u;
    CIoU about 40 fp32 operations on parts (1, iou, centre term, alpha v) that are each <= 1: 512 u per labelled cell.
    Class gradient f (softmax - target): the softmax error above and 2 u of the difference."""
    p = pred.double()
    N, D = p.shape[:2]
    nc = D - 5
    m = lab[:, 0].double()
    lg = p[:, 5:]
    mx = lg.max(1).values
    tgt = lab[:, 5].long().clamp(0, nc - 1)
    lt = lg.gather(1, tgt[:, None])[:, 0]
    e_cell = m * (8 * U * (mx.abs() + lt.abs() + lg.abs().mean(1)) + 2.0 ** -21 + (2 + 0.44 * nc) * U)
    e_iou = w["iou_weight"] / N * 512 * U * float(m.sum())
    e_obj = 4 * U * ref4[2]
    e_cls = w["classify_weight"] / N * float(e_cell.sum())
    e4 = np.array([e_iou + e_obj + e_cls, e_iou, e_obj, e_cls]) + 2 * U * np.abs(ref4)
    sm = torch.softmax(lg, 1)
    s = w["label_smoothing"]
    tdist = torch.full_like(sm, s / nc).scatter_add_(1, tgt[:, None], torch.full_like(sm[:, :1], 1 - s))
    f = (m * w["classify_weight"] / N)[:, None]
    ecls = f * (sm * ((2 + 1.17 * (lg - mx[:, None]).abs()) + (2 + 0.44 * nc) + 4) * U + 2 * U * (sm - tdist).abs())
    return e4, ecls + 1e-300


def _check_loss(pred, lab, w, ref4, dref, alt_smooth, got4, dgot):
    """the four outputs and dpred against the float64 reference; margins against the reference without label smoothing
    (classification) and with the box and objectness terms scaled by 1 + 2^-10."""
    nc = pred.shape[1] - 5
    e4, ecls = _loss_bounds(pred, lab, ref4, w)
    got4 = np.asarray(got4, dtype=np.float64)
    res = {"out4": float(np.max(np.abs(got4 - ref4) / e4))}
    res["dpred_cls"] = _worst(dgot[:, 5:], dref[:, 5:], ecls + U * dref[:, 5:].abs())
    res["dpred_obj"] = _worst(dgot[:, 4], dref[:, 4], 4 * U * dref[:, 4].abs() + 1e-300)
    # box gradients: ~40 fp32 operations, the quotient-rule differences of the CIoU gradient lose up to ~25x: 1024 u
    res["dpred_box"] = _dist(dgot[:, :4], dref[:, :4]) / (1024 * U)
    assert all(v <= 1 for v in res.values()), res
    sc = 1 + 2.0 ** -10
    a4, adref = alt_smooth
    mar = {"out4": max(
        _margin("loss", got4[0], ref4[0], {"box term scaled": ref4[0] + ref4[1] * (sc - 1)} | ({"smoothing dropped": a4[0]} if nc > 1 else {})),
        _margin("iou_loss", got4[1], ref4[1], {"box term scaled": ref4[1] * sc}),
        _margin("objectness_loss", got4[2], ref4[2], {"objectness scaled": ref4[2] * sc}))}
    mar["dpred_box"] = _margin("dpred boxes", dgot[:, :4], dref[:, :4], {"box term scaled": dref[:, :4] * sc})
    mar["dpred_obj"] = _margin("dpred objectness", dgot[:, 4], dref[:, 4], {"objectness scaled": dref[:, 4] * sc})
    mar["dpred_cls"] = 0.0
    if nc > 1:   # the cross-entropy of a single class is 0 whatever the smoothing: nothing can move it
        mar["out4"] = max(mar["out4"], _margin("classification_loss", got4[3], ref4[3], {"smoothing dropped": a4[3]}))
        mar["dpred_cls"] = _margin("dpred classes", dgot[:, 5:], dref[:, 5:], {"smoothing dropped": adref[:, 5:]})
    for k in res:
        _record("fp32", k, res[k], mar[k])
    return res


def _run_loss(pred, lab, w):
    loss_fn = yogo_b200.YOGOLoss(**w).to(DEV)
    loss, comps, dpred = loss_fn.loss_and_grad(pred.to(DEV), lab.to(DEV))
    got4 = [loss.item(), comps["iou_loss"], comps["objectness_loss"], comps["classification_loss"]]
    return got4, dpred


# ============================================================================= CPU: the references themselves
@pytest.mark.parametrize("nc", [1, 2, 7, 12, 27])
def test_loss_reference_class_term_equals_torch_cross_entropy(nc):
    """the class part of the float64 loss reference (classification_loss and gradient planes 5:) is torch's label-smoothed
    cross-entropy, masked to the labelled cells, differentiated by autograd."""
    pred, lab = _loss_case(2, 11, 13, nc, 40, seed=nc)
    for w in (LOSS_W, LOSS_W_ALT):
        _, comps, d = O.yogo_loss_np(pred.numpy(), lab.numpy(), dtype=np.float64, **w)
        lg = pred[:, 5:].double().requires_grad_(True)
        m = lab[:, 0].double()
        ce = F.cross_entropy(lg, lab[:, 5].long(), label_smoothing=w["label_smoothing"], reduction="none") * m
        cls = w["classify_weight"] * ce.sum() / pred.shape[0]
        cls.backward()
        assert abs(comps["classification_loss"] - cls.item()) <= 1e-12 * max(abs(cls.item()), 1.0)
        np.testing.assert_allclose(d[:, 5:], lg.grad.numpy(), rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("inference", [False, True])
@pytest.mark.parametrize("nc", [1, 12, 27])
def test_head_forward_reference_equals_conv_and_head_transform(nc, inference):
    """the NHWC einsum reference of the head is the 1x1 Conv2d + YOGO output transform of the model, with the grid
    offsets added as given."""
    x, w, b, cxs, cys = _head_fwd_case(2, 11, 13, 32, nc, "fp32", seed=nc, with_offsets=True)
    x64, w64, b64 = x.double(), w.double(), b.double()
    out, t = _head_fwd_ref(x64, w64, b64, inference, cxs, cys)
    tn = F.conv2d(x64.permute(0, 3, 1, 2), w64[:, :, None, None], b64)
    exp = O.head_transform(tn, AW, AH, WM, HM, inference=inference).clone()
    exp[:, 0] = torch.sigmoid(tn[:, 0]) / 13 + cxs.double()   # model.py: (1 / Sx) sigmoid(t0) + _Cxs
    exp[:, 1] = torch.sigmoid(tn[:, 1]) / 11 + cys.double()
    torch.testing.assert_close(t.permute(0, 3, 1, 2), tn, rtol=1e-13, atol=1e-13)
    torch.testing.assert_close(out, exp, rtol=1e-13, atol=1e-13)
    assert bool((tn[:, 2:4] > 80).any())   # the cases reach the clamp


@pytest.mark.parametrize("epi_kind", EPILOGUES)
def test_head_backward_reference_equals_autograd(epi_kind):
    """the head backward reference without roundings is float64 autograd of: block output = dropout scale x
    act(BN affine of the saved tensor), 1x1 head, YOGO transform; dx = d/d(BN output or conv output), and the BN sums are
    sum(dx) and sum(dx * xhat)."""
    nc, Cin = 12, 32
    x, w, traw, dpred, epi = _head_bwd_case(2, 5, 7, Cin, nc, torch.float32, epi_kind, seed=3)
    ref, _ = _head_bwd_ref(dpred.double(), traw.double(), x.double(), w.double(), epi, False, torch.float32)
    w64 = w.double().requires_grad_(True)
    b64 = torch.zeros(5 + nc, dtype=torch.float64, requires_grad=True)
    if epi:
        sv = epi["saved"].double()
        if "bn" in epi:
            sc, sh, mu, istd = (v.double() for v in epi["bn"])
            pre = (sv * sc + sh).requires_grad_(True)
        else:
            pre = sv.clone().requires_grad_(True)
        act = F.silu if epi["act"] == L.ACT_SILU else (lambda v: F.leaky_relu(v, 0.01))
        h = act(pre) * (epi["drop"].double()[:, None, None, :] if "drop" in epi else 1.0)
        # the head reads the stored block output x; the chain through act(pre) only supplies the epilogue factor
        h = h + (x.double() - h).detach()
    else:
        pre = h = x.double().requires_grad_(True)
    t = torch.einsum("nyxc,dc->nyxd", h, w64) + b64
    t = t.permute(0, 3, 1, 2)
    # the transform takes the stored raw logits (traw) and passes the gradient of t through it
    t = t + (traw.double().permute(0, 3, 1, 2) - t).detach()
    O.head_transform(t, AW, AH, WM, HM).backward(dpred.double())
    torch.testing.assert_close(ref["g"], pre.grad, rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(ref["dw"], w64.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref["db"], b64.grad, rtol=1e-12, atol=1e-12)
    if "sums" in ref:
        xhat = (epi["saved"].double() - epi["bn"][2].double()) * epi["bn"][3].double()
        exp = torch.cat([pre.grad.sum((0, 1, 2)), (pre.grad * xhat).sum((0, 1, 2))])
        torch.testing.assert_close(ref["sums"], exp, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("nc", [1, 12, 27])
def test_format_preds_and_class_counts_references_agree(nc):
    """prediction_class_counts_np is the histogram of format_preds_np's rows, with and without a class-confidence floor."""
    p = O.synth_sparse_preds(4, 24, 32, nc, 40).numpy()
    for mcc in (0.0, 0.4):
        tot = np.zeros(nc, np.int64)
        for b in range(p.shape[0]):
            rows = O.format_preds_np(p[b], 0.5, 0.5, "cxcywh", mcc)
            if rows.size:
                tot += O.count_cells_np(rows[:, 5:])
        assert np.array_equal(O.prediction_class_counts_np(p, 0.5, 0.5, mcc), tot)
        assert tot.sum() > 0


# ============================================================================= GPU: head forward
@gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("Cin", CINS)
@pytest.mark.parametrize("nc", NCS)
def test_head_forward_every_class_count(nc, Cin, path, impl_guard):
    """odd 13 x 17 grid: tcgen05 epilogue (bf16, D <= 16), head_fwd_kernel<bf16 | float, 16 | 32>; training and
    inference transforms, the grid offsets read from the module's buffers or computed."""
    _set_path(path)
    x, w, b, cxs, cys = _head_fwd_case(3, 13, 17, Cin, nc, path, seed=nc * 1000 + Cin)
    _check_head_fwd(x, w, b, nc, path, inference=False)
    _check_head_fwd(x, w, b, nc, path, inference=True, cxs=cxs, cys=cys)


@pytest.fixture(scope="module")
def big_head_fwd():
    """batch 64 at 97 x 129 (base_model's head, Cin = 128): the inputs are built once per module."""
    cache = {}

    def get(nc, path):
        key = (nc, path == "fp32")
        if key not in cache:
            cache[key] = _head_fwd_case(64, 97, 129, 128, nc, path, seed=nc)
        return cache[key]
    return get


@gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("nc", [7, 27])
def test_head_forward_batch64_full_grid(nc, path, big_head_fwd, impl_guard):
    _set_path(path)
    x, w, b, _, _ = big_head_fwd(nc, path)
    _check_head_fwd(x, w, b, nc, path, inference=False)


# ============================================================================= GPU: head backward
@gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("Cin", CINS)
@pytest.mark.parametrize("nc", NCS)
def test_head_backward_every_class_count(nc, Cin, path, impl_guard):
    """tcgen05 with kmask 1 (D <= 16) and 3; head_bwd_warp_kernel at CPL = Cin / 32 = 1, 2, 4, 8 (SIMT, D <= 16);
    head_bwd_kernel<T, 16> (Cin = 384) and <T, 32> (D > 16).  BatchNorm + SiLU epilogue with both BN sums."""
    dtype = _set_path(path)
    x, w, traw, dpred, epi = _head_bwd_case(3, 13, 17, Cin, nc, dtype, "bn_silu_sums", seed=nc * 1000 + Cin)
    _check_head_bwd(x, w, traw, dpred, epi, nc, path)


@gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("Cin", [128, 384])
@pytest.mark.parametrize("nc", [4, 27])
@pytest.mark.parametrize("epi_kind", EPILOGUES + ["no_param_grads"])
def test_head_backward_epilogues(epi_kind, nc, Cin, path, impl_guard):
    """every backward epilogue engine.py builds, on every dispatch branch; dw = dbias = None computes dx alone."""
    dtype = _set_path(path)
    kind = "silu_drop" if epi_kind == "no_param_grads" else epi_kind
    x, w, traw, dpred, epi = _head_bwd_case(2, 13, 17, Cin, nc, dtype, kind, seed=nc * 7 + Cin)
    _check_head_bwd(x, w, traw, dpred, epi, nc, path, want_params=epi_kind != "no_param_grads")


# batch 64 at 97 x 129 = 800,832 pixels: head_dt_kernel sweeps its 592 x 256 threads 6 times, the warp kernel's 2368 warps
# take 11 runs each, head_bwd_kernel's 296 blocks 22 tiles each.  Cin = 64 keeps the float64 reference small; Cin = 96
# (3 channel chunks, no warp-kernel width) sends D <= 16 to head_bwd_kernel<T, 16> as Cin = 384 does, at a quarter of
# that reference's size.
BIG_BWD = [("bf16-auto", 7, 64, "lrelu_mask_drop"), ("bf16-auto", 27, 64, "bn_silu_sums"), ("fp32", 7, 64, "bn_silu_sums"),
           ("fp32", 27, 64, "silu_drop"), ("bf16-simt", 7, 96, "bn_lrelu_sums")]


@gpu
@pytest.mark.parametrize("path,nc,Cin,kind", BIG_BWD)
def test_head_backward_batch64_full_grid(path, nc, Cin, kind, impl_guard):
    """tcgen05 kmask 1 and 3, warp kernel CPL 2, head_bwd_kernel<float, 32> and <bf16, 16>, each sweeping more than once."""
    dtype = _set_path(path)
    x, w, traw, dpred, epi = _head_bwd_case(64, 97, 129, Cin, nc, dtype, kind, seed=nc)
    _check_head_bwd(x, w, traw, dpred, epi, nc, path)


# ============================================================================= GPU: loss
@gpu
@pytest.mark.parametrize("nc", NCS)
def test_loss_every_class_count(nc):
    """yogo_loss_kernel<MAXC = 4, 8, 16, 27> on a small batch; the `lossw` weights at nc = 9 and 27."""
    w = LOSS_W_ALT if nc in (9, 27) else LOSS_W
    pred, lab = _loss_case(4, 37, 41, nc, 120, seed=nc)
    ref4, dref = _loss_ref(pred, lab, w)
    alt = _loss_ref(pred, lab, dict(w, label_smoothing=0.0))
    got4, dgot = _run_loss(pred, lab, w)
    _check_loss(pred, lab, w, ref4, dref, alt, got4, _cpu64(dgot))


@gpu
@pytest.mark.parametrize("nc", [4, 27])
def test_loss_batch64_full_grid_and_determinism(nc):
    """batch 64 at 97 x 129 with 300 labels per image: 3,129 chunks of 256 cells over 1,184 blocks, so labelled cells wait
    in the per-warp queue from one chunk to the next."""
    pred, lab = _loss_case(64, 97, 129, nc, 300, seed=nc)
    ref4, dref = _loss_ref(pred, lab, LOSS_W)
    alt = _loss_ref(pred, lab, dict(LOSS_W, label_smoothing=0.0))
    got4, dgot = _run_loss(pred, lab, LOSS_W)
    _check_loss(pred, lab, LOSS_W, ref4, dref, alt, got4, _cpu64(dgot))
    got4b, dgotb = _run_loss(pred, lab, LOSS_W)
    assert got4b == got4 and torch.equal(dgotb, dgot)
    # the batch twice: every sum doubles with N, and each cell's gradient halves exactly (1 / (2N) = (1 / N) / 2 in fp32).
    # The fp64 totals are summed in another order (other chunks per thread), so each output may land on the neighbouring
    # fp32 number: one ulp.
    got4d, dgotd = _run_loss(torch.cat([pred, pred]), torch.cat([lab, lab]), LOSS_W)
    for a, b in zip(got4d, got4):
        assert abs(a - b) <= float(np.spacing(np.float32(abs(b)))), (got4d, got4)
    assert torch.equal(dgotd[:64] * 2, dgot) and torch.equal(dgotd[64:] * 2, dgot)


# ============================================================================= GPU: format_preds
@gpu
@pytest.mark.parametrize("mcc", [0.0, 0.4])
@pytest.mark.parametrize("nc", [1, 12, 27])
def test_format_preds_batch64_bit_exact(nc, mcc):
    p = O.synth_sparse_preds(64, 97, 129, nc, 300, seed=nc)
    rows, kc, _, counts = yogo_b200.format_preds_batch(p.to(DEV), min_class_confidence_threshold=mcc)
    rows, kc = rows.cpu().numpy(), kc.cpu().numpy()
    for b in range(64):
        exp = O.format_preds_np(p[b].numpy(), 0.5, 0.5, "cxcywh", mcc)
        assert int(kc[b]) == exp.shape[0], b
        assert np.array_equal(rows[b, : exp.shape[0]].view(np.uint32), exp.view(np.uint32)), b
    assert np.array_equal(counts.cpu().numpy(), O.prediction_class_counts_np(p.numpy(), 0.5, 0.5, mcc))


# ============================================================================= GPU: guard bands
@gpu
@pytest.mark.parametrize("impl", ["auto", "simt"])
@pytest.mark.parametrize("nc", [1, 27])
def test_outputs_stay_inside_their_buffers_at_d6_and_d32(nc, impl, impl_guard):
    """nothing outside the outputs of the head forward and backward (both storage types, with BN sums), the loss and
    format_preds is written at D = 6 and D = 32, on an odd grid."""
    lib = L.lib()
    L.set_conv_impl(impl)
    N, Sy, Sx, Cin = 3, 13, 17, 128
    D = 5 + nc
    for dtype in (torch.bfloat16, torch.float32):
        x, w, traw, dpred, epi = _head_bwd_case(N, Sy, Sx, Cin, nc, dtype, "bn_silu_sums", seed=11)
        xd, wd, bd = x.to(DEV), w.to(DEV), torch.zeros(D, device=DEV)
        obuf, o = guarded((N, D, Sy, Sx), torch.float32, 7.0)
        tbuf, t = guarded((N, Sy, Sx, D), torch.float32, 7.0)
        L.check(lib.yg_head_fwd(xd.data_ptr(), L.dtype_code(dtype), wd.data_ptr(), bd.data_ptr(), o.data_ptr(), t.data_ptr(),
                                N, Sy, Sx, Cin, nc, AW, AH, WM, HM, 0, None, None, L.stream()))
        dxbuf, dx = guarded((N, Sy, Sx, Cin), dtype, 7.0)
        dwbuf, dw = guarded((D, Cin), torch.float32, 7.0)
        dbbuf, db = guarded((D,), torch.float32, 7.0)
        sbuf, sums = guarded((2 * Cin,), torch.float64, 0.0)
        sv = epi["saved"].to(DEV)
        sc, sh, mu, istd = (v.to(DEV) for v in epi["bn"])
        ep = L.BwdEpilogue(sv.data_ptr(), epi["act"], None, sc.data_ptr(), sh.data_ptr(), mu.data_ptr(), istd.data_ptr(),
                           sums.data_ptr(), None)
        nb = lib.yg_head_bwd_workspace(N, Sy, Sx, Cin, nc)
        ws = torch.empty(max(nb, 16), dtype=torch.uint8, device=DEV)
        pd = dpred.to(DEV)
        L.check(lib.yg_head_bwd(pd.data_ptr(), t.data_ptr(), xd.data_ptr(), wd.data_ptr(), dx.data_ptr(), L.dtype_code(dtype),
                                dw.data_ptr(), db.data_ptr(), N, Sy, Sx, Cin, nc, AW, AH, WM, HM, C.byref(ep), 1.0,
                                ws.data_ptr(), nb, L.stream()))
        torch.cuda.synchronize()
        assert intact(obuf, o, 7.0) and intact(tbuf, t, 7.0), dtype
        assert intact(dxbuf, dx, 7.0) and intact(dwbuf, dw, 7.0) and intact(dbbuf, db, 7.0) and intact(sbuf, sums, 0.0), dtype
        assert float(sums.abs().sum()) > 0
    lab = O.synth_labels(N, Sy, Sx, nc, 20).to(DEV)
    pbuf, dp = guarded((N, D, Sy, Sx), torch.float32, 7.0)
    o4buf, o4 = guarded((4,), torch.float32, 7.0)
    nbl = lib.yg_yogo_loss_workspace(N, Sy, Sx)
    wsl = torch.empty(max(nbl, 16), dtype=torch.uint8, device=DEV)
    L.check(lib.yg_yogo_loss_fwd_bwd(o.data_ptr(), lab.data_ptr(), o4.data_ptr(), dp.data_ptr(), N, nc, Sy, Sx, 0.5, 5.0, 1.0, 0.01,
                                     wsl.data_ptr(), nbl, L.stream()))
    torch.cuda.synchronize()
    assert intact(pbuf, dp, 7.0) and intact(o4buf, o4, 7.0) and bool(torch.isfinite(o4).all())
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


# ============================================================================= GPU: one training step per class-count boundary
@gpu
@pytest.mark.parametrize("nc", [1, 12, 27])
def test_train_step_fp32_simt_vs_float64_autograd(nc, impl_guard):
    """silu_model (no LeakyReLU kinks) with Dropout2d p = 0, one fp32 step on the exact SIMT kernels, against float64 CPU
    autograd of a copy of the same torch.nn modules fed the float64 loss gradient: 1e-3 relative per tensor (the conv bias
    in front of BatchNorm has a zero gradient: the project's absolute floor of 1e-3).  Margin: a second float64 copy with
    the head weight rounded to bf16 (the rounding the SIMT path must not do) is at least 10x further from the reference than
    the kernels, for the outputs, the loss and every gradient that is not zero by construction."""
    L.set_conv_impl("simt")
    L.set_fp32_tensor_cores(False)
    torch.manual_seed(nc)
    net = yogo_b200.YOGO((96, 128), O.ANCHOR_W, O.ANCHOR_H, nc, model_func=yogo_b200.get_model_func("silu_model"))
    for m in net.modules():
        if isinstance(m, torch.nn.Dropout2d):
            m.p = 0.0
    with torch.no_grad():
        net.model[-1].weight.mul_(0.05)
    ref = copy.deepcopy(net.model).double().train()
    alt = copy.deepcopy(ref)
    with torch.no_grad():
        alt[-1].weight.copy_(_bf16(alt[-1].weight))
    # conv biases followed by BatchNorm: their gradient is zero by construction, no rounding of W can move it
    zero_grad = {f"{i}.0.bias" for i, blk in enumerate(ref[:-1])
                 if blk[0].bias is not None and isinstance(blk[1], torch.nn.BatchNorm2d)}
    net = net.to(DEV)
    net.compute_dtype = torch.float32
    net.train()
    N = 4
    x = O.synth_images(N, 96, 128, seed=nc).float() / 255.0
    lab = O.synth_labels(N, 12, 16, nc, 10, seed=nc)
    out = net(x.to(DEV))
    loss, _ = yogo_b200.YOGOLoss().to(DEV)(out, lab.to(DEV))
    loss.backward()

    def step64(model):
        o = O.head_transform(model(x.double()), O.ANCHOR_W, O.ANCHOR_H)
        lo, _, dpred = O.yogo_loss_np(o.detach().numpy(), lab.numpy(), dtype=np.float64)
        o.backward(torch.from_numpy(dpred))
        return o.detach(), lo, {k: q.grad.clamp(-1, 1) for k, q in model.named_parameters()}

    ref_out, ref_loss, ref_g = step64(ref)
    alt_out, alt_loss, alt_g = step64(alt)
    got = _cpu64(out)
    assert _dist(got, ref_out) < 1e-3
    assert abs(loss.item() - ref_loss) < 1e-3 * abs(ref_loss)
    # planes 0 and 1 are (1 / S) sigmoid(t) + the grid offset: the offsets are taken out so that the margin sees the logits
    off = torch.zeros_like(ref_out)
    off[:, 0] = torch.linspace(0, 1 - 1 / 16, 16, dtype=torch.float32).double()
    off[:, 1] = torch.linspace(0, 1 - 1 / 12, 12, dtype=torch.float32).double()[:, None]
    margin = {"out": _margin("out", got - off, ref_out - off, {"head W in bf16": alt_out - off}, dim=1, rnd=lambda v: v),
              "loss": _margin("loss", loss.item(), ref_loss, {"head W in bf16": alt_loss})}
    worst = {}
    for k, p in net.model.named_parameters():
        g, r = _cpu64(p.grad), ref_g[k]
        worst[k] = float((g - r).norm()) / max(float(r.norm()), 1e-3)
        if k not in zero_grad:
            margin[k] = _margin(k, g, r, {"head W in bf16": alt_g[k]})
    _record("fp32", "step", max(worst.values()) / 1e-3, max(margin.values()))
    assert max(worst.values()) < 1e-3, worst


if __name__ == "__main__":
    # pytest imports this file under its module name; import it first so that the tests fill that module's MEASURED
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import test_head_loss_classes as mod
    rc = pytest.main(["-m", "gpu", os.path.abspath(__file__), "-q", "-p", "no:cacheprovider"])
    MEASURED = mod.MEASURED
    print("%-48s %-10s %-9s %13s %13s" % ("test", "path", "output", "error/bound", "margin ratio"))
    for (test, path, output), (ratio, margin) in sorted(MEASURED.items()):
        print("%-48s %-10s %-9s %13.3g %13.3g" % (test, path, output, ratio, margin))
    sys.exit(rc)
