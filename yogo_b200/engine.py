"""Plan compiler + executor: turns a YOGO backbone (an ``nn.Sequential`` produced by a
``ModelDefn``) into a sequence of libyogo_b200 kernel launches, forward and backward.

This replaces what ``self.model(x)`` + autograd + cuDNN do in the reference
(/root/reference/yogo/model.py:275, model_defns.py:68-77).  PyTorch is used for memory
(tensors, caching allocator), streams and RNG only; every FLOP runs in our CUDA kernels.

Data layout in HBM: activations NHWC in ``compute_dtype`` (bf16 by default, fp32 for the
tight-parity path); parameters stay fp32 OIHW ``nn.Parameter``s exactly as in the reference
state_dict; the prediction tensor is fp32 NCHW (N, 5+C, Sy, Sx) as the reference returns it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import nn

from . import _lib as L


@dataclass
class ConvBlock:
    conv: nn.Conv2d
    bn: Optional[nn.BatchNorm2d]
    act: int
    p_drop: float
    cin: int
    cout: int
    ksize: int
    stride: int
    drop: Optional[nn.Dropout2d] = None


@dataclass
class Plan:
    blocks: List[ConvBlock]
    head: nn.Conv2d
    params: List[nn.Parameter]  # in the order grads are returned


def _unsupported(what: str) -> NotImplementedError:
    return NotImplementedError(
        f"yogo_b200: {what} cannot be compiled to the sm_100a kernel plan (supported: Conv2d 3x3 pad 1 / 1x1 "
        "pad 0, stride 1|2, BatchNorm2d, LeakyReLU(0.01), SiLU, Dropout2d, final 1x1 Conv2d head)"
    )


def _check_conv(conv: nn.Conv2d) -> Tuple[int, int]:
    k = conv.kernel_size
    if k[0] != k[1] or k[0] not in (1, 3):
        raise _unsupported(f"Conv2d kernel_size {k}")
    s = conv.stride
    if s[0] != s[1] or s[0] not in (1, 2):
        raise _unsupported(f"Conv2d stride {s}")
    pad = conv.padding
    if isinstance(pad, str) or tuple(pad) != (k[0] // 2, k[0] // 2):
        raise _unsupported(f"Conv2d padding {pad} with kernel {k}")
    if tuple(conv.dilation) != (1, 1) or conv.groups != 1 or conv.padding_mode != "zeros":
        raise _unsupported("dilated / grouped / non-zero-padded Conv2d")
    return k[0], s[0]


def compile_plan(model: nn.Module) -> Plan:
    if not isinstance(model, nn.Sequential) or len(model) < 2:
        raise _unsupported(f"backbone of type {type(model).__name__}")
    children = list(model.children())
    head = children[-1]
    if not isinstance(head, nn.Conv2d) or head.kernel_size != (1, 1) or head.stride != (1, 1) or head.bias is None:
        raise _unsupported("a backbone whose last module is not a biased 1x1 Conv2d head")
    blocks: List[ConvBlock] = []
    params: List[nn.Parameter] = []
    for child in children[:-1]:
        mods = list(child.children()) if isinstance(child, nn.Sequential) else [child]
        if not mods or not isinstance(mods[0], nn.Conv2d):
            raise _unsupported(f"block starting with {type(mods[0]).__name__ if mods else 'nothing'}")
        conv = mods[0]
        k, s = _check_conv(conv)
        bn, act, p, drop = None, L.ACT_NONE, 0.0, None
        stage = 1  # 1: expect bn/act/drop, 2: after bn, 3: after act, 4: after drop
        for m in mods[1:]:
            if isinstance(m, nn.BatchNorm2d) and stage == 1:
                if not (m.affine and m.track_running_stats):
                    raise _unsupported("BatchNorm2d without affine/running stats")
                if m.momentum is None:
                    raise _unsupported("BatchNorm2d(momentum=None)")
                bn, stage = m, 2
            elif isinstance(m, nn.LeakyReLU) and stage <= 2:
                if abs(m.negative_slope - 0.01) > 1e-12:
                    raise _unsupported(f"LeakyReLU slope {m.negative_slope}")
                act, stage = L.ACT_LRELU, 3
            elif isinstance(m, nn.SiLU) and stage <= 2:
                act, stage = L.ACT_SILU, 3
            elif isinstance(m, nn.Dropout2d) and stage <= 3:
                p, stage, drop = float(m.p), 4, m
            elif isinstance(m, nn.Identity):
                continue
            else:
                raise _unsupported(f"module {type(m).__name__} at this position")
        blocks.append(ConvBlock(conv, bn, act, p, conv.in_channels, conv.out_channels, k, s, drop))
        params.append(conv.weight)
        if conv.bias is not None:
            params.append(conv.bias)
        if bn is not None:
            params += [bn.weight, bn.bias]
    params += [head.weight, head.bias]
    return Plan(blocks, head, params)


def _out_hw(h: int, w: int, k: int, s: int) -> Tuple[int, int]:
    pad = k // 2
    return (h + 2 * pad - k) // s + 1, (w + 2 * pad - k) // s + 1


def _fwd_ep(scale=None, shift=None, act=L.ACT_NONE, dropscale=None, stats=None, preact=None,
            actmask=None) -> L.FwdEpilogue:
    return L.FwdEpilogue(L.ptr(scale), L.ptr(shift), act, L.ptr(dropscale), L.ptr(stats), L.ptr(preact),
                         L.ptr(actmask))


def _f32(t: torch.Tensor) -> torch.Tensor:
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class Runner:
    """Executes a Plan.  One instance per YOGO module; stateless between calls except for
    scratch buffers."""

    def __init__(self, owner):
        self.owner = owner  # the YOGO module
        self.plan = compile_plan(owner.model)
        self.drop_keep_override: Optional[Dict[int, torch.Tensor]] = None  # tests inject masks here
        # data-parallel trainer plumbing (yogo_b200.train): parameter gradients are written
        # straight into views of a flat bucket, and a callback fires as each one is enqueued
        self.grad_views: Optional[Dict[int, torch.Tensor]] = None
        self.on_grad_ready = None
        # uint8 input normalisation fused into the first layer: the network sees x * input_scale (1/255 = the `/ 255` of
        # the reference's datasets, yogo_dataset.py:280-283, image_path_dataset.py:71-73) without an fp32 copy of the image
        self.input_scale: Optional[float] = None

    # ---------------------------------------------------------------- helpers
    def _zeros64(self, n: int, dev) -> torch.Tensor:
        a = getattr(self, "_arena64", None)
        if a is not None and a.device == dev and self._arena64_pos + n <= a.numel():
            out = a[self._arena64_pos:self._arena64_pos + n]
            self._arena64_pos += n
            return out
        return torch.zeros(n, dtype=torch.float64, device=dev)

    def _step_randoms(self, N: int, device, want_grad: bool) -> Dict[int, torch.Tensor]:
        """Dropout2d keep-scales of every training-mode Dropout2d block and the `num_batches_tracked += 1` of every
        training-mode BatchNorm, in ONE launch (csrc/input.cu: Philox keyed by a seed drawn once from torch's generator and a
        device-side call counter, so CUDA-graph replays draw fresh masks).  The mask values cannot match the reference's
        draw; the distribution does."""
        lib = L.lib()
        blocks = [(i, b) for i, b in enumerate(self.plan.blocks) if b.p_drop > 0 and b.drop is not None and b.drop.training
                  and not (self.drop_keep_override is not None and i in self.drop_keep_override)]
        bns = [b.bn for b in self.plan.blocks if b.bn is not None and b.bn.training and b.bn.num_batches_tracked is not None
               and b.bn.num_batches_tracked.is_cuda]
        key = (N, str(device), tuple(i for i, _ in blocks), tuple(float(b.p_drop) for _, b in blocks),
               tuple(b.num_batches_tracked.data_ptr() for b in bns))
        st = getattr(self, "_rand_state", None)
        if st is None or st["key"] != key:
            import struct
            offs, rows, off = {}, [], 0
            for i, b in blocks:
                cnt = N * b.cout
                offs[i] = (off, cnt, b.cout)
                rows.append([off, cnt, struct.unpack("i", struct.pack("f", float(b.p_drop)))[0], 0])
                off += cnt
            table = torch.tensor(rows if rows else [[0, 0, 0, 0]], dtype=torch.int32).to(device)
            # derived from torch's seed without consuming its generator (reproducible under torch.manual_seed; runners differ)
            Runner._seed_counter = getattr(Runner, "_seed_counter", 0) + 1
            seed = ((torch.initial_seed() * 6364136223846793005 + 1442695040888963407 * Runner._seed_counter) % (2 ** 62)) \
                if (st is None) else st["seed"]
            state = st["state"] if (st is not None and st["state"].device == torch.device(device)) else \
                torch.tensor([seed, 0, 0], dtype=torch.int64).to(device)
            ptrs = torch.tensor([b.num_batches_tracked.data_ptr() for b in bns] or [0], dtype=torch.int64).to(device)
            st = {"key": key, "offs": offs, "table": table, "total": off, "seed": seed, "state": state, "ptrs": ptrs, "nbn": len(bns)}
            self._rand_state = st
        out = torch.empty(max(st["total"], 1), dtype=torch.float32, device=device)
        if st["total"] > 0 or st["nbn"] > 0:
            L.check(lib.yg_dropout_scales(out.data_ptr(), st["table"].data_ptr(), len(st["offs"]), st["total"],
                                          st["state"].data_ptr(), st["ptrs"].data_ptr(), st["nbn"], L.stream()))
        self._bn_counted = {id(b) for b in bns}
        return {i: out[o:o + c].view(N, co) for i, (o, c, co) in st["offs"].items()}

    def _dropscale(self, i: int, blk: ConvBlock, N: int, device, training: bool) -> Optional[torch.Tensor]:
        if blk.p_drop <= 0 or not training:
            return None
        if self.drop_keep_override is not None and i in self.drop_keep_override:
            keep = self.drop_keep_override[i].to(device=device, dtype=torch.float32)
            return (keep / (1.0 - blk.p_drop)).contiguous()
        return self._scales[i]

    def _prep_input(self, x: torch.Tensor) -> Tuple[torch.Tensor, int]:
        if x.ndim == 3:
            x = x.unsqueeze(0)
        if x.ndim != 4:
            raise ValueError(f"expected (N,C,H,W) or (C,H,W) input, got shape {tuple(x.shape)}")
        L.require_cuda(x, "YOGO input")
        if x.dtype == torch.uint8:
            code = L.YG_U8
        else:
            if x.dtype != torch.float32:
                x = x.float()  # model.py:272-273
            code = L.YG_F32
        return x.contiguous(), code

    # ---------------------------------------------------------------- forward
    @L.on_device(lambda self, x, want_grad: x)
    def forward(self, x: torch.Tensor, want_grad: bool):
        own = self.owner
        lib = L.lib()
        st = L.stream()
        plan = self.plan
        x, x_code = self._prep_input(x)
        N, Cx, H, W = x.shape
        dev = x.device
        dt: torch.dtype = own.compute_dtype
        dcode = L.dtype_code(dt)
        if plan.blocks[0].cin != Cx:
            raise RuntimeError(f"expected input with {plan.blocks[0].cin} channels, got {Cx}")
        saved = {"x": x, "x_code": x_code, "blocks": [], "N": N, "dtype": dt}
        self._scales = self._step_randoms(N, dev, want_grad)
        # every fp64 accumulator of the step (BatchNorm statistics forward, BatchNorm sums backward) comes zeroed from one arena:
        # one fill launch per step instead of one per BatchNorm layer and direction
        need64 = (sum(4 * b.cout for b in plan.blocks if b.bn is not None)
                  if (want_grad or any(b.bn is not None and b.bn.training for b in plan.blocks)) else 0)
        self._arena64 = torch.zeros(need64, dtype=torch.float64, device=dev) if need64 else None
        self._arena64_pos = 0
        cur: Optional[torch.Tensor] = None  # NHWC activation
        h, w = H, W
        for i, blk in enumerate(plan.blocks):
            ho, wo = _out_hw(h, w, blk.ksize, blk.stride)
            bn_train = blk.bn is not None and blk.bn.training
            module_training = blk.drop.training if blk.drop is not None else False
            ds = self._dropscale(i, blk, N, dev, module_training)
            wt = _f32(blk.conv.weight)
            bias = _f32(blk.conv.bias) if blk.conv.bias is not None else None
            rec = {"in": cur, "h": h, "w": w, "ho": ho, "wo": wo, "dropscale": ds, "bn_train": bn_train}
            first_direct = i == 0 and blk.ksize == 3 and blk.cin <= 3
            rec["first_direct"] = first_direct
            in_scale = self.input_scale if (i == 0 and x_code == L.YG_U8 and self.input_scale not in (None, 1.0)) else None
            if in_scale is not None:
                # conv(x * s, W) = conv(x, W * s): the first layer runs on the raw bytes with scaled weights (144 floats)
                wt = wt * in_scale
                rec["in_scale"], rec["wt_eff"] = in_scale, wt
            if i == 0 and not first_direct:
                cur = x.permute(0, 2, 3, 1).contiguous().to(dt)  # plumbing: NCHW image -> NHWC
                rec["in"] = cur
                if in_scale is not None:
                    raise _unsupported("input_scale with a first block that is not a 3x3 conv on 1-3 input channels")
            out = torch.empty((N, ho, wo, blk.cout), dtype=dt, device=dev)

            def conv(ep: L.FwdEpilogue, y: Optional[torch.Tensor]):
                if first_direct:
                    L.check(lib.yg_conv_first_fwd(x.data_ptr(), x_code, wt.data_ptr(), L.ptr(y), dcode, N, h, w,
                                                  blk.cin, blk.cout, blk.stride, C.byref(ep), st))
                else:
                    L.check(lib.yg_conv_fwd(cur.data_ptr(), wt.data_ptr(), L.ptr(y), dcode, N, h, w, blk.cin,
                                            blk.cout, blk.ksize, blk.stride, C.byref(ep), st))

            if blk.bn is None:
                pre = None
                if want_grad and blk.act == L.ACT_SILU:
                    pre = torch.empty_like(out)
                mask = None
                if (want_grad and blk.act == L.ACT_LRELU and not first_direct and blk.cout % 32 == 0
                        and dt == torch.bfloat16):
                    # 1 sign bit per element: what the next layer's dgrad epilogue needs of this activation
                    mask = torch.empty(N * ho * wo * blk.cout // 8, dtype=torch.uint8, device=dev)
                conv(_fwd_ep(shift=bias, act=blk.act, dropscale=ds, preact=pre, actmask=mask), out)
                rec["saved"] = pre if pre is not None else out
                rec["actmask"] = mask
            else:
                bn = blk.bn
                g, b = _f32(bn.weight), _f32(bn.bias)
                if not want_grad and not bn_train:
                    # inference: BN folded into the conv epilogue, nothing else touches HBM
                    scale = torch.empty(blk.cout, dtype=torch.float32, device=dev)
                    shift = torch.empty_like(scale)
                    L.check(lib.yg_bn_fold_eval(g.data_ptr(), b.data_ptr(), bn.running_mean.data_ptr(),
                                                bn.running_var.data_ptr(), L.ptr(bias), float(bn.eps),
                                                scale.data_ptr(), shift.data_ptr(), blk.cout, st))
                    conv(_fwd_ep(scale=scale, shift=shift, act=blk.act, dropscale=ds), out)
                else:
                    mean = torch.empty(blk.cout, dtype=torch.float32, device=dev)
                    invstd, scale, shift = torch.empty_like(mean), torch.empty_like(mean), torch.empty_like(mean)
                    use_gram = first_direct and blk.cin == 1
                    if use_gram and want_grad:
                        # 9-tap Gram statistics of the image: BN statistics now, BN backward later (first_layer.cu)
                        gram = torch.empty(54, dtype=torch.float64, device=dev)
                        L.check(lib.yg_conv_first_gram(x.data_ptr(), x_code, N, h, w, blk.stride, gram.data_ptr(), st))
                        rec["gram"] = gram
                    if bn_train:
                        stats = self._zeros64(2 * blk.cout, dev)
                        y_raw = None if first_direct else torch.empty_like(out)
                        if use_gram:
                            if "gram" not in rec:
                                gram = torch.empty(54, dtype=torch.float64, device=dev)
                                L.check(lib.yg_conv_first_gram(x.data_ptr(), x_code, N, h, w, blk.stride,
                                                               gram.data_ptr(), st))
                            L.check(lib.yg_conv_first_stats_from_gram(gram.data_ptr(), wt.data_ptr(), L.ptr(bias),
                                                                      float(N * ho * wo), blk.cout, stats.data_ptr(), st))
                        else:
                            # pass 1: conv (+bias) with the plain epilogue, then one streaming pass for sum / sum of squares
                            # (cheaper than reducing inside the tensor-core epilogue, and keeps the MMAs at full rate).
                            # A direct first layer without Gram statistics (RGB input) uses `out` as the scratch copy: the
                            # stencil is recomputed with the final constants below.
                            y_stat = y_raw if y_raw is not None else out
                            conv(_fwd_ep(shift=bias), y_stat)
                            L.check(lib.yg_bn_stats(y_stat.data_ptr(), dcode, N, ho * wo, blk.cout, stats.data_ptr(), st))
                        L.check(lib.yg_bn_finalize(stats.data_ptr(), float(N * ho * wo), g.data_ptr(), b.data_ptr(),
                                                   bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                                                   float(bn.momentum), float(bn.eps), mean.data_ptr(),
                                                   invstd.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                                   blk.cout, st))
                        if id(bn) not in self._bn_counted:   # (counted by yg_dropout_scales when the buffer is on the GPU)
                            bn.num_batches_tracked += 1
                    else:
                        # BN in eval mode inside a training graph (tuning=True, model.py:69-70)
                        L.check(lib.yg_bn_fold_eval(g.data_ptr(), b.data_ptr(), bn.running_mean.data_ptr(),
                                                    bn.running_var.data_ptr(), None, float(bn.eps),
                                                    scale.data_ptr(), shift.data_ptr(), blk.cout, st))
                        mean.copy_(bn.running_mean)
                        invstd.copy_(torch.rsqrt(bn.running_var + bn.eps))
                        y_raw = None if first_direct else torch.empty_like(out)
                        if y_raw is not None:
                            conv(_fwd_ep(shift=bias), y_raw)
                    if first_direct:
                        # recompute the 9-tap stencil instead of storing the raw conv output
                        sh2 = shift if bias is None else shift + bias * scale
                        conv(_fwd_ep(scale=scale, shift=sh2, act=blk.act, dropscale=ds), out)
                        rec["fwd_shift"] = bias
                    else:
                        mask = None
                        if want_grad and blk.act == L.ACT_LRELU and blk.cout % 32 == 0 and dt == torch.bfloat16:
                            mask = torch.empty(N * ho * wo * blk.cout // 8, dtype=torch.uint8, device=dev)
                        L.check(lib.yg_bn_act_apply(y_raw.data_ptr(), out.data_ptr(), dcode, N, ho * wo, blk.cout,
                                                    scale.data_ptr(), shift.data_ptr(), blk.act, L.ptr(ds), L.ptr(mask), st))
                        rec["actmask"] = mask
                    rec.update(saved=y_raw, mean=mean, invstd=invstd, scale=scale, shift=shift, gamma=g)
            rec["out"] = out
            saved["blocks"].append(rec)
            cur = out
            h, w = ho, wo
        # head
        D = plan.head.out_channels
        nc = D - 5
        outp = torch.empty((N, D, h, w), dtype=torch.float32, device=dev)
        t_raw = torch.empty((N, h, w, D), dtype=torch.float32, device=dev) if want_grad else None
        hw_ = _f32(plan.head.weight)
        hb_ = _f32(plan.head.bias)
        hc = own._hc
        cxs = own._Cxs if own._Cxs.is_cuda and tuple(own._Cxs.shape) == (h, w) else None
        cys = own._Cys if own._Cys.is_cuda and tuple(own._Cys.shape) == (h, w) else None
        if cxs is not None:
            cxs, cys = cxs.contiguous(), cys.contiguous()
        L.check(lib.yg_head_fwd(cur.data_ptr(), dcode, hw_.data_ptr(), hb_.data_ptr(), outp.data_ptr(), L.ptr(t_raw),
                                N, h, w, plan.head.in_channels, nc, hc["anchor_w"], hc["anchor_h"],
                                hc["width_multiplier"], hc["height_multiplier"],
                                1 if own.inference else 0, L.ptr(cxs), L.ptr(cys), st))
        saved.update(t_raw=t_raw, head_in=cur, Sy=h, Sx=w, nc=nc,
                     consts=(hc["anchor_w"], hc["anchor_h"], hc["width_multiplier"], hc["height_multiplier"]))
        return outp, (saved if want_grad else None)

    # ---------------------------------------------------------------- backward
    @L.on_device(lambda self, saved, dpred, **kw: dpred)
    def backward(self, saved, dpred: torch.Tensor, want_params: bool = True,
                 want_input: bool = False) -> Tuple[List[Optional[torch.Tensor]], Optional[torch.Tensor]]:
        """Gradients of the parameters (in plan order; all of them, or none with want_params=False: nothing that only
        produces parameter gradients runs then) and, with want_input, of the fp32 input as (N, Cin, H, W)."""
        own = self.owner
        lib = L.lib()
        st = L.stream()
        plan = self.plan
        N, dt = saved["N"], saved["dtype"]
        dcode = L.dtype_code(dt)
        dev = dpred.device
        clip = float(own._clip_value_f)
        recs = saved["blocks"]
        grads: Dict[int, torch.Tensor] = {}
        dpred = dpred.contiguous().float()
        views = self.grad_views or {}
        dx: Optional[torch.Tensor] = None

        def gbuf(p: torch.Tensor) -> torch.Tensor:
            v = views.get(id(p))
            return v if v is not None else torch.empty(p.shape, dtype=torch.float32, device=dev)

        def done(*ps):
            if self.on_grad_ready is not None:
                for p in ps:
                    if p is not None:
                        self.on_grad_ready(p)

        def bwd_ep(i: int) -> Tuple[Optional[L.BwdEpilogue], Optional[torch.Tensor]]:
            """epilogue turning d(block i output) into d(conv i output) / d(BN i output)."""
            blk, rec = plan.blocks[i], recs[i]
            if rec["first_direct"]:
                return None, None  # handled inside yg_conv_first_bwd (recomputation)
            sums = None
            if blk.bn is not None and rec.get("actmask") is not None:
                # LeakyReLU after BatchNorm with a recorded sign mask: the producer only applies the activation backward
                # (sign(out) = sign(BN output)); sum(g), sum(g*xhat) come from one streaming pass (yg_bn_bwd_sums)
                ep = L.BwdEpilogue(rec["out"].data_ptr(), blk.act, L.ptr(rec["dropscale"]), None, None, None, None, None,
                                   rec["actmask"].data_ptr())
            elif blk.bn is not None:
                # SiLU (or LeakyReLU without a mask) after BatchNorm: the epilogue recomputes the BN output from the saved raw
                # conv output.  With 8-channel-aligned rows the two BN sums come from the streaming pass (yg_bn_bwd_sums),
                # which keeps the epilogue on its straight-line path; otherwise it reduces them itself.
                if blk.cout % 8 != 0:
                    sums = self._zeros64(2 * blk.cout, dev)
                ep = L.BwdEpilogue(rec["saved"].data_ptr(), blk.act, L.ptr(rec["dropscale"]),
                                   rec["scale"].data_ptr(), rec["shift"].data_ptr(), rec["mean"].data_ptr(),
                                   rec["invstd"].data_ptr(), L.ptr(sums))
            else:
                sv = rec["saved"] if blk.act != L.ACT_NONE else None
                # d(bias) of this block comes from its own wgrad call (a ones column in the tcgen05 kernel)
                ep = L.BwdEpilogue(L.ptr(sv), blk.act, L.ptr(rec["dropscale"]), None, None, None, None, L.ptr(sums),
                                   L.ptr(rec.get("actmask")))
            return ep, sums

        # ---- head
        head = plan.head
        Cl = head.in_channels
        Sy, Sx, nc = saved["Sy"], saved["Sx"], saved["nc"]
        aw, ah, wm, hm = saved["consts"]
        if own.inference:
            # the class planes of the output are softmax probabilities: turn their gradient into the logits' gradient
            dlogit = torch.empty_like(dpred)
            L.check(lib.yg_head_softmax_bwd(dpred.data_ptr(), saved["t_raw"].data_ptr(), dlogit.data_ptr(), N, Sy, Sx,
                                            nc, st))
            dpred = dlogit
        last = len(plan.blocks) - 1
        ep, sums = bwd_ep(last)
        g = torch.empty((N, Sy, Sx, Cl), dtype=dt, device=dev)
        dw_h = gbuf(head.weight) if want_params else None
        db_h = gbuf(head.bias) if want_params else None
        nbytes = lib.yg_head_bwd_workspace(N, Sy, Sx, Cl, nc)
        ws = L.workspace.get("head_bwd", nbytes, dev)
        L.check(lib.yg_head_bwd(dpred.data_ptr(), saved["t_raw"].data_ptr(), saved["head_in"].data_ptr(),
                                _f32(head.weight).data_ptr(), g.data_ptr(), dcode, L.ptr(dw_h), L.ptr(db_h),
                                N, Sy, Sx, Cl, nc, aw, ah, wm, hm, C.byref(ep) if ep is not None else None, clip,
                                ws.data_ptr(), nbytes, st))
        if want_params:
            grads[id(head.weight)] = dw_h
            grads[id(head.bias)] = db_h
            done(head.weight, head.bias)

        # ---- conv blocks, last to first
        for i in range(last, -1, -1):
            blk, rec = plan.blocks[i], recs[i]
            h, w, ho, wo = rec["h"], rec["w"], rec["ho"], rec["wo"]
            wt = rec.get("wt_eff") if rec.get("wt_eff") is not None else _f32(blk.conv.weight)
            in_scale = rec.get("in_scale")
            # W_eff = W * s: dL/dW = s * dL/dW_eff, and clamp(s * g, c) = s * clamp(g, c / s)
            clip_w = clip / in_scale if (in_scale and clip > 0) else clip

            def reclamp(*ts):   # the kernels clamp every output of a call with one bound: restore the true one for the others
                if in_scale and clip > 0:
                    for t in ts:
                        if t is not None:
                            t.clamp_(-clip, clip)
            dw = gbuf(blk.conv.weight) if want_params else None
            db = gbuf(blk.conv.bias) if (want_params and blk.conv.bias is not None) else None
            if rec["first_direct"]:
                x, x_code = saved["x"], saved["x_code"]
                nb = lib.yg_conv_first_bwd_workspace(blk.cin, blk.cout)
                ws = L.workspace.get("first_bwd", nb, dev)
                m1 = m2 = None
                bn_train = blk.bn is not None and rec["bn_train"]
                if blk.bn is not None and "gram" in rec:
                    # one pass over (da, image): P = sum g*x_t, Sg = sum g; everything else in closed form
                    P = torch.empty(blk.cout * 9, dtype=torch.float32, device=dev)
                    Sg = torch.empty(blk.cout, dtype=torch.float32, device=dev)
                    epp = L.BwdEpilogue(None, blk.act, L.ptr(rec["dropscale"]), rec["scale"].data_ptr(),
                                        rec["shift"].data_ptr(), rec["mean"].data_ptr(), rec["invstd"].data_ptr(), None)
                    if want_params or bn_train:
                        L.check(lib.yg_conv_first_bwd(x.data_ptr(), x_code, wt.data_ptr(), g.data_ptr(), dcode, N, h, w,
                                                      blk.cin, blk.cout, blk.stride, C.byref(epp),
                                                      L.ptr(rec.get("fwd_shift")), None, None, P.data_ptr(), Sg.data_ptr(),
                                                      0.0, ws.data_ptr(), nb, st))
                    if want_input:
                        if bn_train:
                            m1 = torch.empty(blk.cout, dtype=torch.float32, device=dev)
                            m2 = torch.empty_like(m1)
                            L.check(lib.yg_conv_first_bn_means(P.data_ptr(), Sg.data_ptr(), wt.data_ptr(),
                                                               L.ptr(rec.get("fwd_shift")), rec["mean"].data_ptr(),
                                                               rec["invstd"].data_ptr(), float(N * ho * wo), blk.cout,
                                                               m1.data_ptr(), m2.data_ptr(), st))
                        dx = self._first_dgrad(saved, blk, rec, wt, g, epp, rec.get("fwd_shift"), m1, m2)
                    if not want_params:
                        continue
                    dgam = gbuf(blk.bn.weight)
                    dbet = gbuf(blk.bn.bias)
                    L.check(lib.yg_conv_first_bwd_finalize(P.data_ptr(), Sg.data_ptr(), rec["gram"].data_ptr(),
                                                           wt.data_ptr(), L.ptr(rec.get("fwd_shift")),
                                                           rec["gamma"].data_ptr(), rec["mean"].data_ptr(),
                                                           rec["invstd"].data_ptr(), float(N * ho * wo),
                                                           1 if rec["bn_train"] else 0, clip_w, blk.cout, dw.data_ptr(),
                                                           L.ptr(db), dgam.data_ptr(), dbet.data_ptr(), st))
                    if in_scale:
                        dw.mul_(in_scale)
                        reclamp(db, dgam, dbet)
                    grads[id(blk.bn.weight)] = dgam
                    grads[id(blk.bn.bias)] = dbet
                    grads[id(blk.conv.weight)] = dw
                    if db is not None:
                        grads[id(blk.conv.bias)] = db
                    done(blk.conv.weight, blk.conv.bias, blk.bn.weight, blk.bn.bias)
                    continue
                if blk.bn is not None:
                    if want_params or bn_train:
                        sums = self._zeros64(2 * blk.cout, dev)
                        ep1 = L.BwdEpilogue(None, blk.act, L.ptr(rec["dropscale"]), rec["scale"].data_ptr(),
                                            rec["shift"].data_ptr(), rec["mean"].data_ptr(), rec["invstd"].data_ptr(),
                                            sums.data_ptr())
                        L.check(lib.yg_conv_first_bwd(x.data_ptr(), x_code, wt.data_ptr(), g.data_ptr(), dcode, N, h, w,
                                                      blk.cin, blk.cout, blk.stride, C.byref(ep1),
                                                      L.ptr(rec.get("fwd_shift")), None, None, None, None, clip, None, 0, st))
                    if want_params:
                        dgam = gbuf(blk.bn.weight)
                        dbet = gbuf(blk.bn.bias)
                        L.check(lib.yg_bn_bwd_apply(None, None, dcode, N, ho * wo, blk.cout, sums.data_ptr(),
                                                    rec["gamma"].data_ptr(), rec["mean"].data_ptr(),
                                                    rec["invstd"].data_ptr(), dgam.data_ptr(), dbet.data_ptr(), clip,
                                                    1, st))
                        grads[id(blk.bn.weight)] = dgam
                        grads[id(blk.bn.bias)] = dbet
                    if rec["bn_train"]:
                        M = float(N * ho * wo)
                        m1 = (sums[: blk.cout] / M).float().contiguous()
                        m2 = (sums[blk.cout :] / M).float().contiguous()
                    elif want_params:
                        m1 = torch.zeros(blk.cout, dtype=torch.float32, device=dev)
                        m2 = torch.zeros_like(m1)
                    ep2 = L.BwdEpilogue(None, blk.act, L.ptr(rec["dropscale"]), rec["scale"].data_ptr(),
                                        rec["shift"].data_ptr(), rec["mean"].data_ptr(), rec["invstd"].data_ptr(), None)
                else:
                    ep2 = L.BwdEpilogue(None, blk.act, L.ptr(rec["dropscale"]), None, None, None, None, None)
                fsh = rec.get("fwd_shift") if blk.bn is not None else (_f32(blk.conv.bias) if blk.conv.bias is not None else None)
                if want_input:
                    # running statistics: dz = scale * g' (the zero means above only serve the weight-gradient pass)
                    dx = self._first_dgrad(saved, blk, rec, wt, g, ep2, fsh, m1 if rec["bn_train"] else None,
                                           m2 if rec["bn_train"] else None)
                if not want_params:
                    continue
                L.check(lib.yg_conv_first_bwd(x.data_ptr(), x_code, wt.data_ptr(), g.data_ptr(), dcode, N, h, w,
                                              blk.cin, blk.cout, blk.stride, C.byref(ep2), L.ptr(fsh),
                                              L.ptr(m1), L.ptr(m2), dw.data_ptr(), L.ptr(db), clip_w, ws.data_ptr(), nb, st))
                if in_scale:
                    dw.mul_(in_scale)
                    reclamp(db)
                grads[id(blk.conv.weight)] = dw
                if db is not None:
                    grads[id(blk.conv.bias)] = db
                done(blk.conv.weight, blk.conv.bias, blk.bn.weight if blk.bn is not None else None,
                     blk.bn.bias if blk.bn is not None else None)
                continue
            if blk.bn is not None:
                dgam = gbuf(blk.bn.weight) if want_params else None
                dbet = gbuf(blk.bn.bias) if want_params else None
                if sums is None:
                    sums = self._zeros64(2 * blk.cout, dev)
                    L.check(lib.yg_bn_bwd_sums(g.data_ptr(), rec["saved"].data_ptr(), dcode, N, ho * wo, blk.cout,
                                               rec["mean"].data_ptr(), rec["invstd"].data_ptr(), sums.data_ptr(), st))
                L.check(lib.yg_bn_bwd_apply(g.data_ptr(), rec["saved"].data_ptr(), dcode, N, ho * wo, blk.cout,
                                            sums.data_ptr(), rec["gamma"].data_ptr(), rec["mean"].data_ptr(),
                                            rec["invstd"].data_ptr(), L.ptr(dgam), L.ptr(dbet), clip,
                                            1 if rec["bn_train"] else 0, st))
                if want_params:
                    grads[id(blk.bn.weight)] = dgam
                    grads[id(blk.bn.bias)] = dbet
            # g is now d(loss)/d(conv output of block i)
            if want_params:
                db_from_wgrad = db
                nb = lib.yg_conv_wgrad_workspace(N, h, w, blk.cin, blk.cout, blk.ksize, blk.stride)
                ws = L.workspace.get("wgrad", nb, dev)
                L.check(lib.yg_conv_wgrad(rec["in"].data_ptr(), g.data_ptr(), dw.data_ptr(), L.ptr(db_from_wgrad), dcode, N, h,
                                          w, blk.cin, blk.cout, blk.ksize, blk.stride, clip, ws.data_ptr(), nb, st))
                grads[id(blk.conv.weight)] = dw
                if db is not None:
                    grads[id(blk.conv.bias)] = db
                done(blk.conv.weight, blk.conv.bias, blk.bn.weight if blk.bn is not None else None,
                     blk.bn.bias if blk.bn is not None else None)
            if i > 0 or want_input:
                ep, sums = bwd_ep(i - 1) if i > 0 else (None, None)
                gprev = torch.empty((N, h, w, blk.cin), dtype=dt, device=dev)
                L.check(lib.yg_conv_dgrad(g.data_ptr(), wt.data_ptr(), gprev.data_ptr(), dcode, N, h, w, blk.cin,
                                          blk.cout, blk.ksize, blk.stride, C.byref(ep) if ep is not None else None, st))
                g = gprev
        if want_input and dx is None:
            dx = g.permute(0, 3, 1, 2).float().contiguous()   # plumbing: NHWC gradient of the first conv's input -> NCHW
        # gradients already written into trainer-owned views are not returned through autograd
        return [None if id(p) in views else grads.get(id(p)) for p in plan.params], dx

    def _first_dgrad(self, saved, blk: ConvBlock, rec, wt: torch.Tensor, g: torch.Tensor, ep: L.BwdEpilogue, fwd_shift,
                     m1, m2):
        """d(loss)/d(image) of a direct first block (yg_conv_first_dgrad), fp32 (N, Cin, H, W)."""
        x = saved["x"]   # fp32: a uint8 image cannot require a gradient
        N, H, W = saved["N"], rec["h"], rec["w"]
        dx = torch.empty((N, blk.cin, H, W), dtype=torch.float32, device=x.device)
        L.check(L.lib().yg_conv_first_dgrad(x.data_ptr(), wt.data_ptr(), g.data_ptr(),
                                            L.dtype_code(saved["dtype"]), N, H, W, blk.cin, blk.cout, blk.stride,
                                            C.byref(ep), L.ptr(fwd_shift), L.ptr(m1), L.ptr(m2), dx.data_ptr(),
                                            L.stream()))
        return dx


class _YOGOFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, runner: Runner, x: torch.Tensor, *params):
        out, saved = runner.forward(x, want_grad=True)
        ctx.runner = runner
        ctx.saved = saved
        ctx.x_meta = (x.shape, x.dtype)
        return out

    @staticmethod
    def backward(ctx, dpred):
        # parameter gradients are all or nothing: a frozen model skips every weight-gradient pass
        grads, dx = ctx.runner.backward(ctx.saved, dpred, want_params=any(ctx.needs_input_grad[2:]),
                                        want_input=ctx.needs_input_grad[1])
        ctx.saved = None
        if dx is not None:
            shape, dtype = ctx.x_meta
            dx = dx.reshape(shape).to(dtype)   # (C, H, W) inputs and non-fp32 float inputs, which the engine casts to fp32
        return (None, dx, *grads)


def run(runner: Runner, x: torch.Tensor) -> torch.Tensor:
    params = runner.plan.params
    need_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
    if need_grad:
        return _YOGOFunction.apply(runner, x, *params)
    out, _ = runner.forward(x, want_grad=False)
    return out
