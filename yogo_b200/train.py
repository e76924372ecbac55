"""Data-parallel training step: the hot loop of /root/reference/yogo/train.py:295-339 and the
DDP/optimizer wiring of train.py:152-159, 206-223, re-designed for one process per B200.

What the reference does with ``DistributedDataParallel`` + ``torch.optim.AdamW``:
  * DDP ctor broadcast of parameters/buffers from rank 0 (C1)            -> ``broadcast_state``
  * bucketed gradient all-reduce (SUM, / world) overlapped with backward (C3)
                                                                          -> flat fp32 buckets,
    the weight-gradient kernels write (already clamped) gradients straight into bucket views,
    ``on_grad_ready`` fires as each layer's gradient is enqueued (last layers first), and a
    complete bucket is all-reduced on a side stream while the remaining dgrad/wgrad kernels run
  * per-step buffer broadcast (C2)                                        -> dropped: only BN
    running statistics change, and they are broadcast from rank 0 on demand
    (``sync_bn_buffers``) before eval/checkpoint, which is result-equivalent because rank 0's
    statistics are what the reference checkpoints (train.py:273-288)
  * AdamW + CosineAnnealingLR (train.py:213-223)                          -> one fused kernel over
    the flat parameter buffer (csrc/optim.cu), 1/world folded into the gradient scale.
Semantics preserved: mean over ranks of clamp(local_grad, +-clip) (SURVEY.md 2.4), loss divided
by the local batch, BatchNorm with local statistics (no SyncBN).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib as L
from .model import YOGO
from .yogo_loss import YOGOLoss

FIRST_BUCKET_BYTES = 1 << 20   # DDP: first bucket 1 MiB ...
BUCKET_BYTES = 25 << 20        # ... then bucket_cap_mb = 25


class DataParallelTrainer:
    def __init__(
        self,
        net: YOGO,
        loss_fn: Optional[YOGOLoss] = None,
        lr: float = 3e-4,
        weight_decay: float = 5e-2,
        betas: Tuple[float, float] = (0.9, 0.999),
        eps: float = 1e-8,
        total_steps: Optional[int] = None,
        decay_factor: float = 10.0,
        process_group=None,
        overlap: bool = True,
    ):
        self.net = net
        self.loss_fn = loss_fn if loss_fn is not None else YOGOLoss()
        self.lr0, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.total_steps, self.decay_factor = total_steps, decay_factor
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        self.overlap = overlap
        self.step_count = 0
        self._graph = None
        self._graphs, self._graph_losses, self._static = [], [], []

        runner = net._get_runner()
        params = [p for p in runner.plan.params if p.requires_grad]
        self.params = params
        dev = params[0].device
        n = sum(p.numel() for p in params)
        self.numel = n
        # flat parameter / gradient / optimizer-state buffers; parameters become views
        self.flat_p = torch.empty(n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        # bucket layout follows gradient-ready order: head first, then blocks last -> first
        order = self._ready_order(runner)
        off = 0
        self.offsets: Dict[int, Tuple[int, int]] = {}
        for p in order:
            self.offsets[id(p)] = (off, p.numel())
            off += p.numel()
        assert off == n
        views = {}
        with torch.no_grad():
            for p in order:
                o, k = self.offsets[id(p)]
                self.flat_p[o:o + k].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[o:o + k].view_as(p)
                g = self.flat_g[o:o + k].view_as(p)
                p.grad = g
                views[id(p)] = g
        runner.grad_views = views
        # buckets: contiguous ranges of the flat buffer
        self.buckets: List[Tuple[int, int]] = []
        self.bucket_of: Dict[int, int] = {}
        start, cap = 0, FIRST_BUCKET_BYTES
        cur = 0
        for p in order:
            o, k = self.offsets[id(p)]
            self.bucket_of[id(p)] = len(self.buckets)
            cur = o + k
            if (cur - start) * 4 >= cap:
                self.buckets.append((start, cur))
                start, cap = cur, BUCKET_BYTES
        if cur > start:
            self.buckets.append((start, cur))
        self._bucket_pending = [0] * len(self.buckets)
        self._bucket_size = [0] * len(self.buckets)
        for p in order:
            self._bucket_size[self.bucket_of[id(p)]] += 1
        self.comm_stream = torch.cuda.Stream(device=dev) if (self.world > 1 and dev.type == "cuda") else None
        self._comm_events: List[torch.cuda.Event] = []
        runner.on_grad_ready = self._on_grad_ready if self.world > 1 else None

    @staticmethod
    def _ready_order(runner) -> List[torch.nn.Parameter]:
        plan = runner.plan
        order: List[torch.nn.Parameter] = [plan.head.weight, plan.head.bias]
        for blk in reversed(plan.blocks):
            order.append(blk.conv.weight)
            if blk.conv.bias is not None:
                order.append(blk.conv.bias)
            if blk.bn is not None:
                order += [blk.bn.weight, blk.bn.bias]
        return [p for p in order if p.requires_grad]

    # ------------------------------------------------------------------ distributed plumbing
    def broadcast_state(self, src: int = 0) -> None:
        """C1: every rank starts from rank `src`'s parameters and buffers."""
        if self.world == 1:
            return
        dist.broadcast(self.flat_p, src, group=self.pg)
        for b in self.net.buffers():
            if b.is_floating_point() or b.dtype in (torch.int64, torch.bool):
                t = b if b.dtype != torch.bool else b.to(torch.uint8)
                dist.broadcast(t, src, group=self.pg)
                if b.dtype == torch.bool:
                    b.copy_(t.bool())

    def sync_bn_buffers(self, src: int = 0) -> None:
        """C2-equivalent, on demand: BN running statistics of rank `src` to every rank."""
        if self.world == 1:
            return
        for name, b in self.net.named_buffers():
            if "running_" in name or "num_batches_tracked" in name:
                dist.broadcast(b, src, group=self.pg)

    def _on_grad_ready(self, p) -> None:
        bi = self.bucket_of.get(id(p))
        if bi is None:
            return
        self._bucket_pending[bi] += 1
        if self._bucket_pending[bi] == self._bucket_size[bi]:
            self._launch_bucket(bi)

    def _launch_bucket(self, bi: int) -> None:
        """All-reduce one complete bucket on the side stream while the remaining dgrad / wgrad kernels run on the main
        stream.  Only stream/event dependencies are used, so the same code runs eagerly and under CUDA-graph capture
        (the side stream joins the capture through the event wait; NCCL collectives are capturable)."""
        s, e = self.buckets[bi]
        if self.overlap and self.comm_stream is not None:
            cur = torch.cuda.current_stream()
            ev = torch.cuda.Event()
            ev.record(cur)
            self.comm_stream.wait_event(ev)
            with torch.cuda.stream(self.comm_stream):
                dist.all_reduce(self.flat_g[s:e], op=dist.ReduceOp.SUM, group=self.pg)
                done = torch.cuda.Event()
                done.record(self.comm_stream)
            self._comm_events.append(done)
        else:
            dist.all_reduce(self.flat_g[s:e], op=dist.ReduceOp.SUM, group=self.pg)

    # ------------------------------------------------------------------ one training step
    def lr_at(self, step: int) -> float:
        """CosineAnnealingLR(T_max=total_steps, eta_min=lr/decay_factor) (train.py:219-223)."""
        if not self.total_steps:
            return self.lr0
        eta_min = self.lr0 / self.decay_factor
        t = min(step, self.total_steps)
        return eta_min + (self.lr0 - eta_min) * (1 + math.cos(math.pi * t / self.total_steps)) / 2

    def forward_backward(self, imgs: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        self._bucket_pending = [0] * len(self.buckets)
        self._comm_events = []
        out = self.net(imgs)
        if isinstance(self.loss_fn, YOGOLoss):
            # the kernel already produced d(loss)/d(out): feed it to the network's backward directly (no `ones * grad` pass)
            loss, _, dout = self.loss_fn.loss_and_grad(out, labels)
            torch.autograd.backward(out, dout)
        else:
            loss, _ = self.loss_fn(out, labels)
            loss.backward()
        if self.world > 1:
            cur = torch.cuda.current_stream()
            for ev in self._comm_events:
                cur.wait_event(ev)
        return loss

    def _check_views(self) -> None:
        """`net.to()`, `.half()` or `load_state_dict(assign=True)` after construction re-allocate parameters; AdamW would
        then update a buffer the model no longer reads.  Cheap (one pointer compare per tensor), checked every step."""
        base = self.flat_p.data_ptr()
        for p in self.params:
            o, _ = self.offsets[id(p)]
            if p.data_ptr() != base + 4 * o:
                raise RuntimeError("DataParallelTrainer: a parameter no longer aliases the flat parameter buffer (the model "
                                   "was moved / cast / re-assigned after the trainer was built); build a new trainer")

    def optimizer_step(self) -> None:
        self.step_count += 1
        with torch.cuda.device(self.flat_p.device):
            self._adamw_host()

    def _adamw_host(self) -> None:
        b1, b2 = self.betas
        L.check(L.lib().yg_adamw_flat(self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.exp_avg.data_ptr(),
                                      self.exp_avg_sq.data_ptr(), self.numel, self.lr_at(self.step_count - 1),
                                      b1, b2, self.eps, self.wd, self.step_count, 1.0 / self.world, L.stream()))

    def step(self, imgs: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """zero_grad is implicit: every gradient view is overwritten by its kernel each step."""
        self._check_views()
        if self._graph is not None and imgs.shape == self._static_imgs.shape and labels.shape == self._static_labels.shape:
            return self._graph_step(imgs, labels)
        # eager path (also the ragged last batch of an epoch when a graph of the full batch shape is active)
        loss = self.forward_backward(imgs, labels)
        self.optimizer_step()
        return loss

    # ------------------------------------------------------------------ CUDA-graph replay of the whole step
    def _hyper_host(self, step_count: int) -> torch.Tensor:
        b1, b2 = self.betas
        return torch.tensor([self.lr_at(step_count - 1), b1, b2, self.eps, self.wd, 1.0 - b1 ** step_count,
                             math.sqrt(1.0 - b2 ** step_count), 1.0 / self.world], dtype=torch.float32)

    def enable_cuda_graph(self, imgs: torch.Tensor, labels: torch.Tensor, warmup: int = 2, slots: int = 1) -> None:
        """Capture forward + loss + backward (+ bucketed all-reduces) + AdamW for this input shape into one CUDA graph;
        afterwards `step` copies the batch into static buffers and replays it (launch-bound inner loop:
        ~350 kernel launches and their host-side argument marshalling collapse into one graph launch).

        `slots` > 1 captures one graph per static input buffer set (sharing one memory pool, they never run
        concurrently): `steps_from_host` then copies host batch i+1 straight into the idle slot while the graph of the
        other slot runs, so no device-to-device staging copy is needed."""
        dev = imgs.device
        self._static = [(imgs.clone(), labels.clone()) for _ in range(max(1, slots))]
        self._static_imgs, self._static_labels = self._static[0]
        self._hyper = torch.zeros(8, dtype=torch.float32, device=dev)

        def body(slot=0):
            loss = self.forward_backward(*self._static[slot])
            self._adamw_dev()
            return loss

        # warm-up on a side stream (allocator pools, NCCL communicator and channel setup, library caches); parameters,
        # optimizer state, module buffers and the CUDA RNG stream (Dropout2d masks) are restored afterwards
        snap = self.snapshot()
        rng = torch.cuda.get_rng_state(dev)
        self._hyper.copy_(self._hyper_host(1))
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(warmup):
                body()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        # several ranks: the per-bucket NCCL all-reduces are captured on the side stream (fork / join through events), so
        # one replay runs backward with the communication overlapped and the fused AdamW behind it.  NCCL's watchdog
        # thread polls events of earlier collectives, which a capture in "global" mode would reject: thread-local mode.
        mode = "thread_local" if self.world > 1 else "global"
        self._graphs, self._graph_losses, pool = [], [], None
        for slot in range(len(self._static)):
            graph = torch.cuda.CUDAGraph()
            n0 = L.load().yg_launch_count()
            with torch.cuda.graph(graph, pool=pool, capture_error_mode=mode):
                loss = body(slot)
            self.graph_launches = int(L.load().yg_launch_count() - n0)  # our kernels inside one replay
            pool = graph.pool()
            self._graphs.append(graph)
            self._graph_losses.append(loss)
        self.restore(snap)
        torch.cuda.set_rng_state(rng, dev)
        torch.cuda.synchronize()
        self._graph = self._graphs[0]

    def snapshot(self):
        """Copies of the step count, parameters, gradients, optimizer state and module buffers, for `restore`."""
        return (self.step_count, [t.clone() for t in (self.flat_p, self.flat_g, self.exp_avg, self.exp_avg_sq)],
                [b.clone() for b in self.net.buffers()])

    def restore(self, snap) -> None:
        """Puts back what `snapshot` copied (stream-ordered copies on the current stream)."""
        self.step_count = snap[0]
        for t, v in zip((self.flat_p, self.flat_g, self.exp_avg, self.exp_avg_sq), snap[1]):
            t.copy_(v)
        for b, v in zip(self.net.buffers(), snap[2]):
            b.copy_(v)

    def disable_cuda_graph(self) -> None:
        """Drop the captured graphs and the memory pool they pin.  With several ranks the graphs hold captured NCCL work and
        destroying them has been seen to block inside NCCL's cleanup: keep them until the process exits instead."""
        self._graph = None
        self._graphs, self._graph_losses = [], []
        torch.cuda.synchronize()

    def _adamw_dev(self) -> None:
        # current stream has already joined the side stream (forward_backward waits on the bucket events)
        L.check(L.lib().yg_adamw_flat_dev(self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.exp_avg.data_ptr(),
                                          self.exp_avg_sq.data_ptr(), self.numel, self._hyper.data_ptr(), L.stream()))

    def _graph_step(self, imgs: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        self._static_imgs.copy_(imgs, non_blocking=True)
        self._static_labels.copy_(labels, non_blocking=True)
        return self.step_static(0)

    def step_static(self, slot: int = 0) -> torch.Tensor:
        """Replay the graph of `slot` on whatever its static input buffers (`static_inputs(slot)`) hold."""
        self.step_count += 1
        self._hyper.copy_(self._hyper_host(self.step_count))  # 32 bytes from pageable memory: staged, race-free
        self._graphs[slot].replay()
        return self._graph_losses[slot].clone()   # callers may keep losses across steps; the graph's tensor is overwritten

    def static_inputs(self, slot: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._static[slot]

    def steps_from_host(self, batches):
        """Generator: one training step per pinned host batch `(images, labels)`, yielding the loss tensor.  In graph mode
        batch i+1 is copied host->device straight into the idle static slot on a copy stream while step i replays (the
        reference's `pin_memory` + `non_blocking` loader pattern, train.py:288-291, without a staging copy); otherwise it
        falls back to `DevicePrefetcher` + `step`."""
        if self._graph is None:
            for x, y in DevicePrefetcher(batches, self.flat_p.device):
                yield self.step(x, y)
            return
        dev = self.flat_p.device
        nslot = len(self._static)
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        copy = self._copy_stream
        cur = torch.cuda.current_stream(dev)
        free_ev = [None] * nslot
        ready_ev = [None] * nslot

        def issue(slot, batch):
            with torch.cuda.stream(copy):
                if free_ev[slot] is not None:
                    copy.wait_event(free_ev[slot])      # the replay that last read this slot has finished
                self._static[slot][0].copy_(batch[0], non_blocking=True)
                self._static[slot][1].copy_(batch[1], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
                ready_ev[slot] = ev

        def fits(batch):
            return batch is not None and tuple(batch[0].shape) == tuple(self._static_imgs.shape) and \
                tuple(batch[1].shape) == tuple(self._static_labels.shape)

        it = iter(batches)
        nxt = next(it, None)
        slot = 0
        if fits(nxt):
            ev0 = torch.cuda.Event()
            ev0.record(cur)
            free_ev = [ev0] * nslot                     # earlier work on the main stream may still read the slots
            issue(0, nxt)
        while nxt is not None:
            if not fits(nxt):
                # a batch of another shape (the ragged last batch of an epoch): eager step, no prefetch
                yield self.step(nxt[0].to(dev, non_blocking=True), nxt[1].to(dev, non_blocking=True))
                nxt = next(it, None)
                if fits(nxt):
                    ev0 = torch.cuda.Event()
                    ev0.record(cur)
                    free_ev[slot] = ev0
                    issue(slot, nxt)
                continue
            nxt2 = next(it, None)
            if fits(nxt2) and nslot > 1:
                issue((slot + 1) % nslot, nxt2)         # overlaps with the replay below
            cur.wait_event(ready_ev[slot])
            loss = self.step_static(slot)
            ev = torch.cuda.Event()
            ev.record(cur)
            free_ev[slot] = ev
            if fits(nxt2) and nslot == 1:
                issue(0, nxt2)
            yield loss
            nxt = nxt2
            slot = (slot + 1) % nslot

    def steps_from_device(self, dd, epoch: int):
        """Generator: one training step per batch of `epoch` of the device-resident dataset `dd`
        (`yogo_b200.data.DeviceResidentDataset`), yielding the loss tensor.  In graph mode (after `enable_cuda_graph`
        with `dd`'s batch shape) every full batch is one replay of a graph that draws the flips, gathers the images, builds
        the labels into the static input slot 0 and then runs the captured step; the host only stages the 32 hyper-parameter
        bytes and launches it.  The ragged last batch, and every batch without graph mode, runs eagerly through the same
        kernels."""
        dev = self.flat_p.device
        with torch.cuda.device(dev):
            dd.begin_epoch(epoch)
        graph = self._device_graph(dd) if self._graph is not None else None
        for n in dd.batch_sizes(epoch):
            if graph is not None and n == dd.batch_size:
                self._check_views()
                self.step_count += 1
                self._hyper.copy_(self._hyper_host(self.step_count))
                graph[2].replay()
                yield graph[3].clone()
            else:
                yield self.step(*dd.next_batch(n))

    def _device_graph(self, dd):
        """(dd, step graph it was captured beside, graph, loss) of `dd`'s batch step, captured on first use with the warm-up / snapshot / restore discipline
        of `enable_cuda_graph`, in the memory pool of its graphs.  `dd`'s draw counter and cursor are restored too."""
        cached = getattr(self, "_dev_graph", None)
        if cached is not None and cached[0] is dd and cached[1] is self._graphs[0]:
            return cached
        imgs, labels = self._static[0]
        if tuple(imgs.shape) != (dd.batch_size,) + tuple(dd.image_shape) or imgs.dtype != dd.image_dtype or \
                tuple(labels.shape) != (dd.batch_size, 6) + tuple(dd.grid):
            raise ValueError(f"steps_from_device: the captured step takes images {tuple(imgs.shape)} {imgs.dtype} and labels "
                             f"{tuple(labels.shape)}, the dataset's batches are ({dd.batch_size}, {dd.image_shape}) "
                             f"{dd.image_dtype} and ({dd.batch_size}, 6, {dd.grid})")
        dev = self.flat_p.device

        def body():
            dd.next_batch_into(imgs, labels)
            loss = self.forward_backward(imgs, labels)
            self._adamw_dev()
            return loss

        snap, dd_state, rng = self.snapshot(), dd.state(), torch.cuda.get_rng_state(dev)
        self._hyper.copy_(self._hyper_host(1))
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            body()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, pool=self._graphs[0].pool(), capture_error_mode="thread_local" if self.world > 1 else "global"):
            loss = body()
        self.restore(snap)
        dd.set_state(dd_state)
        torch.cuda.set_rng_state(rng, dev)
        torch.cuda.synchronize()
        self._dev_graph = (dd, self._graphs[0], graph, loss)
        return self._dev_graph

    # ------------------------------------------------------------------ checkpoint state (train.py:262-293)
    def optimizer_state_dict(self) -> Dict:
        """`torch.optim.AdamW.state_dict()` layout (what the reference stores under "optimizer_state_dict"): per-parameter
        `step` / `exp_avg` / `exp_avg_sq` in `net.parameters()` order, one param group with the current learning rate."""
        params = list(self.net.parameters())
        state = {}
        for i, p in enumerate(params):
            if id(p) not in self.offsets:
                continue
            o, k = self.offsets[id(p)]
            state[i] = {"step": torch.tensor(float(self.step_count)),
                        "exp_avg": self.exp_avg[o:o + k].view_as(p).clone(),
                        "exp_avg_sq": self.exp_avg_sq[o:o + k].view_as(p).clone()}
        group = {"lr": self.lr_at(self.step_count), "betas": self.betas, "eps": self.eps, "weight_decay": self.wd,
                 "amsgrad": False, "maximize": False, "foreach": None, "capturable": False, "differentiable": False,
                 "fused": None, "initial_lr": self.lr0, "params": list(range(len(params)))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd: Dict) -> None:
        params = list(self.net.parameters())
        steps = set()
        with torch.no_grad():
            for i, st in sd["state"].items():
                p = params[int(i)]
                if id(p) not in self.offsets:
                    continue
                o, k = self.offsets[id(p)]
                self.exp_avg[o:o + k].copy_(st["exp_avg"].reshape(-1))
                self.exp_avg_sq[o:o + k].copy_(st["exp_avg_sq"].reshape(-1))
                steps.add(int(float(st["step"])))
        if len(steps) > 1:
            raise ValueError(f"per-parameter step counts differ ({sorted(steps)}); the fused AdamW keeps one")
        if steps:
            self.step_count = steps.pop()   # drives the bias correction and the cosine schedule

    def state_dict(self) -> Dict:
        return {"step": self.step_count, "total_steps": self.total_steps,
                "optimizer_state_dict": self.optimizer_state_dict()}

    def load_state_dict(self, sd: Dict) -> None:
        self.load_optimizer_state_dict(sd["optimizer_state_dict"])
        if "step" in sd:
            self.step_count = int(sd["step"])

    def checkpoint(self, filename, model_name: str, epoch: int = 0, normalize_images: bool = False, classes=None,
                   **kwargs) -> None:
        """The reference's checkpoint dict (train.py:266-293), loadable by `YOGO.from_pth` of either implementation and by
        `torch.optim.AdamW.load_state_dict`.  BN running statistics of rank 0 are broadcast first (the per-step buffer
        broadcast of DDP, done on demand)."""
        self.sync_bn_buffers()
        if self.world > 1 and dist.get_rank(self.pg) != 0:
            return
        torch.save({"epoch": epoch, "step": self.step_count, "normalize_images": normalize_images, "classes": classes,
                    "model_name": model_name,
                    "model_state_dict": {k: v.detach().clone() for k, v in self.net.state_dict().items()},
                    "optimizer_state_dict": self.optimizer_state_dict(),
                    "model_version": getattr(self.net, "model_version", None), **kwargs}, str(filename))


class DevicePrefetcher:
    """Feeds pinned host batches to the GPU one step ahead of the consumer (what `DataLoader(pin_memory=True)` +
    `.to(device, non_blocking=True)` does in the reference's training loop, train.py:288-291, made explicit): the
    host->device copy of batch i+1 runs on a side stream while step i computes, so the copy leaves the critical path.
    Iterating yields `(images, labels)` device tensors that are safe to use on the current stream."""

    def __init__(self, batches, device):
        self.batches = iter(batches)
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self._next = None
        self._fetch()

    def _fetch(self):
        try:
            img, lab = next(self.batches)
        except StopIteration:
            self._next = None
            return
        with torch.cuda.stream(self.stream):
            x = img.to(self.device, non_blocking=True)
            y = lab.to(self.device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self._next = (x, y, ev)

    def __iter__(self):
        return self

    def __next__(self):
        if self._next is None:
            raise StopIteration
        x, y, ev = self._next
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(ev)
        x.record_stream(cur)
        y.record_stream(cur)
        self._fetch()   # the next copy overlaps with the step the caller is about to run
        return x, y
