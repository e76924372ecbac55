"""Sharded device-resident stores (a dataset larger than one GPU): the placement decision and the collective teardown
protocol on the CPU (the latter with a fake library); on a B200 the peer gather kernel against torch indexing +
flip_batch with local allocations standing in for the shards; on boxes with several GPUs the torchrun check
tests/ddp_sharded_dataset_check.py (sharded against replicated batches, training and teardown)."""
import gc
import os
import subprocess
import sys

import pytest
import torch

from yogo_b200.data.device_dataset import ShardMemory, placement

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GiB = 1 << 30


# ----------------------------------------------------------------------------- CPU: placement
ONE_HOST = [("a", "boot-a")] * 4
TWO_HOSTS = [("a", "boot-a")] * 2 + [("b", "boot-b")] * 2


@pytest.mark.parametrize("full,shard,free,reserve,hosts,expect", [
    (10 * GiB, 3 * GiB, [20 * GiB] * 4, [8 * GiB] * 4, ONE_HOST, "replicated"),           # fits everywhere
    (10 * GiB, 3 * GiB, [20 * GiB] * 4, [8 * GiB] * 4, TWO_HOSTS, "replicated"),          # fits: hosts do not matter
    (10 * GiB, 3 * GiB, [20 * GiB, 20 * GiB, 17 * GiB, 20 * GiB], [8 * GiB] * 4, ONE_HOST, "sharded"),  # one rank short
    (10 * GiB, 3 * GiB, [12 * GiB] * 4, [8 * GiB] * 4, ONE_HOST, "sharded"),
    (10 * GiB, 3 * GiB, [20 * GiB] * 4, [8 * GiB, 8 * GiB, 8 * GiB, 15 * GiB], ONE_HOST, "sharded"),   # per-rank reserve
    (10 * GiB, 3 * GiB, [12 * GiB] * 4, [8 * GiB] * 4, TWO_HOSTS, "ranks 0-1 on host a, 2-3 on host b"),
    (10 * GiB, 3 * GiB, [10 * GiB] * 4, [8 * GiB] * 4, ONE_HOST, "does not fit either"),     # nothing fits
    (10 * GiB, 3 * GiB, [12 * GiB, 12 * GiB, 10 * GiB, 12 * GiB], [8 * GiB] * 4, ONE_HOST, "rank 2 has"),
    (10 * GiB, 10 * GiB, [12 * GiB], [8 * GiB], [None], "kept for training"),                # world 1 never shards
    (10 * GiB, 10 * GiB, [18 * GiB], [8 * GiB], [None], "replicated"),
])
def test_placement(full, shard, free, reserve, hosts, expect):
    if expect in ("replicated", "sharded"):
        assert placement(full, shard, free, reserve, hosts) == expect
        return
    with pytest.raises(ValueError) as e:
        placement(full, shard, free, reserve, hosts)
    msg = str(e.value)
    assert expect in msg and f"needs {full} bytes" in msg, msg
    if len(free) > 1:
        assert str(shard) in msg and str(min(free)) in msg, msg


def test_world_one_raises_the_capacity_message():
    with pytest.raises(ValueError, match=r"needs 100 bytes .* but the device has 150 bytes free .* of which 60 are kept"):
        placement(100, 10, [150], [60], [None])


# ----------------------------------------------------------------------------- CPU: teardown protocol (fake library)
class FakeLib:
    def __init__(self, log):
        self.log = log
        self.next = 0x7000

    def yg_dd_shard_alloc(self, nbytes, pref):
        pref._obj.value = 0x1000
        self.log.append(("alloc", nbytes))
        return 0

    def yg_dd_shard_export(self, ptr, buf):
        buf.value = b"H%d" % ptr
        self.log.append(("export", ptr))
        return 0

    def yg_dd_shard_open(self, handle, pref):
        self.next += 0x100
        pref._obj.value = self.next
        self.log.append(("open", self.next))
        return 0

    def yg_dd_shard_close(self, ptr):
        self.log.append(("close", ptr))
        return 0

    def yg_dd_shard_free(self, ptr):
        self.log.append(("free", ptr))
        return 0


def _mem(log):
    return ShardMemory(FakeLib(log), 4096, barrier=lambda: log.append(("barrier",)),
                       synchronize=lambda: log.append(("sync",)))


def test_close_is_barrier_close_imports_barrier_free_own():
    log = []
    mem = _mem(log)
    assert mem.export().startswith(b"H4096")
    a, b = mem.open(b"peer1"), mem.open(b"peer2")
    log.clear()
    mem.close()
    assert log == [("sync",), ("barrier",), ("close", b), ("close", a), ("barrier",), ("free", 0x1000)]
    log.clear()
    mem.close()                      # a second close does nothing
    del mem
    gc.collect()
    assert log == []


def test_collected_without_close_closes_imports_and_never_frees():
    log = []
    mem = _mem(log)
    mem.export()
    mem.open(b"peer1")
    log.clear()
    with pytest.warns(UserWarning, match="without close"):
        del mem
        gc.collect()
    assert [e[0] for e in log] == ["sync", "close"]


def test_failed_build_frees_directly_before_sharing_and_by_protocol_after():
    log = []
    _mem(log).release_after_failed_build()
    assert [e[0] for e in log] == ["alloc", "free"]
    # this rank's export succeeded but another rank's did not: nothing was shared, so no barrier may be entered
    log.clear()
    mem = _mem(log)
    mem.export()
    mem.release_after_failed_build()
    assert [e[0] for e in log] == ["alloc", "export", "free"]
    # every rank exported (mark_shared on all of them), then mapping failed somewhere: every rank runs the protocol
    log.clear()
    mem = _mem(log)
    mem.export()
    mem.mark_shared()
    mem.open(b"peer1")
    mem.release_after_failed_build()
    assert [e[0] for e in log] == ["alloc", "export", "open", "sync", "barrier", "close", "barrier", "free"]


def test_failed_export_frees_without_barrier():
    log = []
    lib = FakeLib(log)

    def fail(ptr, buf):
        log.append(("export failed",))
        raise RuntimeError("cudaIpcGetMemHandle failed")

    lib.yg_dd_shard_export = fail
    mem = ShardMemory(lib, 4096, barrier=lambda: log.append(("barrier",)), synchronize=lambda: log.append(("sync",)))
    with pytest.raises(RuntimeError):
        mem.export()
    assert not mem.shared
    mem.release_after_failed_build()
    assert [e[0] for e in log] == ["alloc", "export failed", "free"]


def test_failed_allocation_leaves_nothing_to_release():
    log = []
    lib = FakeLib(log)

    def fail(nbytes, pref):
        raise RuntimeError("cudaMalloc failed")

    lib.yg_dd_shard_alloc = fail
    import warnings
    with warnings.catch_warnings(record=True) as seen:
        warnings.simplefilter("always")
        try:
            ShardMemory(lib, 4096, barrier=lambda: log.append(("barrier",)), synchronize=lambda: log.append(("sync",)))
        except RuntimeError:
            pass
        else:
            raise AssertionError("the failed allocation did not raise")
        gc.collect()
    assert log == [] and not [w for w in seen if "without close" in str(w.message)], (log, [str(w.message) for w in seen])


# ----------------------------------------------------------------------------- GPU: the peer gather kernel
def _gather_peers(shards, shard_items, out, table, flags, stride, n, C, H, W, dtype):
    from yogo_b200 import _lib as L
    ptrs = torch.tensor([s.data_ptr() for s in shards], dtype=torch.int64, device=DEV)
    rc = L.lib().yg_dd_gather_images_peers(ptrs.data_ptr(), shard_items, out.data_ptr(), L.dtype_code(dtype),
                                           table.data_ptr(), flags.data_ptr(), stride, n, C, H, W, L.stream())
    torch.cuda.synchronize()
    return rc


def _expected(store, idx, h, v):
    from yogo_b200.data import flip_batch
    x = store[torch.tensor(idx, device=DEV)]
    y = torch.zeros((len(idx), 6, 2, 3), device=DEV)
    return flip_batch(x, y, h, v)[0]


def _same(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


def _check(W_shards, n_items, C, H, W, dtype, N, seed):
    g = torch.Generator().manual_seed(seed)
    if dtype == torch.uint8:
        store = torch.randint(0, 256, (n_items, C, H, W), dtype=torch.uint8, generator=g).to(DEV)
    else:
        store = torch.randn((n_items, C, H, W), generator=g).to(DEV)
    shard_items = -(-n_items // W_shards)
    assert n_items % shard_items != 0          # the last shard is partial
    shards = [store[i:i + shard_items].clone() for i in range(0, n_items, shard_items)]
    assert len(shards) == W_shards
    # two batches per table, stride > N; batch 1 hits every shard's first slot and the last slot
    stride = N + 3
    b1 = [s * shard_items for s in range(W_shards)] + [n_items - 1]
    b1 += torch.randint(0, n_items, (N - len(b1),), generator=g).tolist()
    b0 = torch.randint(0, n_items, (N,), generator=g).tolist()
    table = torch.tensor(b0 + [0] * 3 + b1 + [0] * 3, dtype=torch.int32, device=DEV)
    pad = 64
    fill = 0xA5 if dtype == torch.uint8 else float("nan")
    for batch, idx in ((0, b0), (1, b1)):
        for h in (0, 1):
            for v in (0, 1):
                flags = torch.tensor([h, v, batch, 0], dtype=torch.int32, device=DEV)
                buf = torch.full((2 * pad + N * C * H * W,), fill, dtype=dtype, device=DEV)
                out = buf[pad:pad + N * C * H * W].view(N, C, H, W)
                assert _gather_peers(shards, shard_items, out, table, flags, stride, N, C, H, W, dtype) == 0
                assert _same(out, _expected(store, idx, bool(h), bool(v))), (W_shards, C, H, W, dtype, batch, h, v)
                for m in (buf[:pad], buf[-pad:]):
                    assert (m == 0xA5).all() if dtype == torch.uint8 else m.isnan().all()


@pytest.mark.gpu
@pytest.mark.parametrize("W_shards", [2, 3, 8])
@pytest.mark.parametrize("C,H,W,dtype", [
    (1, 20, 64, torch.uint8),      # 16-byte vectors
    (3, 13, 40, torch.uint8),      # 8-byte vectors
    (1, 9, 37, torch.uint8),       # odd width: bytes
    (3, 7, 24, torch.float32),     # 4-float vectors
    (1, 11, 37, torch.float32),    # odd width: floats
])
def test_gather_peers_bit_identical(W_shards, C, H, W, dtype):
    _check(W_shards, 5 * W_shards - 1, C, H, W, dtype, 12, seed=W_shards * 100 + W)


@pytest.mark.gpu
def test_gather_peers_full_size_batch():
    _check(8, 70, 1, 772, 1032, torch.uint8, 64, seed=1)


@pytest.mark.gpu
def test_gather_peers_argument_checks():
    from yogo_b200 import _lib as L
    shards = [torch.zeros((4, 1, 8, 16), dtype=torch.uint8, device=DEV) for _ in range(2)]
    out = torch.empty((4, 1, 8, 16), dtype=torch.uint8, device=DEV)
    table = torch.zeros(8, dtype=torch.int32, device=DEV)
    flags = torch.zeros(4, dtype=torch.int32, device=DEV)
    ok = dict(shard_items=4, stride=4, n=4, C=1, dtype=torch.uint8)

    def call(**kw):
        a = {**ok, **kw}
        return _gather_peers(shards, a["shard_items"], out, table, flags, a["stride"], a["n"], a["C"], 8, 16, a["dtype"])

    assert call() == 0
    for bad in (dict(stride=3), dict(C=2), dict(shard_items=0), dict(dtype=torch.bfloat16)):
        assert call(**bad) != 0, bad
        assert "dd_gather_images_peers" in L.load().yg_last_error().decode()
    rc = L.lib().yg_dd_gather_images_peers(None, 4, out.data_ptr(), L.YG_U8, table.data_ptr(), flags.data_ptr(), 4, 4, 1,
                                           8, 16, L.stream())
    assert rc != 0
    rc = L.lib().yg_dd_gather_images_peers(out.data_ptr(), 4, out.data_ptr(), L.YG_U8, table.data_ptr(), flags.data_ptr(),
                                           1 << 30, 1 << 30, 3, 1024, 16, L.stream())
    assert rc != 0 and "too many rows" in L.load().yg_last_error().decode()


# ----------------------------------------------------------------------------- GPU: shard memory on one device
@pytest.mark.gpu
def test_shard_memory_view_write_read_and_free():
    """A yg_dd_shard_alloc buffer: the tensor view the build writes through, a read by the peer gather kernel, the
    export, and the free giving the memory back."""
    from yogo_b200 import _lib as L
    from yogo_b200.data.device_dataset import _CudaBuffer
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(DEV)[0]
    n, C, H, W = 40, 1, 772, 1032
    nbytes = n * C * H * W
    mem = ShardMemory(L.lib(), nbytes, barrier=lambda: None, synchronize=torch.cuda.synchronize)
    assert free0 - torch.cuda.mem_get_info(DEV)[0] >= nbytes
    view = torch.as_tensor(_CudaBuffer(mem.ptr, nbytes), device=DEV)
    assert view.data_ptr() == mem.ptr and view.numel() == nbytes and view.dtype == torch.uint8 and view.device == torch.device(DEV)
    src = torch.randint(0, 256, (n, C, H, W), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    view.view(n, C, H, W).copy_(src)
    other = torch.randint(0, 256, (n, C, H, W), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).to(DEV)
    store = torch.cat([src.to(DEV), other])
    idx = [0, n - 1, n, 2 * n - 1, 7, n + 5]
    table = torch.tensor(idx, dtype=torch.int32, device=DEV)
    flags = torch.tensor([1, 0, 0, 0], dtype=torch.int32, device=DEV)
    out = torch.empty((len(idx), C, H, W), dtype=torch.uint8, device=DEV)
    ptrs = torch.tensor([mem.ptr, other.data_ptr()], dtype=torch.int64, device=DEV)
    L.check(L.lib().yg_dd_gather_images_peers(ptrs.data_ptr(), n, out.data_ptr(), L.YG_U8, table.data_ptr(),
                                              flags.data_ptr(), len(idx), len(idx), C, H, W, L.stream()))
    assert torch.equal(out, _expected(store, idx, True, False))
    handle = mem.export()
    assert len(handle) == L.YG_IPC_HANDLE_BYTES and any(handle)
    del view, store, other, out
    mem.mark_shared()
    mem.close()
    assert mem.closed and not mem.peers
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    assert torch.cuda.mem_get_info(DEV)[0] >= free0 - (4 << 20)


_IPC_CHILD = """
import sys, hashlib, ctypes
sys.path.insert(0, sys.argv[1])
import torch
from yogo_b200 import _lib as L
from yogo_b200.data.device_dataset import _CudaBuffer
torch.cuda.set_device(0)
lib = L.lib()
p = ctypes.c_void_p()
L.check(lib.yg_dd_shard_open(bytes.fromhex(sys.argv[2]), ctypes.byref(p)))
view = torch.as_tensor(_CudaBuffer(p.value, int(sys.argv[3])), device="cuda:0")
digest = hashlib.sha256(view.cpu().numpy().tobytes()).hexdigest()
del view
torch.cuda.synchronize()
L.check(lib.yg_dd_shard_close(p.value))
print("digest", digest)
"""


@pytest.mark.gpu
def test_shard_shared_with_another_process():
    """CUDA IPC between two processes, in the teardown order of a sharded store: the owner allocates, writes and exports;
    the other process maps the shard, reads it and unmaps it; only after that process has exited does the owner free."""
    import hashlib
    from yogo_b200 import _lib as L
    from yogo_b200.data.device_dataset import _CudaBuffer
    nbytes = 3 * 772 * 1032 + 5
    mem = ShardMemory(L.lib(), nbytes, barrier=lambda: None, synchronize=torch.cuda.synchronize)
    data = torch.randint(0, 256, (nbytes,), dtype=torch.uint8, generator=torch.Generator().manual_seed(4))
    torch.as_tensor(_CudaBuffer(mem.ptr, nbytes), device=DEV).copy_(data)
    torch.cuda.synchronize()
    handle = mem.export()
    mem.mark_shared()
    try:
        r = subprocess.run([sys.executable, "-c", _IPC_CHILD, ROOT, handle.hex(), str(nbytes)], capture_output=True,
                           text=True, timeout=300)
    finally:
        mem.close()          # the other process has exited (or timed out and been killed): nothing maps the shard
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert ("digest " + hashlib.sha256(data.numpy().tobytes()).hexdigest()) in r.stdout, r.stdout


# ----------------------------------------------------------------------------- several GPUs
def _torchrun(n):
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                        "--master-addr", "127.0.0.1", "--master-port", str(29541 + n),
                        os.path.join(ROOT, "tests", "ddp_sharded_dataset_check.py")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ddp_sharded_dataset_check ok" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]


@pytest.mark.gpu
def test_sharded_store_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    _torchrun(2)


@pytest.mark.gpu
def test_sharded_store_on_every_gpu():
    n = min(torch.cuda.device_count(), 8)
    if n < 3:
        pytest.skip("needs >= 3 GPUs (two are covered by test_sharded_store_on_two_gpus)")
    _torchrun(n)
