"""PNG decoding on the GPU for 8-bit grayscale files, with torchvision for every other file.

``decode_png_batch(inputs, device)`` returns what ``torch.stack([torchvision.io.decode_png(x, ImageReadMode.GRAY) for x
in inputs])`` returns, on ``device``, and raises what it raises.  The path is chosen per file from what the file says:

* device: a valid signature, IHDR first with bit depth 8, colour type 0 and compression / filter / interlace 0, no PLTE
  or tRNS, consecutive IDAT chunks, and a chunk walk that reaches IEND inside the file.  The host checks the IHDR and IEND
  CRCs, skips ancillary chunks as libpng does, and lists the IDAT chunks; the kernels of csrc/png.cu check the IDAT
  CRCs, inflate, unfilter and check the Adler-32.
* host: every other file (16-bit, palette, alpha, RGB, interlaced, unparseable) is decoded by torchvision.
* a file whose device decode reports an error is decoded again by torchvision, and its result or exception is what the
  caller gets, so corrupt files behave exactly as they do with libpng.
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .. import _lib as L

PNG_SIGNATURE = b"\x89PNG\r\n\x1a\n"
MAX_SIDE = 1_000_000   # libpng's default limit on width and height; larger files go to libpng, which rejects them

STATUS_NAMES = {
    0: "ok", 1: "bad IDAT CRC", 2: "bad zlib header", 3: "block type 3", 4: "stored length mismatch",
    5: "invalid code lengths", 6: "invalid symbol", 7: "distance too far back", 8: "output overflow",
    9: "stream ends early", 10: "data after the final block", 11: "Adler-32 mismatch", 12: "filter byte > 4",
    13: "chunk table outside the buffers",
}

CHUNK_DTYPE = np.dtype([("src", "<i8"), ("dst", "<i8"), ("length", "<i4"), ("crc", "<u4")])              # yg_png_chunk
IMAGE_DTYPE = np.dtype([("stream", "<i8"), ("length", "<i8"), ("chunk_begin", "<i4"), ("chunk_end", "<i4")])  # yg_png_image

Input = Union[bytes, bytearray, memoryview, torch.Tensor]


@dataclass
class PngInfo:
    """Result of the host chunk walk.  ``idat`` lists (offset of the chunk type, payload length, stored CRC)."""

    device: bool
    reason: str = ""
    height: int = 0
    width: int = 0
    idat: List[Tuple[int, int, int]] = field(default_factory=list)


def parse_png(data: Union[bytes, memoryview]) -> PngInfo:
    """Walk the chunks of one file and decide whether the device decodes it.  No decompression and no CRC beyond IHDR
    and IEND; ``reason`` says why a file goes to the host."""
    mv = memoryview(data)
    n = len(mv)
    if n < 8 or mv[:8] != PNG_SIGNATURE:
        return PngInfo(False, "no PNG signature")
    pos = 8
    info = PngInfo(False)
    seen_ihdr = idat_closed = False
    while True:
        if pos + 8 > n:
            return PngInfo(False, "chunk header past the end of the file")
        length, ctype = struct.unpack_from(">I4s", mv, pos)
        if length > 0x7FFFFFFF:
            return PngInfo(False, "chunk length over 2^31 - 1")
        end = pos + 12 + length
        if end > n:
            return PngInfo(False, "chunk past the end of the file")
        if not ctype.isalpha():
            return PngInfo(False, "invalid chunk type")
        if not seen_ihdr:
            if ctype != b"IHDR" or length != 13:
                return PngInfo(False, "IHDR is not the first chunk")
            if zlib.crc32(mv[pos + 4:pos + 21]) != struct.unpack_from(">I", mv, pos + 21)[0]:
                return PngInfo(False, "IHDR CRC")
            w, h, depth, color, comp, filt, inter = struct.unpack_from(">IIBBBBB", mv, pos + 8)
            if (depth, color, comp, filt, inter) != (8, 0, 0, 0, 0):
                return PngInfo(False, "not 8-bit grayscale, non-interlaced")
            if not (1 <= w <= MAX_SIDE and 1 <= h <= MAX_SIDE):
                return PngInfo(False, "image size outside libpng's limits")
            info.width, info.height = w, h
            seen_ihdr = True
        elif ctype == b"IDAT":
            if idat_closed:
                return PngInfo(False, "IDAT chunks are not consecutive")
            info.idat.append((pos + 4, length, struct.unpack_from(">I", mv, end - 4)[0]))
        elif ctype == b"IEND":
            if length != 0 or zlib.crc32(mv[pos + 4:pos + 8]) != struct.unpack_from(">I", mv, pos + 8)[0]:
                return PngInfo(False, "bad IEND")
            break
        elif ctype in (b"PLTE", b"tRNS"):
            return PngInfo(False, f"{ctype.decode()} chunk")
        elif not ctype[0] & 0x20:
            return PngInfo(False, f"critical chunk {ctype!r}")
        else:
            idat_closed = idat_closed or bool(info.idat)   # ancillary: skipped
        pos = end
    if not info.idat:
        return PngInfo(False, "no IDAT")
    info.device = True
    return info


def _view(x: Input) -> Optional[memoryview]:
    """Bytes of one input, or None when it is not something the device path reads (torchvision then decides)."""
    if isinstance(x, torch.Tensor):
        if x.dtype != torch.uint8 or x.dim() != 1 or x.device.type != "cpu":
            return None
        return memoryview(x.contiguous().numpy())
    try:
        return memoryview(x).cast("B")
    except TypeError:
        return None


def _as_tensor(x: Input):
    if isinstance(x, torch.Tensor):
        return x
    v = _view(x)
    return x if v is None else torch.from_numpy(np.frombuffer(v, dtype=np.uint8).copy())


def _host_decode_png(x: torch.Tensor) -> torch.Tensor:
    from torchvision.io import ImageReadMode, decode_png

    return decode_png(x, ImageReadMode.GRAY)


def stage_gray8(views: Sequence[memoryview], infos: Sequence[PngInfo], device) -> dict:
    """Pack the IDAT runs of a group of same-size files and their chunk / image tables into one pinned buffer and upload
    it with one copy.  Returns the device buffer and the offsets and sizes yg_png_decode_gray8 takes."""
    n = len(views)
    lo = np.array([i.idat[0][0] for i in infos], np.int64)
    hi = np.array([i.idat[-1][0] + 4 + i.idat[-1][1] for i in infos], np.int64)
    size = hi - lo
    file_off = np.zeros(n, np.int64)
    np.cumsum(size[:-1], out=file_off[1:])
    files_bytes = int(size.sum())
    tabs = [np.array(i.idat, np.int64).reshape(-1, 3) for i in infos]
    counts = np.array([len(t) for t in tabs], np.int64)
    idat = np.concatenate(tabs)
    stream_len = np.array([int(t[:, 1].sum()) for t in tabs], np.int64)
    stream_off = np.zeros(n, np.int64)
    np.cumsum((stream_len[:-1] + 15) // 16 * 16, out=stream_off[1:])
    stream_bytes = int(stream_off[-1] + (stream_len[-1] + 15) // 16 * 16)
    first = np.zeros(n, np.int64)
    np.cumsum(counts[:-1], out=first[1:])
    owner = np.repeat(np.arange(n), counts)
    run = np.cumsum(idat[:, 1]) - idat[:, 1]   # payload bytes before each chunk, over all files
    chunks = np.empty(len(idat), CHUNK_DTYPE)
    chunks["src"] = file_off[owner] - lo[owner] + idat[:, 0]
    chunks["dst"] = stream_off[owner] + run - run[first[owner]]
    chunks["length"] = idat[:, 1]
    chunks["crc"] = idat[:, 2]
    images = np.empty(n, IMAGE_DTYPE)
    images["stream"] = stream_off
    images["length"] = stream_len
    images["chunk_begin"] = first
    images["chunk_end"] = first + counts
    chunk_at = (files_bytes + 15) // 16 * 16
    image_at = chunk_at + chunks.nbytes
    total = image_at + images.nbytes
    host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    a = host.numpy()
    for k, v in enumerate(views):
        a[file_off[k]:file_off[k] + size[k]] = np.frombuffer(v, np.uint8, count=int(size[k]), offset=int(lo[k]))
    a[chunk_at:image_at] = chunks.view(np.uint8)
    a[image_at:total] = images.view(np.uint8)
    buf = torch.empty(total, dtype=torch.uint8, device=device)
    buf.copy_(host, non_blocking=True)
    return dict(buf=buf, files_bytes=files_bytes, chunk_at=chunk_at, image_at=image_at, stream_bytes=stream_bytes, n=n)


def workspace_bytes(n: int, H: int, W: int, stream_bytes: int) -> int:
    return int(L.load().yg_png_gray8_workspace(n, H, W, stream_bytes))


def launch_gray8(staged: dict, H: int, W: int, out: torch.Tensor, status: torch.Tensor,
                 workspace: Optional[torch.Tensor] = None) -> None:
    """Decode a staged group into out (n, 1, H, W) uint8 and status (n,) int32, on the current stream."""
    n = staged["n"]
    ws_need = workspace_bytes(n, H, W, staged["stream_bytes"])
    if workspace is None:   # per call, from the caching allocator: a group's workspace is GBs and is not kept
        workspace = torch.empty(ws_need, dtype=torch.uint8, device=out.device)
    if workspace.numel() < ws_need:
        raise L.YogoB200Error(f"PNG workspace of {workspace.numel()} bytes, {ws_need} needed")
    base = staged["buf"].data_ptr()
    L.check(L.lib().yg_png_decode_gray8(
        base, staged["files_bytes"], base + staged["chunk_at"], base + staged["image_at"], n, H, W, out.data_ptr(),
        status.data_ptr(), workspace.data_ptr(), workspace.numel(), L.stream()))


Entry = Union[Tuple[torch.Tensor, int], BaseException]


def decode_entries(inputs: Sequence[Input], device, host_decode: Callable = _host_decode_png
                   ) -> Tuple[List[Entry], Dict[int, int]]:
    """Decode every input: entry i is (tensor of shape (m, 1, H, W), index) for a decoded file, or the exception its host
    decode raised.  Files of the same size that the device decodes share one output tensor, in input order.  Also returns
    the device status of each file that went to the device."""
    device = torch.device(device)
    views = [_view(x) for x in inputs]
    infos = [parse_png(v) if v is not None else PngInfo(False, "not a byte buffer") for v in views]
    entries: List[Optional[Entry]] = [None] * len(inputs)
    groups: Dict[Tuple[int, int], List[int]] = {}
    for i, info in enumerate(infos):
        if info.device:
            groups.setdefault((info.height, info.width), []).append(i)
    dev_status: Dict[int, int] = {}
    if groups:
        with torch.cuda.device(device):
            order = [i for idx in groups.values() for i in idx]
            status = torch.empty(len(order), dtype=torch.int32, device=device)
            at = 0
            for (H, W), idx in groups.items():
                out = torch.empty((len(idx), 1, H, W), dtype=torch.uint8, device=device)
                staged = stage_gray8([views[i] for i in idx], [infos[i] for i in idx], device)
                launch_gray8(staged, H, W, out, status[at:at + len(idx)])
                at += len(idx)
                for j, i in enumerate(idx):
                    entries[i] = (out, j)
            for i, s in zip(order, status.cpu().tolist()):   # the one device-to-host read of the call
                dev_status[i] = s
                if s != 0:
                    entries[i] = None
    for i, x in enumerate(inputs):
        if entries[i] is None:
            try:
                entries[i] = (host_decode(_as_tensor(x)).unsqueeze(0).to(device), 0)
            except Exception as e:   # re-raised by the caller in input order
                entries[i] = e
    return entries, dev_status


def stack_entries(entries: Sequence[Entry]) -> torch.Tensor:
    """torch.stack of the entries' images, raising the first exception in order; a run of consecutive images of one
    device group is returned as a view without a copy."""
    for e in entries:
        if isinstance(e, BaseException):
            raise e
    if entries:
        base, i0 = entries[0]
        if all(b is base and i == i0 + k for k, (b, i) in enumerate(entries)):
            return base if i0 == 0 and len(entries) == base.shape[0] else base[i0:i0 + len(entries)]
    return torch.stack([b[i] for b, i in entries])


def decode_png_batch(inputs: Sequence[Input], device=None) -> torch.Tensor:
    """``torch.stack([torchvision.io.decode_png(x, ImageReadMode.GRAY) for x in inputs])`` on ``device`` (default: the
    current CUDA device), bit for bit, raising what that expression raises.  ``inputs`` are encoded files as bytes-like
    objects or 1-D uint8 CPU tensors.  8-bit grayscale files are decoded on the GPU, all others by torchvision."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise L.YogoB200Error(f"decode_png_batch decodes on a CUDA device, not {dev}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    entries, _ = decode_entries(inputs, dev)
    return stack_entries(entries)
