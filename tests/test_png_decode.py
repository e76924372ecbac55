"""PNG decoding on the GPU (yogo_b200.data.decode_png_batch, csrc/png.cu): the host chunk walk and the device / host
decision on the CPU, bit-exactness against torchvision.io.decode_png on the GPU, corrupt files, and predict over a
folder.  Every fixture is generated from a seed."""
import struct
import warnings
import zlib

import numpy as np
import pytest
import torch

from yogo_b200.data.png import decode_entries, decode_png_batch, launch_gray8, parse_png, stage_gray8, workspace_bytes

DEV = "cuda"
SIG = b"\x89PNG\r\n\x1a\n"


# ---- a small PNG writer ---------------------------------------------------------------------------------------------
def chunk(ctype: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + ctype + data + struct.pack(">I", zlib.crc32(ctype + data))


def ihdr(h, w, depth=8, color=0, interlace=0):
    return chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, color, 0, 0, interlace))


def filter_rows(img: np.ndarray, filters) -> bytes:
    """Filtered scanlines of an (H, W) uint8 image; filters is one type for all rows or one per row."""
    h, w = img.shape
    x = img.astype(np.int32)
    out = []
    for r in range(h):
        ft = filters if isinstance(filters, int) else filters[r]
        cur = x[r]
        up = x[r - 1] if r else np.zeros(w, np.int32)
        left = np.concatenate([[0], cur[:-1]])
        ul = np.concatenate([[0], up[:-1]])
        if ft == 0:
            f = cur
        elif ft == 1:
            f = cur - left
        elif ft == 2:
            f = cur - up
        elif ft == 3:
            f = cur - ((left + up) >> 1)
        else:
            p = left + up - ul
            pa, pb, pc = np.abs(p - left), np.abs(p - up), np.abs(p - ul)
            f = cur - np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, up, ul))
        out.append(bytes([ft]) + (f & 255).astype(np.uint8).tobytes())
    return b"".join(out)


def split(stream: bytes, sizes) -> list:
    """IDAT payloads: fixed-size pieces (int), or the given sizes cycled (list; 0 inserts an empty IDAT)."""
    if isinstance(sizes, int):
        return [stream[i:i + sizes] for i in range(0, len(stream), sizes)] or [b""]
    out, i, k = [], 0, 0
    while i < len(stream):
        s = sizes[k % len(sizes)]
        out.append(stream[i:i + s])
        i += s
        k += 1
    return out


def make_png(img=None, filters=1, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15, idat=8192, stream=None,
             before=(), between=(), after=(), head=None):
    """A grayscale 8-bit PNG of img (or of a given zlib stream); before / between / after are extra chunks placed after
    IHDR, between the first and second IDAT, and before IEND."""
    if stream is None:
        c = zlib.compressobj(level, zlib.DEFLATED, wbits, 9, strategy)
        stream = c.compress(filter_rows(img, filters)) + c.flush()
    h, w = img.shape if img is not None else (1, 1)
    parts = split(stream, idat)
    body = b"".join(chunk(*c) for c in before)
    for i, p in enumerate(parts):
        body += chunk(b"IDAT", p)
        if i == 0:
            body += b"".join(chunk(*c) for c in between)
    return SIG + (head if head is not None else ihdr(h, w)) + body + b"".join(chunk(*c) for c in after) + chunk(b"IEND", b"")


def noise_image(h, w, sigma=8.0, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    a, b = rng.random(2) * 0.05
    return (128 + 60 * np.sin(a * xx + b * yy) + sigma * rng.standard_normal((h, w))).clip(0, 255).astype(np.uint8)


def tv_encode(img: np.ndarray, level=6) -> bytes:
    from torchvision.io import encode_png

    return encode_png(torch.from_numpy(img)[None], compression_level=level).numpy().tobytes()


def stream_of(data: bytes) -> bytes:
    info = parse_png(data)
    return b"".join(data[t + 4:t + 4 + n] for t, n, _ in info.idat)


# ---- CPU: chunk walk and device / host decision ---------------------------------------------------------------------
@pytest.mark.parametrize("idat", [1, 7, 8192, [0, 5, 1000, 0, 3, 77], "random"])
def test_chunk_walk_lists_every_idat(idat):
    img = noise_image(23, 41, seed=1)
    if idat == "random":
        idat = [int(s) for s in np.random.default_rng(5).integers(0, 300, 50)]
    stream = zlib.compress(filter_rows(img, 3), 6)
    data = make_png(img, stream=stream, idat=idat)
    info = parse_png(data)
    assert info.device and (info.height, info.width) == (23, 41)
    assert stream_of(data) == stream
    for t, n, crc in info.idat:
        assert data[t:t + 4] == b"IDAT" and zlib.crc32(data[t:t + 4 + n]) == crc


def test_chunk_walk_of_libpng_files():
    for level in (0, 6, 9):
        data = tv_encode(noise_image(40, 50, seed=level), level)
        info = parse_png(data)
        assert info.device and (info.height, info.width) == (40, 50)
        assert len(zlib.decompress(stream_of(data))) == 40 * 51


ANC = [(b"tEXt", b"Comment\x00seeded"), (b"gAMA", struct.pack(">I", 45455)), (b"prIv", b"\x01\x02\x03")]


def test_ancillary_chunks_are_skipped():
    img = noise_image(9, 17, seed=2)
    assert parse_png(make_png(img, before=ANC, after=ANC)).device
    # an ancillary chunk between two IDATs makes them non-consecutive: libpng decides
    info = parse_png(make_png(img, idat=7, between=ANC[:1]))
    assert not info.device and "consecutive" in info.reason
    # a bad CRC on an ancillary chunk is libpng's business (it warns and skips); the walk does not check it
    bad = make_png(img, before=ANC[:1])
    i = bad.index(b"tEXt") + 4
    assert parse_png(bad[:i] + bytes([bad[i] ^ 1]) + bad[i + 1:]).device


@pytest.mark.parametrize("depth,color,interlace,extra", [
    (16, 0, 0, ()), (8, 2, 0, ()), (8, 3, 0, ((b"PLTE", bytes(range(6))),)), (8, 4, 0, ()), (8, 6, 0, ()),
    (8, 0, 1, ()), (1, 0, 0, ()), (4, 0, 0, ()), (8, 0, 0, ((b"tRNS", b"\x00\x05"),)), (8, 0, 0, ((b"XXXX", b""),)),
])
def test_unsupported_formats_go_to_the_host(depth, color, interlace, extra):
    data = make_png(noise_image(5, 6), head=ihdr(5, 6, depth, color, interlace), before=extra)
    assert not parse_png(data).device


def test_truncated_and_malformed_files_go_to_the_host():
    data = make_png(noise_image(20, 30, seed=3), idat=100)
    assert parse_png(data).device
    for cut in range(len(data)):
        assert not parse_png(data[:cut]).device, cut
    assert parse_png(data + b"trailing bytes after IEND").device   # libpng stops reading at IEND
    assert not parse_png(b"\x89PNG\r\n\x1a\x0b" + data[8:]).device
    bad_ihdr = bytearray(data)
    bad_ihdr[16] ^= 1
    assert not parse_png(bytes(bad_ihdr)).device
    bad_iend = bytearray(data)
    bad_iend[-1] ^= 1
    assert not parse_png(bytes(bad_iend)).device
    no_idat = SIG + ihdr(2, 2) + chunk(b"IEND", b"")
    assert not parse_png(no_idat).device
    assert not parse_png(SIG + ihdr(2, 2) + ihdr(2, 2) + data[33:]).device   # a second IHDR


# ---- GPU: bit-exact against torchvision -----------------------------------------------------------------------------
def tv_stack(files):
    from torchvision.io import ImageReadMode, decode_png

    return torch.stack([decode_png(torch.frombuffer(bytearray(f), dtype=torch.uint8), ImageReadMode.GRAY) for f in files])


def check_equal(files):
    got = decode_png_batch(files, DEV)
    assert got.device.type == "cuda" and got.dtype == torch.uint8
    ref = tv_stack(files)
    assert got.shape == ref.shape and torch.equal(got.cpu(), ref)
    return got


@pytest.mark.gpu
def test_libpng_files_at_every_compression_level():
    for level in range(10):
        files = [tv_encode(noise_image(61, 97, sigma=s, seed=level * 3 + i), level) for i, s in enumerate((8, 2, 0.5))]
        entries, st = decode_entries(files, DEV)
        assert st == {0: 0, 1: 0, 2: 0}, (level, st)
        check_equal(files)


@pytest.mark.gpu
def test_every_filter_and_zlib_strategy_and_window():
    img = noise_image(37, 53, sigma=4, seed=4)
    mixed = [int(v) for v in np.random.default_rng(6).integers(0, 5, 37)]
    files = [make_png(img, filters=f) for f in (0, 1, 2, 3, 4, mixed)]
    for strat in (zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED):
        files += [make_png(img, filters=mixed, strategy=strat, level=lv) for lv in (1, 9)]
    for wbits in range(9, 16):
        files.append(make_png(noise_image(37, 53, sigma=1, seed=wbits), filters=mixed, wbits=wbits, idat=[0, 1, 7, 300]))
    _, st = decode_entries(files, DEV)
    assert set(st.values()) == {0}
    check_equal(files)


@pytest.mark.gpu
def test_constant_images_and_long_runs():
    files = [make_png(np.full((33, 700), v, np.uint8), filters=f, level=9) for v, f in ((0, 0), (255, 1), (17, 2), (200, 4))]
    _, st = decode_entries(files, DEV)
    assert set(st.values()) == {0}
    check_equal(files)


class BitWriter:
    def __init__(self):
        self.bits, self.n = 0, 0

    def put(self, v, n):   # LSB first
        self.bits |= v << self.n
        self.n += n

    def code(self, c, n):  # Huffman codes go MSB first
        self.put(int(format(c, f"0{n}b")[::-1], 2), n)

    def bytes(self):
        return self.bits.to_bytes((self.n + 7) // 8, "little")


LBASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
DBASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145,
         8193, 12289, 16385, 24577]


def fixed_match_stream(row: bytes, copies: int) -> bytes:
    """zlib stream of `row` (a stored block) followed by `copies` repeats of it as fixed-Huffman matches at distance
    len(row) (zlib's own encoder never reaches 32768)."""
    dist = len(row)
    out = bytearray(b"\x78\x01")
    out += b"\x00" + struct.pack("<HH", len(row), len(row) ^ 0xFFFF) + row   # not final, stored
    bw = BitWriter()
    bw.put(1, 1)
    bw.put(1, 2)   # final, fixed
    dcode = max(i for i in range(30) if DBASE[i] <= dist)
    left = dist * copies
    while left:
        n = min(258, left) if left - 258 not in (1, 2) else left - 3
        li = 28 if n == 258 else max(i for i in range(28) if LBASE[i] <= n)
        sym = 257 + li
        if sym < 280:
            bw.code(sym - 256, 7)
        else:
            bw.code(0b11000000 + sym - 280, 8)
        bw.put(n - LBASE[li], 0 if li < 8 or li == 28 else (li - 4) >> 2)
        bw.code(dcode, 5)
        bw.put(dist - DBASE[dcode], 0 if dcode < 4 else (dcode - 2) >> 1)
        left -= n
    bw.code(0, 7)   # end of block
    out += bw.bytes()
    return bytes(out) + struct.pack(">I", zlib.adler32(row * (copies + 1)))


@pytest.mark.gpu
def test_distance_32768_in_a_hand_built_fixed_block():
    row = bytes([0]) + noise_image(1, 32767, seed=9).tobytes()
    data = make_png(np.zeros((2, 32767), np.uint8), stream=fixed_match_stream(row, 1))
    assert zlib.decompress(stream_of(data)) == row * 2
    _, st = decode_entries([data], DEV)
    assert st == {0: 0}
    check_equal([data])


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", [(1, 1), (1, 333), (300, 1), (17, 31), (19, 129), (772, 1032)])
def test_sizes(h, w):
    files = [tv_encode(noise_image(h, w, seed=s)) for s in range(3)] + [make_png(noise_image(h, w, seed=9), filters=4)]
    _, st = decode_entries(files, DEV)
    assert set(st.values()) == {0}
    check_equal(files)


@pytest.mark.gpu
def test_mixed_device_and_host_files():
    from torchvision.io import encode_png

    rng = np.random.default_rng(11)
    rgb = encode_png(torch.from_numpy(rng.integers(0, 256, (3, 20, 30), dtype=np.uint8))).numpy().tobytes()
    palette = make_png(None, head=ihdr(20, 30, 8, 3), before=((b"PLTE", rng.bytes(768)),),
                       stream=zlib.compress(b"".join(b"\x00" + rng.bytes(30) for _ in range(20))))
    files = [tv_encode(noise_image(20, 30, seed=1)), rgb, make_png(noise_image(20, 30, seed=2), filters=3), palette,
             tv_encode(noise_image(20, 30, seed=3))]
    _, st = decode_entries(files, DEV)
    assert st == {0: 0, 2: 0, 4: 0}
    check_equal(files)
    # tensors in, as torchvision.io.read_file returns them
    check_equal([torch.frombuffer(bytearray(f), dtype=torch.uint8) for f in files])
    with pytest.raises(RuntimeError):   # two sizes: torch.stack's error
        decode_png_batch([files[0], tv_encode(noise_image(21, 30))], DEV)
    with pytest.raises(RuntimeError):
        decode_png_batch([], DEV)


# ---- GPU: corrupt files ---------------------------------------------------------------------------------------------
def corrupt_cases():
    img = noise_image(48, 77, sigma=6, seed=21)
    good = make_png(img, filters=3, idat=500)
    stream = stream_of(good)
    raw = filter_rows(img, 3)
    cases = {}
    b = bytearray(good)
    i = parse_png(good).idat[1][0] + 40
    b[i] ^= 0x10
    cases["flipped bit"] = (bytes(b), 1)
    s = bytearray(stream)
    s[len(s) // 2] ^= 0x10
    cases["flipped bit, CRC recomputed"] = (make_png(img, stream=bytes(s), idat=500), None)
    s = bytearray(stream)
    s[-1] ^= 1
    cases["bad Adler-32"] = (make_png(img, stream=bytes(s), idat=500), 11)
    bad_filter = bytearray(raw)
    bad_filter[5 * 78] = 5
    cases["filter byte 5"] = (make_png(img, stream=zlib.compress(bytes(bad_filter)), idat=500), 12)
    cases["truncated stream"] = (make_png(img, stream=stream[:len(stream) // 2], idat=500), 9)
    cases["too much data"] = (make_png(img, stream=stream + b"\x00\x01\x02", idat=500), 10)
    cases["short image data"] = (make_png(img, stream=zlib.compress(raw[:-78]), idat=500), 9)
    return good, cases


@pytest.mark.gpu
def test_corrupt_files_match_torchvision_and_stay_inside_their_buffers():
    from torchvision.io import ImageReadMode, decode_png

    good, cases = corrupt_cases()
    H, W = 48, 77
    GUARD = 4096
    for name, (bad, want) in cases.items():
        files = [good, bad, good]
        # the device status
        views = [memoryview(f) for f in files]
        infos = [parse_png(v) for v in views]
        assert all(i.device for i in infos), name
        staged = stage_gray8(views, infos, DEV)
        n = len(files)
        ws_need = workspace_bytes(n, H, W, staged["stream_bytes"])
        wbuf = torch.full((ws_need + 2 * GUARD,), 0xA5, dtype=torch.uint8, device=DEV)
        obuf = torch.full((n * H * W + 2 * GUARD,), 0x5A, dtype=torch.uint8, device=DEV)
        sbuf = torch.full((n + 2 * GUARD,), 77, dtype=torch.int32, device=DEV)
        out = obuf[GUARD:GUARD + n * H * W].view(n, 1, H, W)
        launch_gray8(staged, H, W, out, sbuf[GUARD:GUARD + n], wbuf[GUARD:GUARD + ws_need])
        torch.cuda.synchronize()
        status = sbuf[GUARD:GUARD + n].cpu().tolist()
        assert status[0] == 0 and status[2] == 0, (name, status)
        assert status[1] != 0 and (want is None or status[1] == want), (name, status)
        for buf, fill in ((wbuf, 0xA5), (obuf, 0x5A), (sbuf, 77)):
            assert bool((buf[:GUARD] == fill).all()) and bool((buf[-GUARD:] == fill).all()), name
        ref_good = decode_png(torch.frombuffer(bytearray(good), dtype=torch.uint8), ImageReadMode.GRAY)
        assert torch.equal(out[0].cpu(), ref_good) and torch.equal(out[2].cpu(), ref_good), name
        # the public function: what torchvision returns or raises
        try:
            ref = tv_stack(files)
        except Exception as e:
            with pytest.raises(type(e)) as got:
                decode_png_batch(files, DEV)
            assert str(got.value) == str(e), name
        else:
            assert torch.equal(decode_png_batch(files, DEV).cpu(), ref), name


# ---- GPU: predict over a folder -------------------------------------------------------------------------------------
def small_checkpoint(tmp_path, H, W, C):
    import yogo_b200

    torch.manual_seed(3)
    net = yogo_b200.YOGO((H, W), 0.1, 0.1, C, inference=True)
    with torch.no_grad():
        net.model[-1].bias[4] = 1.0
    pth = tmp_path / "m.pth"
    torch.save({"step": 5, "model_state_dict": net.state_dict(), "model_version": "base_model", "class_names": list("abcd"),
                "normalize_images": True}, pth)
    return pth


# images per SM of the decode groups: the default (one group here), groups of two batches, groups of one batch
@pytest.mark.gpu
@pytest.mark.parametrize("per_sm", [None, 0.04, 0.01])
def test_predict_from_a_folder_matches_predict_on_decoded_images(tmp_path, capsys, monkeypatch, per_sm):
    import yogo_b200
    import yogo_b200.infer as infer
    from yogo_b200.infer import _list_images, _read_image

    if per_sm is not None:
        monkeypatch.setattr(infer, "DECODE_IMAGES_PER_SM", per_sm)
    H, W, C = 96, 128, 4
    pth = small_checkpoint(tmp_path, H, W, C)
    idir = tmp_path / "images"
    idir.mkdir()
    N, bs = 14, 3
    good, cases = corrupt_cases()
    for i in range(N):
        img = noise_image(H, W, sigma=(8, 2, 20)[i % 3], seed=100 + i)
        data = tv_encode(img, i % 10) if i % 2 else make_png(img, filters=i % 5)
        if i == 4:   # batch 1: a file libpng rejects
            data = cases["flipped bit"][0]
        if i == 7:   # batch 2: a file of another size
            data = tv_encode(noise_image(50, 60))
        (idir / f"img_{i:03d}.png").write_bytes(data)
    paths = _list_images(idir)
    expected_errors = []
    for lo in range(0, N, bs):
        try:
            torch.stack([_read_image(q) for q in paths[lo:lo + bs]])
        except RuntimeError as e:
            expected_errors.append(f"got error {e}; continuing")
    assert len(expected_errors) == 2
    odir = tmp_path / "out"
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        res = yogo_b200.predict(str(pth), path_to_images=idir, output_dir=str(odir), save_preds=True, batch_size=bs,
                                return_full_predictions=True, half=True)
    got_errors = [str(x.message) for x in w if str(x.message).startswith("got error")]
    assert got_errors == expected_errors
    # the reference: the same files decoded by torchvision, the skipped batches replaced by any image of the right size
    imgs = [_read_image(q) for q in paths if q.name not in ("img_004.png", "img_007.png")]
    imgs.insert(4, imgs[0])
    imgs.insert(7, imgs[0])
    rdir = tmp_path / "ref"
    ref = yogo_b200.predict(str(pth), images=torch.stack(imgs), output_dir=str(rdir), save_preds=True, batch_size=bs,
                            return_full_predictions=True, half=True)
    ref[3:9] = 0
    assert torch.equal(res, ref)
    for i in range(N):
        written = odir / f"img_{i:03d}.txt"
        if 3 <= i < 9:
            assert not written.exists()
        else:
            assert written.read_text() == (rdir / f"image_{i:06d}.txt").read_text()

    # per-class counts over a folder without bad files: the same as over the decoded stack
    cdir = tmp_path / "clean"
    cdir.mkdir()
    for q in paths[8:]:
        (cdir / q.name).write_bytes(q.read_bytes())
    capsys.readouterr()
    yogo_b200.predict(str(pth), path_to_images=cdir, batch_size=bs, count_predictions=True, half=True)
    from_files = capsys.readouterr().out
    yogo_b200.predict(str(pth), images=torch.stack([_read_image(q) for q in paths[8:]]), batch_size=bs,
                      count_predictions=True, half=True)
    assert from_files == capsys.readouterr().out and from_files.startswith("[(")


@pytest.mark.gpu
def test_predict_raises_when_a_decode_group_fails(tmp_path, monkeypatch):
    """An error of a whole decode group (not of a file) ends predict; no later batch sees another group's images."""
    import yogo_b200
    import yogo_b200.data.png as png
    import yogo_b200.infer as infer

    monkeypatch.setattr(infer, "DECODE_IMAGES_PER_SM", 0.04)   # groups of two batches of 3
    pth = small_checkpoint(tmp_path, 96, 128, 4)
    idir = tmp_path / "images"
    idir.mkdir()
    for i in range(12):
        (idir / f"img_{i:03d}.png").write_bytes(tv_encode(noise_image(96, 128, seed=i)))
    real, calls = png.decode_entries, []

    def failing(*args, **kw):
        calls.append(len(args[0]))
        if len(calls) == 1:
            raise png.L.YogoB200Error("simulated launch failure")
        return real(*args, **kw)

    monkeypatch.setattr(png, "decode_entries", failing)
    with pytest.raises(png.L.YogoB200Error, match="simulated launch failure"):
        yogo_b200.predict(str(pth), path_to_images=idir, batch_size=3, return_full_predictions=True)
    assert calls == [6]
