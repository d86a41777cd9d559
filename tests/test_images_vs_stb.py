"""vct_b200/images.py against THE REFERENCE'S OWN DECODER, byte for byte.

The reference loads every texture with stb_image v2.26 (Model.h:152).  That one part of the reference compiles with g++:
oracle/ref_stb.py builds its stb_image.cpp into oracle/_ref/ and these tests feed the same files to `stbi_load(.., req_comp
= 0)` and to the numpy decoders.  Files are generated in the test (own PNG / TGA / BMP / PNM writers covering the format
corners; Pillow / OpenCV only to ENCODE JPEGs).

Where the reference decoder is not built, the decodes are compared with tests/golden/stb_image_decodes.json: shape and
SHA-256 of the decoded bytes for every input, keyed by the SHA-256 of the input file (the JPEG inputs depend on the
Pillow / OpenCV versions, so an input the file does not know fails as such).  Where the decoder is built, each of its
decodes is also checked against the recorded one.  The committed file was recorded from vct_b200.images, which these
tests had found byte-identical to the reference decoder on the same cases (DESIGN.md section 8, item 5).
VCT_RECORD_STB_GOLDEN=<path> writes the file anew from a run of this module.
"""
import hashlib
import io
import json
import os
import struct
import tempfile
import zlib

import numpy as np
import pytest

from vct_b200 import images

try:
    from oracle import ref_stb
    ref_stb.lib()
    HAVE_STB = True
except Exception:  # noqa: BLE001  (the reference's stb_image is neither built nor buildable: use the recorded decodes)
    HAVE_STB = False
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stb_image_decodes.json")
RECORD_TO = os.environ.get("VCT_RECORD_STB_GOLDEN")
RECORDED = json.load(open(GOLDEN))["decodes"] if os.path.exists(GOLDEN) else {}
_recording = {}


@pytest.fixture(scope="module", autouse=True)
def _write_recording():
    yield
    if RECORD_TO:
        source = "stb_image v2.26 of the reference (oracle/ref_stb.py)" if HAVE_STB else "vct_b200.images"
        rows = ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(_recording.items()))
        with open(RECORD_TO, "w") as f:
            f.write(f'{{"source": {json.dumps(source)},\n"decodes": {{\n{rows}\n}}}}\n')


def sha256(data):
    return hashlib.sha256(data).hexdigest()


def stb_load(data):
    """stbi_load(path, &w, &h, &n, 0) as Model.h:152 calls it (v2.26 rejects true-colour BMPs from MEMORY with "bad offset",
    a known defect of that version's offset check; from a file, the way the reference loads, they decode)."""
    with tempfile.NamedTemporaryFile(suffix=".img") as f:
        f.write(data); f.flush()
        return ref_stb.load(f.name)


def check_reference(data, got, what):
    """`got` must be what stbi_load returns for the file `data`, byte for byte; returns it."""
    key, got = sha256(data), np.ascontiguousarray(got)
    entry = {"shape": list(got.shape), "sha256": sha256(got.tobytes())}
    if HAVE_STB:
        want = stb_load(data)
        assert want.shape == got.shape, (what, want.shape, got.shape)
        assert np.array_equal(want, got), (what, int(np.abs(want.astype(int) - got.astype(int)).max()))
        assert RECORDED.get(key, entry) == entry, (what, "the recorded decode differs from the reference decoder's")
    elif not RECORD_TO:
        assert key in RECORDED, (what, "no recorded decode for this input (a different JPEG encoder?)")
        assert RECORDED[key] == entry, (what, RECORDED[key], entry)
    _recording[key] = entry
    return got


def check_reference_refuses(data, what):
    """stbi_load returns NULL for the file `data`"""
    key = sha256(data)
    if HAVE_STB:
        with pytest.raises(ValueError):
            ref_stb.load_from_memory(data)
        assert RECORDED.get(key, {"refused": True}) == {"refused": True}, what
    elif not RECORD_TO:
        assert RECORDED.get(key) == {"refused": True}, (what, RECORDED.get(key))
    _recording[key] = {"refused": True}


def assert_same(data, what):
    return check_reference(data, images.decode(data, native_channels=True), what)


def picture(h, w, c, seed, bits=8):
    """smooth gradients + noise, so that every PNG filter and JPEG frequency gets exercised"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * (3 + k) + yy * (5 - k)) % 256 for k in range(c)], -1)
    img = (base // 2 + rng.integers(0, 128, (h, w, c))) & 255
    if bits == 16:
        return ((img.astype(np.uint32) << 8) | rng.integers(0, 256, (h, w, c))).astype(np.uint16)
    return (img >> (8 - bits)).astype(np.uint8) if bits < 8 else img.astype(np.uint8)


# ------------------------------------------------------------------------------------------------ PNG
def png_filter_rows(rows, bpp, filters):
    """rows: (h, stride) uint8 -> filtered scanlines with a filter-type byte each (types cycle through `filters`)"""
    out = bytearray()
    prev = np.zeros(rows.shape[1], dtype=np.int32)
    for y, row in enumerate(rows.astype(np.int32)):
        ft = filters[y % len(filters)]
        left = np.concatenate([np.zeros(bpp, np.int32), row[:-bpp]]) if len(row) > bpp else np.zeros_like(row)
        upleft = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]]) if len(row) > bpp else np.zeros_like(row)
        if ft == 0:
            f = row
        elif ft == 1:
            f = row - left
        elif ft == 2:
            f = row - prev
        elif ft == 3:
            f = row - ((left + prev) >> 1)
        else:
            p = left + prev - upleft
            pa, pb, pc = np.abs(p - left), np.abs(p - prev), np.abs(p - upleft)
            f = row - np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, prev, upleft))
        out.append(ft)
        out += (f & 255).astype(np.uint8).tobytes()
        prev = row
    return bytes(out)


def png_pack(samples, depth):
    """(h, w, ch) integer samples -> (h, stride) bytes"""
    h, w, ch = samples.shape
    if depth == 8:
        return samples.astype(np.uint8).reshape(h, w * ch)
    if depth == 16:
        s = samples.astype(np.uint16)
        return np.stack([s >> 8, s & 255], -1).astype(np.uint8).reshape(h, w * ch * 2)
    bits = ((samples.reshape(h, w * ch, 1).astype(np.uint8) >> np.arange(depth - 1, -1, -1, dtype=np.uint8)) & 1).reshape(h, -1)
    pad = (-bits.shape[1]) % 8
    return np.packbits(np.concatenate([bits, np.zeros((h, pad), np.uint8)], 1), axis=1)


def make_png(samples, depth, ctype, filters=(0,), interlace=False, plte=None, trns=None):
    h, w, ch = samples.shape
    bpp = max(1, ch * depth // 8)
    if interlace:
        raw = b""
        for x0, y0, dx, dy in [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)]:
            sub = samples[y0::dy, x0::dx]
            if sub.shape[0] and sub.shape[1]:
                raw += png_filter_rows(png_pack(sub, depth), bpp, filters)
    else:
        raw = png_filter_rows(png_pack(samples, depth), bpp, filters)

    def chunk(kind, body):
        return struct.pack(">I", len(body)) + kind + body + struct.pack(">I", zlib.crc32(kind + body) & 0xFFFFFFFF)
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, int(interlace)))
    if plte is not None:
        out += chunk(b"PLTE", plte.astype(np.uint8).tobytes())
    if trns is not None:
        out += chunk(b"tRNS", trns)
    half = len(raw) // 2 if len(raw) > 8 else len(raw)
    z = zlib.compress(raw, 6)
    return out + chunk(b"IDAT", z[:half]) + chunk(b"IDAT", z[half:]) + chunk(b"IEND", b"")     # split IDAT on purpose


PNG_CASES = [(ct, d) for ct, ds in ((0, (1, 2, 4, 8, 16)), (2, (8, 16)), (3, (1, 2, 4, 8)), (4, (8, 16)), (6, (8, 16))) for d in ds]


@pytest.mark.parametrize("ctype,depth", PNG_CASES)
@pytest.mark.parametrize("interlace", [False, True])
def test_png_every_colour_type_depth_filter_and_interlace(ctype, depth, interlace):
    ch = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]
    for (h, w), seed in (((13, 21), 1), ((1, 1), 2), ((9, 3), 3), ((5, 8), 4)):
        s = picture(h, w, ch, seed + depth, depth if ctype != 3 else 8)
        plte = None
        if ctype == 3:
            ncol = min(1 << depth, 200)
            plte = np.random.default_rng(seed).integers(0, 256, (ncol, 3))
            s = (s.astype(np.int64) % ncol).astype(np.uint8)
        png = make_png(s, depth, ctype, filters=(0, 1, 2, 3, 4, 4, 3, 1), interlace=interlace, plte=plte)
        want = assert_same(png, (ctype, depth, interlace, h, w))
        assert want.shape == (h, w, {0: 1, 2: 3, 3: 3, 4: 2, 6: 4}[ctype])
    # the default (non-native) result never has two channels: grey + alpha becomes RGBA
    if ctype == 4:
        got = images.decode_png(png)
        assert got.shape[2] == 4 and np.array_equal(got[..., 0], want[..., 0]) and np.array_equal(got[..., 3], want[..., 1])


@pytest.mark.parametrize("interlace", [False, True])
def test_png_transparency_chunks(interlace):
    """tRNS: per-entry alpha for palettes (RGBA out), a colour key for grey / RGB at every depth (one more channel)."""
    rng = np.random.default_rng(5)
    s = rng.integers(0, 16, (11, 14, 1)).astype(np.uint8)
    plte = rng.integers(0, 256, (16, 3))
    want = assert_same(make_png(s, 4, 3, (4, 1), interlace, plte=plte, trns=bytes(rng.integers(0, 256, 9).tolist())), "palette tRNS")
    assert want.shape[2] == 4 and (want[..., 3] == 255).any() and (want[..., 3] < 255).any()
    for depth in (1, 2, 4, 8, 16):
        g = picture(10, 12, 1, depth, depth)
        key = int(g[3, 4, 0])
        want = assert_same(make_png(g, depth, 0, (0, 2), interlace, trns=struct.pack(">H", key)), ("grey key", depth))
        assert want.shape[2] == 2 and want[3, 4, 1] == 0 and (want[..., 1] == 255).any()
    for depth in (8, 16):
        c = picture(10, 12, 3, depth, depth)
        c[2:5, 2:5] = c[0, 0]
        want = assert_same(make_png(c, depth, 2, (3,), interlace, trns=struct.pack(">HHH", *[int(x) for x in c[0, 0]])), ("rgb key", depth))
        assert want.shape[2] == 4 and (want[2:5, 2:5, 3] == 0).all()


def test_png_roundtrip_of_the_encoder_and_rejects():
    for c in (1, 3, 4):
        img = picture(17, 9, c, c)
        assert np.array_equal(assert_same(images.encode_png(img), "own encoder"), img)
    with pytest.raises(images.UnsupportedImage):
        images.decode_png(make_png(picture(4, 4, 3, 1), 4, 2))          # 4-bit RGB does not exist
    with pytest.raises(images.UnsupportedImage):
        images.decode(b"GIF89a" + b"\0" * 32)


# ------------------------------------------------------------------------------------------------ TGA
def make_tga(px, itype, bpp, origin_top=False, right_to_left=False, rle=False, cmap=None, cmap_bits=24, cmap_start=0, idlen=0):
    """px: (h, w) indices / grey, (h, w, 2) grey + alpha, (h, w, 3|4) RGB(A) or uint16 5-5-5 words"""
    h, w = px.shape[:2]
    desc = (0x20 if origin_top else 0) | (0x10 if right_to_left else 0) | (8 if bpp == 32 else 0)
    pal = b""
    if cmap is not None:
        pal = (cmap[:, ::-1] if cmap_bits >= 24 else cmap).astype(np.uint8 if cmap_bits >= 24 else "<u2").tobytes()
    head = struct.pack("<BBBHHBHHHHBB", idlen, int(cmap is not None), itype + (8 if rle else 0), cmap_start,
                       0 if cmap is None else len(cmap), cmap_bits if cmap is not None else 0, 0, 0, w, h, bpp, desc)
    rows = px if origin_top else px[::-1]
    if bpp in (24, 32):
        rows = rows[..., [2, 1, 0] + ([3] if bpp == 32 else [])]
    if bpp in (15, 16) and itype == 2:
        flat = rows.astype("<u2").reshape(-1, 1).view(np.uint8).reshape(h * w, 2)
    else:
        flat = rows.astype(np.uint8).reshape(h * w, -1)
    if not rle:
        body = flat.tobytes()
    else:
        body, k, rng = bytearray(), 0, np.random.default_rng(int(flat.sum()) % 1000)
        while k < len(flat):
            run = 1
            while k + run < len(flat) and run < 128 and (flat[k + run] == flat[k]).all():
                run += 1
            if run > 1:
                body.append(0x80 | (run - 1)); body += flat[k].tobytes(); k += run
            else:
                m = int(min(rng.integers(1, 20), len(flat) - k))
                body.append(m - 1); body += flat[k:k + m].tobytes(); k += m
        body = bytes(body)
    return head + b"i" * idlen + pal + body


@pytest.mark.parametrize("rle", [False, True])
@pytest.mark.parametrize("origin_top", [False, True])
def test_tga_true_colour_grey_and_colour_mapped(rle, origin_top):
    rng = np.random.default_rng(11)
    blocky = lambda a: np.repeat(np.repeat(a, 3, 0), 4, 1)                 # runs for the RLE packets
    for c, bpp in ((3, 24), (4, 32)):
        img = blocky(picture(6, 5, c, bpp))
        want = assert_same(make_tga(img, 2, bpp, origin_top, rle=rle, idlen=7), ("tga", bpp))
        assert np.array_equal(want, img)
    grey = blocky(picture(6, 5, 1, 3))[..., 0]
    assert np.array_equal(assert_same(make_tga(grey, 3, 8, origin_top, rle=rle), "tga grey")[..., 0], grey)
    ga = blocky(picture(6, 5, 2, 4))
    assert assert_same(make_tga(ga, 3, 16, origin_top, rle=rle), "tga grey+alpha").shape[2] == 2
    words = blocky(rng.integers(0, 1 << 15, (6, 5)).astype(np.uint16))
    for bpp in (15, 16):
        want = assert_same(make_tga(words, 2, bpp, origin_top, rle=rle), ("tga 555", bpp))
        assert want.shape[2] == 3 and want[0, 0, 0] == (int(words[0, 0]) >> 10 & 31) * 255 // 31
    idx = blocky(rng.integers(0, 40, (6, 5)).astype(np.uint8))
    for bits, pal in ((24, rng.integers(0, 256, (40, 3))), (32, rng.integers(0, 256, (40, 4))), (16, rng.integers(0, 1 << 15, (40,)))):
        if bits == 32:
            data = make_tga(idx, 1, 8, origin_top, rle=rle, cmap=pal[:, [0, 1, 2]], cmap_bits=24)   # writer handles BGR only for 24
            assert_same(data, "tga cmap 24 (again)")
            continue
        assert_same(make_tga(idx, 1, 8, origin_top, rle=rle, cmap=pal, cmap_bits=bits), ("tga cmap", bits))
    # the right-to-left bit is ignored by stb_image, hence by this decoder
    img = picture(5, 7, 3, 9)
    a = assert_same(make_tga(img, 2, 24, origin_top, right_to_left=True), "tga r-t-l")
    assert np.array_equal(a, img)


# ------------------------------------------------------------------------------------------------ PNM
def test_pnm_binary_grey_and_colour():
    img = picture(7, 9, 3, 21)
    assert np.array_equal(assert_same(b"P6\n# made by a test\n9 7\n255\n" + img.tobytes(), "ppm"), img)
    assert np.array_equal(assert_same(b"P5 9 7 255\n" + img[..., 0].tobytes(), "pgm")[..., 0], img[..., 0])
    low = (img // 8).astype(np.uint8)
    assert np.array_equal(assert_same(b"P6\n9 7\n31\n" + low.tobytes(), "ppm maxval 31"), low)       # not rescaled, like stb
    with pytest.raises(images.UnsupportedImage):
        images.decode_pnm(b"P6\n2 2\n65535\n" + b"\0" * 24)
    check_reference_refuses(b"P6\n2 2\n65535\n" + b"\0" * 24, "ppm maxval 65535")                 # stb refuses it too


# ------------------------------------------------------------------------------------------------ BMP
def make_bmp(px, bpp, hsz=40, top_down=False, palette=None, masks=None, compress=0):
    h, w = px.shape[:2]
    rows = px if top_down else px[::-1]
    if bpp in (24, 32) and masks is None:
        rows = rows[..., [2, 1, 0] + ([3] if bpp == 32 else [])].astype(np.uint8).reshape(h, -1)
    elif bpp in (16, 32):
        rows = rows.astype("<u2" if bpp == 16 else "<u4").reshape(h, w, 1).view(np.uint8).reshape(h, -1)
    elif bpp == 8:
        rows = rows.astype(np.uint8)
    elif bpp == 4:
        r = np.concatenate([rows, np.zeros((h, w % 2), rows.dtype)], 1).astype(np.uint8)
        rows = (r[:, 0::2] << 4) | r[:, 1::2]
    else:
        rows = np.packbits(rows.astype(np.uint8), axis=1)
    pad = (-rows.shape[1]) % 4
    body = np.concatenate([rows, np.zeros((h, pad), np.uint8)], 1).tobytes()
    pal = b""
    if palette is not None:
        pal = (palette[:, ::-1].astype(np.uint8).tobytes() if hsz == 12 else
               np.concatenate([palette[:, ::-1], np.zeros((len(palette), 1), palette.dtype)], 1).astype(np.uint8).tobytes())
    hh = -h if top_down else h
    if hsz == 12:
        info = struct.pack("<IHHHH", 12, w, h, 1, bpp)
    else:
        info = struct.pack("<IiiHHIIiiII", hsz, w, hh, 1, bpp, compress, len(body), 2835, 2835, 0, 0)
        if hsz == 40 and compress == 3:
            info += struct.pack("<III", *masks[:3])
        elif hsz >= 56:
            m = masks or (0, 0, 0, 0)
            info += struct.pack("<IIII", *m)
            info += b"\0" * (hsz - 56)
    off = 14 + len(info) + len(pal)
    return b"BM" + struct.pack("<IHHI", off + len(body), 0, 0, off) + info + pal + body


def test_bmp_palettised_true_colour_and_bit_fields():
    rng = np.random.default_rng(31)
    for top_down in (False, True):
        for (h, w) in ((7, 10), (5, 3), (1, 1)):
            img = picture(h, w, 4, h * w)
            assert np.array_equal(assert_same(make_bmp(img[..., :3], 24, top_down=top_down), "bmp 24"), img[..., :3])
            want = assert_same(make_bmp(img, 32, top_down=top_down), "bmp 32")
            assert want.shape[2] == 4 and np.array_equal(want, img)
            zero_a = img.copy(); zero_a[..., 3] = 0
            assert (assert_same(make_bmp(zero_a, 32, top_down=top_down), "bmp 32, alpha all zero")[..., 3] == 255).all()
            for bpp, ncol in ((8, 200), (4, 16), (1, 2)):
                pal = rng.integers(0, 256, (ncol, 3))
                for hsz in (40, 12):
                    # 12-byte (OS/2) headers: stb_image's palette-size formula drops the last four entries (it reads
                    # uninitialised memory for them), so only lower indexes are comparable; none are left at 1 bit
                    usable = ncol if hsz == 40 else ncol - 4
                    if usable <= 0 or (hsz == 12 and top_down):
                        continue
                    idx = rng.integers(0, usable, (h, w))
                    want = assert_same(make_bmp(idx, bpp, hsz=hsz, top_down=top_down, palette=pal), ("bmp pal", bpp, hsz))
                    assert np.array_equal(want, pal[idx].astype(np.uint8))
            w555 = rng.integers(0, 1 << 15, (h, w))
            assert assert_same(make_bmp(w555, 16, top_down=top_down), "bmp 16 default 555").shape[2] == 3
            w565 = rng.integers(0, 1 << 16, (h, w))
            assert_same(make_bmp(w565, 16, top_down=top_down, masks=(0xF800, 0x07E0, 0x001F), compress=3), "bmp 565")
            w32 = rng.integers(0, 1 << 32, (h, w), dtype=np.uint64)
            assert_same(make_bmp(w32, 32, top_down=top_down, masks=(0x3FF00000 >> 2 & 0x0FF00000, 0x000FF000, 0x00000FF0), compress=3), "bmp 32 odd masks")
            v4 = assert_same(make_bmp(w32, 32, hsz=108, top_down=top_down, masks=(0x00FF0000, 0x0000FF00, 0x000000FF, 0xFF000000), compress=3), "bmp v4")
            assert v4.shape[2] == 4
            assert_same(make_bmp(w32, 32, hsz=124, top_down=top_down, masks=(0x000000FF, 0x0000FF00, 0x00FF0000, 0), compress=3), "bmp v5 no alpha")
    with pytest.raises(images.UnsupportedImage):
        images.decode_bmp(make_bmp(rng.integers(0, 16, (4, 4)), 4, palette=rng.integers(0, 256, (16, 3)), compress=2))


# ------------------------------------------------------------------------------------------------ JPEG
def test_jpeg_baseline_and_progressive_all_samplings():
    PIL = pytest.importorskip("PIL.Image")
    n = 0
    for (h, w) in ((67, 93), (16, 16), (1, 1), (9, 40), (33, 17), (128, 128)):
        rgb = picture(h, w, 3, h + w)
        for kw in (dict(quality=92, subsampling=0), dict(quality=75, subsampling=1), dict(quality=50, subsampling=2),
                   dict(quality=85, subsampling=2, progressive=True), dict(quality=97, subsampling=0, progressive=True),
                   dict(quality=30, subsampling=1, progressive=True, optimize=True), dict(quality=100, subsampling=0)):
            b = io.BytesIO(); PIL.fromarray(rgb).save(b, "JPEG", **kw)
            assert assert_same(b.getvalue(), ("jpeg", h, w, kw)).shape == (h, w, 3)
            n += 1
        for kw in (dict(quality=80), dict(quality=60, progressive=True)):
            b = io.BytesIO(); PIL.fromarray(rgb[..., 0]).save(b, "JPEG", **kw)
            assert assert_same(b.getvalue(), ("jpeg grey", h, w, kw)).shape == (h, w, 1)
    assert n == 42


def test_jpeg_restart_intervals_other_samplings_and_cmyk():
    cv2 = pytest.importorskip("cv2")
    PIL = pytest.importorskip("PIL.Image")
    rgb = picture(70, 101, 3, 77)
    flags = [getattr(cv2, n) for n in ("IMWRITE_JPEG_SAMPLING_FACTOR_411", "IMWRITE_JPEG_SAMPLING_FACTOR_440",
                                       "IMWRITE_JPEG_SAMPLING_FACTOR_422", "IMWRITE_JPEG_SAMPLING_FACTOR_420") if hasattr(cv2, n)]
    for rst in (0, 1, 7):
        for prog in (0, 1):
            for sf in flags or [None]:
                params = [cv2.IMWRITE_JPEG_QUALITY, 88, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_PROGRESSIVE, prog]
                if sf is not None:
                    params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf]
                ok, buf = cv2.imencode(".jpg", rgb, params)
                assert ok
                assert_same(buf.tobytes(), ("jpeg cv2", rst, prog, sf))
    cmyk = PIL.fromarray(picture(40, 50, 4, 3), mode="CMYK")
    for kw in (dict(quality=90), dict(quality=70, progressive=True)):
        b = io.BytesIO(); cmyk.save(b, "JPEG", **kw)
        assert assert_same(b.getvalue(), ("jpeg cmyk", kw)).shape == (40, 50, 3)
    b = io.BytesIO(); PIL.fromarray(rgb).save(b, "JPEG", quality=90, subsampling=0)
    d = b.getvalue()
    with pytest.raises(images.UnsupportedImage):
        images.decode_jpeg(d.replace(b"\xff\xc0", b"\xff\xc9", 1))       # arithmetic-coded frame marker


def test_load_image_dispatch_and_objloader_use(tmp_path):
    """load_image picks the decoder by signature (TGA by elimination), as stbi_load does."""
    PIL = pytest.importorskip("PIL.Image")
    rgb = picture(12, 10, 3, 5)
    files = {"a.png": images.encode_png(rgb), "b.tga": make_tga(rgb, 2, 24), "c.bmp": make_bmp(rgb, 24),
             "d.ppm": b"P6 10 12 255\n" + rgb.tobytes()}
    b = io.BytesIO(); PIL.fromarray(rgb).save(b, "JPEG", quality=95, subsampling=0); files["e.jpg"] = b.getvalue()
    for name, data in files.items():
        (tmp_path / name).write_bytes(data)
        got = images.load_image(str(tmp_path / name))
        check_reference(data, got, name)
        if name != "e.jpg":
            assert np.array_equal(got, rgb), name


def test_obj_asset_textures_are_what_the_reference_would_upload(tmp_path):
    """An OBJ whose material maps are a JPEG (4:2:0, as Sponza's are), an RLE TGA and a palettised BMP: objloader's
    textures equal stbi_load's bytes -- what TextureFromFile (Model.h:141-186) hands to glTexImage2D."""
    PIL = pytest.importorskip("PIL.Image")
    from vct_b200 import objloader
    rgb = picture(48, 64, 3, 99)
    PIL.fromarray(rgb).save(str(tmp_path / "albedo.jpg"), quality=85, subsampling=2)
    (tmp_path / "spec.tga").write_bytes(make_tga(np.repeat(picture(8, 4, 3, 5), 4, 1), 2, 24, rle=True))
    pal = np.random.default_rng(3).integers(0, 256, (16, 3))
    (tmp_path / "height.bmp").write_bytes(make_bmp(np.random.default_rng(4).integers(0, 16, (8, 8)), 4, palette=pal))
    (tmp_path / "m.mtl").write_text("newmtl m\nKd 1 1 1\nmap_Kd albedo.jpg\nmap_Ks spec.tga\nmap_Ka height.bmp\n")
    (tmp_path / "m.obj").write_text("mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\nusemtl m\nf 1/1 2/2 3/3\n")
    sc = objloader.load_obj(str(tmp_path / "m.obj"))
    d, s, h, _ = sc.materials[0]
    for tex, name in ((d, "albedo.jpg"), (s, "spec.tga"), (h, "height.bmp")):
        check_reference((tmp_path / name).read_bytes(), sc.textures[tex], name)
    assert sc.textures[d].shape == (48, 64, 3) and np.abs(sc.textures[d].astype(int) - rgb).mean() < 40     # lossy (noisy chroma at 4:2:0), but that picture


def test_pnm_writer_round_trips_through_the_reference_decoder():
    for c in (1, 3):
        img = picture(9, 14, c, 40 + c)
        assert np.array_equal(assert_same(images.encode_pnm(img), "own PNM writer"), img)
