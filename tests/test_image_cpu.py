"""Image ingestion (minigpt4_image_load_from_file / minigpt4_preprocess_image, reference minigpt4.cpp:2576-2651) against Pillow:
the PNG decoder byte for byte, the bicubic resize bit for bit (the reference resizes with a C++ port of Pillow's ImagingResample),
the normalisation against the same expression in numpy.  Host-only code: no GPU needed."""
import ctypes
import io
from pathlib import Path

import numpy as np
import pytest

PIL = pytest.importorskip("PIL")
from PIL import Image  # noqa: E402

import minigpt4_cpp_b200 as m  # noqa: E402

MEAN = np.array([0.48145466, 0.4578275, 0.40821073])
STD = np.array([0.26862954, 0.26130258, 0.27577711])
NULL = m.MiniGPT4Context(None)


def load(lib, path):
    img = lib.minigpt4_image_load_from_file(NULL, str(path), 0)
    assert img.format == 2 and img.channels == 3
    a = np.ctypeslib.as_array(ctypes.cast(img.data, ctypes.POINTER(ctypes.c_uint8)), shape=(img.height, img.width, 3)).copy()
    return img, a


def preprocess(lib, img):
    out = lib.minigpt4_preprocess_image(NULL, img, 0)
    assert out.format == 1 and out.width * out.height * out.channels == 3 * 224 * 224
    a = np.ctypeslib.as_array(ctypes.cast(out.data, ctypes.POINTER(ctypes.c_float)), shape=(3, 224, 224)).copy()
    lib.minigpt4_free_image(out)
    return a


def expected_preprocess(rgb_u8):
    small = np.asarray(Image.fromarray(rgb_u8, "RGB").resize((224, 224), Image.BICUBIC))
    f = small.astype(np.float32) * np.float32(1.0 / 255.0)
    d = (f.astype(np.float64) - MEAN).astype(np.float32)
    return small, (d.astype(np.float64) / STD).astype(np.float32).transpose(2, 0, 1)


def as_image(rgb_u8):
    rgb_u8 = np.ascontiguousarray(rgb_u8)
    img = m.MiniGPT4Image()
    img.data = rgb_u8.ctypes.data_as(ctypes.c_void_p); img.width = rgb_u8.shape[1]; img.height = rgb_u8.shape[0]; img.channels = 3; img.format = 2
    return img, rgb_u8


def textured(rng, h, w, ch, top=256):
    """smooth ramp + noise: exercises every PNG filter type and real Huffman trees"""
    yy, xx = np.mgrid[0:h, 0:w]
    return ((((xx * 3 + yy * 5) % top)[..., None] + rng.integers(0, max(2, top // 10), (h, w, ch))) % top)


@pytest.mark.parametrize("mode,size,kw", [
    ("RGB", (37, 23), {}), ("RGB", (640, 480), {"compress_level": 9}), ("RGB", (300, 200), {"compress_level": 0}),
    ("RGBA", (65, 33), {}), ("L", (50, 41), {}), ("LA", (31, 17), {}), ("P", (99, 77), {}), ("1", (45, 19), {}), ("I;16", (40, 30), {}),
])
def test_png_decoder_matches_pillow(lib, tmp_path, mode, size, kw):
    rng = np.random.default_rng(sum(mode.encode()) * 1000 + size[0])
    w, h = size
    if mode == "I;16":
        pil = Image.fromarray(textured(rng, h, w, 1, 65536)[..., 0].astype(np.uint16))
        want = np.repeat((np.asarray(pil) >> 8).astype(np.uint8)[..., None], 3, 2)   # 16-bit samples: the high byte
    elif mode == "P":
        pil = Image.fromarray(textured(rng, h, w, 1, 200)[..., 0].astype(np.uint8), "P")
        pil.putpalette(rng.integers(0, 256, 768, dtype=np.uint8).tobytes())
        want = np.asarray(pil.convert("RGB"))
    elif mode == "1":
        pil = Image.fromarray(rng.integers(0, 2, (h, w), dtype=np.uint8) * 255).convert("1")
        want = np.asarray(pil.convert("RGB"))
    else:
        ch = {"RGB": 3, "RGBA": 4, "L": 1, "LA": 2}[mode]
        arr = textured(rng, h, w, ch).astype(np.uint8)
        pil = Image.fromarray(arr[..., 0] if ch == 1 else arr, mode)
        # alpha is dropped, not blended (cv::imread IMREAD_COLOR); grey is replicated
        want = arr[..., :3] if ch >= 3 else np.repeat(arr[..., :1], 3, 2)
    p = tmp_path / f"t_{mode.replace(';', '')}.png"
    pil.save(p, **kw)
    img, got = load(lib, p)
    assert got.shape == want.shape and np.array_equal(got, want)
    lib.minigpt4_free_image(img)


def write_png(path, samples, depth, ctype, interlace, palette=None, filters=(0, 1, 2, 3, 4)):
    """A minimal PNG writer for the cases Pillow cannot produce (Adam7, 2- and 4-bit grey, 16-bit RGB): samples [h][w][channels] ints."""
    import struct
    import zlib
    h, w, ch = samples.shape

    def pack_row(px):   # px [n][ch] -> bytes at `depth` bits per sample, most significant bit first
        flat = px.reshape(-1).astype(np.uint32)
        if depth == 16:
            return flat.astype(">u2").tobytes()
        if depth == 8:
            return flat.astype(np.uint8).tobytes()
        bits = np.zeros(((flat.size * depth + 7) // 8) * 8, np.uint8)
        for b in range(depth):
            bits[b:flat.size * depth:depth] = (flat >> (depth - 1 - b)) & 1
        return np.packbits(bits).tobytes()

    bpp = max(1, ch * depth // 8)

    def filt(rows):
        out = bytearray(); prev = None
        for y, raw in enumerate(rows):
            ft = filters[y % len(filters)]
            cur = np.frombuffer(raw, np.uint8).astype(np.int32)
            up = np.zeros_like(cur) if prev is None else prev
            left = np.concatenate([np.zeros(bpp, np.int32), cur[:-bpp]]) if cur.size > bpp else np.zeros_like(cur)
            ul = np.concatenate([np.zeros(bpp, np.int32), up[:-bpp]]) if cur.size > bpp else np.zeros_like(cur)
            if ft == 0: enc = cur
            elif ft == 1: enc = cur - left
            elif ft == 2: enc = cur - up
            elif ft == 3: enc = cur - ((left + up) >> 1)
            else:
                pa, pb, pc = np.abs(up - ul), np.abs(left - ul), np.abs(left + up - 2 * ul)
                enc = cur - np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, up, ul))
            out.append(ft); out += (enc & 255).astype(np.uint8).tobytes(); prev = cur
        return bytes(out)

    passes = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)] if interlace else [(0, 0, 1, 1)]
    data = b""
    for x0, y0, dx, dy in passes:
        sub = samples[y0::dy, x0::dx]
        if sub.shape[0] and sub.shape[1]:
            data += filt([pack_row(r) for r in sub])

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d))
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, int(interlace)))
    if palette is not None:
        out += chunk(b"PLTE", palette.astype(np.uint8).tobytes())
    out += chunk(b"tEXt", b"Comment\0ancillary chunks are skipped")
    comp = zlib.compress(data, 6)
    out += chunk(b"IDAT", comp[: len(comp) // 3]) + chunk(b"IDAT", comp[len(comp) // 3:]) + chunk(b"IEND", b"")   # split IDAT
    Path(path).write_bytes(out)


@pytest.mark.parametrize("name,depth,ctype,ch,interlace,size", [
    ("adam7_rgb8", 8, 2, 3, True, (131, 71)), ("adam7_rgba16", 16, 6, 4, True, (37, 29)), ("adam7_tiny", 8, 2, 3, True, (3, 2)),
    ("adam7_grey1", 1, 0, 1, True, (53, 19)), ("grey2", 2, 0, 1, False, (41, 13)), ("grey4", 4, 0, 1, False, (40, 12)),
    ("pal4", 4, 3, 1, False, (39, 11)), ("adam7_pal2", 2, 3, 1, True, (21, 17)), ("rgb16", 16, 2, 3, False, (25, 18)), ("ga16", 16, 4, 2, False, (14, 9)),
])
def test_png_cases_pillow_cannot_write(lib, tmp_path, name, depth, ctype, ch, interlace, size):
    rng = np.random.default_rng(len(name) * 131 + depth)
    w, h = size
    pal = rng.integers(0, 256, (1 << depth, 3)) if ctype == 3 else None
    s = textured(rng, h, w, ch, 1 << depth)
    p = tmp_path / f"{name}.png"
    write_png(p, s, depth, ctype, interlace, pal)
    if ctype == 3:
        want = pal[s[..., 0]].astype(np.uint8)
    else:
        v = (s >> 8) if depth == 16 else (s * 255 // ((1 << depth) - 1) if depth < 8 else s)
        want = (v[..., :3] if ch >= 3 else np.repeat(v[..., :1], 3, 2)).astype(np.uint8)
    img, got = load(lib, p)
    assert got.shape == want.shape and np.array_equal(got, want)
    lib.minigpt4_free_image(img)
    # Pillow reads the same file to the same pixels where its conversion is the same rule (8-bit RGB / palette)
    if (depth == 8 and ctype == 2) or ctype == 3:
        assert np.array_equal(np.asarray(Image.open(p).convert("RGB")), want)


# (Pillow's Python layer swaps the pass order for images more than 100 x taller than wide - a speed-up newer than the C++ port of
# ImagingResample the reference links; sizes here stay below that aspect ratio, where Pillow = its C core = horizontal pass, then vertical)
@pytest.mark.parametrize("size", [(224, 224), (500, 375), (1920, 1080), (100, 60), (224, 500), (33, 224), (3001, 2000), (1, 1), (2, 3), (5, 3),
                                  (223, 225), (224, 1), (10000, 2), (448, 448), (7, 600)])
def test_preprocess_is_pillow_bicubic_then_clip_normalisation(lib, size):
    w, h = size
    rng = np.random.default_rng(w * 7919 + h)
    yy, xx = np.mgrid[0:h, 0:w]
    rgb = ((np.stack([xx * 2 + yy, xx + yy * 3, 255 - xx], -1) % 256) + rng.integers(-20, 20, (h, w, 3))).clip(0, 255).astype(np.uint8)
    img, keep = as_image(rgb)
    got = preprocess(lib, img)
    small, want = expected_preprocess(keep)
    # undo the normalisation to compare the resized bytes exactly
    back = np.rint((got.transpose(1, 2, 0).astype(np.float64) * STD + MEAN) * 255.0).astype(np.int64)
    assert np.array_equal(back, small.astype(np.int64))
    assert np.array_equal(got, want)


def test_reference_sample_images_end_to_end(lib):
    """The original project's sample images (minigpt4/images/), stored under tests/golden/images by tools/make_reference_fixtures.py:
    llama.png as shipped (RGBA screenshot with ICC / EXIF / XMP chunks), and a 64-row band of story.png with its original filtered scanlines."""
    files = sorted((Path(__file__).resolve().parent / "golden" / "images").glob("*.png"))
    assert [f.name for f in files] == ["llama.png", "story_rows84-147.png"]
    for f in files:
        img, got = load(lib, f)
        want = np.asarray(Image.open(f).convert("RGB")) if Image.open(f).mode in ("RGB", "L", "P") else np.asarray(Image.open(f))[..., :3]
        assert np.array_equal(got, want), f.name
        _, want_pre = expected_preprocess(np.ascontiguousarray(want))
        assert np.array_equal(preprocess(lib, img), want_pre), f.name
        lib.minigpt4_free_image(img)


def test_ppm_and_errors(lib, tmp_path):
    rgb = np.random.default_rng(5).integers(0, 256, (9, 13, 3), dtype=np.uint8)
    p = tmp_path / "a.ppm"
    p.write_bytes(b"P6\n# comment\n13 9\n255\n" + rgb.tobytes())
    img, got = load(lib, p)
    assert np.array_equal(got, rgb)
    lib.minigpt4_free_image(img)
    with pytest.raises(RuntimeError, match="OpenImage"):
        lib.minigpt4_image_load_from_file(NULL, str(tmp_path / "missing.png"), 0)
    bad = tmp_path / "bad.png"
    buf = io.BytesIO(); Image.fromarray(rgb).save(buf, "PNG"); raw = bytearray(buf.getvalue())
    raw[len(raw) // 2] ^= 0x55   # checksum must catch it
    bad.write_bytes(bytes(raw))
    with pytest.raises(RuntimeError, match="OpenImage"):
        lib.minigpt4_image_load_from_file(NULL, str(bad), 0)
    (tmp_path / "cut.png").write_bytes(buf.getvalue()[:60])
    with pytest.raises(RuntimeError, match="OpenImage"):
        lib.minigpt4_image_load_from_file(NULL, str(tmp_path / "cut.png"), 0)
    f32, _ = as_image(rgb); f32.format = 1
    with pytest.raises(RuntimeError, match="ImageFormatExpectedU8"):
        lib.minigpt4_preprocess_image(NULL, f32, 0)
    c1, _ = as_image(rgb); c1.channels = 1
    with pytest.raises(RuntimeError, match="ImageChannelsExpectedRGB"):
        lib.minigpt4_preprocess_image(NULL, c1, 0)


FUZZ_CHILD = r'''
import ctypes, io, struct, sys, zlib
import numpy as np
sys.path.insert(0, sys.argv[2])
import minigpt4_cpp_b200 as m
from PIL import Image
lib = m.load_library()
rng = np.random.default_rng(int(sys.argv[1]))
yy, xx = np.mgrid[0:48, 0:64]
arr = (((xx * 3 + yy * 5) % 256)[..., None] + rng.integers(0, 24, (48, 64, 3))).astype(np.uint8)
buf = io.BytesIO(); Image.fromarray(arr).save(buf, "PNG"); good = buf.getvalue()
def chunks(b):
    pos, out = 8, []
    while pos < len(b):
        n = struct.unpack(">I", b[pos:pos + 4])[0]; out.append((b[pos + 4:pos + 8], bytearray(b[pos + 8:pos + 8 + n]))); pos += 12 + n
    return out
def build(cs):
    return good[:8] + b"".join(struct.pack(">I", len(d)) + t + bytes(d) + struct.pack(">I", zlib.crc32(t + bytes(d))) for t, d in cs)
img = m.MiniGPT4Image(); ok = bad = 0
for it in range(400):
    cs = chunks(good)
    mode = it % 4
    if mode == 0:     # damage the compressed stream, checksums re-computed so that the inflater sees it
        for t, d in cs:
            if t == b"IDAT":
                for _ in range(int(rng.integers(1, 6))): d[int(rng.integers(0, len(d)))] = int(rng.integers(0, 256))
        b = build(cs)
    elif mode == 1:   # wild header fields
        t, d = cs[0]; i = int(rng.integers(0, 13)); d[i] = int(rng.integers(0, 256)); b = build(cs)
    elif mode == 2:   # truncation
        b = good[:int(rng.integers(0, len(good)))]
    else:             # a shorter / longer stream than the header promises
        t, d = cs[0]; d[0:8] = struct.pack(">II", int(rng.integers(1, 200)), int(rng.integers(1, 200))); b = build(cs)
    open(sys.argv[3], "wb").write(b)
    rc = lib.library.minigpt4_image_load_from_file(None, sys.argv[3].encode(), ctypes.pointer(img), 0)
    assert rc in (0, 5), rc
    if rc == 0: ok += 1; lib.library.minigpt4_free_image(ctypes.pointer(img))
    else: bad += 1
print("ok", ok, "bad", bad)
'''


def test_damaged_png_files_are_rejected_not_crashed_on(tmp_path):
    import subprocess
    import sys
    root = Path(__file__).resolve().parent.parent
    child = tmp_path / "child.py"; child.write_text(FUZZ_CHILD)
    for seed in (0, 1):
        r = subprocess.run([sys.executable, str(child), str(seed), str(root), str(tmp_path / "f.png")], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (r.returncode, r.stdout[-200:], r.stderr[-600:])
        ok, bad = int(r.stdout.split()[1]), int(r.stdout.split()[3])
        assert bad > 200, (ok, bad)


# ---------------------------------------------------------------------------------------------------------------------------------------
# JPEG (csrc/jpeg.cpp).  Pillow decodes with libjpeg-turbo's defaults - the library and settings behind cv::imread in the reference -
# so equality with Pillow is equality with the reference's pixels.
# ---------------------------------------------------------------------------------------------------------------------------------------
def photo(rng, h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([128 + 100 * np.sin(xx / 17.0) * np.cos(yy / 23.0), 128 + 90 * np.cos(xx / 11.0 + yy / 31.0), (xx * 2 + yy * 3) % 256], -1)
    return (base + rng.normal(0, 12, (h, w, 3))).clip(0, 255).astype(np.uint8)


def load_pixels(lib, path):
    img, a = load(lib, path)
    lib.minigpt4_free_image(img)
    return a


@pytest.mark.parametrize("size", [(64, 48), (65, 49), (17, 9), (1, 1), (8, 8), (257, 131), (640, 427)])
def test_jpeg_written_by_pillow(lib, tmp_path, size):
    w, h = size
    a = photo(np.random.default_rng(w * 31 + h), h, w)
    p = tmp_path / "t.jpg"
    for kw in (dict(quality=90, subsampling=0), dict(quality=75, subsampling=1), dict(quality=75, subsampling=2), dict(quality=30, subsampling=2, optimize=True),
               dict(quality=85, subsampling=2, progressive=True), dict(quality=95, subsampling=0, progressive=True),
               dict(quality=60, subsampling=1, progressive=True, optimize=True), dict(quality=80, subsampling=2, restart_marker_blocks=2),
               dict(quality=80, subsampling=1, progressive=True, restart_marker_rows=1), dict(quality=90, subsampling=0, keep_rgb=True)):
        Image.fromarray(a).save(p, "JPEG", **kw)
        if "restart_marker_blocks" in kw and w * h > 256:
            assert b"\xff\xd0" in p.read_bytes()
        assert np.array_equal(load_pixels(lib, p), np.asarray(Image.open(p).convert("RGB"))), (size, kw)
    Image.fromarray(a[..., 0]).save(p, "JPEG", quality=80)
    assert np.array_equal(load_pixels(lib, p), np.asarray(Image.open(p).convert("RGB")))


def test_jpeg_exif_orientation_is_applied_like_imread(lib, tmp_path):
    from PIL import ImageOps
    a = photo(np.random.default_rng(8), 75, 103)
    p = tmp_path / "o.jpg"
    for o in range(1, 9):
        ex = Image.Exif(); ex[0x0112] = o
        Image.fromarray(a).save(p, "JPEG", quality=85, exif=ex.tobytes())
        want = np.asarray(ImageOps.exif_transpose(Image.open(p)).convert("RGB"))
        got = load_pixels(lib, p)
        assert got.shape == want.shape and np.array_equal(got, want), o


ZZ = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
      35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
AC_SYMS = [0x00, 0xF0] + [(r << 4) | s for r in range(16) for s in range(1, 11)]


def write_jpeg(path, rgb, samp, interleaved=True, restart=0, q16=False, ids=(1, 2, 3), jfif=True):
    """A minimal baseline JPEG writer (flat Huffman codes: 4-bit DC categories, 8-bit AC symbols) for the layouts Pillow cannot write:
    4:4:0, 4:1:1, 4:1:0, chroma at 2x1 under 2x2 luma, one scan per component, 16-bit quantisation tables, fill bytes, odd component ids."""
    import struct
    from scipy.fft import dctn

    class BitW:
        def __init__(s): s.out = bytearray(); s.acc = 0; s.n = 0

        def put(s, v, k):
            for i in range(k - 1, -1, -1):
                s.acc = (s.acc << 1) | ((v >> i) & 1); s.n += 1
                if s.n == 8:
                    s.out.append(s.acc)
                    if s.acc == 0xFF: s.out.append(0)
                    s.acc = 0; s.n = 0

        def flush(s):
            while s.n: s.put(1, 1)

    def cat(v): return 0 if v == 0 else abs(v).bit_length()

    def enc_block(bw, q, pred):
        d = int(q[0]) - pred; c = cat(d); bw.put(c, 4)
        if c: bw.put(d if d > 0 else d + (1 << c) - 1, c)
        run = 0
        last = max([k for k in range(1, 64) if q[ZZ[k]] != 0], default=0)
        for k in range(1, last + 1):
            v = int(q[ZZ[k]])
            if v == 0: run += 1; continue
            while run > 15: bw.put(AC_SYMS.index(0xF0), 8); run -= 16
            c = cat(v); bw.put(AC_SYMS.index((run << 4) | c), 8); bw.put(v if v > 0 else v + (1 << c) - 1, c); run = 0
        if last < 63: bw.put(AC_SYMS.index(0x00), 8)
        return int(q[0])

    H, W, _ = rgb.shape; f = rgb.astype(np.float64)
    ycc = np.stack([0.299 * f[..., 0] + 0.587 * f[..., 1] + 0.114 * f[..., 2], -0.168736 * f[..., 0] - 0.331264 * f[..., 1] + 0.5 * f[..., 2] + 128,
                    0.5 * f[..., 0] - 0.418688 * f[..., 1] - 0.081312 * f[..., 2] + 128], -1)
    hmax = max(s[0] for s in samp); vmax = max(s[1] for s in samp)
    mcux = -(-W // (8 * hmax)); mcuy = -(-H // (8 * vmax))
    qt = (np.arange(64).reshape(8, 8) // 4 + 3).astype(np.int64) + (260 if q16 else 0)
    comps = []
    for i, (h, v) in enumerate(samp):
        fx, fy = hmax // h, vmax // v
        dw, dh = -(-W * h // hmax), -(-H * v // vmax)
        pl = np.pad(ycc[..., i], ((0, dh * fy - H), (0, dw * fx - W)), mode="edge").reshape(dh, fy, dw, fx).mean((1, 3))
        bw_, bh_ = mcux * h, mcuy * v
        pl = np.pad(pl, ((0, bh_ * 8 - dh), (0, bw_ * 8 - dw)), mode="edge")
        blocks = np.zeros((bh_, bw_, 64), np.int64)
        for by in range(bh_):
            for bx in range(bw_):
                blocks[by, bx] = np.rint(dctn(pl[by * 8:by * 8 + 8, bx * 8:bx * 8 + 8] - 128, norm="ortho") / qt).astype(np.int64).reshape(64)
        comps.append(dict(h=h, v=v, blocks=blocks, cw=-(-dw // 8), ch=-(-dh // 8)))
    out = bytearray(b"\xff\xd8")
    if jfif: out += b"\xff\xe0" + struct.pack(">H", 16) + b"JFIF\0\1\1\0\0\1\0\1\0\0"
    qz = [int(qt.reshape(64)[ZZ[i]]) for i in range(64)]
    if q16: out += b"\xff\xdb" + struct.pack(">H", 2 + 1 + 128) + bytes([0x10]) + b"".join(struct.pack(">H", x) for x in qz)
    else: out += b"\xff\xdb" + struct.pack(">H", 2 + 1 + 64) + bytes([0]) + bytes(qz)
    out += b"\xff\xc0" + struct.pack(">HBHHB", 8 + 3 * 3, 8, H, W, 3) + b"".join(bytes([ids[i], (samp[i][0] << 4) | samp[i][1], 0]) for i in range(3))
    out += b"\xff\xc4" + struct.pack(">H", 2 + 17 + 12) + bytes([0x00]) + bytes([0, 0, 0, 12] + [0] * 12) + bytes(range(12))
    out += b"\xff\xc4" + struct.pack(">H", 2 + 17 + 162) + bytes([0x10]) + bytes([0] * 7 + [162] + [0] * 8) + bytes(AC_SYMS)
    if restart: out += b"\xff\xdd" + struct.pack(">HH", 4, restart)

    def scan(cis):
        nonlocal out
        out += b"\xff\xff\xda" + struct.pack(">HB", 6 + 2 * len(cis), len(cis)) + b"".join(bytes([ids[c], 0x00]) for c in cis) + bytes([0, 63, 0])
        bw = BitW(); st = dict(pred=[0, 0, 0], cnt=0, rst=0)

        def maybe_restart():
            if restart and st["cnt"] == restart:
                bw.flush(); bw.out += bytes([0xFF, 0xD0 + st["rst"]]); st["rst"] = (st["rst"] + 1) & 7; st["pred"] = [0, 0, 0]; st["cnt"] = 0
        if len(cis) == 1:
            c = comps[cis[0]]
            for by in range(c["ch"]):
                for bx in range(c["cw"]):
                    maybe_restart(); st["pred"][cis[0]] = enc_block(bw, c["blocks"][by, bx], st["pred"][cis[0]]); st["cnt"] += 1
        else:
            for my in range(mcuy):
                for mx in range(mcux):
                    maybe_restart()
                    for ci in cis:
                        c = comps[ci]
                        for v in range(c["v"]):
                            for h in range(c["h"]):
                                st["pred"][ci] = enc_block(bw, c["blocks"][my * c["v"] + v, mx * c["h"] + h], st["pred"][ci])
                    st["cnt"] += 1
        bw.flush(); out += bw.out
    if interleaved: scan([0, 1, 2])
    else:
        for c in (0, 1, 2): scan([c])
    out += b"\xff\xd9"
    Path(path).write_bytes(bytes(out))


JPEG_LAYOUTS = [("444", [(1, 1)] * 3, {}), ("420", [(2, 2), (1, 1), (1, 1)], {}), ("422", [(2, 1), (1, 1), (1, 1)], {}), ("440", [(1, 2), (1, 1), (1, 1)], {}),
                ("411", [(4, 1), (1, 1), (1, 1)], {}), ("410", [(4, 2), (1, 1), (1, 1)], {}), ("420_scan_per_component", [(2, 2), (1, 1), (1, 1)], dict(interleaved=False)),
                ("440_restart2", [(1, 2), (1, 1), (1, 1)], dict(restart=2)), ("420_scan_per_component_restart3", [(2, 2), (1, 1), (1, 1)], dict(interleaved=False, restart=3)),
                ("422_q16", [(2, 1), (1, 1), (1, 1)], dict(q16=True)), ("chroma2x1_luma2x2", [(2, 2), (2, 1), (2, 1)], {}),
                ("ids_10_20_30_no_jfif", [(2, 2), (1, 1), (1, 1)], dict(ids=(10, 20, 30), jfif=False))]


@pytest.mark.parametrize("name,samp,kw", JPEG_LAYOUTS, ids=[c[0] for c in JPEG_LAYOUTS])
def test_jpeg_layouts_pillow_cannot_write(lib, tmp_path, name, samp, kw):
    pytest.importorskip("scipy")
    for (w, h) in [(61, 45), (16, 16), (33, 7)]:
        a = photo(np.random.default_rng(w + h), h, w)
        p = tmp_path / f"{name}.jpg"
        write_jpeg(p, a, samp, **kw)
        want = np.asarray(Image.open(p).convert("RGB"))
        assert np.abs(want.astype(int) - a.astype(int)).mean() < (25 if kw.get("q16") else 12)   # (the writer produced the picture it was given)
        got = load_pixels(lib, p)
        assert got.shape == want.shape and np.array_equal(got, want), (name, w, h)


JPEG_FUZZ_CHILD = r'''
import ctypes, io, sys
import numpy as np
sys.path.insert(0, sys.argv[2])
import minigpt4_cpp_b200 as m
from PIL import Image
lib = m.load_library()
rng = np.random.default_rng(int(sys.argv[1]))
yy, xx = np.mgrid[0:48, 0:64]
arr = (np.stack([128 + 100 * np.sin(xx / 7.0), 128 + 90 * np.cos(yy / 5.0), (xx * 3 + yy * 5) % 256], -1) + rng.normal(0, 10, (48, 64, 3))).clip(0, 255).astype(np.uint8)
goods = []
for kw in (dict(subsampling=2), dict(subsampling=1, progressive=True), dict(subsampling=2, restart_marker_blocks=2)):
    b = io.BytesIO(); Image.fromarray(arr).save(b, "JPEG", quality=80, **kw); goods.append(b.getvalue())
img = m.MiniGPT4Image(); ok = bad = 0
for it in range(900):
    b = bytearray(goods[it % 3])
    for _ in range(int(rng.integers(1, 5))):
        i = int(rng.integers(2, min(len(b), 700) if it & 1 else len(b)))
        b[i] = int(rng.integers(0, 256)) if rng.integers(0, 3) == 0 else b[i] ^ (1 << int(rng.integers(0, 8)))
    if it % 7 == 0: b = b[:int(rng.integers(2, len(b)))]
    open(sys.argv[3], "wb").write(bytes(b))
    rc = lib.library.minigpt4_image_load_from_file(None, sys.argv[3].encode(), ctypes.pointer(img), 0)
    assert rc in (0, 5), rc
    if rc == 0: ok += 1; lib.library.minigpt4_free_image(ctypes.pointer(img))
    else: bad += 1
print("ok", ok, "bad", bad)
'''


def test_damaged_jpeg_files_do_not_crash_the_process(tmp_path):
    import subprocess
    import sys
    root = Path(__file__).resolve().parent.parent
    child = tmp_path / "child.py"; child.write_text(JPEG_FUZZ_CHILD)
    for seed in (0, 1):
        r = subprocess.run([sys.executable, str(child), str(seed), str(root), str(tmp_path / "f.jpg")], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (r.returncode, r.stdout[-200:], r.stderr[-600:])
        ok, bad = int(r.stdout.split()[1]), int(r.stdout.split()[3])
        assert ok > 50 and bad > 50, (ok, bad)   # (a damaged scan still decodes to some picture, as with libjpeg; damaged headers are errors)


def test_chatbot_preprocess_accepts_a_file_path(lib, tmp_path):
    """MiniGPT4ChatBot.upload_image(path) goes through the C ABI's decode + preprocess (no model needed for this half)."""
    a = photo(np.random.default_rng(4), 120, 200)
    p = tmp_path / "x.jpg"
    Image.fromarray(a).save(p, "JPEG", quality=90)
    bot = m.MiniGPT4ChatBot.__new__(m.MiniGPT4ChatBot)
    bot.library = lib; bot.ctx = NULL
    got = bot._preprocess(str(p))
    _, want = expected_preprocess(np.asarray(Image.open(p).convert("RGB")))
    assert got.shape == (1, 3, 224, 224) and np.array_equal(got[0], want)
