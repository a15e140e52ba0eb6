"""`.sens` payload codecs pinned against the REFERENCE's own: mLib's ml::SensorData decodes colour with stbi_load_from_memory and depth with stbi_zlib_decode_malloc and
compresses depth with stbi_zlib_compress (external/mLib/include/ext-depthcamera/sensorData.h:540-668) -- the stb_image v2.08 / stb_image_write it vendors under
ext-depthcamera/sensorData/.  oracle/build_ref.py (build_sens_host) compiles those two headers where they lie -> oracle/_ref/libref_sens_host.so;
scripts/make_golden_sens_stb.py ran it on the streams below and stored streams + outputs in tests/golden/sens_reference_stb.npz.

JPEG decoding is not normative in its last bit (IDCT, chroma up-sampling, colour conversion), and the frame loop's SIFT sees that bit: csrc/sens_io.cu restates the
reference decoder's fixed-point pipeline, and the bar here is bit-exact on every stream (odd sizes, every sub-sampling up to 2x2, restart intervals, grey, baseline
and progressive)."""
import ctypes as C
import io
import os
import struct
import zlib

import numpy as np

from bundlefusion_b200 import sens
from tests._golden import load, matches

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "sens_reference_stb.npz")
REF_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_sens_host.so")

SIZES = ((37, 53), (48, 64), (1, 1), (2, 3), (17, 16), (16, 17), (111, 159), (8, 8), (9, 33), (120, 160))
VARIANTS = (dict(quality=90, subsampling=2), dict(quality=50, subsampling=1), dict(quality=92, subsampling=0), dict(quality=75, subsampling=2, restart_marker_blocks=2),
            dict(quality=30, subsampling=2), dict(quality=100, subsampling=0))


def picture(rng, h, w):
    """smooth colour picture with some texture (JPEG-typical content), deterministic in rng"""
    from PIL import Image
    low = (rng.random((max(h // 3, 1), max(w // 3, 1), 3)) * 255).astype(np.uint8)
    img = np.asarray(Image.fromarray(low).resize((w, h), Image.BILINEAR)).astype(np.int32)
    return np.clip(img + rng.integers(-6, 7, img.shape), 0, 255).astype(np.uint8)


def handmade_png(arr, ctype, depth, palette=None, interlace=True):
    """a PNG assembled by hand, filter type 0 on every row, optionally Adam7-interlaced (PIL writes neither interlaced files nor 2-bit grey); arr: [h, w] samples
    (colour type 0 / 3) or [h, w, c] bytes"""
    import zlib

    def chunk(t, b):
        return struct.pack(">I", len(b)) + t + b + struct.pack(">I", zlib.crc32(t + b) & 0xffffffff)
    h, w = arr.shape[:2]
    raw = b""
    for x0, y0, dx, dy in (((0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)) if interlace else ((0, 0, 1, 1),)):
        sub = arr[y0::dy, x0::dx]
        if sub.size == 0:
            continue
        for row in sub:
            if row.ndim == 1 and depth < 8:
                bits = np.zeros(((len(row) * depth + 7) // 8) * 8, np.uint8)
                for i, v in enumerate(row):
                    for k in range(depth):
                        bits[i * depth + k] = (int(v) >> (depth - 1 - k)) & 1
                data = np.packbits(bits).tobytes()
            else:
                data = np.ascontiguousarray(row, np.uint8).tobytes()
            raw += b"\x00" + data
    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 1 if interlace else 0))
    if palette is not None:
        out += chunk(b"PLTE", np.ascontiguousarray(palette, np.uint8).tobytes())
    return out + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b"")


def make_streams():
    """the streams of the golden file (encoded by libjpeg / libpng through PIL; the bytes are stored, so another libjpeg version does not change the test)"""
    from PIL import Image
    rng = np.random.default_rng(20240611)
    jpegs, pngs = [], []
    for (h, w) in SIZES:
        img = picture(rng, h, w)
        for kw in VARIANTS if h * w <= 64 * 64 else VARIANTS[:4]:
            bio = io.BytesIO(); Image.fromarray(img).save(bio, "JPEG", **kw); jpegs.append(bio.getvalue())
        bio = io.BytesIO(); Image.fromarray(img[..., 0]).save(bio, "JPEG", quality=80); jpegs.append(bio.getvalue())          # one component
        if h * w <= 64 * 64 or (h, w) == (120, 160):                                                                     # progressive (SOF2): DC / AC first and refinement scans, end-of-band runs
            for kw in (dict(quality=88, subsampling=2, progressive=True), dict(quality=40, subsampling=0, progressive=True)):
                bio = io.BytesIO(); Image.fromarray(img).save(bio, "JPEG", **kw); jpegs.append(bio.getvalue())
            bio = io.BytesIO(); Image.fromarray(img[..., 1]).save(bio, "JPEG", quality=70, progressive=True); jpegs.append(bio.getvalue())
        if (h, w) in ((37, 53), (2, 3), (48, 64)):
            for mode in ("RGB", "RGBA", "L", "LA", "P"):
                bio = io.BytesIO(); Image.fromarray(img).convert(mode).save(bio, "PNG"); pngs.append(bio.getvalue())
            # Adam7 and the 1 / 2 / 4-bit layouts, rows unfiltered: with Up / Average / Paeth rows stb_image v2.08 reads the "prior row" of a sub-byte image from the
            # wrong place (it unfilters in place at the right end of the row buffer and looks for the previous row at the left end) -- the reference's pixels are
            # undefined there, and tests/test_sens_io.py holds this decoder to the PNG specification (PIL) for those files
            pal = rng.integers(0, 256, (16, 3)).astype(np.uint8)
            for il in (True, False):
                pngs += [handmade_png(img[..., 0] >> 6, 0, 2, None, il), handmade_png(img[..., 1] >> 4, 3, 4, pal, il), handmade_png(img[..., 2] >> 7, 3, 1, pal[:2], il),
                         handmade_png(img[..., 0] >> 4, 0, 4, None, il)]
            pngs += [handmade_png(img, 2, 8), handmade_png(np.dstack([img, img[..., :1]]), 6, 8), handmade_png(img[..., 0], 0, 8), handmade_png(np.dstack([img[..., 0], img[..., 1]]), 4, 8)]
    depth = (1000.0 + 600.0 * np.sin(np.arange(120)[:, None] / 17.0) * np.cos(np.arange(160)[None, :] / 23.0)).astype(np.uint16)
    depth[rng.random(depth.shape) < 0.07] = 0
    return jpegs, pngs, depth


class RefStb:
    def __init__(self):
        self.L = C.CDLL(REF_SO)
        vp = C.c_void_p
        self.L.ref_stb_decode.argtypes = [vp, C.c_int, vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        self.L.ref_stb_zlib_compress.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int]
        self.L.ref_stb_zlib_decode.argtypes = [vp, C.c_int, vp, C.c_int]

    def decode(self, data: bytes) -> np.ndarray:
        w, h = C.c_int(0), C.c_int(0)
        buf = np.frombuffer(data, np.uint8)
        assert self.L.ref_stb_decode(buf.ctypes.data, len(data), None, C.byref(w), C.byref(h)) == 0
        out = np.zeros((h.value, w.value, 3), np.uint8)
        assert self.L.ref_stb_decode(buf.ctypes.data, len(data), out.ctypes.data, C.byref(w), C.byref(h)) == 0
        return out

    def zlib_compress(self, raw: bytes, quality: int = 8) -> bytes:
        src = np.frombuffer(raw, np.uint8); out = np.zeros(len(raw) * 2 + 1024, np.uint8)
        n = self.L.ref_stb_zlib_compress(src.ctypes.data, len(raw), out.ctypes.data, out.size, quality)
        assert n > 0
        return out[:n].tobytes()

    def zlib_decode(self, z: bytes, cap: int) -> bytes:
        src = np.frombuffer(z, np.uint8); out = np.zeros(cap, np.uint8)
        n = self.L.ref_stb_zlib_decode(src.ctypes.data, len(z), out.ctypes.data, cap)
        assert n >= 0
        return out[:n].tobytes()


def assemble_sens(path, w, h, color_blobs, depth_blobs, cc, dc):
    """a version-4 file byte by byte, as ml::SensorData::saveToFile lays it out (sensorData.h:1040-1048, RGBDFrame::saveToFile :686-700)"""
    K = np.eye(4, dtype=np.float32)
    with open(path, "wb") as f:
        f.write(struct.pack("<IQ", 4, 3) + b"stb")
        for _ in range(4):
            f.write(K.tobytes())
        f.write(struct.pack("<iiIIIIf", cc, dc, w, h, w, h, 1000.0))
        f.write(struct.pack("<Q", len(color_blobs)))
        for i, (cb, db) in enumerate(zip(color_blobs, depth_blobs)):
            f.write(K.tobytes() + struct.pack("<QQQQ", i, i, len(cb), len(db)) + cb + db)
        f.write(struct.pack("<Q", 0))


def test_jpeg_and_png_decoders_bit_exact_with_the_references_stb_golden():
    g = np.load(GOLDEN)
    n = int(g["num_jpeg"])
    assert n >= 80 and sum(1 for i in range(n) if b"\xff\xc2" in g[f"jpeg_{i}"].tobytes()) >= 20
    for i in range(n):
        got = sens.decode_jpeg(g[f"jpeg_{i}"].tobytes())
        assert matches(got, g, f"jpeg_rgb_{i}"), i
    for i in range(int(g["num_png"])):
        assert np.array_equal(sens.decode_png(g[f"png_{i}"].tobytes()), g[f"png_rgb_{i}"]), i


def test_reader_on_a_file_with_the_references_payloads(tmp_path):
    """JPEG colour + depth compressed by the reference's stbi_zlib_compress (its own deflate, not zlib's): the reader must give the reference's pixels"""
    g = np.load(GOLDEN)
    depth = g["depth"]
    h, w = depth.shape
    ids = [int(i) for i in g["sens_jpeg_ids"]]
    p = str(tmp_path / "ref_payload.sens")
    assemble_sens(p, w, h, [g[f"jpeg_{i}"].tobytes() for i in ids], [g["depth_stb_zlib"].tobytes()] * len(ids), sens.COLOR_JPEG, sens.DEPTH_ZLIB_USHORT)
    r = sens.SensorDataReader(p)
    assert len(r) == len(ids)
    for k, i in enumerate(ids):
        du, cu = r.frame_raw(k)
        assert np.array_equal(du, depth) and matches(cu, g, f"jpeg_rgb_{i}")
        d, c, _, _ = r.frame(k)
        assert matches(c[..., :3], g, f"jpeg_rgb_{i}") and np.array_equal(np.isfinite(d), depth > 0)
    r.close()


def more_jpegs():
    """60 more random streams (Pillow's libjpeg: sizes, qualities, subsampling, restart markers, progressive); the tests read the streams stored in
    reference_host_cases.npz, the encoder's output being version dependent"""
    from PIL import Image
    rng = np.random.default_rng(77)
    out = []
    for _ in range(60):
        h, w = int(rng.integers(1, 90)), int(rng.integers(1, 90))
        img = picture(rng, h, w)
        bio = io.BytesIO()
        Image.fromarray(img).save(bio, "JPEG", quality=int(rng.integers(5, 101)), subsampling=int(rng.integers(0, 3)), restart_marker_blocks=int(rng.integers(0, 4)),
                                  progressive=bool(rng.integers(0, 2)))
        out.append(bio.getvalue())
    return out


def library_zlib_depth(path, depth):
    """the depth payload of a file this library's writer (system zlib) makes"""
    K = np.eye(4, dtype=np.float32)
    wr = sens.SensorDataWriter(path, 160, 120, K, depth_shift=1000.0, zlib_depth=True)
    wr.append(depth, np.zeros((120, 160, 3), np.uint8), K)
    wr.finish()
    from tests.test_sens_io import python_reader
    _, fr = python_reader(path)
    return fr[0][4]


def test_live_against_the_references_stb(tmp_path):
    """more random streams decode as the reference's stb_image decodes them, and depth written by this library's writer is read back by the reference's
    inflate.  The reference's results are stored in tests/golden/reference_host_cases.npz (scripts/make_golden_reference_host_cases.py); where its codecs
    are built, they compute them again, and the golden file above is checked to be what they produce now."""
    g, h = np.load(GOLDEN), load("reference_host_cases.npz")
    jpegs, pngs, depth = make_streams()
    more = [h[f"stb_jpeg{i}"].tobytes() for i in range(int(h["stb_num_jpeg"]))]
    assert len(more) == 60
    for i, b in enumerate(more):
        assert matches(sens.decode_jpeg(b), h, f"stb_jpeg_rgb{i}"), i
    z = library_zlib_depth(str(tmp_path / "w.sens"), depth)
    assert z == h["stb_lib_zlib"].tobytes(), "the library writes another payload than the reference read"
    assert int(h["stb_lib_zlib_decoded_crc"]) == zlib.crc32(depth.tobytes())        # the reference's inflate gave back the depth
    if os.path.exists(REF_SO):
        R = RefStb()
        for i in (0, 7, len(jpegs) - 1):
            assert matches(R.decode(g[f"jpeg_{i}"].tobytes()), g, f"jpeg_rgb_{i}")
        for i, b in enumerate(more):
            assert matches(R.decode(b), h, f"stb_jpeg_rgb{i}"), i
        assert R.zlib_decode(z, depth.nbytes) == depth.tobytes()
