"""`.sens` container pinned against the REFERENCE's own class: oracle/build_ref.py (build_sensordata_host) compiles ml::SensorData
(external/mLib/include/ext-depthcamera/sensorData.h) with g++ -> oracle/_ref/libref_sensordata_host.so; scripts/make_golden_sensordata.py had it WRITE the files stored in
tests/golden/sens_reference_sensordata.npz (raw colour with raw and with stb-zlib depth -- JPEG / PNG can only be written through the reference's Windows-only uplink codec).
  * the library's reader on the reference's files: every header field and every frame;
  * the library's writer: with raw depth the FILE is the reference's, byte for byte; with zlib depth (another deflate encoder) the reference's loadFromFile + decompress
    give back the frames;
  * a file with JPEG colour is read by both readers into the same pixels.
What the reference's reader made of the last two files is stored in tests/golden/reference_host_cases.npz (scripts/make_golden_reference_host_cases.py), with
the files; where oracle/_ref is built, the reference reads them again."""
import ctypes as C
import io
import os
import struct

import numpy as np
import pytest

from bundlefusion_b200 import sens, synth
from tests._golden import load

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "sens_reference_sensordata.npz")
REF_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_sensordata_host.so")
W, H, N = 64, 48, 3
NAME = "StructureSensor"


def sequence():
    K = np.array([[52.5, 0, 31.5, 0], [0, 52.5, 23.5, 0], [0, 0, 1, 0], [0, 0, 0, 1]], np.float32)
    rgb, depth, poses, ts = [], [], [], []
    for i in range(N):
        d, c, T = synth.make_frame(7 * i, W, H, texture="rich")
        depth.append(np.where(np.isfinite(d), np.clip(np.round(d * 1000.0), 1, 65535), 0).astype(np.uint16)); rgb.append(np.ascontiguousarray(c[..., :3]))
        poses.append(T.astype(np.float32)); ts.append((1000 + 33 * i, 1007 + 33 * i))
    poses[1] = np.full((4, 4), -np.inf, np.float32)                       # a frame without a pose, as the reference's recorder stores it
    return K, np.stack(rgb), np.stack(depth), np.stack(poses), np.array(ts, np.uint64)


class RefSensorData:
    def __init__(self):
        self.L = C.CDLL(REF_SO)
        vp = C.c_void_p
        self.L.ref_sensordata_write.argtypes = [C.c_char_p, C.c_uint, C.c_uint, vp, C.c_float, C.c_int, C.c_char_p, C.c_uint, vp, vp, vp, vp]
        self.L.ref_sensordata_read.argtypes = [C.c_char_p, vp, vp, vp, C.c_char_p, C.c_uint, C.c_uint, vp, vp, vp, vp]

    def write(self, path, K, rgb, depth, poses, ts, depth_type):
        n, h, w = depth.shape
        arrs = [np.ascontiguousarray(a) for a in (K, rgb, depth, poses, ts)]
        assert self.L.ref_sensordata_write(path.encode(), w, h, arrs[0].ctypes.data, 1000.0, depth_type, NAME.encode(), n, arrs[1].ctypes.data, arrs[2].ctypes.data, arrs[3].ctypes.data,
                                           arrs[4].ctypes.data) == 0

    READ = ("dims", "calib", "shift", "name", "rgb", "depth", "poses", "ts")

    def read(self, path, w, h, cap):
        dims = np.zeros(8, np.uint32); calib = np.zeros((4, 4, 4), np.float32); shift = C.c_float(0); name = C.create_string_buffer(256)
        rgb = np.zeros((cap, h, w, 3), np.uint8); depth = np.zeros((cap, h, w), np.uint16); poses = np.zeros((cap, 4, 4), np.float32); ts = np.zeros((cap, 2), np.uint64)
        assert self.L.ref_sensordata_read(path.encode(), dims.ctypes.data, calib.ctypes.data, C.byref(shift), name, 256, cap, rgb.ctypes.data, depth.ctypes.data, poses.ctypes.data,
                                          ts.ctypes.data) == 0
        return dims, calib, shift.value, name.value.decode(), rgb, depth, poses, ts


def library_write(path, K, rgb, depth, poses, ts, zl):
    w = sens.SensorDataWriter(path, W, H, K, depth_shift=1000.0, zlib_depth=zl, sensor_name=NAME)
    for i in range(len(depth)):
        w.append(depth[i], rgb[i], poses[i], int(ts[i, 0]), int(ts[i, 1]))
    w.finish()


@pytest.mark.parametrize("zl", [0, 1])
def test_reader_on_the_references_files_and_writer_byte_for_byte(tmp_path, zl):
    g = np.load(GOLDEN)
    K, rgb, depth, poses, ts = sequence()
    p = str(tmp_path / "ref.sens")
    open(p, "wb").write(g[f"file_depth{zl}"].tobytes())
    r = sens.SensorDataReader(p)
    hd = r.header
    assert len(r) == N and (hd.version, hd.sensorName.decode(), hd.colorCompression, hd.depthCompression) == (4, NAME, sens.COLOR_RAW, zl)
    assert (hd.colorWidth, hd.colorHeight, hd.depthWidth, hd.depthHeight, hd.depthShift, hd.numIMUFrames) == (W, H, W, H, 1000.0, 0)
    assert np.array_equal(np.array(hd.colorIntrinsic[:], np.float32).reshape(4, 4), K) and np.array_equal(np.array(hd.depthIntrinsic[:], np.float32).reshape(4, 4), K)
    assert np.array_equal(np.array(hd.colorExtrinsic[:], np.float32).reshape(4, 4), np.eye(4)) and np.array_equal(np.array(hd.depthExtrinsic[:], np.float32).reshape(4, 4), np.eye(4))
    for i in range(N):
        du, cu = r.frame_raw(i)
        d, c, T, t = r.frame(i)
        assert np.array_equal(du, depth[i]) and np.array_equal(cu, rgb[i]) and np.array_equal(c[..., :3], rgb[i])
        assert np.array_equal(T.view(np.uint32), poses[i].view(np.uint32)) and tuple(int(x) for x in t) == tuple(int(x) for x in ts[i])
    r.close()
    if zl == 0:                                                          # nothing in the file depends on an encoder: the library's writer must produce the same bytes
        q = str(tmp_path / "lib.sens")
        library_write(q, K, rgb, depth, poses, ts, False)
        assert open(q, "rb").read() == g["file_depth0"].tobytes()


def jpeg_blobs(rgb):
    """the colour of sequence() encoded by libjpeg (through Pillow); the tests read the blobs stored in reference_host_cases.npz, the encoder's output being version dependent"""
    from PIL import Image
    blobs = []
    for i in range(N):
        bio = io.BytesIO(); Image.fromarray(rgb[i]).save(bio, "JPEG", quality=85 + 5 * i, subsampling=i % 3); blobs.append(bio.getvalue())
    return blobs


def write_library_and_jpeg_files(d, blobs):
    """the two files the reference's reader is given: the library's zlib-depth file and a file with JPEG colour laid out as saveToFile lays it out"""
    from tests.test_sens_reference_stb import assemble_sens
    K, rgb, depth, poses, ts = sequence()
    q, j = os.path.join(d, "libz.sens"), os.path.join(d, "jpeg.sens")
    library_write(q, K, rgb, depth, poses, ts, True)
    assemble_sens(j, W, H, blobs, [depth[i].tobytes() for i in range(N)], sens.COLOR_JPEG, sens.DEPTH_RAW_USHORT)
    return q, j


def test_live_against_the_references_sensor_data_class(tmp_path):
    g, h = np.load(GOLDEN), load("reference_host_cases.npz")
    K, rgb, depth, poses, ts = sequence()
    q, j = write_library_and_jpeg_files(str(tmp_path), [h[f"sd_jpeg{i}"].tobytes() for i in range(N)])
    assert open(q, "rb").read() == h["sd_libz_file"].tobytes(), "the library writes another file than the reference read"
    stored = {f: tuple(h[f"sd_{f}_{k}"] for k in RefSensorData.READ) for f in ("libz", "jpeg")}
    if os.path.exists(REF_SO):
        R = RefSensorData()
        for zl in (0, 1):                                                # the golden files are what the reference writes now
            p = str(tmp_path / f"r{zl}.sens")
            R.write(p, K, rgb, depth, poses, ts, zl)
            assert open(p, "rb").read() == g[f"file_depth{zl}"].tobytes()
        for f, path in (("libz", q), ("jpeg", j)):                       # the stored reads are what the reference's reader returns now
            assert all(np.array_equal(a, b) for a, b in zip(R.read(path, W, H, N), stored[f]))
    # the library's zlib-depth file through the reference's loadFromFile / decompress*
    dims, calib, shift, name, rrgb, rdepth, rposes, rts = stored["libz"]
    assert list(dims) == [W, H, W, H, 0, 1, N, 0] and shift == 1000.0 and str(name) == NAME and np.array_equal(calib[0], K) and np.array_equal(calib[3], np.eye(4))
    assert np.array_equal(rrgb, rgb) and np.array_equal(rdepth, depth) and np.array_equal(rposes.view(np.uint32), poses.view(np.uint32)) and np.array_equal(rts, ts)
    # JPEG colour: both readers decode the same pixels
    dims, _, _, _, rrgb, rdepth, _, _ = stored["jpeg"]
    r = sens.SensorDataReader(j)
    assert list(dims[:7]) == [W, H, W, H, 2, 0, N]
    for i in range(N):
        du, cu = r.frame_raw(i)
        assert np.array_equal(cu, rrgb[i]) and np.array_equal(du, rdepth[i]) and np.array_equal(du, depth[i])
    r.close()


def test_reader_survives_corrupt_files(tmp_path):
    """sizes a corrupt file claims (frame count, payload bytes, image dimensions) must end in an error code, not an allocation failure that takes the process down"""
    g = np.load(GOLDEN)
    rng = np.random.default_rng(1)
    p = str(tmp_path / "f.sens")
    rejected = 0
    for it in range(600):
        b = bytearray(g[f"file_depth{it % 2}"].tobytes())
        mode = it % 4
        if mode == 0:
            for _ in range(int(rng.integers(1, 5))):
                b[int(rng.integers(0, 600))] = int(rng.integers(0, 256))                    # header and first frame record
        elif mode == 1:
            b = b[: int(rng.integers(1, len(b)))]
        elif mode == 2:
            for _ in range(int(rng.integers(1, 5))):
                b[int(rng.integers(0, len(b)))] = int(rng.integers(0, 256))
        else:
            i = int(rng.integers(2, len(b))); del b[i:i + int(rng.integers(1, 30))]
        open(p, "wb").write(bytes(b))
        try:
            r = sens.SensorDataReader(p)
            for i in range(min(len(r), 4)):
                r.frame(i); r.frame_raw(i)
            r.close()
        except (RuntimeError, MemoryError, ValueError):
            rejected += 1
    assert rejected > 100
    b = bytearray(g["file_depth0"].tobytes())
    at = 4 + 8 + len(NAME) + 4 * 64 + 8 + 16 + 4                                            # numFrames: a count the file cannot hold
    b[at:at + 8] = (1 << 40).to_bytes(8, "little")
    open(p, "wb").write(bytes(b))
    with pytest.raises(RuntimeError):
        sens.SensorDataReader(p)
