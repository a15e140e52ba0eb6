"""Generates tests/golden/sens_reference_stb.npz: the streams of tests/test_sens_reference_stb.py (make_streams) and what the REFERENCE's codecs make of them --
the stb_image v2.08 / stb_image_write mLib vendors under external/mLib/include/ext-depthcamera/sensorData/, compiled from there into
oracle/_ref/libref_sens_host.so by oracle/build_ref.py (build_sens_host).

    python oracle/build_ref.py && python scripts/make_golden_sens_stb.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests._golden import as_crc                                                 # noqa: E402
from tests.test_sens_reference_stb import GOLDEN, RefStb, make_streams              # noqa: E402


def main():
    R = RefStb()
    jpegs, pngs, depth = make_streams()
    out = {"num_jpeg": np.int32(len(jpegs)), "num_png": np.int32(len(pngs)), "depth": depth}
    for i, b in enumerate(jpegs):
        out[f"jpeg_{i}"] = np.frombuffer(b, np.uint8)
        out.update(as_crc(f"jpeg_rgb_{i}", R.decode(b)))                            # shape + CRC32: the decoded pixels whole would pass 1 MB
    for i, b in enumerate(pngs):
        out[f"png_{i}"] = np.frombuffer(b, np.uint8)
        out[f"png_rgb_{i}"] = R.decode(b)
    z = R.zlib_compress(depth.tobytes(), 8)                                          # RGBDFrame::compressDepth's quality
    assert R.zlib_decode(z, depth.nbytes) == depth.tobytes()
    out["depth_stb_zlib"] = np.frombuffer(z, np.uint8)
    out["sens_jpeg_ids"] = np.array([i for i, b in enumerate(jpegs) if tuple(out[f"jpeg_rgb_{i}_shape"]) == (120, 160, 3)], np.int32)
    np.savez_compressed(GOLDEN, **out)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes;", len(jpegs), "jpeg,", len(pngs), "png streams")


if __name__ == "__main__":
    main()
