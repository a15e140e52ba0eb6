"""Generates tests/golden/reference_host_cases.npz: what the REFERENCE's host-side classes and codecs (oracle/_ref, built by oracle/build_ref.py from the
reference's sources) return on the inputs of
  tests/test_fuse_reference_emulated.py::test_live_against_the_references_manager_class  (SIFTImageManager::fuseToGlobal, keys "fuse<seed>_*"),
  tests/test_mat4_inverse_reference.py::test_live_against_the_reference_classes          (float4x4 / mat4f inverses, "mat4_*"),
  tests/test_mesh_reference_host.py::test_live_against_the_references_mesh_classes       (MeshData clean-up + PLY writer, "mesh<i>_*"),
  tests/test_sens_reference_sensordata.py::test_live_against_the_references_sensor_data_class  (ml::SensorData's reader, "sd_*"),
  tests/test_sens_reference_stb.py::test_live_against_the_references_stb                 (stb_image's JPEG decoder and inflate, "stb_*").
Inputs the tests regenerate are tied to the stored results by a CRC; inputs made by third-party encoders (JPEG streams through Pillow) and the files of
this library's writer the reference read are stored with them.

    python oracle/build_ref.py && python scripts/make_golden_reference_host_cases.py
"""
import os
import sys
import tempfile
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import test_fuse_reference_emulated as fuse                              # noqa: E402
from tests import test_mat4_inverse_reference as mat4                               # noqa: E402
from tests import test_mesh_reference_host as mesh                                  # noqa: E402
from tests import test_sens_reference_sensordata as sd                              # noqa: E402
from tests import test_sens_reference_stb as stb                                    # noqa: E402
from tests._golden import GOLD, as_crc, input_crc                                   # noqa: E402


def main():
    out = {}
    for seed in fuse.LIVE_SEEDS:
        pb = fuse.live_problem(seed)
        out[f"fuse{seed}_keys"], out[f"fuse{seed}_descs"] = fuse.reference_fuse(pb)
        out[f"fuse{seed}_input_crc"] = np.uint32(input_crc(pb))
    M = mat4.matrices(seed=99, n=300)
    out["mat4_float4x4"], out["mat4_mat4f"] = mat4.ref_inverses(M)
    out["mat4_input_crc"] = np.uint32(input_crc(M))
    with tempfile.TemporaryDirectory() as d:
        for it, (tri, transform) in enumerate(mesh.live_soups()):
            path = os.path.join(d, f"r{it}.ply")
            out[f"mesh{it}_pos"], out[f"mesh{it}_col"], out[f"mesh{it}_faces"] = mesh.reference_save(tri, transform, path)
            out[f"mesh{it}_ply"] = np.frombuffer(open(path, "rb").read(), np.uint8)
            out[f"mesh{it}_input_crc"] = np.uint32(input_crc(tri))
        R = sd.RefSensorData()
        blobs = sd.jpeg_blobs(sd.sequence()[1])
        q, j = sd.write_library_and_jpeg_files(d, blobs)
        for i, b in enumerate(blobs):
            out[f"sd_jpeg{i}"] = np.frombuffer(b, np.uint8)
        out["sd_libz_file"] = np.frombuffer(open(q, "rb").read(), np.uint8)
        for f, path in (("libz", q), ("jpeg", j)):
            for k, v in zip(sd.RefSensorData.READ, R.read(path, sd.W, sd.H, sd.N)):
                out[f"sd_{f}_{k}"] = np.asarray(v)
        S = stb.RefStb()
        more = stb.more_jpegs()
        out["stb_num_jpeg"] = np.int32(len(more))
        for i, b in enumerate(more):
            out[f"stb_jpeg{i}"] = np.frombuffer(b, np.uint8)
            out.update(as_crc(f"stb_jpeg_rgb{i}", S.decode(b)))
        depth = stb.make_streams()[2]
        z = stb.library_zlib_depth(os.path.join(d, "w.sens"), depth)
        out["stb_lib_zlib"] = np.frombuffer(z, np.uint8)
        out["stb_lib_zlib_decoded_crc"] = np.uint32(zlib.crc32(S.zlib_decode(z, depth.nbytes)))
    path = os.path.join(GOLD, "reference_host_cases.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
