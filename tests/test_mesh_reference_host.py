"""The host half of the mesh export pinned against the REFERENCE's own classes: oracle/build_ref.py (build_mesh_host) compiles mLib's MeshDataf / MeshIOf from
/root/reference/external/mLib/include (g++, a scratch copy with the few one-line patches g++ needs) behind the statements of
CUDAMarchingCubesHashSDF::copyTrianglesToCPU / ::saveMesh (FL/DepthSensing/CUDAMarchingCubesHashSDF.cpp:26-46, 70-100) -> oracle/_ref/libref_mesh_host.so;
scripts/make_golden_mesh_host.py ran it on the triangle soups below and stored merged vertices, colours, faces and the PLY FILE BYTES in
tests/golden/mesh_reference_host.npz.  The library's bfMesh* functions and bfMarchingCubesSaveMesh's writer (host code: runs without a GPU) must reproduce all of it."""
import ctypes as C
import os

import numpy as np
import pytest

from bundlefusion_b200 import marching_cubes as mc
from oracle import oracle as orc
from tests._golden import input_crc, load

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "mesh_reference_host.npz")
REF_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_mesh_host.so")
TRANSFORM = np.array([[0.0, -1.0, 0.0, 0.25], [1.0, 0.0, 0.0, -0.5], [0.0, 0.0, 1.0, 2.0], [0.0, 0.0, 0.0, 1.0]], np.float32)


def soups():
    """(a) marching-cubes output of the seeded scene (shared edge vertices, bit-equal); (b) the same with jitter below / around the merge threshold, duplicated and
    rotated faces, degenerate faces, negative coordinates -- what exercises the 27-cell probe order and the sign-aware rounding of mergeCloseVertices"""
    from tests.test_marchingcubes_reference_emulated import golden_params, golden_scene, scene_box
    sc, cam, frames = golden_scene()
    tri, _ = orc.marchingcubes_extract(sc, golden_params(sc.hp, scene_box(sc)))
    a = np.ascontiguousarray(tri[:1200])
    rng = np.random.default_rng(5)
    b = a[:500].copy()
    b[..., :3] -= np.float32(0.8)                                                          # straddle the origin
    b[..., :3] += rng.uniform(-8e-6, 8e-6, b[..., :3].shape).astype(np.float32)           # around the 1e-5 cell
    b = np.concatenate([b, b[40:60][:, [1, 2, 0]], b[100:103], np.repeat(b[7:8, :1], 3, axis=1)])
    return {"a": a, "b": np.ascontiguousarray(b)}


def library_save(tri, transform, path):
    """what bfMarchingCubesSaveMesh does with a soup, through the exported pieces"""
    pos = np.ascontiguousarray(tri[..., :3].reshape(-1, 3)); col = np.concatenate([tri[..., 3:].reshape(-1, 3), np.ones((len(pos), 1), np.float32)], axis=1)
    faces = np.arange(len(pos), dtype=np.uint32).reshape(-1, 3)
    p, c, f = mc.merge_close_vertices(pos, col, faces, 0.00001)
    f = mc.remove_duplicate_faces(f)
    if transform is not None:
        h = np.concatenate([p, np.ones((len(p), 1), np.float32)], axis=1)
        r = np.stack([(transform[k, 0] * h[:, 0] + transform[k, 1] * h[:, 1] + transform[k, 2] * h[:, 2] + transform[k, 3]).astype(np.float32) for k in range(4)], axis=1)
        p = (r[:, :3] / r[:, 3:4]).astype(np.float32)
    mc.save_ply(path, p, c, f)
    return p, c, f


def reference_save(tri, transform, path):
    R = C.CDLL(REF_SO)
    vp = C.c_void_p
    R.ref_mesh_save.argtypes = [vp, C.c_uint, vp, C.c_char_p, vp, vp, vp, vp]
    n = len(tri)
    pos = np.zeros((3 * n, 3), np.float32); col = np.zeros((3 * n, 4), np.float32); faces = np.zeros((3 * n, 3), np.uint32); counts = np.zeros(2, np.uint32)
    t = None if transform is None else np.ascontiguousarray(transform, np.float32)
    rc = R.ref_mesh_save(np.ascontiguousarray(tri, np.float32).ctypes.data, n, None if t is None else t.ctypes.data, path.encode(), pos.ctypes.data, col.ctypes.data, faces.ctypes.data,
                         counts.ctypes.data)
    assert rc == 0
    return pos[:counts[0]].copy(), col[:counts[0]].copy(), faces[:counts[1]].copy()


@pytest.mark.parametrize("name,transform", [("a", None), ("b", None), ("b", TRANSFORM)])
def test_mesh_cleanup_and_ply_equal_the_references_golden(tmp_path, name, transform):
    g = np.load(GOLDEN)
    key = name + ("_t" if transform is not None else "")
    tri = soups()[name]
    assert np.array_equal(tri, g["soup_" + name])
    path = str(tmp_path / "lib.ply")
    p, c, f = library_save(tri, transform, path)
    assert len(p) == len(g["pos_" + key]) < 3 * len(tri) / 2 and len(f) == len(g["faces_" + key])
    assert np.array_equal(p.view(np.uint32), g["pos_" + key].view(np.uint32)) and np.array_equal(c, g["col_" + key]) and np.array_equal(f, g["faces_" + key])
    assert open(path, "rb").read() == g["ply_" + key].tobytes()                            # the file the reference writes, byte for byte


def live_soups():
    """four more soups: other visiting orders (which vertex of a cluster survives depends on it), jitter, mirrored through the origin, a transform"""
    rng = np.random.default_rng(11)
    out = []
    for it in range(4):
        tri = soups()["a"][rng.permutation(1200)[:400]].copy()
        tri[..., :3] += rng.uniform(-1.2e-5, 1.2e-5, tri[..., :3].shape).astype(np.float32) * (it % 2)
        tri[..., :3] *= np.float32(1 - 2 * (it // 2))
        out.append((tri, TRANSFORM if it == 3 else None))
    return out


def test_live_against_the_references_mesh_classes(tmp_path):
    """the reference's results on live_soups() -- merged vertices, colours, faces, PLY bytes -- are stored in tests/golden/reference_host_cases.npz
    (scripts/make_golden_reference_host_cases.py); where oracle/_ref is built, its classes compute them again"""
    g, h = np.load(GOLDEN), load("reference_host_cases.npz")
    live = os.path.exists(REF_SO)
    for it, (tri, transform) in enumerate(live_soups()):
        assert int(h[f"mesh{it}_input_crc"]) == input_crc(tri), it
        wp, wc, wf, wply = (h[f"mesh{it}_{k}"] for k in ("pos", "col", "faces", "ply"))
        lp = str(tmp_path / "l.ply")
        p, c, f = library_save(tri, transform, lp)
        assert np.array_equal(p.view(np.uint32), wp.view(np.uint32)) and np.array_equal(c, wc) and np.array_equal(f, wf)
        assert open(lp, "rb").read() == wply.tobytes()
        if live:
            rp = str(tmp_path / "r.ply")
            rp_, rc_, rf_ = reference_save(tri, transform, rp)
            assert np.array_equal(rp_.view(np.uint32), wp.view(np.uint32)) and np.array_equal(rc_, wc) and np.array_equal(rf_, wf) and open(rp, "rb").read() == wply.tobytes()
    if live:
        assert np.array_equal(reference_save(soups()["b"], None, str(tmp_path / "g.ply"))[2], g["faces_b"])       # the golden file is what the reference produces now
