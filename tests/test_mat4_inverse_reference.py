"""The host-side 4x4 inverse (bfMat4Inverse; what forms m_rigidTransformInverse for every TSDF operation and the ray cast's view matrix) pinned against BOTH of the
reference's implementations, compiled by g++ from /root/reference: float4x4::getInverse (FL/SiftGPU/cuda_SimpleMatrixUtil.h:980-1100, in oracle/_ref/libref_kabsch_host.so)
and mLib's mat4f::getInverse (core-math/matrix4x4.h:587-710, in libref_mesh_host.so).  scripts/make_golden_mat4_inverse.py stored their outputs on the matrices below in
tests/golden/mat4_inverse_reference.npz.  Bit for bit: an inverse that differs in the last place moves TSDF voxel words (round 2 found one block in 4 478 differing
on the golden scene when the inverse was formed through 2x2 sub-determinants instead)."""
import ctypes as C
import os

import numpy as np

from bundlefusion_b200 import scene_rep
from oracle import oracle as orc
from tests._golden import input_crc, load

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "mat4_inverse_reference.npz")
KABSCH_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_kabsch_host.so")
MESH_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_mesh_host.so")


def matrices(seed=3, n=600):
    """rigid poses (the application's case), intrinsics-shaped matrices, and general well-conditioned ones"""
    from bundlefusion_b200 import synth
    rng = np.random.default_rng(seed)
    out = [synth.make_frame(i, 32, 24)[2].astype(np.float32) for i in range(0, 200, 5)]
    for _ in range(n):
        ax = rng.normal(size=3); ax /= np.linalg.norm(ax); th = rng.uniform(-3.1, 3.1)
        Kx = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
        T = np.eye(4); T[:3, :3] = np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx; T[:3, 3] = rng.uniform(-4, 4, 3)
        out.append(T.astype(np.float32))
    for fx, mx in ((525.0, 319.5), (583.0, 320.0), (131.25, 79.5), (1170.2, 647.75)):
        out.append(np.array([[fx, 0, mx, 0], [0, fx * 1.01, mx * 0.75, 0], [0, 0, 1, 0], [0, 0, 0, 1]], np.float32))
    for _ in range(100):
        out.append((np.eye(4) * 2 + rng.normal(size=(4, 4)) * 0.4).astype(np.float32))
    return np.stack(out)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def ref_inverses(M):
    fp = C.c_void_p
    K, S = C.CDLL(KABSCH_SO), C.CDLL(MESH_SO)
    a, b = np.zeros_like(M), np.zeros_like(M)
    for i in range(len(M)):
        m = np.ascontiguousarray(M[i])
        K.refHostFloat4x4Inverse(fp(m.ctypes.data), fp(a[i].ctypes.data)); S.ref_mlib_mat4_inverse(fp(m.ctypes.data), fp(b[i].ctypes.data))
    return a, b


def test_host_inverse_equals_both_reference_implementations():
    g = np.load(GOLDEN)
    M = matrices()
    assert np.array_equal(bits(M), bits(g["matrices"]))
    assert np.array_equal(bits(g["float4x4"]), bits(g["mat4f"]))                              # the reference's two classes agree with each other
    lib = np.stack([scene_rep.mat4_inverse_f32(m) for m in M])                                 # bfMat4Inverse: host code of the library
    oracle = np.stack([orc.mat4_inverse(m) for m in M])
    assert np.array_equal(bits(lib), bits(g["float4x4"])) and np.array_equal(bits(oracle), bits(g["float4x4"]))
    assert np.abs(np.einsum("nij,njk->nik", lib[:640].astype(np.float64), M[:640].astype(np.float64)) - np.eye(4)).max() < 1e-5


def test_live_against_the_reference_classes():
    """another 344 matrices: both classes' inverses are stored in tests/golden/reference_host_cases.npz (scripts/make_golden_reference_host_cases.py);
    where oracle/_ref is built, the classes compute them again"""
    g = load("reference_host_cases.npz")
    M = matrices(seed=99, n=300)
    assert int(g["mat4_input_crc"]) == input_crc(M)
    a, b = g["mat4_float4x4"], g["mat4_mat4f"]
    if os.path.exists(KABSCH_SO) and os.path.exists(MESH_SO):
        la, lb = ref_inverses(M)
        assert np.array_equal(bits(la), bits(a)) and np.array_equal(bits(lb), bits(b))
    lib = np.stack([scene_rep.mat4_inverse_f32(m) for m in M])
    assert np.array_equal(bits(a), bits(b)) and np.array_equal(bits(lib), bits(a))
