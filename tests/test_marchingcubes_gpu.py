"""Iso-surface extraction on the GPU (csrc/marching_cubes.cu behind include/bf_marchingcubes.h) against oracle/marchingcubes_oracle.c: the multiset of triangles --
positions and colours bit for bit, the three vertices of a triangle in the reference's order (the order of the soup itself is undefined in the reference, which appends
with atomics).  The model is fused by the library's bit-exact TSDF kernels (arithmetic="exact"), the oracle's by its own: hash slots differ, voxel values do not."""
import ctypes as C
import os

import numpy as np
import pytest

from bundlefusion_b200 import _capi as capi
from bundlefusion_b200 import synth
from bundlefusion_b200.marching_cubes import CUDAMarchingCubesHashSDF, marching_cubes_params, merge_close_vertices, remove_duplicate_faces
from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params
from oracle import oracle as orc
from tests.test_marchingcubes_reference_emulated import canon

pytestmark = pytest.mark.gpu
W, H = 160, 120
BUCKETS, BLOCKS = 50021, 40000


def build(dev, n_frames=3, first=5):
    import torch
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=BUCKETS, num_sdf_blocks=BLOCKS)
    gpu = CUDASceneRepHashSDF(hp, dev, arithmetic="exact")
    cpu = orc.OracleSceneRepHashSDF(hp)
    for i in range(n_frames):
        d, c, T = synth.make_frame(first + i, W, H)
        gpu.integrate(T, torch.from_numpy(d).to(dev), torch.from_numpy(c).to(dev), cam)
        cpu.integrate(T, d, c, cam)
    return gpu, cpu


def soup_triangles(mc):
    pos, col = mc.soup()
    return np.concatenate([pos, col[:, :3]], axis=1).reshape(-1, 3, 6), col


def test_marching_cubes_matches_oracle_bit_for_bit(cuda_device, tmp_path):
    gpu, cpu = build(cuda_device)
    p = marching_cubes_params(BUCKETS, voxel_size=float(cpu.hp.m_virtualVoxelSize), max_num_triangles=600000)
    want, found = orc.marchingcubes_extract(cpu, p)
    assert found == len(want) and 20000 < len(want) < 600000
    mc = CUDAMarchingCubesHashSDF(p, cuda_device)
    assert mc.extractIsoSurface(gpu) == 3 * len(want)
    got, col = soup_triangles(mc)
    assert np.array_equal(canon(got), canon(want)) and np.all(col[:, 3] == 1.0)
    # an axis-aligned box through the scene: only cells whose centre is inside; the triangles are appended to the buffer
    lo, hi = want[..., :3].reshape(-1, 3).min(0), want[..., :3].reshape(-1, 3).max(0)
    box = ((float(lo[0]) - 1.0, float(lo[1]) - 1.0, float(lo[2]) - 1.0), (float(0.5 * (lo[0] + hi[0])), float(hi[1]) + 1.0, float(hi[2]) + 1.0))
    pb = marching_cubes_params(BUCKETS, voxel_size=float(cpu.hp.m_virtualVoxelSize), max_num_triangles=600000)
    pb.m_boxEnabled = 1
    for k in range(3):
        pb.m_minCorner[k], pb.m_maxCorner[k] = box[0][k], box[1][k]
    wantb, _ = orc.marchingcubes_extract(cpu, pb)
    assert 0 < len(wantb) < len(want)
    assert mc.extractIsoSurface(gpu, box[0], box[1], True) == 3 * (len(want) + len(wantb))
    got2, _ = soup_triangles(mc)
    assert np.array_equal(canon(got2[len(want):]), canon(wantb)) and np.array_equal(got2[:len(want)], got)
    # saveMesh: merge / de-duplicate / PLY; an existing file is kept and the name counts up; the buffer is cleared.  The soup's order is the
    # order of the atomic appends, so it differs between extractions, and with it which vertex of a merged cluster survives: each file is
    # checked against the soup it was made from.
    mc.clearMeshBuffer()
    mc.extractIsoSurface(gpu)
    soup1 = mc.soup()
    path = str(tmp_path / "scans" / "scan.ply")
    first = mc.saveMesh(path)
    assert first == path and os.path.exists(path) and mc.soup()[0].shape[0] == 0
    mc.extractIsoSurface(gpu)
    soup2 = mc.soup()
    assert np.array_equal(canon(soup_triangles(mc)[0]), canon(want))
    second = mc.saveMesh(path, transform=np.diag([2.0, 2.0, 2.0, 1.0]).astype(np.float32))
    assert second == str(tmp_path / "scans" / "scan1.ply") and os.path.exists(second)

    def merged(soup):
        pos, col = soup
        p, c, f = merge_close_vertices(pos, col, np.arange(len(pos), dtype=np.uint32).reshape(-1, 3), 0.00001)
        return p, (c * 255).astype(np.uint8), remove_duplicate_faces(f)

    def read_ply(f):
        head, body = open(f, "rb").read().split(b"end_header\n", 1)
        lines = head.decode().splitlines()
        nv = int([l for l in lines if l.startswith("element vertex")][0].split()[-1]); nf = int([l for l in lines if l.startswith("element face")][0].split()[-1])
        v = np.frombuffer(body[:16 * nv], np.dtype([("p", "<f4", 3), ("c", "u1", 4)]))
        fa = np.frombuffer(body[16 * nv:], np.dtype([("n", "u1"), ("i", "<i4", 3)]))
        assert len(fa) == nf
        return v, fa
    v1, f1 = read_ply(first)
    v2, f2 = read_ply(second)
    # the merged mesh: every cell edge vertex once instead of once per adjoining triangle; (almost) every triangle survives
    assert len(v1) < len(want) and 0.98 * len(want) < len(f1) <= len(want) and f1["i"].max() <= len(v1) - 1 and f1["i"].min() == 0
    for (v, fa), soup, scale in (((v1, f1), soup1, 1.0), ((v2, f2), soup2, 2.0)):
        p, c, f = merged(soup)
        assert len(v) == len(p) and np.allclose(v["p"], scale * p, rtol=1e-6, atol=0) and np.array_equal(v["c"], c) and np.array_equal(fa["i"], f.astype(np.int32))
    assert abs(len(v2) - len(v1)) <= 1e-3 * len(v1) and abs(len(f2) - len(f1)) <= 1e-3 * len(f1)
    mc.close(); gpu.close()


def test_full_buffer_reference_named_stubs_and_empty_model(cuda_device):
    import torch
    gpu, cpu = build(cuda_device, n_frames=2, first=30)
    L = capi.lib()
    vp = C.c_void_p
    L.bfMarchingCubesExtract.argtypes = [vp] * 5
    L.resetMarchingCubesCUDA.argtypes = [vp]; L.resetMarchingCubesCUDA.restype = None
    L.extractIsoSurfaceCUDA.argtypes = [vp] * 4; L.extractIsoSurfaceCUDA.restype = None
    L.updateConstantHashParams.argtypes = [vp]
    L.bfSetStream(C.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream))
    p = marching_cubes_params(BUCKETS, voxel_size=float(cpu.hp.m_virtualVoxelSize), max_num_triangles=600000)
    want, _ = orc.marchingcubes_extract(cpu, p)
    full = {r.tobytes() for r in canon(want)}
    # a buffer of 5000 triangles: the count stops at the capacity, what is written are triangles of the model
    cap = 5000
    pc = marching_cubes_params(BUCKETS, voxel_size=float(cpu.hp.m_virtualVoxelSize), max_num_triangles=cap)
    tri = torch.zeros(cap + 16, 18, device=cuda_device); n = torch.full((1,), 9, dtype=torch.int32, device=cuda_device)
    tri[cap:] = 7.0
    assert L.bfMarchingCubesExtract(C.byref(gpu.getHashData()), C.byref(gpu.getHashParams()), C.byref(pc), tri.data_ptr(), n.data_ptr()) == 0
    torch.cuda.synchronize()
    assert int(n.item()) == cap and bool((tri[cap:] == 7.0).all())                       # nothing past the capacity
    rows = canon(tri[:cap].cpu().numpy().reshape(cap, 3, 6))
    assert all(r.tobytes() in full for r in rows)
    # the reference's call sequence with the parameters in device memory
    dparams = torch.from_numpy(np.frombuffer(bytes(p), np.uint8).copy()).to(cuda_device)
    big = torch.zeros(len(want) + 8, 18, device=cuda_device)
    p.m_maxNumTriangles = len(want) + 8
    dparams = torch.from_numpy(np.frombuffer(bytes(p), np.uint8).copy()).to(cuda_device)
    data = capi.BFMarchingCubesData(dparams.data_ptr(), n.data_ptr(), big.data_ptr(), 1)
    L.updateConstantHashParams(C.byref(gpu.getHashParams()))
    L.resetMarchingCubesCUDA(C.byref(data))
    torch.cuda.synchronize()
    assert int(n.item()) == 0
    L.extractIsoSurfaceCUDA(C.byref(gpu.getHashData()), None, C.byref(p), C.byref(data))
    torch.cuda.synchronize()
    assert int(n.item()) == len(want)
    assert np.array_equal(canon(big[:len(want)].cpu().numpy().reshape(-1, 3, 6)), canon(want))
    gpu.close()
    # an empty model has no surface
    hp = default_hash_params(num_buckets=BUCKETS, num_sdf_blocks=BLOCKS)
    empty = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="exact")
    mc = CUDAMarchingCubesHashSDF(pc, cuda_device)
    assert mc.extractIsoSurface(empty) == 0
    mc.close(); empty.close()
