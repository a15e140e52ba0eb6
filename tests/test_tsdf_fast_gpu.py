"""The TOLERANCE-arithmetic stencil (bundlefusion_b200/csrc/tsdf_fast.cu, the library default and the path bench.py times) against
the oracle, against the library's own bit-exact kernels and against the reference's CUDA build -- both of its builds: IEEE and the
--use_fast_math one FriedLiver ships.

Contract (include/bf_tsdf.h, bfTsdfSetArithmetic):
* allocated block set, in-frustum list, heap count: identical (allocation and list building do not change with the arithmetic);
* weights identical, |d sdf| <= 1e-5 m, colour within 1 level -- for all voxels but a counted fraction <= 1e-4 whose projected pixel or
  truncation test sits within float rounding distance of its decision boundary (such a voxel samples the neighbouring depth pixel, or is
  / is not updated: weight differs by one).  The reference's own fast-math build differs from its IEEE build in the same way
  (profiles/r1_tsdf_parity_vs_reference_cuda.txt: 1.1e-5 flips, 5e-7 weight mismatches)."""
import numpy as np
import pytest

from bundlefusion_b200 import _capi as capi
from bundlefusion_b200 import synth
from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params
from oracle import oracle as orc
from tests._golden import block_crcs
from tests.test_tsdf_vs_reference_gpu import compare_states, compare_with_reference, reference_stream

pytestmark = pytest.mark.gpu
F = np.float32
SDF_TOL = 1e-5


def _frames(torch, dev, n, W, H, step=30):
    frames = [synth.make_frame(step * i, W, H) for i in range(n)]
    return frames, [torch.from_numpy(f[0]).to(dev) for f in frames], [torch.from_numpy(f[1]).to(dev) for f in frames]


def test_fast_stream_matches_oracle(cuda_device):
    """integrate x 6, separate de-integrate / integrate at updated poses, lone de-integration, GC -- fast kernels vs the CPU oracle."""
    import torch
    W, H = 320, 240
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=100003, num_sdf_blocks=60000)
    gpu, cpu = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast"), orc.OracleSceneRepHashSDF(hp)
    frames, dl, cl = _frames(torch, cuda_device, 6, W, H)
    for (d, c, T), dd, dc in zip(frames, dl, cl):
        gpu.integrate(T, dd, dc, cam)
        cpu.integrate(T, d, c, cam)
    s1 = compare_states(gpu.download(), cpu.download(), SDF_TOL)
    assert gpu.getNumOccupiedBlocks() == cpu.num_occupied and gpu.getHeapFreeCount() == cpu.getHeapFreeCount()
    st = gpu.getLastFrameStats()
    assert st["E"] == cpu.num_occupied and abs(int(st["U"]) - int(cpu.last_U)) <= max(4, 1e-4 * cpu.last_U)
    for k in (1, 4):
        d, c, T = frames[k]
        T2 = T.copy(); T2[:3, 3] += np.array([0.011, -0.006, 0.004], F)
        gpu.deIntegrate(T, dl[k], cl[k], cam); gpu.integrate(T2, dl[k], cl[k], cam)
        cpu.deIntegrate(T, d, c, cam); cpu.integrate(T2, d, c, cam)
    gpu.deIntegrate(frames[0][2], dl[0], cl[0], cam); cpu.deIntegrate(frames[0][2], frames[0][0], frames[0][1], cam)
    gpu.garbageCollect(); cpu.garbageCollect()
    s2 = compare_states(gpu.download(), cpu.download(), 10 * SDF_TOL)       # de-integration divides by (w - 1): differences grow a little
    assert gpu.getHeapFreeCount() == cpu.getHeapFreeCount()
    print("fast vs oracle:", s1, s2)


def test_fast_fused_reintegration_matches_oracle_and_exact_kernels(cuda_device):
    """bfTsdfRunOps with fused (de-integrate old pose, integrate new pose) pairs: the fast fused kernel vs the oracle's two passes and vs
    the library's own bit-exact kernels on the same op list."""
    import torch
    W, H = 320, 240
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=100003, num_sdf_blocks=60000)
    fast = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast")
    exact = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="exact")
    cpu = orc.OracleSceneRepHashSDF(hp)
    frames, dl, cl = _frames(torch, cuda_device, 6, W, H, step=35)
    ops = [(capi.BF_TSDF_OP_INTEGRATE, i, frames[i][2]) for i in range(6)]
    for d, c, T in frames:
        cpu.integrate(T, d, c, cam)
    rng = np.random.default_rng(4)
    for k in (4, 2, 0, 5, 2):
        T = frames[k][2]
        T2 = (synth.se3_exp(rng.standard_normal(3) * 0.01, rng.standard_normal(3) * 0.02) @ T.astype(np.float64)).astype(F)
        ops += [(capi.BF_TSDF_OP_DEINTEGRATE, k, T), (capi.BF_TSDF_OP_INTEGRATE, k, T2)]
        cpu.deIntegrate(T, frames[k][0], frames[k][1], cam); cpu.integrate(T2, frames[k][0], frames[k][1], cam)
        frames[k] = (frames[k][0], frames[k][1], T2)
    ops.append((capi.BF_TSDF_OP_GARBAGE_COLLECT, 0, None))
    cpu.garbageCollect()
    fast.runOps(ops, dl, cl, cam)
    exact.runOps(ops, dl, cl, cam)
    fs, es = fast.download(), exact.download()
    s_orc = compare_states(fs, cpu.download(), 10 * SDF_TOL)
    s_exact = compare_states(fs, es, 10 * SDF_TOL)
    eb, ev = orc.canonical_blocks(es); cb, cv = orc.canonical_blocks(cpu.download())
    np.testing.assert_array_equal(ev, cv)                                  # the exact kernels stay bit-identical to the oracle
    assert fast.getHeapFreeCount() == exact.getHeapFreeCount() == cpu.getHeapFreeCount()
    print("fast fused vs oracle / exact:", s_orc, s_exact)


@pytest.mark.parametrize("fast_math", [False, True])
def test_fast_stream_matches_reference_cuda(cuda_device, fast_math):
    """the same statement against the reference's own CUDA kernels, IEEE build and --use_fast_math build, through their stored states
    (tests/test_tsdf_vs_reference_gpu.py): the IEEE build's state is the oracle's -- every block's CRC equals the stored one -- and is compared
    whole; the fast-math build's on its stored sample of blocks"""
    import torch
    W, H = 320, 240
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=100003, num_sdf_blocks=60000)
    ours = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast")
    frames, dl, cl = _frames(torch, cuda_device, 6, W, H)
    g = reference_stream(fast_math, frames)
    cpu = None if fast_math else orc.OracleSceneRepHashSDF(hp)
    tol = 1e-4 if fast_math else SDF_TOL          # the reference's fast-math build is itself ~1e-5 away from IEEE

    def compare(stage, sdf_tol):
        if fast_math:
            return compare_with_reference(ours.download(), g, stage, sdf_tol, exact=False)
        rb, rv = orc.canonical_blocks(cpu.download())
        np.testing.assert_array_equal(rb, g[f"blocks{stage}"]); np.testing.assert_array_equal(block_crcs(rv), g[f"crcs{stage}"])
        return compare_states(ours.download(), (rb, rv), sdf_tol)

    for (d, c, T), dd, dc in zip(frames, dl, cl):
        ours.integrate(T, dd, dc, cam)
        if cpu is not None: cpu.integrate(T, d, c, cam)
    s1 = compare(1, tol)
    assert ours.getNumOccupiedBlocks() == int(g["occupied1"]) and ours.getHeapFreeCount() == int(g["heap_free1"])
    for k in (1, 4):
        d, c, T = frames[k]
        T2 = T.copy(); T2[:3, 3] += np.array([0.011, -0.006, 0.004], F)
        ours.runOps([(capi.BF_TSDF_OP_DEINTEGRATE, k, T), (capi.BF_TSDF_OP_INTEGRATE, k, T2)], dl, cl, cam)       # fused pass
        if cpu is not None: cpu.deIntegrate(T, d, c, cam); cpu.integrate(T2, d, c, cam)
    ours.deIntegrate(frames[0][2], dl[0], cl[0], cam); ours.garbageCollect()
    if cpu is not None: cpu.deIntegrate(frames[0][2], frames[0][0], frames[0][1], cam); cpu.garbageCollect()
    s2 = compare(2, 10 * tol)
    assert ours.getHeapFreeCount() == int(g["heap_free2"])
    print("fast vs reference CUDA (fast_math=%s):" % fast_math, s1, s2)


def test_fast_full_size_round_trip_properties(cuda_device):
    """BASELINE size (640x480, 1 cm voxels), size-independent properties: integrate then de-integrate the same frames at the same poses
    and garbage-collect -> every block is freed (weights are whole numbers in both arithmetics) and every voxel word is zero;
    integrating a frame twice doubles every touched weight."""
    import torch
    W, H = 640, 480
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=400009, num_sdf_blocks=120000)
    gpu = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast")
    frames, dl, cl = _frames(torch, cuda_device, 3, W, H, step=25)
    free0 = gpu.getHeapFreeCount()
    for (d, c, T), dd, dc in zip(frames, dl, cl):
        gpu.integrate(T, dd, dc, cam)
    assert gpu.getHeapFreeCount() < free0
    w1 = gpu.d_SDFBlocks.view(torch.float32).reshape(-1, 3)[:, 1].clone()
    gpu.integrate(frames[0][2], dl[0], cl[0], cam)
    w2 = gpu.d_SDFBlocks.view(torch.float32).reshape(-1, 3)[:, 1]
    dw = (w2 - w1)
    assert set(torch.unique(dw).tolist()) <= {0.0, 1.0} and int((dw == 1).sum()) == gpu.getLastFrameStats()["U"]
    gpu.deIntegrate(frames[0][2], dl[0], cl[0], cam)
    for (d, c, T), dd, dc in zip(frames, dl, cl):
        gpu.deIntegrate(T, dd, dc, cam)
        gpu.garbageCollect()
    assert gpu.getHeapFreeCount() == free0
    assert int(gpu.d_SDFBlocks.abs().max()) == 0
    h = gpu.download()["hash"]
    assert (h[:, 3] == -2).all()


def test_batched_reintegration_equals_pair_by_pair(cuda_device):
    """bfTsdfRunOps with batching (n alloc launches, one union list, one multi-op stencil pass per run of re-integration pairs) against the same
    op list replayed pair by pair, both in fast arithmetic: voxels, block set and heap must be IDENTICAL bit for bit -- the batch changes how
    often a voxel travels, not what happens to it; a block inserted by pair k's alloc stays invisible to the pairs before k."""
    import torch
    W, H = 320, 240
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=100003, num_sdf_blocks=60000)
    L = capi.lib()
    frames, dl, cl = _frames(torch, cuda_device, 8, W, H, step=35)
    rng = np.random.default_rng(11)
    ops = [(capi.BF_TSDF_OP_INTEGRATE, i, frames[i][2]) for i in range(6)]
    cur = [f[2] for f in frames]
    def pair(k, big=False):
        T = cur[k]
        s = 0.05 if big else 0.01
        T2 = (synth.se3_exp(rng.standard_normal(3) * s, rng.standard_normal(3) * 2 * s) @ T.astype(np.float64)).astype(F)
        cur[k] = T2
        return [(capi.BF_TSDF_OP_DEINTEGRATE, k, T), (capi.BF_TSDF_OP_INTEGRATE, k, T2)]
    for k in (4, 2, 0, 5, 2, 1, 3):                      # frame 2 moves twice inside one batch
        ops += pair(k)
    ops.append((capi.BF_TSDF_OP_GARBAGE_COLLECT, 0, None))
    ops.append((capi.BF_TSDF_OP_INTEGRATE, 6, frames[6][2]))
    for k in (6, 0, 3):
        ops += pair(k, big=True)                         # large moves: their allocs insert blocks the earlier pairs of the batch must not see
    ops += [(capi.BF_TSDF_OP_GARBAGE_COLLECT, 0, None), (capi.BF_TSDF_OP_INTEGRATE, 7, frames[7][2])]
    states = []
    for batching in (1, 0):
        prev = L.bfTsdfSetBatching(batching)
        try:
            sc = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast")
            l0 = L.bfGetLaunchCount()
            sc.runOps(ops, dl, cl, cam)
            torch.cuda.synchronize()
            states.append((orc.canonical_blocks(sc.download()), sc.getHeapFreeCount(), L.bfGetLaunchCount() - l0, sc.getLastFrameStats()))
        finally:
            L.bfTsdfSetBatching(prev)
    (b1, v1), h1, n1, st1 = states[0]
    (b0, v0), h0, n0, st0 = states[1]
    np.testing.assert_array_equal(b1, b0)
    np.testing.assert_array_equal(v1, v0)
    assert h1 == h0 and n1 < n0
    # and the whole thing within the tolerance contract of the oracle's pair-by-pair replay
    cpu = orc.OracleSceneRepHashSDF(hp)
    for kind, f, T in ops:
        if kind == capi.BF_TSDF_OP_GARBAGE_COLLECT: cpu.garbageCollect()
        elif kind == capi.BF_TSDF_OP_DEINTEGRATE: cpu.deIntegrate(T, frames[f][0], frames[f][1], cam)
        else: cpu.integrate(T, frames[f][0], frames[f][1], cam)
    sc = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="fast")
    sc.runOps(ops, dl, cl, cam)
    print("batched fast vs oracle:", compare_states(sc.download(), cpu.download(), 10 * SDF_TOL), "launches batched / pair by pair:", n1, n0)
    assert sc.getHeapFreeCount() == cpu.getHeapFreeCount()
