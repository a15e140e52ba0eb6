"""Parity of the bundle-adjustment solver against the REFERENCE'S OWN CUDA solver (FL/Solver/SolverBundling.cu + FL/SBA.cu built for sm_100a
with the compatibility patch of oracle/build_ref.py), on identical correspondences, cache frames and initial poses, on the GPU.  The reference's
results are stored in tests/golden/solver_vs_reference_cuda.npz (scripts/make_golden_reference_cuda.py ran its kernels on a B200, IEEE and
--use_fast_math builds), each with a CRC of the inputs it was computed from.  This is what pins the CPU oracle (oracle/solver_oracle.c) too: the
same cases are run through it and compared with the reference's output.

Tolerance (BASELINE.json north_star): solved poses within 1e-4 relative L2.  The reference accumulates with float atomics, so its
own result moves in the last bits from run to run; the PCG early-out |p.Ap| < 5e-7 is absolute (see tests/test_solver_gpu.py)."""
import ctypes as C

import numpy as np
import pytest

from bundlefusion_b200 import _capi as capi
from bundlefusion_b200 import synth
from bundlefusion_b200.solver import CUDASolverBundling, DeviceCache
from oracle import oracle as orc
from tests._golden import input_crc, load

pytestmark = pytest.mark.gpu
TOL = 1e-4


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-12)


def _dev_inputs(dev, prob, corr):
    import torch
    c = np.ascontiguousarray(corr)
    corr_t = torch.from_numpy(c.view(np.uint8).reshape(-1).copy()).to(dev) if len(c) else torch.zeros(32, dtype=torch.uint8, device=dev)
    rot = torch.from_numpy(prob["init_rot"].copy()).to(dev)
    trans = torch.from_numpy(prob["init_trans"].copy()).to(dev)
    valid = torch.ones(len(prob["init_rot"]), dtype=torch.int32, device=dev)
    return corr_t, rot, trans, valid


def run_ours(dev, prob, corr, n_gn, n_pcg, wS, wD=None, wC=None, cache=None):
    import torch
    N = len(prob["init_rot"])
    corr_t, rot, trans, valid = _dev_inputs(dev, prob, corr)
    s = CUDASolverBundling(N, max(len(corr), 1000 * N), dev)
    s.solve(corr_t, len(corr), valid, N, n_gn, n_pcg, wS, wD, wC, d_rotationAnglesUnknowns=rot, d_translationUnknowns=trans, cudaCache=cache)
    torch.cuda.synchronize()
    return np.c_[rot.cpu().numpy(), trans.cpu().numpy()], s.getStats()


def reference(key, prob):
    """the reference's stored results of case `key`, after checking they were computed from these inputs"""
    g = load("solver_vs_reference_cuda.npz")
    assert int(g[key + "_input_crc"]) == input_crc(prob), f"the stored reference results of {key} were computed from other inputs"
    return lambda name: g[f"{key}_{name}"]


@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("n_images,degree,n_gn,n_pcg", [(2, 1, 4, 50), (11, 10, 2, 100), (60, 8, 3, 150), (200, 12, 4, 150)])
def test_sparse_solve_matches_reference_cuda(cuda_device, n_images, degree, n_gn, n_pcg, fast):
    cpp = 256 if n_images == 2 else 25
    prob = synth.make_ba_problem(n_images, degree=degree, corr_per_pair=cpp, noise=0.002, seed=5)
    w = [1.0] * n_gn
    ref = reference(f"sparse_{n_images}_{int(fast)}", prob)
    x_ref, conv = ref("x"), ref("conv")
    x_our, st = run_ours(cuda_device, prob, prob["corr"], n_gn, n_pcg, w)
    o = orc.solve_sparse(prob["corr"], prob["init_rot"], prob["init_trans"], n_gn, n_pcg)
    x_orc = np.c_[o["rot"], o["trans"]]
    assert st["error"] == 0
    assert np.isfinite(x_ref).all()
    assert rel_l2(x_our, x_ref) < TOL, "CUDA path vs reference CUDA"
    assert rel_l2(x_orc, x_ref) < TOL, "CPU oracle vs reference CUDA (pins the oracle)"
    # the reference's own energy record (EvalResidual after each GN iteration) agrees with the oracle's energy of our result
    e_ref_final = float(conv[conv >= 0][-1])
    e_our = orc.energy(prob["corr"], x_our[:, :3].astype(np.float32), x_our[:, 3:].astype(np.float32))
    assert e_our <= e_ref_final * 1.02 + 1e-7
    np.testing.assert_array_equal(x_ref[0], x_our[0])                       # variable 0 is fixed in both


def _ulp_perturbed(prob, seed):
    """initial poses moved by at most 2 ulp (variable 0 untouched): the size of the perturbation a different float summation order is"""
    rng = np.random.default_rng(seed)
    r, t = prob["init_rot"].copy(), prob["init_trans"].copy()
    r = (r * (1 + rng.integers(-2, 3, r.shape) * 6e-8)).astype(np.float32)
    t = (t * (1 + rng.integers(-2, 3, t.shape) * 6e-8)).astype(np.float32)
    r[0], t[0] = prob["init_rot"][0], prob["init_trans"][0]
    return r, t


def oracle_sensitivity(prob, corr, n_gn, n_pcg, wS, wD, wC, n=4):
    """Largest relative-L2 move of the ORACLE's solution under 2-ulp perturbations of the initial poses.  The reference sums with float
    atomics in scheduling order (SURVEY.md Q14), i.e. it perturbs itself by about this much from run to run; a problem whose solution
    moves more than the parity tolerance under such a perturbation cannot pin anything at that tolerance."""
    o = orc.solve(corr, prob["init_rot"], prob["init_trans"], n_gn, n_pcg, wS, wD, wC, prob["caches"], prob["intrinsics"])
    x0 = np.c_[o["rot"], o["trans"]]
    worst = 0.0
    for k in range(n):
        r, t = _ulp_perturbed(prob, k)
        q = orc.solve(corr, r, t, n_gn, n_pcg, wS, wD, wC, prob["caches"], prob["intrinsics"])
        worst = max(worst, rel_l2(np.c_[q["rot"], q["trans"]], x0))
    return worst, o


def test_dense_only_matches_reference_cuda(cuda_device):
    """Dense depth term alone (PCGIteration<false,true>, SolverBundling.cu:1181-1184).  The problem is CERTIFIED well-posed by the oracle
    before it is used: its solution moves < 1e-5 under 2-ulp input perturbations and every early-out decision (|p.Ap| vs 5e-7 / 1e-6,
    max|delta| vs 0.005) is at least 30 % clear of its threshold."""
    prob = synth.make_dense_ba_problem(8, stride=2, perturb_rot=0.004, perturb_trans=0.008, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], cuda_device)
    wS, wD, wC = [0.0] * 2, [1.0, 2.0], [0.0] * 2
    empty = prob["corr"][:0]
    sens, o = oracle_sensitivity(prob, empty, 2, 10, wS, wD, wC)
    assert sens < 1e-5 and orc.decision_margin(o["trace"]) > 0.3, "test problem is not well-posed"
    ref = reference("dense_only", prob)
    x_ref, x_ref2 = ref("x"), ref("x2")                                     # two runs of the reference
    x_our, st = run_ours(cuda_device, prob, empty, 2, 10, wS, wD, wC, cache=cache)
    n_overlap_ref = int(ref("overlap"))
    assert st["dense_overlap_pairs"] == n_overlap_ref == o["overlap_pairs"]
    assert rel_l2(x_ref2, x_ref) < TOL, "the reference does not reproduce itself on this problem"
    assert rel_l2(x_our, x_ref) < TOL
    assert rel_l2(np.c_[o["rot"], o["trans"]], x_ref) < TOL


def test_dense_only_chaotic_configuration_is_bounded_by_its_own_sensitivity(cuda_device):
    """Round 1's dense-only case (5 frames, 3 GN x 60 PCG) FAILED on the driver's box at 2.1e-2 after passing on another.  Cause, found
    with the oracle: with weightSparse == 0 the preconditioner is the identity, PCG stagnates with |p.Ap| hovering around the 5e-7 / 1e-6
    guards, and whether iteration 16 of the first Gauss-Newton step takes the early-out decides between two end points 2e-2 apart -- a
    2-ulp change of the input flips it (the oracle shows the same 2.1e-2 against itself).  The reference's float atomics are such a
    change.  So here the bound is the problem's own measured sensitivity, and the fixed-order implementations (library, oracle) must
    still agree with each other."""
    prob = synth.make_dense_ba_problem(5, stride=3, perturb_rot=0.004, perturb_trans=0.008, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], cuda_device)
    wS, wD, wC = [0.0] * 3, [1.0, 2.0, 3.0], [0.0] * 3
    empty = prob["corr"][:0]
    sens, o = oracle_sensitivity(prob, empty, 3, 60, wS, wD, wC, n=6)
    assert sens > 1e-3, "this configuration is expected to be chaotic (documented above)"
    ref = reference("chaotic", prob)
    x_ref = ref("x")
    x_our, _ = run_ours(cuda_device, prob, empty, 3, 60, wS, wD, wC, cache=cache)
    assert rel_l2(x_our, x_ref) < max(TOL, 3 * sens)
    # the first Gauss-Newton step truncated before the stagnation (10 PCG iterations) is decided identically by everyone
    x_ref1 = ref("x1")
    x_our1, _ = run_ours(cuda_device, prob, empty, 1, 10, wS[:1], wD[:1], wC[:1], cache=cache)
    assert rel_l2(x_our1, x_ref1) < 2e-4


@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("wC", [[0.0, 0.0], [0.1, 0.1]])
def test_local_chunk_sparse_plus_dense_matches_reference_cuda(cuda_device, wC, fast):
    """The reference's local BA configuration (FL/SBA.cpp:28-31): 11 frames, 2 GN x 100 PCG, sparse 1, dense depth 1 -> 2."""
    prob = synth.make_dense_ba_problem(11, stride=3, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], cuda_device)
    wS, wD = [1.0, 1.0], [1.0, 2.0]
    ref = reference("local", prob)
    x_ref = ref(f"{int(wC[0] > 0)}_{int(fast)}_x")
    x_our, st = run_ours(cuda_device, prob, prob["corr"], 2, 100, wS, wD, wC, cache=cache)
    o = orc.solve(prob["corr"], prob["init_rot"], prob["init_trans"], 2, 100, wS, wD, wC, prob["caches"], prob["intrinsics"])
    assert st["dense_overlap_pairs"] == int(ref(f"{int(wC[0] > 0)}_{int(fast)}_overlap"))
    assert rel_l2(x_our, x_ref) < TOL
    assert rel_l2(np.c_[o["rot"], o["trans"]], x_ref) < TOL


def test_dense_system_matches_reference_cuda(cuda_device):
    """The assembled dense normal equations themselves: the reference's d_denseJtJ (6N x 6N) / d_denseJtr after BuildDenseSystem
    against THIS LIBRARY's (bfSolverDebugDenseSystem) and the oracle's, entry for entry (float-atomic summation order differs: relative
    Frobenius 1e-4).  This is the deterministic parity statement for row a13: no solver dynamics in between."""
    import torch
    prob = synth.make_dense_ba_problem(6, stride=3, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], cuda_device)
    N = 6
    # one GN iteration with zero PCG iterations leaves the poses untouched and the system of iteration 0 in the buffers
    ref = reference("dense_system", prob)
    x_ref = ref("x")
    np.testing.assert_array_equal(x_ref, np.c_[prob["init_rot"], prob["init_trans"]])
    JtJ_ref = ref("JtJ")
    Jtr_ref = ref("Jtr")
    JtJ, Jtr, _ = orc.build_dense(prob["init_rot"], prob["init_trans"], prob["caches"], prob["intrinsics"], 1.0, 0.1)
    assert np.linalg.norm(JtJ_ref) > 0
    assert rel_l2(JtJ, JtJ_ref) < TOL
    assert rel_l2(Jtr, Jtr_ref) < TOL
    # the library's own system
    corr_t, rot, trans, valid = _dev_inputs(cuda_device, prob, prob["corr"][:0])
    sv = CUDASolverBundling(N, 1000 * N, cuda_device)
    sv.solve(corr_t, 0, valid, N, 1, 0, [0.0], [1.0], [0.1], d_rotationAnglesUnknowns=rot, d_translationUnknowns=trans, cudaCache=cache)
    d_JtJ = torch.zeros(36 * N * N, device=cuda_device); d_Jtr = torch.zeros(6 * N, device=cuda_device)
    capi.check(sv.lib.bfSolverDebugDenseSystem(C.byref(sv.m_solverState), N, C.c_void_p(d_JtJ.data_ptr()), C.c_void_p(d_Jtr.data_ptr())), "bfSolverDebugDenseSystem")
    torch.cuda.synchronize()
    np.testing.assert_array_equal(np.c_[rot.cpu().numpy(), trans.cpu().numpy()], np.c_[prob["init_rot"], prob["init_trans"]])
    JtJ_our, Jtr_our = d_JtJ.cpu().numpy().reshape(6 * N, 6 * N), d_Jtr.cpu().numpy()
    # rows / columns of the fixed variable 0 are never read by either PCG; compare the part that is (and all of J^T r)
    assert rel_l2(JtJ_our[6:, 6:], JtJ_ref[6:, 6:]) < TOL, "library's dense J^T J vs the reference's"
    assert rel_l2(Jtr_our[6:], Jtr_ref[6:]) < TOL, "library's dense J^T r vs the reference's"
    blk = np.abs(JtJ_our[6:, 6:] - JtJ_ref[6:, 6:]).max() / np.abs(JtJ_ref[6:, 6:]).max()
    assert blk < 1e-4


def test_dense_term_beyond_64_images_matches_reference_cuda(cuda_device):
    """The dense term at N = 72 (> the 64 images the first version stopped at), where the reference's dense (6N)^2 matrix still fits comfortably:
    (a) this library's block-sparse system, scattered into the reference's layout, against the reference's d_denseJtJ / d_denseJtr entry for entry;
    (b) the solved poses of a sparse + dense depth + colour solve."""
    import torch
    N = 72
    prob = synth.make_dense_ba_problem(N, stride=1, start=60, corr_per_pair=8, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], cuda_device)
    ref = reference("beyond64", prob)
    JtJ_ref = np.zeros((6 * N, 6 * N), np.float32); JtJ_ref[6:, 6:] = ref("JtJ"); Jtr_ref = ref("Jtr")      # stored without the fixed variable 0's rows / columns
    corr_t, rot, trans, valid = _dev_inputs(cuda_device, prob, prob["corr"][:0])
    sv = CUDASolverBundling(N, 1000 * N, cuda_device)
    sv.solve(corr_t, 0, valid, N, 1, 0, [0.0], [1.0], [0.1], d_rotationAnglesUnknowns=rot, d_translationUnknowns=trans, cudaCache=cache)
    d_JtJ = torch.zeros(36 * N * N, device=cuda_device); d_Jtr = torch.zeros(6 * N, device=cuda_device)
    capi.check(sv.lib.bfSolverDebugDenseSystem(C.byref(sv.m_solverState), N, C.c_void_p(d_JtJ.data_ptr()), C.c_void_p(d_Jtr.data_ptr())), "bfSolverDebugDenseSystem")
    torch.cuda.synchronize()
    JtJ_our, Jtr_our = d_JtJ.cpu().numpy().reshape(6 * N, 6 * N), d_Jtr.cpu().numpy()
    assert np.count_nonzero(JtJ_ref[6:, 6:]) > 36 * 500
    assert rel_l2(JtJ_our[6:, 6:], JtJ_ref[6:, 6:]) < TOL and rel_l2(Jtr_our[6:], Jtr_ref[6:]) < TOL
    assert np.array_equal(JtJ_our[6:, 6:] != 0, JtJ_ref[6:, 6:] != 0), "same block sparsity as the reference's dense matrix"
    wS, wD, wC = [1.0, 1.0], [1.0, 2.0], [0.1, 0.1]
    x_ref = ref("x")
    x_our, st = run_ours(cuda_device, prob, prob["corr"], 2, 15, wS, wD, wC, cache=cache)
    assert st["dense_overlap_pairs"] == int(ref("overlap"))
    assert rel_l2(x_our, x_ref) < TOL


def test_max_residual_and_pose_stubs_match_reference_cuda(cuda_device):
    import torch
    dev = cuda_device
    prob = synth.make_ba_problem(8, degree=7, corr_per_pair=25, noise=0.0, perturb_rot=0.0, perturb_trans=0.0)
    prob["corr"]["pj"][333] += np.array([0.0, 0.4, 0.0], np.float32)
    ref = reference("maxres", prob)
    x_ref = ref("x")
    v_ref, i_ref = float(ref("v")), int(ref("i"))
    v_orc, i_orc = orc.max_residual(prob["corr"], x_ref[:, :3].astype(np.float32).copy(), x_ref[:, 3:].astype(np.float32).copy())
    assert i_ref == i_orc and abs(v_ref - v_orc) < 1e-5
    # pose <-> matrix stubs, ours against the reference's, on poses with small, moderate and near-pi rotations
    rng = np.random.default_rng(2)
    N = 64
    rot = (rng.standard_normal((N, 3)) * np.r_[np.full(16, 1e-4), np.full(32, 0.5), np.full(16, 1.6)][:, None]).astype(np.float32)
    trans = rng.standard_normal((N, 3)).astype(np.float32)
    L = capi.lib()
    L.bfSetStream(None)
    r = torch.from_numpy(rot).to(dev); t = torch.from_numpy(trans).to(dev)
    T = torch.zeros(N * 16, device=dev); Ti = torch.zeros(N * 16, device=dev); T2 = torch.zeros(N * 16, device=dev)
    r2 = torch.zeros_like(r); t2 = torch.zeros_like(t); valid = torch.ones(N, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    P = C.c_void_p
    L.convertLiePosesToMatricesCU(P(r.data_ptr()), P(t.data_ptr()), C.c_uint(N), P(T.data_ptr()), P(Ti.data_ptr()))
    L.convertMatricesToPosesCU(P(T.data_ptr()), C.c_uint(N), P(r2.data_ptr()), P(t2.data_ptr()), P(valid.data_ptr()))
    L.convertPosesToMatricesCU(P(r2.data_ptr()), P(t2.data_ptr()), C.c_uint(N), P(T2.data_ptr()), P(valid.data_ptr()))
    torch.cuda.synchronize()
    stubs = reference("stubs", (rot, trans))
    for name, x, tol in zip(("T", "Ti", "r2", "t2", "T2"), (T, Ti, r2, t2, T2), (2e-6, 1e-5, 2e-4, 2e-4, 2e-4)):
        np.testing.assert_allclose(x.cpu().numpy(), stubs(name), atol=tol)
