"""Generates the golden files of the GPU tests that compare this library with the REFERENCE'S OWN CUDA (oracle/_ref: its TSDF and solver
sources built for sm_100a by oracle/build_ref.py, IEEE and --use_fast_math builds):
  tests/golden/tsdf_stream_reference_ieee.npz, tsdf_stream_reference_fastmath.npz -- tests/test_tsdf_vs_reference_gpu.py, tests/test_tsdf_fast_gpu.py;
  tests/golden/solver_vs_reference_cuda.npz                                      -- tests/test_solver_vs_reference_gpu.py.
Each case runs the inputs the tests regenerate (bundlefusion_b200/synth.py, seeded) through the reference, and stores what the tests compare
against together with a CRC of those inputs, which the tests check before they use the stored results.
Needs a GPU and oracle/_ref.  Run:  python scripts/make_golden_reference_cuda.py OUTDIR   (then copy OUTDIR/*.npz into tests/golden/)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bundlefusion_b200 import synth
from bundlefusion_b200.scene_rep import camera_params, default_hash_params
from bundlefusion_b200.solver import DeviceCache
from oracle import oracle as orc
from oracle import ref_solver, ref_tsdf
from tests._golden import block_crcs, input_crc

F = np.float32
# the TSDF stream of the tests: 6 frames (synth.make_frame(30 i), 320 x 240) integrated, frames 1 and 4 re-integrated at shifted poses, frame 0
# de-integrated, garbage collection
TSDF_STREAM = {"W": 320, "H": 240, "frames": [0, 30, 60, 90, 120, 150], "num_buckets": 100003, "num_sdf_blocks": 60000, "reint": [1, 4],
               "shift": [0.011, -0.006, 0.004], "deint": 0}
SAMPLE_BLOCKS = 56          # blocks whose voxel words are stored whole (fast-math build), per stage


def tsdf_frames():
    c = TSDF_STREAM
    return [synth.make_frame(i, c["W"], c["H"]) for i in c["frames"]]


def sample_blocks(n_blocks: int) -> np.ndarray:
    return np.sort(np.random.default_rng(7).choice(n_blocks, min(SAMPLE_BLOCKS, n_blocks), replace=False))


def tsdf_stream(dev, fast_math):
    c = TSDF_STREAM
    cam = camera_params(c["W"], c["H"])
    hp = default_hash_params(num_buckets=c["num_buckets"], num_sdf_blocks=c["num_sdf_blocks"])
    ref = ref_tsdf.ReferenceSceneRepHashSDF(hp, dev, fast_math=fast_math)
    frames = tsdf_frames()
    devf = [(torch.from_numpy(d).to(dev), torch.from_numpy(col).to(dev)) for d, col, _ in frames]
    out = {"case": np.bytes_(repr(c)), "input_crc": np.uint32(input_crc([f[:2] for f in frames], [f[2] for f in frames]))}
    for (_, _, T), (dd, dc) in zip(frames, devf):
        ref.integrate(T, dd, dc, cam)
    stages = [(ref.download(), ref.getHeapFreeCount(), int(ref.hp.m_numOccupiedBlocks))]
    out["alloc_rounds"] = np.int64(ref.alloc_rounds)
    for k in c["reint"]:
        T = frames[k][2]
        T2 = T.copy(); T2[:3, 3] += np.array(c["shift"], F)
        ref.deIntegrate(T, devf[k][0], devf[k][1], cam); ref.integrate(T2, devf[k][0], devf[k][1], cam)
    k = c["deint"]
    ref.deIntegrate(frames[k][2], devf[k][0], devf[k][1], cam)
    ref.garbageCollect()
    stages.append((ref.download(), ref.getHeapFreeCount(), int(ref.hp.m_numOccupiedBlocks)))
    for s, (snap, heap_free, occupied) in enumerate(stages, 1):
        b, v = orc.canonical_blocks(snap)
        out[f"blocks{s}"], out[f"crcs{s}"] = b, block_crcs(v)
        out[f"heap_free{s}"], out[f"occupied{s}"] = np.int64(heap_free), np.int64(occupied)
        if fast_math:
            idx = sample_blocks(len(b))
            out[f"sample{s}"], out[f"sample_voxels{s}"] = idx.astype(np.int32), v[idx]
    return out


# ---- solver ------------------------------------------------------------------------------------------------------------------------------
def _dev_inputs(dev, prob, corr):
    c = np.ascontiguousarray(corr)
    corr_t = torch.from_numpy(c.view(np.uint8).reshape(-1).copy()).to(dev) if len(c) else torch.zeros(32, dtype=torch.uint8, device=dev)
    rot = torch.from_numpy(prob["init_rot"].copy()).to(dev)
    trans = torch.from_numpy(prob["init_trans"].copy()).to(dev)
    valid = torch.ones(len(prob["init_rot"]), dtype=torch.int32, device=dev)
    return corr_t, rot, trans, valid


def run_ref(dev, prob, corr, n_gn, n_pcg, wS, wD=None, wC=None, cache=None, fast=True):
    N = len(prob["init_rot"])
    corr_t, rot, trans, valid = _dev_inputs(dev, prob, corr)
    s = ref_solver.ReferenceSolverBundling(N, max(len(corr), 1000 * N), dev, fast_math=fast)
    conv = s.solve(corr_t, len(corr), valid, N, n_gn, n_pcg, wS, wD, wC, d_rot=rot, d_trans=trans, cudaCache=cache,
                   record_convergence=len(corr) > 0)    # EvalResidual launches a 0-block grid when there are no correspondences
    return np.c_[rot.cpu().numpy(), trans.cpu().numpy()], conv, s


def overlap(s):
    return np.int64(s._bufs["d_numDenseOverlappingImages"].cpu().numpy()[0])


def solver_cases(dev):
    g = {}
    for fast in (True, False):
        for n_images, degree, n_gn, n_pcg in ((2, 1, 4, 50), (11, 10, 2, 100), (60, 8, 3, 150), (200, 12, 4, 150)):
            cpp = 256 if n_images == 2 else 25
            prob = synth.make_ba_problem(n_images, degree=degree, corr_per_pair=cpp, noise=0.002, seed=5)
            key = f"sparse_{n_images}_{int(fast)}"
            x, conv, _ = run_ref(dev, prob, prob["corr"], n_gn, n_pcg, [1.0] * n_gn, fast=fast)
            g[key + "_x"], g[key + "_conv"], g[key + "_input_crc"] = x, conv, np.uint32(input_crc(prob))
    prob = synth.make_dense_ba_problem(8, stride=2, perturb_rot=0.004, perturb_trans=0.008, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], dev)
    wS, wD, wC = [0.0] * 2, [1.0, 2.0], [0.0] * 2
    g["dense_only_x"], _, s = run_ref(dev, prob, prob["corr"][:0], 2, 10, wS, wD, wC, cache=cache, fast=False)
    g["dense_only_x2"], _, _ = run_ref(dev, prob, prob["corr"][:0], 2, 10, wS, wD, wC, cache=cache, fast=False)
    g["dense_only_overlap"], g["dense_only_input_crc"] = overlap(s), np.uint32(input_crc(prob))
    prob = synth.make_dense_ba_problem(5, stride=3, perturb_rot=0.004, perturb_trans=0.008, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], dev)
    wS, wD, wC = [0.0] * 3, [1.0, 2.0, 3.0], [0.0] * 3
    g["chaotic_x"], _, _ = run_ref(dev, prob, prob["corr"][:0], 3, 60, wS, wD, wC, cache=cache, fast=False)
    g["chaotic_x1"], _, _ = run_ref(dev, prob, prob["corr"][:0], 1, 10, wS[:1], wD[:1], wC[:1], cache=cache, fast=False)
    g["chaotic_input_crc"] = np.uint32(input_crc(prob))
    prob = synth.make_dense_ba_problem(11, stride=3, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], dev)
    g["local_input_crc"] = np.uint32(input_crc(prob))
    for fast in (True, False):
        for c, wC in enumerate(([0.0, 0.0], [0.1, 0.1])):
            key = f"local_{c}_{int(fast)}"
            g[key + "_x"], _, s = run_ref(dev, prob, prob["corr"], 2, 100, [1.0, 1.0], [1.0, 2.0], wC, cache=cache, fast=fast)
            g[key + "_overlap"] = overlap(s)
    N = 6
    prob = synth.make_dense_ba_problem(N, stride=3, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], dev)
    g["dense_system_x"], _, s = run_ref(dev, prob, prob["corr"][:0], 1, 0, [0.0], [1.0], [0.1], cache=cache, fast=False)
    g["dense_system_JtJ"] = s._bufs["d_denseJtJ"].cpu().numpy().reshape(6 * N, 6 * N)
    g["dense_system_Jtr"] = s._bufs["d_denseJtr"].cpu().numpy()
    g["dense_system_input_crc"] = np.uint32(input_crc(prob))
    N = 72
    prob = synth.make_dense_ba_problem(N, stride=1, start=60, corr_per_pair=8, W=320, H=240)
    cache = DeviceCache(prob["caches"], prob["intrinsics"], dev)
    _, _, s = run_ref(dev, prob, prob["corr"][:0], 1, 0, [0.0], [1.0], [0.1], cache=cache, fast=False)
    g["beyond64_JtJ"] = s._bufs["d_denseJtJ"].cpu().numpy().reshape(6 * N, 6 * N)[6:, 6:]     # rows / columns of the fixed variable 0 are never read
    g["beyond64_Jtr"] = s._bufs["d_denseJtr"].cpu().numpy()
    g["beyond64_x"], _, s = run_ref(dev, prob, prob["corr"], 2, 15, [1.0, 1.0], [1.0, 2.0], [0.1, 0.1], cache=cache, fast=False)
    g["beyond64_overlap"], g["beyond64_input_crc"] = overlap(s), np.uint32(input_crc(prob))
    prob = synth.make_ba_problem(8, degree=7, corr_per_pair=25, noise=0.0, perturb_rot=0.0, perturb_trans=0.0)
    prob["corr"]["pj"][333] += np.array([0.0, 0.4, 0.0], np.float32)
    g["maxres_x"], _, s = run_ref(dev, prob, prob["corr"], 1, 1, [1.0], fast=False)
    v, i = s.max_residual()
    g["maxres_v"], g["maxres_i"], g["maxres_input_crc"] = np.float32(v), np.int64(i), np.uint32(input_crc(prob))
    # pose <-> matrix stubs of the reference on poses with small, moderate and near-pi rotations (the inputs are regenerated by the test)
    import ctypes as C
    rng = np.random.default_rng(2)
    N = 64
    rot = (rng.standard_normal((N, 3)) * np.r_[np.full(16, 1e-4), np.full(32, 0.5), np.full(16, 1.6)][:, None]).astype(np.float32)
    trans = rng.standard_normal((N, 3)).astype(np.float32)
    r = torch.from_numpy(rot).to(dev); t = torch.from_numpy(trans).to(dev)
    T = torch.zeros(N * 16, device=dev); Ti = torch.zeros(N * 16, device=dev); T2 = torch.zeros(N * 16, device=dev)
    r2 = torch.zeros_like(r); t2 = torch.zeros_like(t); valid = torch.ones(N, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    P, L = C.c_void_p, s.L
    L.convertLiePosesToMatricesCU(P(r.data_ptr()), P(t.data_ptr()), C.c_uint(N), P(T.data_ptr()), P(Ti.data_ptr()))
    L.convertMatricesToPosesCU(P(T.data_ptr()), C.c_uint(N), P(r2.data_ptr()), P(t2.data_ptr()), P(valid.data_ptr()))
    L.convertPosesToMatricesCU(P(r2.data_ptr()), P(t2.data_ptr()), C.c_uint(N), P(T2.data_ptr()), P(valid.data_ptr()))
    torch.cuda.synchronize()
    for name, x in zip(("T", "Ti", "r2", "t2", "T2"), (T, Ti, r2, t2, T2)):
        g["stubs_" + name] = x.cpu().numpy()
    g["stubs_input_crc"] = np.uint32(input_crc(rot, trans))
    return g


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "golden_out"
    os.makedirs(out, exist_ok=True)
    dev = torch.device("cuda:0")
    if not (ref_tsdf.available(True) and ref_tsdf.available(False) and ref_solver.available(True) and ref_solver.available(False)):
        raise SystemExit("oracle/_ref is not built: python oracle/build_ref.py on a machine with the reference sources")
    np.savez_compressed(os.path.join(out, "tsdf_stream_reference_ieee.npz"), **tsdf_stream(dev, False))
    np.savez_compressed(os.path.join(out, "tsdf_stream_reference_fastmath.npz"), **tsdf_stream(dev, True))
    np.savez_compressed(os.path.join(out, "solver_vs_reference_cuda.npz"), **solver_cases(dev))
    for f in sorted(os.listdir(out)):
        print(f, os.path.getsize(os.path.join(out, f)))


if __name__ == "__main__":
    main()
