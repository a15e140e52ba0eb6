"""Pins the oracles of rows a19 - a22 against the REFERENCE's own kernels executed on the CPU: FL/SiftGPU/SIFTImageManager.cu (Kabsch
filter in its DEVICE flavour, surface-area filter, dense verification, residual assembly), FL/CUDAImageUtil.cu (called in the order of
CUDACache::storeFrame and CUDAImageManager::process) and FL/OnlineBundler.cu (the three trajectory kernels), compiled by g++ against the
CUDA emulation (oracle/build_ref.py build_mgr_emulated -> oracle/_ref/libref_mgr_emulated.so); outputs on seeded inputs are committed as
tests/golden/manager_reference_emulated.npz (scripts/make_golden_manager_emulated.py).
Not covered: SortKeyPointMatchesCU_Kernel -- its termination flag is a shared-memory race that only lock-step warps survive, it cannot
run under the emulation (inputs are sorted by the oracle instead; an odd-even transposition sort is a stable sort by distance)."""
import os

import numpy as np

from bundlefusion_b200 import synth
from oracle import oracle as orc
from tests._golden import matches
from tests.test_verify_filters_oracle import VERIFY

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "manager_reference_emulated.npz")
F = np.float32


def filter_problems():
    for seed, n_in, n_out, noise in ((1, 40, 12, 0.002), (2, 20, 30, 0.004), (4, 6, 3, 0.002), (7, 50, 5, 0.0005)):
        pb = synth.make_filter_problem(n_pairs=5, n_inliers=n_in, n_outliers=n_out, noise=noise, seed=seed)
        rng = np.random.default_rng(seed)
        d, ix = pb["dists"].copy(), pb["idxs"].copy()
        for p in range(pb["P"] - 1):
            perm = rng.permutation(pb["num"][p]); d[p, :pb["num"][p]] = d[p, perm]; ix[p, :pb["num"][p]] = ix[p, perm]
        sd, si = orc.sift_sort_matches(pb["cur"], 0, pb["P"], pb["num"], d, ix)
        yield pb, np.ascontiguousarray(sd, F), np.ascontiguousarray(si, np.uint32)


def area_problems():
    """(problem, thresholds): for each pair the thresholds bracket the oracle's two areas within 1e-4 relative, so that the reference's
    yes / no decisions pin its areas (it does not output them)."""
    for seed in range(3):
        pb = synth.make_area_problem(seed)
        _, areas = orc.sift_filter_surface_area(pb["cur"], 0, pb["P"], pb["keys"], pb["num"], pb["fidx"], pb["Kinv"], 0.0)
        big = np.maximum(areas[:, 0], areas[:, 1])
        ths = [0.032] + [float(F(b * (1 - 1e-4))) for b in big if b > 0] + [float(F(b * (1 + 1e-4))) for b in big if b > 0]
        yield pb, ths


def dense_problem():
    dv = synth.make_dense_verify_problem()
    opts = [VERIFY, dict(VERIFY, errThresh=0.0215, corrThresh=0.86), dict(VERIFY, errThresh=0.024, corrThresh=0.80), dict(VERIFY, corrThresh=0.45, errThresh=0.5)]
    # thresholds that bracket every pair's (err, corr) of the oracle within 1e-3 relative: the reference's yes / no answers pin its two numbers
    _, st = orc.sift_filter_dense_verify(dv["cur"], 0, dv["P"], dv["W"], dv["H"], dv["K"], np.full(dv["P"], 7, np.int32), dv["T"], dv["caches"], **VERIFY)
    for p in range(dv["P"] - 1):
        e, c = float(st[p, 0]), float(st[p, 1])
        if np.isfinite(e) and c > 0:
            opts += [dict(VERIFY, errThresh=e * (1 + 1e-3), corrThresh=c * (1 - 1e-3)), dict(VERIFY, errThresh=e * (1 - 1e-3), corrThresh=c * (1 - 1e-3)),
                     dict(VERIFY, errThresh=e * (1 + 1e-3), corrThresh=c * (1 + 1e-3))]
    return dv, opts


def image_cases():
    for frame, (W, H) in ((100, (320, 240)), (250, (160, 120))):
        depth, color, _ = synth.make_frame(frame, W, H)
        fx = 525.0 * W / 640.0
        K = np.array([[fx, 0, (W - 1) / 2.0, 0], [0, fx, (H - 1) / 2.0, 0], [0, 0, 1, 0], [0, 0, 0, 1]])
        yield np.ascontiguousarray(depth, F), np.ascontiguousarray(color, np.uint8), K, W, H


INGEST = ((1.0, 1.0, 1, 2.0), (0.5, 0.5, 1, 2.0), (1.0, 1.0, 0, 0.0), (0.5, 0.5, 0, 2.0))          # (width factor, height factor, erode, sigmaD)


def poses(n, seed):
    rng = np.random.default_rng(seed)
    return np.stack([synth.se3_exp(rng.standard_normal(3) * 0.3, rng.standard_normal(3)) for _ in range(n)]).astype(F)


def trajectory_case():
    G, per = 5, 11
    glob, loc = poses(G + 1, 1), poses(G * per, 2)
    inval = np.ones(G * (per - 1), np.int32); inval[[3, 17]] = 0
    n_all, cur, cur_all = 40, 7, 27
    sift, comp, finv = poses(n_all, 3), poses(n_all, 4), poses(cur, 5)
    nf = np.zeros(cur, np.int32); nf[[2, 4]] = 30
    prev = cur_all - (cur - 4)
    return dict(G=G, per=per, glob=glob, loc=loc, inval=inval, n_all=n_all, cur=cur, cur_all=cur_all, sift=sift, comp=comp, finv=finv, nf=nf,
                last_valids=(0, prev + 5, prev - 3))


def bits(a):
    return np.ascontiguousarray(a, F).view(np.uint32)


def test_kabsch_filter_device_flavour_and_residuals():
    g = np.load(GOLDEN)
    for k, (pb, sd, si) in enumerate(filter_problems()):
        P, cur = pb["P"], pb["cur"]
        o = orc.sift_filter_matches(cur, 0, P, pb["keys"], pb["num"], sd, si, pb["Kinv"])
        pairs = [p for p in range(P) if p != cur]
        assert np.array_equal(o[0][pairs], g[f"filter{k}_nf"][pairs])
        assert np.array_equal(o[2][pairs], g[f"filter{k}_fi"][pairs]) and np.array_equal(bits(o[1][pairs]), bits(g[f"filter{k}_fd"][pairs]))
        assert np.array_equal(bits(o[3][pairs]), bits(g[f"filter{k}_T"][pairs])) and np.array_equal(bits(o[4][pairs]), bits(g[f"filter{k}_Ti"][pairs]))
        nf = o[0].copy(); nf[cur] = 0
        ent, _ = orc.sift_add_residuals(cur, 0, P, nf, o[2], pb["keys"], pb["Kinv"])
        mine = sorted(bytes(e) for e in ent.view(np.uint8).reshape(-1, 32)); ref = sorted(bytes(e) for e in g[f"filter{k}_entries"])
        assert mine == ref                                                 # the reference appends pairs in atomicAdd order: same set


def test_surface_area_decisions_pin_the_areas():
    g = np.load(GOLDEN)
    for k, (pb, ths) in enumerate(area_problems()):
        for t, th in enumerate(ths):
            nf, _ = orc.sift_filter_surface_area(pb["cur"], 0, pb["P"], pb["keys"], pb["num"], pb["fidx"], pb["Kinv"], th)
            assert np.array_equal(nf, g[f"area{k}_nf"][t]), (k, th, nf, g[f"area{k}_nf"][t])


def reference_reduction(pix, W, H):
    """What FilterMatchesByDenseVerifyCU_Kernel actually adds up (FL/SiftGPU/SIFTImageManager.cu:520-565) for a block of (W, ceil(H / 32)) threads:
    thread (x, ty) sums its rows ty * 32 .. in order; warps are cut from the LINEAR thread id; `val += __shfl_down(val, offset)` doubles a
    lane's value when the source lane is past the warp's end; and the lanes that add their result to the block total are those with
    threadIdx.x % 32 == 0 -- lane 0 of a warp only in the first thread row.  For the 80 x 60 cache (block 80 x 2 = five warps) the total is
    lane 0 of warps 0 - 2 plus lane 16 of warps 2 - 4: part of the image counts twice or more, part of it not at all."""
    by = (H + 31) // 32
    local = np.zeros((by * W, 3), F)
    for ty in range(by):
        for x in range(W):
            acc = np.zeros(3, F)
            for i in range(32):
                y = ty * 32 + i
                if y < H:
                    acc = (acc + pix[y * W + x]).astype(F)
            local[ty * W + x] = acc
    assert (by * W) % 32 == 0
    total = np.zeros(3, F)
    warps = local.reshape(-1, 32, 3).copy()
    for off in (16, 8, 4, 2, 1):
        src = np.arange(32) + off
        src = np.where(src < 32, src, np.arange(32))
        warps = (warps + warps[:, src]).astype(F)
    red = warps.reshape(-1, 3)
    for ty in range(by):
        for x in range(0, W, 32):
            total = (total + red[ty * W + x]).astype(F)
    return total


def test_dense_verify_pixels_and_the_reference_reduction():
    """The reference's decisions follow from THIS oracle's per-pixel residual / weight / count when they are added up the way the reference's
    kernel adds them -- which is not a plain sum (see reference_reduction).  orc_sift_filter_dense_verify and the CUDA path form the total the
    same way (a plain sum would change one decision in twenty on these inputs: a pair whose overlap sits at the threshold)."""
    import ctypes as C
    from oracle.oracle import _CachedFrame
    g = np.load(GOLDEN)
    dv, opts = dense_problem()
    P, cur, W, H = dv["P"], dv["cur"], dv["W"], dv["H"]
    L = orc.lib()
    keep = [{n: np.ascontiguousarray(fr[n], F) for n in ("depth", "campos", "normals")} for fr in dv["caches"]]
    recs = (_CachedFrame * P)()
    for r, fr in zip(recs, keep):
        r.depth, r.campos, r.normals = fr["depth"].ctypes.data, fr["campos"].ctypes.data, fr["normals"].ctypes.data
    L.orc_sift_dense_verify_pixels.argtypes = [C.c_uint] * 4 + [C.c_void_p] * 3 + [C.c_float] * 4 + [C.c_void_p]
    L.orc_sift_dense_verify_pixels.restype = None
    K, T = np.ascontiguousarray(dv["K"], F), np.ascontiguousarray(dv["T"], F)
    plain_differs = 0
    for t, o in enumerate(opts):
        nf_plain, _ = orc.sift_filter_dense_verify(cur, 0, P, W, H, dv["K"], np.full(P, 7, np.int32), dv["T"], dv["caches"], **o)
        for p in range(P - 1):
            pix = np.zeros((W * H, 3), F)
            L.orc_sift_dense_verify_pixels(p, cur, W, H, K.ctypes.data, T.ctypes.data, C.addressof(recs), o["distThresh"], o["normalThresh"], o["dMin"], o["dMax"], pix.ctypes.data)
            tot = reference_reduction(pix, W, H)
            with np.errstate(all="ignore"):
                err = F(tot[0]) / F(tot[1]); corr = F(0.5) * tot[2] / F(W * H)
            keepit = not (corr < o["corrThresh"] or err > o["errThresh"] or np.isnan(err))
            assert (7 if keepit else 0) == g["dense_nf"][t][p], (t, p, err, corr)
            plain_differs += int(nf_plain[p] != g["dense_nf"][t][p])
    assert plain_differs == 0


def test_cache_frame_and_ingest():
    g = np.load(GOLDEN)
    for k, (depth, color, K, W, H) in enumerate(image_cases()):
        o = orc.cache_store_frame(depth, color, K, 80, 60, 2.5, 1.0, 0.05)
        for name, mine in (("depth", "depth"), ("campos", "campos"), ("normals", "normals")):
            assert np.array_equal(bits(o[mine]).reshape(-1), bits(g[f"cache{k}_{name}"]).reshape(-1)), (k, name)      # bit for bit, -inf included
        assert np.array_equal(np.asarray(o["normalsU"]).reshape(-1), g[f"cache{k}_normalsU"].reshape(-1))
        # intensity: the oracle places the fused multiply-adds nvcc emits for the reference's expressions; the emulation is built without
        # contraction, which moves a few hundred pixels by one unit in the last place
        for name, mine in (("intensity", "intensity"), ("derivs", "intensityDerivs")):
            a, b = np.asarray(o[mine], F).reshape(-1), g[f"cache{k}_{name}"].reshape(-1)
            fin = np.isfinite(b)
            assert np.array_equal(np.isfinite(a), fin) and np.abs(a[fin] - b[fin]).max() < 3e-7
        for c, (fw, fh, erode, sig) in enumerate(INGEST):
            wi, hi = int(W * fw), int(H * fh)
            d, col = orc.ingest_frame(depth, color, wi, hi, erode=bool(erode), depth_filter=sig > 0, sigmaD=sig if sig > 0 else 2.0)
            assert matches(np.asarray(d, F), g, f"ingest{k}_{c}_depth") and matches(col, g, f"ingest{k}_{c}_color"), (k, c)       # bit for bit (stored as CRC32)


def close_ulps(a, b):
    """Same -inf pattern, finite entries within a couple of units in the last place: the oracle multiplies 4x4s with the fused multiply-adds
    nvcc emits for the reference's float4x4::operator* (its contract with the CUDA path), the emulation is built without contraction."""
    a, b = np.ascontiguousarray(a, F), np.ascontiguousarray(b, F)
    fa, fb = np.isfinite(a), np.isfinite(b)
    return np.array_equal(fa, fb) and np.array_equal(a[~fa], b[~fb]) and bool(np.all(np.abs(a[fa] - b[fb]) <= 4e-7 * np.maximum(1.0, np.abs(b[fb]))))


def test_trajectory_kernels():
    g = np.load(GOLDEN)
    tc = trajectory_case()
    out = orc.update_trajectory(tc["glob"], tc["loc"], tc["per"], tc["inval"])
    assert close_ulps(out, g["traj_complete"])
    assert np.array_equal(np.isneginf(out[:, 0, 0]), tc["inval"] == 0)
    g2 = orc.init_next_global(tc["glob"], 3, 2, tc["loc"], 9, tc["per"])
    assert close_ulps(g2, g["traj_global"]) and np.array_equal(bits(g2[:3]), bits(g["traj_global"][:3]))
    for t, lv in enumerate(tc["last_valids"]):
        traj, cur = orc.compute_sift_transform(tc["finv"], tc["nf"], tc["comp"], lv, tc["sift"], tc["cur_all"], tc["cur"])
        assert close_ulps(traj, g[f"traj_sift{t}"]) and close_ulps(cur, g[f"traj_cur{t}"]), t
        assert np.array_equal(np.delete(traj, tc["cur_all"], 0), np.delete(g[f"traj_sift{t}"], tc["cur_all"], 0))      # only the current frame's slot is written
