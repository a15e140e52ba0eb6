"""Generates tests/golden/manager_reference_emulated.npz: outputs of the REFERENCE's own match-manager, image and trajectory kernels executed on
the CPU (oracle/_ref/libref_mgr_emulated.so, built by oracle/build_ref.py build_mgr_emulated from FL/SiftGPU/SIFTImageManager.cu,
FL/CUDAImageUtil.cu, FL/OnlineBundler.cu against the CUDA emulation) on the seeded inputs of tests/test_manager_reference_emulated.py.

    python oracle/build_ref.py && python scripts/make_golden_manager_emulated.py
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bundlefusion_b200 import _capi as capi                                                                                   # noqa: E402
from tests._golden import as_crc                                                                                                 # noqa: E402
from tests.test_manager_reference_emulated import INGEST, area_problems, dense_problem, filter_problems, image_cases, trajectory_case    # noqa: E402

F = np.float32


class RefFrame(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("depth", "campos", "intensity", "derivs", "normalsU", "normals")]


def f16(m):
    return np.ascontiguousarray(m, F).reshape(16).ctypes.data_as(C.POINTER(C.c_float))


def main():
    R = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_mgr_emulated.so"))
    vp, u, f, i = C.c_void_p, C.c_uint, C.c_float, C.c_int
    PF = C.POINTER(f)
    R.refFilterKeyPointMatches.argtypes = [u, u, u] + [vp] * 9 + [PF, u, f]
    R.refFilterMatchesBySurfaceArea.argtypes = [u, u, u, vp, vp, vp, PF, f]
    R.refFilterMatchesByDenseVerify.argtypes = [u] * 5 + [PF, vp, vp, vp, vp] + [f] * 7
    R.refAddCurrToResiduals.argtypes = [u, u, u] + [vp] * 6 + [u, PF]
    R.refCacheStoreFrame.argtypes = [vp, u, u, vp, u, u, u, u, PF, f, f, f, RefFrame, vp, vp, vp, vp]
    R.refIngestFrame.argtypes = [vp, vp, u, u, vp, u, u, u, u, i, i, f, f, f, f, vp, vp]
    R.updateTrajectoryCU.argtypes = [vp, u, vp, u, vp, u, u, vp]; R.updateTrajectoryCU.restype = None
    R.initNextGlobalTransformCU.argtypes = [vp, u, u, vp, u, u]; R.initNextGlobalTransformCU.restype = None
    R.computeSiftTransformCU.argtypes = [vp, vp, vp, u, vp, u, u, vp]; R.computeSiftTransformCU.restype = None
    out = {}
    for k, (pb, sd, si) in enumerate(filter_problems()):
        P, cur = pb["P"], pb["cur"]
        keys, num = np.ascontiguousarray(pb["keys"], F), np.ascontiguousarray(pb["num"], np.int32)
        nf = np.zeros(P, np.int32); fd = np.zeros((P, 25), F); fi = np.zeros((P, 25, 2), np.uint32); T = np.zeros((P, 4, 4), F); Ti = np.zeros((P, 4, 4), F)
        R.refFilterKeyPointMatches(cur, 0, P, keys.ctypes.data, num.ctypes.data, sd.ctypes.data, si.ctypes.data, nf.ctypes.data, fd.ctypes.data, fi.ctypes.data,
                                   T.ctypes.data, Ti.ctypes.data, f16(pb["Kinv"]), 5, 0.0004)
        ent = np.zeros((25 * P, 32), np.uint8); eidx = np.zeros((25 * P, 2), np.uint32); cnt = np.zeros(1, np.int32)
        nfc = nf.copy(); nfc[cur] = 0
        R.refAddCurrToResiduals(cur, 0, P, ent.ctypes.data, eidx.ctypes.data, cnt.ctypes.data, nfc.ctypes.data, fi.ctypes.data, keys.ctypes.data, 1024, f16(pb["Kinv"]))
        out.update({f"filter{k}_nf": nf, f"filter{k}_fd": fd, f"filter{k}_fi": fi, f"filter{k}_T": T, f"filter{k}_Ti": Ti, f"filter{k}_entries": ent[:cnt[0]].copy()})
        print("filter", k, nf.tolist(), int(cnt[0]))
    for k, (pb, ths) in enumerate(area_problems()):
        keys, fidx = np.ascontiguousarray(pb["keys"], F), np.ascontiguousarray(pb["fidx"], np.uint32)
        rows = []
        for th in ths:
            num = np.ascontiguousarray(pb["num"], np.int32).copy()
            R.refFilterMatchesBySurfaceArea(pb["cur"], 0, pb["P"], keys.ctypes.data, num.ctypes.data, fidx.ctypes.data, f16(pb["Kinv"]), th)
            rows.append(num)
        out[f"area{k}_nf"] = np.stack(rows)
        print("area", k, len(ths), "thresholds")
    dv, opts = dense_problem()
    P, cur = dv["P"], dv["cur"]
    Tinv = np.stack([np.linalg.inv(t.astype(np.float64)).astype(F) for t in dv["T"]])
    keep = [{n: np.ascontiguousarray(fr[n], F) for n in ("depth", "campos", "normals")} for fr in dv["caches"]]
    recs = (capi.BFCUDACachedFrame * P)()
    for r, fr in zip(recs, keep):
        r.d_depthDownsampled, r.d_cameraposDownsampled, r.d_normalsDownsampled = fr["depth"].ctypes.data, fr["campos"].ctypes.data, fr["normals"].ctypes.data
    rows = []
    T = np.ascontiguousarray(dv["T"], F)
    for o in opts:
        num = np.full(P, 7, np.int32)
        R.refFilterMatchesByDenseVerify(cur, 0, P, dv["W"], dv["H"], f16(dv["K"]), num.ctypes.data, T.ctypes.data, Tinv.ctypes.data, C.addressof(recs), o["distThresh"], o["normalThresh"],
                                        o["colorThresh"], o["errThresh"], o["corrThresh"], o["dMin"], o["dMax"])
        rows.append(num)
    out["dense_nf"] = np.stack(rows)
    print("dense", out["dense_nf"].tolist())
    for k, (depth, color, K, W, H) in enumerate(image_cases()):
        cw, ch = 80, 60
        from oracle import oracle as orc
        Kinv = orc.mat4_inverse(np.asarray(K, F))                      # m_inputIntrinsics.getInverse() as the reference's host forms it (FL/CUDACache.cpp:38)
        b = {"depth": np.zeros((ch, cw), F), "campos": np.zeros((ch, cw, 4), F), "intensity": np.zeros((ch, cw), F), "derivs": np.zeros((ch, cw, 2), F),
             "normalsU": np.zeros((ch, cw, 4), np.uint8), "normals": np.zeros((ch, cw, 4), F)}
        fr = RefFrame(*[b[n].ctypes.data for n in ("depth", "campos", "intensity", "derivs", "normalsU", "normals")])
        h1, h2, h3, h4 = np.zeros((H, W), F), np.zeros((H, W, 4), F), np.zeros((H, W, 4), F), np.zeros((ch, cw), F)
        R.refCacheStoreFrame(depth.ctypes.data, W, H, color.ctypes.data, W, H, cw, ch, Kinv.reshape(16).ctypes.data_as(PF), 2.5, 1.0, 0.05, fr,
                             h1.ctypes.data, h2.ctypes.data, h3.ctypes.data, h4.ctypes.data)
        for n, a in b.items():
            out[f"cache{k}_{n}"] = a
        for c, (fw, fh, erode, sig) in enumerate(INGEST):
            wi, hi = int(W * fw), int(H * fh)
            raw, filt, od, oc = depth.copy(), np.zeros((H, W), F), np.zeros((hi, wi), F), np.zeros((hi, wi, 4), np.uint8)
            R.refIngestFrame(raw.ctypes.data, filt.ctypes.data, W, H, color.ctypes.data, W, H, wi, hi, erode, 3, 0.05, 0.3, sig, 0.05, od.ctypes.data, oc.ctypes.data)
            out.update(as_crc(f"ingest{k}_{c}_depth", od)); out.update(as_crc(f"ingest{k}_{c}_color", oc))      # shape + CRC32: whole frames would pass 1 MB
        print("images", k, W, H)
    tc = trajectory_case()
    n = len(tc["inval"])
    comp = np.zeros((n, 4, 4), F); inval = tc["inval"].copy()
    R.updateTrajectoryCU(tc["glob"].ctypes.data, tc["G"], comp.ctypes.data, n, tc["loc"].ctypes.data, tc["per"], tc["G"], inval.ctypes.data)
    out["traj_complete"] = comp
    g2 = tc["glob"].copy()
    R.initNextGlobalTransformCU(g2.ctypes.data, 3, 2, tc["loc"].ctypes.data, 9, tc["per"])
    out["traj_global"] = g2
    for t, lv in enumerate(tc["last_valids"]):
        sift = tc["sift"].copy(); cur = np.zeros((4, 4), F)
        R.computeSiftTransformCU(tc["finv"].ctypes.data, tc["nf"].ctypes.data, tc["comp"].ctypes.data, lv, sift.ctypes.data, tc["cur_all"], tc["cur"], cur.ctypes.data)
        out[f"traj_sift{t}"], out[f"traj_cur{t}"] = sift, cur
    path = os.path.join(ROOT, "tests", "golden", "manager_reference_emulated.npz")
    np.savez_compressed(path, **out)
    print("written", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
