"""Pins oracle/fuse_oracle.c (row N2: chunk -> keyframe fusion of the sparse features) against the REFERENCE's own code: SIFTImageManager::fuseToGlobal / computeTracks /
findTrack (FL/SiftGPU/SIFTImageManager.cpp:366-476) is host code of the reference's manager class; oracle/build_ref.py (build_fuse_emulated) compiles the class with its
kernels against the CUDA emulation -> oracle/_ref/libref_fuse_emulated.so, scripts/make_golden_fuse_emulated.py fed it the solved chunks below through the class's own
interface and stored the fused keyframe's keys and descriptors in tests/golden/fuse_reference_emulated.npz.  The oracle must reproduce them bit for bit: which key
represents a track, which correspondences contribute to its position, the order of the fused keys."""
import ctypes as C
import os

import numpy as np

from bundlefusion_b200 import synth
from oracle import oracle as orc
from tests._golden import input_crc, load

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "fuse_reference_emulated.npz")
REF_SO = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "libref_fuse_emulated.so")
CASES = [dict(seed=0), dict(seed=1), dict(seed=2), dict(seed=5, n_images=11, n_points=150), dict(seed=7, n_images=3, n_points=20), dict(seed=9, n_images=10, n_points=60, outlier_frac=0.3)]
LIVE_SEEDS = (21, 22, 23, 24)


def live_problem(seed):
    return synth.make_fuse_problem(seed=seed, n_images=int(4 + seed % 7), n_points=80 + 5 * (seed % 5), invalid_frac=0.1)


def reference_fuse(pb, max_keys=1024):
    """the reference's manager, filled through createSIFTImageGPU / finalizeSIFTImageGPU; its global key indices are packed by a prefix sum over the images"""
    R = C.CDLL(REF_SO)
    vp = C.c_void_p
    R.ref_fuse_to_global.argtypes = [C.c_uint, vp, C.c_uint, vp, vp, C.c_uint, vp, vp, vp, vp, C.c_uint, vp, vp]
    ks = int(pb["keyStride"]); num = np.ascontiguousarray(pb["numKeys"], np.uint32); n_img = len(num)
    prefix = np.concatenate([[0], np.cumsum(num)[:-1]]).astype(np.uint32)
    ki = np.ascontiguousarray(pb["keyIdx"], np.uint32)
    packed = (prefix[ki // ks] + ki % ks).astype(np.uint32)
    keys = np.ascontiguousarray(pb["keys"], np.float32); descs = np.ascontiguousarray(pb["descs"], np.uint8)
    corr = np.ascontiguousarray(pb["corr"]); T = np.ascontiguousarray(pb["transforms"], np.float32); K = np.ascontiguousarray(pb["K"], np.float32)
    ok, od = np.zeros((max_keys, 4), np.float32), np.zeros((max_keys, 128), np.uint8)
    n = R.ref_fuse_to_global(n_img, num.ctypes.data, ks, keys.ctypes.data, descs.ctypes.data, len(corr), corr.ctypes.data, packed.ctypes.data, T.ctypes.data, K.ctypes.data, max_keys,
                             ok.ctypes.data, od.ctypes.data)
    return ok[:n].copy(), od[:n].copy()


def oracle_fuse(pb):
    return orc.sift_fuse_to_global(pb["corr"], pb["keyIdx"], pb["transforms"], pb["keys"], pb["descs"], pb["numKeys"], pb["keyStride"], pb["K"])


def test_oracle_reproduces_the_reference_fusion_bit_for_bit():
    g = np.load(GOLDEN)
    for c, kw in enumerate(CASES):
        pb = synth.make_fuse_problem(**kw)
        k, d = oracle_fuse(pb)
        assert len(k) == len(g[f"keys_{c}"]) > 5, c
        assert np.array_equal(k.view(np.uint32), g[f"keys_{c}"].view(np.uint32)) and np.array_equal(d, g[f"descs_{c}"]), c


def test_live_against_the_references_manager_class():
    """four more problems, with invalid correspondences: the manager class's results are stored in tests/golden/reference_host_cases.npz
    (scripts/make_golden_reference_host_cases.py); where oracle/_ref is built, the class computes them again"""
    g = load("reference_host_cases.npz")
    for seed in LIVE_SEEDS:
        pb = live_problem(seed)
        assert int(g[f"fuse{seed}_input_crc"]) == input_crc(pb), seed
        (k, d), rk, rd = oracle_fuse(pb), g[f"fuse{seed}_keys"], g[f"fuse{seed}_descs"]
        assert len(k) == len(rk) > 5 and np.array_equal(k.view(np.uint32), rk.view(np.uint32)) and np.array_equal(d, rd)
        if os.path.exists(REF_SO):
            lk, ld = reference_fuse(pb)
            assert np.array_equal(lk.view(np.uint32), rk.view(np.uint32)) and np.array_equal(ld, rd)


def filter_frames_cases():
    rng = np.random.default_rng(4)
    out = []
    for _ in range(40):
        n = int(rng.integers(1, 12)); cur = int(rng.integers(0, n + 1)); start = int(rng.integers(0, n))
        nf = (rng.integers(0, 4, n) * rng.integers(0, 2, n)).astype(np.int32); valid = rng.integers(0, 2, n + 2).astype(np.int32)
        out.append((cur, start, n, nf, valid))
    return out


def test_filter_frames_oracle_equals_the_references_member_function():
    """SIFTImageManager::filterFrames (FL/SiftGPU/SIFTImageManager.cpp:551-575), host code of the same class: last matched frame and the validity it writes"""
    g = np.load(GOLDEN)
    for k, (cur, start, n, nf, valid) in enumerate(filter_frames_cases()):
        last, v = orc.sift_filter_frames(cur, start, n, nf, valid.copy())
        assert (last & 0xFFFFFFFF) == int(g["ff_last"][k]) and np.array_equal(v, g["ff_valid"][k][:len(v)]), k
    if os.path.exists(REF_SO):                                                  # the stored outputs are what the member function returns now
        last, valid = reference_filter_frames()
        assert np.array_equal(last, g["ff_last"]) and np.array_equal(valid, g["ff_valid"])


def reference_filter_frames():
    R = C.CDLL(REF_SO)
    R.ref_filter_frames.argtypes = [C.c_uint, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_uint]; R.ref_filter_frames.restype = C.c_uint
    lasts, valids = [], []
    for cur, start, n, nf, valid in filter_frames_cases():
        v = np.zeros(16, np.int32); v[:len(valid)] = valid
        lasts.append(R.ref_filter_frames(cur, start, n, nf.ctypes.data, v.ctypes.data, len(valid))); valids.append(v)
    return np.array(lasts, np.uint32), np.stack(valids)
