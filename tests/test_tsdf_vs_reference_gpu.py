"""Parity of this implementation against the REFERENCE'S OWN CUDA kernels (FL/DepthSensing/CUDASceneRepHashSDF.cu built for sm_100a with the
compatibility patch of oracle/build_ref.py), on identical frames and poses, on the GPU.  The reference's states are stored in
tests/golden/tsdf_stream_reference_{ieee,fastmath}.npz (scripts/make_golden_reference_cuda.py ran its kernels on a B200): the block set and a CRC of
every block's voxel words after each stage, and, for the --use_fast_math build, the voxel words of a seeded sample of blocks.

* block coordinates (the allocated set): bit-exact, both builds;
* IEEE build of the reference (no --use_fast_math): EVERY voxel word -- sdf, weight, colour -- bit-identical (every block's CRC), also after
  re-integration, de-integration and GC (the library's arithmetic contract places its FMAs where nvcc places them in the
  reference's expressions, oracle/tsdf_oracle.c header);
* --use_fast_math build (the configuration the reference ships): weights exact, sdf within 1e-4, colours +-1 at rounding ties,
  for all but a vanishing fraction (~1e-5) of voxels whose projected pixel or truncation test sits on a decision boundary
  (approximate division rounds differently there); counted on the stored sample of blocks."""
import numpy as np
import pytest

from bundlefusion_b200 import synth
from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params
from oracle import oracle as orc
from tests._golden import block_crcs, input_crc, load

pytestmark = pytest.mark.gpu
F = np.float32


def compare_states(ours, ref, sdf_tol, exact=False):
    """ours, ref: snapshots (download()) or canonical (blocks, voxels) pairs"""
    ob, ov = ours if isinstance(ours, tuple) else orc.canonical_blocks(ours)
    rb, rv = ref if isinstance(ref, tuple) else orc.canonical_blocks(ref)
    np.testing.assert_array_equal(ob, rb)                                  # block set bit-exact
    if exact:                                                              # IEEE build: every sdf / weight / colour word bit-identical
        np.testing.assert_array_equal(ov, rv)
    o_sdf, o_w, o_c = ov[..., 0].view(F), ov[..., 1].view(F), ov[..., 2].copy().view(np.uint8).reshape(ov.shape[:-1] + (4,))
    r_sdf, r_w, r_c = rv[..., 0].view(F), rv[..., 1].view(F), rv[..., 2].copy().view(np.uint8).reshape(rv.shape[:-1] + (4,))
    n = o_w.size
    w_mismatch = np.count_nonzero(o_w != r_w)
    assert w_mismatch <= max(2, 2e-5 * n), f"{w_mismatch} of {n} voxel weights differ"      # decision-boundary voxels only
    same = o_w == r_w
    touched = same & (o_w > 0)
    dsdf = np.abs(o_sdf[touched] - r_sdf[touched])
    # A voxel whose projection lands within rounding distance of a pixel boundary reads the neighbouring depth pixel in one
    # implementation and not the other (IEEE vs FMA-contracted / fast-math projection): same weight, different sample.  Those
    # are counted, not tolerated silently: they must stay below 1e-4 of the touched voxels; everything else is within sdf_tol.
    flips = np.count_nonzero(dsdf > sdf_tol)
    assert flips <= max(3, 1e-4 * dsdf.size), f"{flips} of {dsdf.size} touched voxels differ by more than {sdf_tol}"
    dc = np.abs(o_c[touched].astype(np.int32) - r_c[touched].astype(np.int32)).max(axis=-1)
    assert np.count_nonzero(dc > 1) <= max(3, 1e-4 * dsdf.size) + flips
    return {"weight_mismatch_frac": w_mismatch / n, "pixel_flip_frac": flips / max(1, dsdf.size), "median_dsdf": float(np.median(dsdf)),
            "p999_dsdf": float(np.quantile(dsdf, 0.999)), "colour_differs_frac": float((dc > 0).mean()), "touched": int(dsdf.size)}


def reference_stream(fast_math, frames):
    """the reference's stored states of the tests' stream (6 frames integrated; frames 1, 4 re-integrated at shifted poses, frame 0 de-integrated, GC)"""
    g = load("tsdf_stream_reference_fastmath.npz" if fast_math else "tsdf_stream_reference_ieee.npz")
    assert int(g["input_crc"]) == input_crc([f[:2] for f in frames], [f[2] for f in frames]), "the stored reference states were made from other frames"
    return g


def compare_with_reference(ours, g, stage, sdf_tol, exact):
    """ours (a snapshot) against the reference's stored state after `stage`: the block set, every block's CRC (IEEE build) or the stored sample
    of blocks (fast-math build) under compare_states' tolerances"""
    ob, ov = orc.canonical_blocks(ours)
    np.testing.assert_array_equal(ob, g[f"blocks{stage}"])                 # block set bit-exact
    if exact:
        np.testing.assert_array_equal(block_crcs(ov), g[f"crcs{stage}"])
        return {"bit_identical_blocks": len(ob)}
    idx = g[f"sample{stage}"]
    return compare_states((ob[idx], ov[idx]), (g[f"blocks{stage}"][idx], g[f"sample_voxels{stage}"]), sdf_tol)


@pytest.mark.parametrize("fast_math", [False, True])
def test_stream_with_reintegration_matches_reference_cuda(cuda_device, fast_math):
    import torch
    W, H = 320, 240
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=100003, num_sdf_blocks=60000)
    ours = CUDASceneRepHashSDF(hp, cuda_device, arithmetic="exact")
    frames = [synth.make_frame(30 * i, W, H) for i in range(6)]
    ref = reference_stream(fast_math, frames)
    dev = [(torch.from_numpy(f[0]).to(cuda_device), torch.from_numpy(f[1]).to(cuda_device)) for f in frames]
    tol = 1e-4 if fast_math else 1e-5
    for (d, c, T), (dd, dc) in zip(frames, dev):
        ours.integrate(T, dd, dc, cam)
    stats = compare_with_reference(ours.download(), ref, 1, tol, exact=not fast_math)
    assert ours.getNumOccupiedBlocks() == int(ref["occupied1"])
    assert ours.getHeapFreeCount() == int(ref["heap_free1"])
    assert int(ref["alloc_rounds"]) >= 2 * len(frames)     # the reference needs >= 2 alloc launches (+ D2H) per frame; we need 1
    # re-integration of two frames at updated poses + GC, as DepthSensing.cpp:854-902
    for k in (1, 4):
        d, c, T = frames[k]
        T2 = T.copy(); T2[:3, 3] += np.array([0.011, -0.006, 0.004], F)
        ours.deIntegrate(T, dev[k][0], dev[k][1], cam); ours.integrate(T2, dev[k][0], dev[k][1], cam)
    ours.deIntegrate(frames[0][2], dev[0][0], dev[0][1], cam)
    ours.garbageCollect()
    stats2 = compare_with_reference(ours.download(), ref, 2, 10 * tol, exact=not fast_math)     # fast-math: de-integration divides by (w - 1), errors grow a little
    assert ours.getHeapFreeCount() == int(ref["heap_free2"])
    print("weight-mismatch fraction, max |dsdf|, colour-differs fraction:", stats, stats2)
