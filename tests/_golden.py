"""Stored outputs of the reference's CUDA (tests/golden/*.npz, written by scripts/make_golden_reference_cuda.py) and the CRCs that tie them to the
inputs the tests regenerate."""
import os
import zlib

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLD, name))


def input_crc(*arrays) -> int:
    """CRC32 of test inputs: arrays, and lists / tuples / dicts of them (synth's problems and cache frames)"""
    c = 0

    def add(a):
        nonlocal c
        if isinstance(a, dict):
            for k in sorted(a):
                add(a[k])
        elif isinstance(a, (list, tuple)):
            for x in a:
                add(x)
        elif a is not None:
            c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    for a in arrays:
        add(a)
    return c


def block_crcs(vox):
    """CRC32 of every block's voxel words, (N, 512, 3) -> (N,)"""
    return np.array([zlib.crc32(np.ascontiguousarray(v).tobytes()) for v in vox], np.uint32)


def as_crc(key, a) -> dict:
    """an array stored by its shape and CRC32 (`key_shape`, `key_crc`) where storing it whole would make the golden file too large"""
    a = np.asarray(a)
    return {key + "_shape": np.array(a.shape, np.int64), key + "_crc": np.uint32(zlib.crc32(a.tobytes()))}


def matches(a, g, key) -> bool:
    """a equals the stored array `key` of golden file g, stored whole or by as_crc"""
    a = np.asarray(a)
    if key in g.files:
        return a.shape == g[key].shape and a.dtype == g[key].dtype and a.tobytes() == g[key].tobytes()
    return a.shape == tuple(g[key + "_shape"]) and zlib.crc32(a.tobytes()) == int(g[key + "_crc"])
