#!/usr/bin/env python
"""Pins oracle/nrc.cpp's input encoding against the reference's own tiny-cuda-nn kernels (oracle/_ref/libtcnn_ref.so, built by
oracle/ref_tcnn/Makefile from the reference's vendored tiny-cuda-nn).  Prints one JSON line and exits 0 when every compared half
is bit-identical.

  python tests/tcnn_ref_check.py                      live: runs the tiny-cuda-nn kernels (GPU, oracle/_ref/libtcnn_ref.so)
  python tests/tcnn_ref_check.py --write-golden PATH  live, and stores what the kernels computed in PATH (.npz)
  python tests/tcnn_ref_check.py --golden PATH        against the stored kernel outputs: CPU only, no oracle/_ref needed

The stored file keeps the SHA-256 of both full outputs (every one of the 8192 rows) and the first GOLDEN_ROWS rows, which
hold all the hand-picked edge cases, so that a mismatch can be located.  Run the live check in a process of its own (it
launches third-party kernels: a fault there must not take another session's CUDA context with it)."""
import argparse
import ctypes as C
import hashlib
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

import oracle_lib as O
from gfxexp_b200 import engine

LEVELS, FEATURES, LOG2_HASHMAP, BASE_RES, PER_LEVEL_SCALE = 16, 2, 15, 16, 2.0   # network_interface.cu:100-107
GOLDEN_ROWS = 128


def level_offsets():
    """GridEncodingTemplated's constructor (grid.h:885-922): entries per level, multiple of 8, capped at 2^log2_hashmap_size"""
    offsets = [0]
    for level in range(LEVELS):
        scale = np.float32(np.exp2(np.float32(level * math.log2(PER_LEVEL_SCALE))) * BASE_RES - 1.0)
        res = int(math.ceil(float(scale))) + 1
        n = min(res ** 3, 0xFFFFFFFF // 2)
        n = (n + 7) // 8 * 8
        n = min(n, 1 << LOG2_HASHMAP)
        offsets.append(offsets[-1] + n)
    return np.asarray(offsets, dtype=np.uint32)


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def tcnn_encodings(q, grid):
    """the reference kernels' hash-grid and one-blob encodings of the queries q (uint16 halves)"""
    ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libtcnn_ref.so"))
    vp = C.c_void_p
    ref.tcnn_ref_grid_forward.argtypes = [C.c_uint32, C.c_uint32, vp, C.c_uint32, C.c_float, vp, C.c_size_t, vp, vp]
    ref.tcnn_ref_oneblob_forward.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, vp, vp]
    n = q.shape[0]
    offsets = level_offsets()
    positions = np.ascontiguousarray(q[:, :3])
    got_grid = np.zeros((n, LEVELS * FEATURES), dtype=np.uint16)
    rc = ref.tcnn_ref_grid_forward(n, LEVELS, offsets.ctypes.data, BASE_RES, C.c_float(math.log2(PER_LEVEL_SCALE)), grid.ctypes.data,
                                   grid.size, positions.ctypes.data, got_grid.ctypes.data)
    assert rc == 0, "tcnn_ref_grid_forward failed"
    blob_in = np.ascontiguousarray(q[:, 3:8])
    got_blob = np.zeros((n, 20), dtype=np.uint16)
    rc = ref.tcnn_ref_oneblob_forward(n, 2, 5, blob_in.ctypes.data, got_blob.ctypes.data)
    assert rc == 0, "tcnn_ref_oneblob_forward failed"
    return got_grid, got_blob


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--golden", help="compare against the kernel outputs stored in this .npz instead of running the kernels")
    ap.add_argument("--write-golden", help="store the kernel outputs in this .npz")
    args = ap.parse_args()

    net = O.OracleNrc(2, 1e-2)
    params = engine.random_nrc_params(net.num_params, net.num_matrix_weights, seed=31, grid_amplitude=0.5)
    net.set_params(params)
    offsets = level_offsets()
    num_grid_params = int(offsets[-1]) * FEATURES
    assert net.num_matrix_weights + num_grid_params == net.num_params, "level table differs from the oracle's"
    grid = np.ascontiguousarray(np.asarray(params).view(np.uint16)[net.num_matrix_weights:])

    rng = np.random.default_rng(17)
    n = 128 * 64
    q = rng.uniform(0.0, 1.0, size=(n, 14)).astype(np.float32)
    q[:16, :3] = 0.0                       # cell corners and the upper boundary of the grid
    q[16:32, :3] = 1.0
    q[32:64, :3] = (rng.integers(0, 17, size=(32, 3)) / 16.0).astype(np.float32)
    q[64:96, 3:8] = rng.choice([0.0, 0.25, 0.5, 0.75, 1.0], size=(32, 5)).astype(np.float32)
    want = net.encode(q).view(np.uint16).reshape(n, 64)
    want_grid, want_blob = np.ascontiguousarray(want[:, :32]), np.ascontiguousarray(want[:, 32:52])

    if args.golden:
        g = np.load(args.golden)
        got_grid, got_blob = g["grid"], g["oneblob"]
        digests = {"grid": str(g["grid_sha256"]), "oneblob": str(g["oneblob_sha256"])}
    else:
        got_grid, got_blob = tcnn_encodings(q, grid)
        digests = {"grid": digest(got_grid), "oneblob": digest(got_blob)}
        if args.write_golden:
            np.savez_compressed(args.write_golden, grid=got_grid[:GOLDEN_ROWS], oneblob=got_blob[:GOLDEN_ROWS],
                                grid_sha256=digests["grid"], oneblob_sha256=digests["oneblob"])

    def compare(got, exp, sha):
        """got: the kernel's rows (all, or the stored first ones); sha: the digest of all its rows"""
        part = exp[:got.shape[0]]
        bad = got != part
        diff = np.abs(got.view(np.float16).astype(np.float64) - part.view(np.float16).astype(np.float64))
        return {"mismatches": int(bad.sum()), "of": int(bad.size), "max_abs_diff": float(diff.max()),
                "first": np.argwhere(bad)[:3].tolist(), "all_rows_equal": digest(exp) == sha}
    result = {"grid": compare(got_grid, want_grid, digests["grid"]), "oneblob": compare(got_blob, want_blob, digests["oneblob"])}
    print(json.dumps(result))
    ok = all(r["mismatches"] == 0 and r["all_rows_equal"] for r in result.values())
    return 0 if ok else 3


if __name__ == "__main__":
    sys.exit(main())
