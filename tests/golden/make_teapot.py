#!/usr/bin/env python
"""Writes tests/golden/teapot.npz, config 1's teapot, from a Wavefront OBJ (the reference's data/teapot.obj, which comes from the
McGuire Computer Graphics Archive):  python tests/golden/make_teapot.py path/to/teapot.obj

positions     float32 [V, 3], as scenes.load_obj reads them
face_deltas   int32, the differences of the flattened triangle index list (load_obj's fan split), which compress far better than
              the indices; np.cumsum gives the indices back"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from gfxexp_b200 import scenes  # noqa: E402


def main():
    verts, faces = scenes.load_obj(sys.argv[1])
    deltas = np.diff(faces.reshape(-1).astype(np.int64), prepend=0).astype(np.int32)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "teapot.npz"), positions=verts, face_deltas=deltas)


if __name__ == "__main__":
    main()
