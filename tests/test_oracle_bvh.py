"""The CPU oracle pinned against reference-independent ground truth (no GPU needed):
 * struct sizes of the reference node formats,
 * the restated SBVH builder produces a valid BVH within the reference's budget,
 * bvh::traverse (first-found and canonical tie-break) equals the exhaustive brute-force closest hit,
 * any-hit equals "brute-force closest hit exists in range".
"""
import os

import numpy as np
import pytest

from gfxexp_b200 import abi, scenes


@pytest.fixture(scope="module")
def tiny(oracle):
    scene = scenes.tiny_city_scene()
    return scene, oracle.OracleScene(scene)


def _rays(oracle, scene, oscene, n=6000, seed=3):
    info = oscene.info()
    rng = np.random.default_rng(seed)
    lo, hi = np.array(info.sceneMin), np.array(info.sceneMax)
    rays = np.zeros(n, dtype=abi.RAY_DTYPE)
    rays["org"] = (lo + (hi - lo) * rng.uniform(-0.2, 1.2, size=(n, 3))).astype(np.float32)
    d = rng.normal(size=(n, 3))
    rays["dir"] = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    rays["tmax"] = np.float32(3.402823466e+38)
    p = abi.default_frame_params(scene, 64, 40)
    return np.concatenate([rays, oracle.primary_rays(p, 64, 40)])


def test_sbvh_build_invariants(tiny):
    scene, oscene = tiny
    info = oscene.info()
    assert info.numTriangles == scene.num_triangles
    # splittingBudget 0.3 (nrtdsm_sandbox.cpp:3177-3184): at most floor(1.3 N) references
    assert info.numTriangles <= info.numPrimRefs <= int(1.3 * info.numTriangles)
    assert oscene.validate() == ""
    nodes, refs, tris = oscene.export_bvh()
    # root is node 0, internal children are contiguous blocks (intNodeChildBaseIndex)
    assert nodes["intNodeChildBaseIndex"][0] == 1
    # every leaf chain ends with isLeafEnd
    assert (refs >> 31).sum() > 0 and (refs[-1] >> 31) == 1


def test_traverse_equals_brute_force(oracle, tiny):
    scene, oscene = tiny
    rays = _rays(oracle, scene, oscene)
    brute = oscene.trace(rays, oracle.TRACE_BRUTE_FORCE)
    canon = oscene.trace(rays, oracle.TRACE_CANONICAL)
    first, stats = oscene.trace(rays, oracle.TRACE_FIRST_FOUND, want_stats=True)
    for name, got in (("canonical", canon), ("first-found", first)):
        same = (got["dist"].view(np.uint32) == brute["dist"].view(np.uint32)) & (got["primIndex"] == brute["primIndex"]) \
            & (got["geomIndex"] == brute["geomIndex"])
        if name == "first-found":
            # ties in distance may resolve to another triangle; the distance itself must still match
            assert np.array_equal(got["dist"].view(np.uint32), brute["dist"].view(np.uint32))
        else:
            assert same.all(), f"{name}: {np.count_nonzero(~same)} rays differ from brute force"
    assert stats.numHits == np.count_nonzero(brute["primIndex"] != 0xFFFFFFFF)
    assert stats.numIntNodes > 0 and stats.maxStackDepth < 32


def test_any_hit_equals_brute_force(oracle, tiny):
    scene, oscene = tiny
    rays = _rays(oracle, scene, oscene, seed=9)
    rays["tmax"] = np.random.default_rng(2).uniform(0.5, 25.0, size=len(rays)).astype(np.float32)
    brute = oscene.trace(rays, oracle.TRACE_BRUTE_FORCE)
    anyhit = oscene.trace(rays, oracle.TRACE_ANY)
    assert np.array_equal(anyhit["primIndex"] != 0xFFFFFFFF, brute["primIndex"] != 0xFFFFFFFF)


def test_node_codec_is_conservative(tiny):
    """setChildAabb (common_shared.h:839-851): decoded child boxes contain the exact ones (checked by
    orc_bvh_validate for un-split references) and quantised coordinates stay within 8 bits."""
    _, oscene = tiny
    nodes, _, _ = oscene.export_bvh()
    valid = (nodes["childQMin"][:, 0, :] != 255) | (nodes["childQMax"][:, 0, :] != 0)
    assert (nodes["childQMin"][:, :, :].transpose(0, 2, 1)[valid] <= nodes["childQMax"].transpose(0, 2, 1)[valid]).all()


def test_teapot_config1_build(oracle, tmp_path):
    """config 1's teapot (tests/golden/teapot.npz, written by make_teapot.py), written back as an OBJ so that it goes through
    scenes.load_obj like the original file"""
    teapot = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "teapot.npz"))
    faces = np.cumsum(teapot["face_deltas"].astype(np.int64)).reshape(-1, 3) + 1
    path = tmp_path / "teapot.obj"
    with open(path, "w") as fh:
        fh.writelines("v %.9g %.9g %.9g\n" % tuple(float(x) for x in v) for v in teapot["positions"])
        fh.writelines("f %d %d %d\n" % tuple(f) for f in faces)
    scene = scenes.teapot_like_scene(str(path))
    oscene = oracle.OracleScene(scene)
    info = oscene.info()
    assert info.numTriangles == 15704 + 2  # SURVEY.md §0: 15 704 faces + the rectangle light
    assert oscene.validate() == ""
