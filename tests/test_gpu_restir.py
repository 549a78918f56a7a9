"""GPU parity: light distributions, G-buffer and the ReSTIR DI passes vs the CPU oracle, bit-exact
(SURVEY.md §8a rows G1, S1-S5, B1-B2, R1-R4)."""
import numpy as np
import pytest

from gfxexp_b200 import abi, engine, scenes

pytestmark = pytest.mark.gpu

ALL_BUFFERS = [(abi.BUF_GBUFFER0, 2), (abi.BUF_GBUFFER1, 2), (abi.BUF_GBUFFER2, 2), (abi.BUF_GBUFFER3, 2),
               (abi.BUF_RNG, 1), (abi.BUF_RESERVOIR, 2), (abi.BUF_RESERVOIR_INFO, 2), (abi.BUF_BEAUTY_ACCUM, 1),
               (abi.BUF_ALBEDO_ACCUM, 1), (abi.BUF_NORMAL_ACCUM, 1)]


def _compare_all(ctx, oframe, tag):
    for buf, count in ALL_BUFFERS:
        for idx in range(count):
            got = ctx.download(buf, idx)
            want = oframe.buffer(buf, idx)
            g = got.view(np.uint32) if got.dtype != np.uint64 else got
            w = want.view(np.uint32) if want.dtype != np.uint64 else want
            if not np.array_equal(g, w):
                bad = np.argwhere(g != w)
                raise AssertionError(f"{tag}: buffer {buf}[{idx}] differs at {len(bad)} elements, first {bad[:4].tolist()}: "
                                     f"{got[tuple(bad[0][:-1])] if got.ndim > 2 else got[tuple(bad[0])]} vs "
                                     f"{want[tuple(bad[0][:-1])] if want.ndim > 2 else want[tuple(bad[0])]}")


def _setup(ctx, oracle, scene, w, h):
    ctx.upload_scene(scene)
    ctx.build_bvh()
    ctx.create_frame(w, h)
    oscene = oracle.OracleScene(scene)
    oframe = oracle.OracleFrame(oscene, w, h)
    return oscene, oframe


def test_light_distributions(gfx_ctx, oracle):
    scene = scenes.small_city_scene()
    gfx_ctx.upload_scene(scene)
    gfx_ctx.build_light_distributions()
    oscene = oracle.OracleScene(scene)
    w, cdf, integ = gfx_ctx.light_dist()
    ow, ocdf, ointeg = oscene.light_dist()
    assert np.array_equal(w.view(np.uint32), ow.view(np.uint32))
    assert np.array_equal(cdf.view(np.uint32), ocdf.view(np.uint32))
    assert np.float32(integ).view(np.uint32) == np.float32(ointeg).view(np.uint32)
    assert integ > 0


_THREE_FRAME_CASES = [(False, "small_city_scene", 1), (True, "small_city_scene", 1),
                      (False, "small_interior_scene", 1),
                      # environment light: importance-map candidates, atInfinity samples through
                      # temporal / spatial reuse, the environment behind miss pixels
                      (False, "small_city_scene_env", 1), (True, "small_city_scene_env", 1),
                      (False, "env_only_scene", 1),
                      # image textures on the BSDF parameters (software tex2DLod, repeat addressing)
                      (False, "small_city_scene_textured", 1),
                      # no visibility reuse: the RIS pass is one kernel without a ray queue (with and without the
                      # environment light), the spatial passes evaluate unshadowed target densities
                      (False, "small_city_scene", 0), (True, "small_city_scene", 0), (False, "small_city_scene_env", 0)]


@pytest.mark.parametrize("unbiased,scene_name,reuse_visibility", _THREE_FRAME_CASES,
                         ids=[f"{u}-{s}" + ("" if v else "-no_reuse_visibility") for u, s, v in _THREE_FRAME_CASES])
def test_restir_three_frames_bit_exact(gfx_ctx, oracle, unbiased, scene_name, reuse_visibility):
    # small_interior_scene: config 3's ingredients - a closed room, 96 two-triangle emitters, SimplePBR materials
    # (common/common_device.cuh:767-776, 806-826)
    scene = getattr(scenes, scene_name)()
    w, h = 192, 108
    oscene, oframe = _setup(gfx_ctx, oracle, scene, w, h)
    p = abi.default_frame_params(scene, w, h)
    p.reuseVisibility = reuse_visibility
    for frame in range(3):
        gfx_ctx.build_light_distributions(frame % 2)
        for kind, pass_id in engine.restir_frame_passes(p, frame, num_spatial_passes=2 if not unbiased else 1,
                                                        temporal=True, unbiased=unbiased):
            if kind == "gbuffer":
                gfx_ctx.gbuffer(p)
                oframe.gbuffer(p)
            else:
                gfx_ctx.restir(p, pass_id)
                oframe.restir(p, pass_id)
        gfx_ctx.synchronize()
        _compare_all(gfx_ctx, oframe, f"frame {frame} unbiased={unbiased}")
    beauty = gfx_ctx.download(abi.BUF_BEAUTY_ACCUM)
    assert np.isfinite(beauty).all() and beauty[..., :3].mean() > 0


def test_restir_random_neighbors_and_jitter(gfx_ctx, oracle):
    scene = scenes.tiny_city_scene()
    w, h = 128, 72
    oscene, oframe = _setup(gfx_ctx, oracle, scene, w, h)
    p = abi.default_frame_params(scene, w, h)
    p.useLowDiscrepancyNeighbors = 0
    p.enableJittering = 1
    p.log2NumCandidateSamples = 3
    p.numSpatialNeighbors = 3
    # moving camera: temporal reprojection through the motion vectors
    for frame in range(3):
        p.prevCamera = abi.make_camera(scene, w, h) if frame == 0 else p.camera
        cam = abi.make_camera(scene, w, h)
        cam.position[0] += 0.05 * frame
        p.camera = cam
        if frame == 0:
            p.prevCamera = cam
        gfx_ctx.build_light_distributions(frame % 2)
        for kind, pass_id in engine.restir_frame_passes(p, frame, 1):
            if kind == "gbuffer":
                gfx_ctx.gbuffer(p)
                oframe.gbuffer(p)
            else:
                gfx_ctx.restir(p, pass_id)
                oframe.restir(p, pass_id)
        gfx_ctx.synchronize()
        _compare_all(gfx_ctx, oframe, f"jitter frame {frame}")


def test_tile_sharded_launch_matches_full_frame(gfx_ctx, oracle):
    """Screen-strip sharding (SURVEY.md §8e): rendering rows [0,h/2) and [h/2,h) in two launches of
    the passes without cross-pixel reads gives the full-frame result."""
    scene = scenes.tiny_city_scene()
    w, h = 96, 64
    oscene, oframe = _setup(gfx_ctx, oracle, scene, w, h)
    p = abi.default_frame_params(scene, w, h)
    gfx_ctx.build_light_distributions()
    passes = list(engine.restir_frame_passes(p, 0, 0))
    for kind, pass_id in passes:
        for (y0, rows) in ((0, h // 2), (h // 2, h - h // 2)):
            p.tileOriginY, p.tileRows = y0, rows
            if kind == "gbuffer":
                gfx_ctx.gbuffer(p)
            else:
                gfx_ctx.restir(p, pass_id)
        p.tileOriginY, p.tileRows = 0, 0
        if kind == "gbuffer":
            oframe.gbuffer(p)
        else:
            oframe.restir(p, pass_id)
    gfx_ctx.synchronize()
    _compare_all(gfx_ctx, oframe, "tiled")
