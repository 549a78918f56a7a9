"""ctypes mirror of include/gfxb200.h (the C ABI) — PODs, enums and the library loader.

The Python host side plays the role the reference's C++ hosts play (restir_di_main.cpp etc.):
it owns scene arrays, fills the per-frame parameter block and calls the launch entry points.
There is no Python fallback: if libgfxb200.so is missing, loading raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgfxb200.so")

c_f = C.c_float
c_u32 = C.c_uint32


class GfxMeshDesc(C.Structure):
    _fields_ = [("positions", C.POINTER(c_f)), ("normals", C.POINTER(c_f)), ("tangents", C.POINTER(c_f)),
                ("texcoords", C.POINTER(c_f)), ("triangles", C.POINTER(c_u32)),
                ("numVertices", c_u32), ("numTriangles", c_u32), ("materialSlot", c_u32), ("reserved", c_u32)]


class GfxMaterialDesc(C.Structure):
    _fields_ = [("p0", c_f * 3), ("p2", c_f), ("p1", c_f * 3), ("bsdfType", c_u32),
                ("emittance", c_f * 3), ("hasEmittance", c_u32)]


class GfxInstanceDesc(C.Structure):
    _fields_ = [("transform", c_f * 12), ("curToPrevTransform", c_f * 12), ("normalMatrix", c_f * 9),
                ("uniformScale", c_f), ("firstMeshSlot", c_u32), ("numMeshSlots", c_u32)]


class GfxTextureDesc(C.Structure):
    _fields_ = [("texels", C.POINTER(c_f)), ("width", c_u32), ("height", c_u32)]


class GfxSceneDesc(C.Structure):
    _fields_ = [("meshes", C.POINTER(GfxMeshDesc)), ("materials", C.POINTER(GfxMaterialDesc)),
                ("instances", C.POINTER(GfxInstanceDesc)), ("instanceMeshSlots", C.POINTER(c_u32)),
                ("numMeshes", c_u32), ("numMaterials", c_u32), ("numInstances", c_u32),
                ("numInstanceMeshSlots", c_u32),
                ("envTexels", C.POINTER(c_f)), ("envWidth", c_u32), ("envHeight", c_u32),
                ("textures", C.POINTER(GfxTextureDesc)), ("materialTextures", C.POINTER(c_u32)), ("numTextures", c_u32)]


class GfxBvhInfo(C.Structure):
    _fields_ = [("numNodes", c_u32), ("numPrimRefs", c_u32), ("numTriangles", c_u32), ("numGeoms", c_u32),
                ("sceneMin", c_f * 3), ("sceneMax", c_f * 3)]


class GfxCamera(C.Structure):
    _fields_ = [("aspect", c_f), ("fovY", c_f), ("position", c_f * 3), ("orientation", c_f * 9)]


class GfxPresentParams(C.Structure):
    _fields_ = [("sourceBuffer", C.c_int32), ("sourceIndex", c_u32), ("mode", C.c_int32), ("flags", c_u32),
                ("brightnessScale", c_f), ("alphaForOverride", c_f)]


class GfxKernelTiming(C.Structure):
    _fields_ = [("label", C.c_char * 48), ("totalMs", c_f), ("launches", c_u32)]


class GfxFrameParams(C.Structure):
    _fields_ = [("camera", GfxCamera), ("prevCamera", GfxCamera),
                ("numAccumFrames", c_u32), ("frameIndex", c_u32), ("bufferIndex", c_u32),
                ("spatialNeighborRadius", c_f),
                ("log2NumCandidateSamples", c_u32), ("numSpatialNeighbors", c_u32),
                ("useLowDiscrepancyNeighbors", c_u32), ("reuseVisibility", c_u32),
                ("enableTemporalReuse", c_u32), ("enableSpatialReuse", c_u32),
                ("useUnbiasedEstimator", c_u32), ("resetFlowBuffer", c_u32), ("enableJittering", c_u32),
                ("currentReservoirIndex", c_u32), ("spatialNeighborBaseIndex", c_u32),
                ("tileOriginY", c_u32), ("tileRows", c_u32), ("svgfFlags", c_u32), ("taaHistoryLength", c_u32),
                ("maxPathLength", c_u32),
                ("sceneAabbMin", c_f * 3), ("sceneAabbMax", c_f * 3), ("radianceScale", c_f),
                ("regirGridDim", c_u32 * 3), ("regirLog2NumCandidatesPerLightSlot", c_u32),
                ("regirLog2NumCandidatesPerCell", c_u32), ("regirEnableCellRandomization", c_u32),
                ("reuseVisibilityForTemporal", c_u32), ("reuseVisibilityForSpatiotemporal", c_u32),
                ("radiusThresholdForSpatialVisReuse", c_f),
                ("enableEnvLight", c_u32), ("envLightPowerCoeff", c_f), ("envLightRotation", c_f)]


NODE_DTYPE = np.dtype([("quantBoxOrigin", np.float32, 3), ("quantBoxExpScale", np.uint8, 3),
                       ("internalMask", np.uint8), ("intNodeChildBaseIndex", np.uint32),
                       ("leafBaseIndex", np.uint32), ("childMetas", np.uint8, 8),
                       ("childQMin", np.uint8, (3, 8)), ("childQMax", np.uint8, (3, 8))])
TRI_DTYPE = np.dtype([("pA", np.float32, 3), ("pB", np.float32, 3), ("pC", np.float32, 3),
                      ("geomIndex", np.uint32), ("primIndex", np.uint32), ("padding", np.uint32)])
HIT_DTYPE = np.dtype([("dist", np.float32), ("instIndex", np.uint32), ("instUserData", np.uint32),
                      ("geomIndex", np.uint32), ("primIndex", np.uint32),
                      ("bcA", np.float32), ("bcB", np.float32), ("bcC", np.float32)])
RAY_DTYPE = np.dtype([("org", np.float32, 3), ("tmin", np.float32), ("dir", np.float32, 3), ("tmax", np.float32)])
assert NODE_DTYPE.itemsize == 80 and TRI_DTYPE.itemsize == 48 and HIT_DTYPE.itemsize == 32 and RAY_DTYPE.itemsize == 32

# enums
TRACE_CLOSEST, TRACE_ANY, TRACE_STATS = 0, 1, 2
PT_BASELINE, PT_NRC, PT_REGIR = 0, 1, 2  # GfxPathTraceVariant
NRC_READ_MASTER, NRC_READ_TRAINING, NRC_READ_INFERENCE, NRC_READ_GRADIENTS = 0, 1, 2, 3  # gfx_nrc_read
(RESTIR_INITIAL_RIS, RESTIR_INITIAL_AND_TEMPORAL_BIASED, RESTIR_INITIAL_AND_TEMPORAL_UNBIASED,
 RESTIR_SPATIAL_BIASED, RESTIR_SPATIAL_UNBIASED, RESTIR_SHADING, RESTIR_PRESAMPLE_LIGHTS, RESTIR_PER_PIXEL_RIS,
 RESTIR_TRACE_SHADOW_RAYS, RESTIR_SHADE_AND_RESAMPLE) = range(10)
(SVGF_TEMPORAL_ACCUMULATE, SVGF_ESTIMATE_VARIANCE, SVGF_ATROUS, SVGF_FILL_BACKGROUND, SVGF_MODULATE_TAA) = range(5)
SVGF_IS_FIRST_FRAME, SVGF_ENABLE_TEMPORAL_ACCUMULATION, SVGF_FEEDBACK_1ST, SVGF_ENABLE_TAA, SVGF_MODULATE_ALBEDO = 1, 2, 4, 8, 16
(BUF_GBUFFER0, BUF_GBUFFER1, BUF_GBUFFER2, BUF_GBUFFER3, BUF_RNG, BUF_RESERVOIR, BUF_RESERVOIR_INFO,
 BUF_BEAUTY_ACCUM, BUF_ALBEDO_ACCUM, BUF_NORMAL_ACCUM, BUF_SVGF_LIGHTING_VARIANCE, BUF_SVGF_FINAL,
 BUF_SVGF_MOMENTS, BUF_SVGF_PREV_LIGHTING, BUF_SVGF_ALBEDO, BUF_SVGF_DEPTH,
 BUF_NRC_INFERENCE_QUERY, BUF_NRC_TERMINAL_INFO, BUF_NRC_INFERRED_RADIANCE, BUF_NRC_FRAME_CONTRIBUTION,
 BUF_NRC_TRAIN_QUERY, BUF_NRC_TRAIN_TARGET, BUF_NRC_TRAIN_VERTEX_INFO, BUF_NRC_TRAIN_SUFFIX_TERMINAL,
 BUF_NRC_STATE, BUF_REGIR_SLOTS, BUF_REGIR_SLOT_RNG, BUF_REGIR_CELL_ACCESSES, BUF_REGIR_LAST_ACCESS,
 BUF_REGIR_NUM_ACTIVE_CELLS, BUF_SAMPLE_VISIBILITY, BUF_PRESAMPLED_LIGHTS, BUF_PRESAMPLE_RNG) = range(33)

# logical per-pixel layout of each downloadable buffer: (numpy dtype, elements per pixel, planes)
BUF_PRESENT_RGBA8 = 33
PRESENT_COLOR, PRESENT_NORMAL = 0, 1
PRESENT_TONE_MAP, PRESENT_SRGB_GAMMA, PRESENT_FLIP_Y = 1, 2, 4
BUF_PEER_FLAGS = -1  # GFX_BUF_PEER_FLAGS: the flag block of the peer exchange (csrc/peer.cu)

BUFFER_LAYOUT = {
    BUF_GBUFFER0: (np.uint32, 4, 1), BUF_GBUFFER1: (np.float32, 2, 1), BUF_GBUFFER2: (np.uint32, 4, 1),
    BUF_GBUFFER3: (np.uint32, 4, 1), BUF_RNG: (np.uint64, 1, 1), BUF_RESERVOIR: (np.uint32, 4, 3),
    BUF_RESERVOIR_INFO: (np.float32, 2, 1), BUF_BEAUTY_ACCUM: (np.float32, 4, 1),
    BUF_ALBEDO_ACCUM: (np.float32, 4, 1), BUF_NORMAL_ACCUM: (np.float32, 4, 1), BUF_SAMPLE_VISIBILITY: (np.uint32, 1, 1),
    BUF_SVGF_LIGHTING_VARIANCE: (np.float32, 4, 1), BUF_SVGF_FINAL: (np.float32, 4, 1),
    BUF_SVGF_MOMENTS: (np.uint32, 4, 1), BUF_SVGF_PREV_LIGHTING: (np.float32, 4, 1),
    BUF_SVGF_ALBEDO: (np.float32, 4, 1), BUF_SVGF_DEPTH: (np.float32, 1, 1), BUF_PRESENT_RGBA8: (np.uint32, 1, 1),
}


def _fp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(c_f))


def _up(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(c_u32))


class SceneArrays:
    """Keeps the numpy arrays of a scenes.Scene alive and exposes them as a GfxSceneDesc."""

    def __init__(self, scene):
        self.scene = scene
        self._keep: List[np.ndarray] = []
        meshes = (GfxMeshDesc * len(scene.meshes))()
        for i, m in enumerate(scene.meshes):
            arrs = [np.ascontiguousarray(a) for a in (m.positions, m.normals, m.tangents, m.texcoords, m.triangles)]
            self._keep.extend(arrs)
            meshes[i].positions = _fp(arrs[0])
            meshes[i].normals = _fp(arrs[1])
            meshes[i].tangents = _fp(arrs[2])
            meshes[i].texcoords = _fp(arrs[3])
            meshes[i].triangles = _up(arrs[4])
            meshes[i].numVertices = arrs[0].shape[0]
            meshes[i].numTriangles = arrs[4].shape[0]
            meshes[i].materialSlot = m.material
        self.meshes = meshes
        mats = np.ascontiguousarray(scene.materials)
        assert mats.dtype.itemsize == C.sizeof(GfxMaterialDesc)
        self._keep.append(mats)
        self.materials = mats
        insts = (GfxInstanceDesc * len(scene.instances))()
        slots: List[int] = []
        for i, inst in enumerate(scene.instances):
            insts[i].transform = (c_f * 12)(*np.asarray(inst.transform, dtype=np.float32).reshape(-1))
            insts[i].curToPrevTransform = (c_f * 12)(*np.asarray(inst.cur_to_prev, dtype=np.float32).reshape(-1))
            insts[i].normalMatrix = (c_f * 9)(*np.asarray(inst.normal_matrix, dtype=np.float32).reshape(-1))
            insts[i].uniformScale = inst.uniform_scale
            insts[i].firstMeshSlot = len(slots)
            insts[i].numMeshSlots = len(inst.mesh_slots)
            slots.extend(inst.mesh_slots)
        self.instances = insts
        self.slots = np.asarray(slots, dtype=np.uint32)
        self.desc = GfxSceneDesc()
        self.desc.meshes = C.cast(meshes, C.POINTER(GfxMeshDesc))
        self.desc.materials = mats.ctypes.data_as(C.POINTER(GfxMaterialDesc))
        self.desc.instances = C.cast(insts, C.POINTER(GfxInstanceDesc))
        self.desc.instanceMeshSlots = _up(self.slots)
        self.desc.numMeshes = len(scene.meshes)
        self.desc.numMaterials = mats.shape[0]
        self.desc.numInstances = len(scene.instances)
        self.desc.numInstanceMeshSlots = self.slots.shape[0]
        env = getattr(scene, "env_map", None)  # float32 [H, W, 4] equirectangular map, or None
        if env is not None:
            self.env = np.ascontiguousarray(env, dtype=np.float32)
            assert self.env.ndim == 3 and self.env.shape[2] == 4
            self.desc.envTexels = self.env.ctypes.data_as(C.POINTER(c_f))
            self.desc.envHeight, self.desc.envWidth = self.env.shape[0], self.env.shape[1]
        textures = getattr(scene, "textures", None)  # list of float32 [H, W, 4] images, already decoded to linear floats
        if textures:
            self.textures = [np.ascontiguousarray(t, dtype=np.float32) for t in textures]
            self.texture_descs = (GfxTextureDesc * len(self.textures))()
            for d, t in zip(self.texture_descs, self.textures):
                assert t.ndim == 3 and t.shape[2] == 4
                d.texels = t.ctypes.data_as(C.POINTER(c_f))
                d.height, d.width = t.shape[0], t.shape[1]
            self.material_textures = np.ascontiguousarray(scene.material_textures, dtype=np.uint32).reshape(-1, 4)
            assert self.material_textures.shape[0] == mats.shape[0]
            self.desc.textures = C.cast(self.texture_descs, C.POINTER(GfxTextureDesc))
            self.desc.materialTextures = self.material_textures.ctypes.data_as(C.POINTER(c_u32))
            self.desc.numTextures = len(self.textures)


def make_instance_descs(instances):
    """GfxInstanceDesc[] for gfx_scene_update_instances: same (firstMeshSlot, numMeshSlots) numbering as SceneArrays"""
    insts = (GfxInstanceDesc * len(instances))()
    first = 0
    for i, inst in enumerate(instances):
        insts[i].transform = (c_f * 12)(*np.asarray(inst.transform, dtype=np.float32).reshape(-1))
        insts[i].curToPrevTransform = (c_f * 12)(*np.asarray(inst.cur_to_prev, dtype=np.float32).reshape(-1))
        insts[i].normalMatrix = (c_f * 9)(*np.asarray(inst.normal_matrix, dtype=np.float32).reshape(-1))
        insts[i].uniformScale = inst.uniform_scale
        insts[i].firstMeshSlot = first
        insts[i].numMeshSlots = len(inst.mesh_slots)
        first += len(inst.mesh_slots)
    return insts


def make_camera(scene, width: int, height: int) -> GfxCamera:
    cam = GfxCamera()
    cam.aspect = float(np.float32(width) / np.float32(height))
    cam.fovY = float(np.float32(scene.fov_y))
    cam.position = (c_f * 3)(*np.asarray(scene.camera_position, dtype=np.float32))
    cam.orientation = (c_f * 9)(*np.asarray(scene.camera_orientation, dtype=np.float32).reshape(-1))
    return cam


def default_frame_params(scene, width: int, height: int) -> GfxFrameParams:
    """restir_di defaults: ReSTIRConfigs(5, passes, neighbours), radius 20, low-discrepancy neighbours,
    reuseVisibility (restir_di_main.cpp:1938-1966), config 2 uses 1 spatial pass x 4 neighbours."""
    p = GfxFrameParams()
    p.camera = make_camera(scene, width, height)
    p.prevCamera = make_camera(scene, width, height)
    p.numAccumFrames = 0
    p.frameIndex = 0
    p.bufferIndex = 0
    p.spatialNeighborRadius = 20.0
    p.log2NumCandidateSamples = 5
    p.numSpatialNeighbors = 4
    p.useLowDiscrepancyNeighbors = 1
    p.reuseVisibility = 1
    p.enableTemporalReuse = 1
    p.enableSpatialReuse = 1
    p.useUnbiasedEstimator = 0
    p.resetFlowBuffer = 1
    p.enableJittering = 0
    p.currentReservoirIndex = 0
    p.spatialNeighborBaseIndex = 0
    p.tileOriginY = 0
    p.tileRows = 0
    p.svgfFlags = SVGF_ENABLE_TEMPORAL_ACCUMULATION | SVGF_FEEDBACK_1ST | SVGF_ENABLE_TAA | SVGF_MODULATE_ALBEDO
    p.taaHistoryLength = 16
    p.maxPathLength = 5
    lo, hi = scene_aabb(scene)
    p.sceneAabbMin = (c_f * 3)(*lo)
    p.sceneAabbMax = (c_f * 3)(*hi)
    p.radianceScale = 1.0
    p.enableEnvLight = 1  # used when the scene has an environment map (restir_di_main.cpp: enableEnvLight = true,
    p.envLightPowerCoeff = 1.0  # log10EnvLightPowerCoeff = 0, envLightRotation = 0 by default)
    p.envLightRotation = 0.0
    p.regirGridDim = (c_u32 * 3)(32, 8, 32)
    p.regirLog2NumCandidatesPerLightSlot = 3
    p.regirLog2NumCandidatesPerCell = 2
    p.regirEnableCellRandomization = 1
    p.reuseVisibilityForTemporal = 1
    p.reuseVisibilityForSpatiotemporal = 0
    p.radiusThresholdForSpatialVisReuse = 10.0
    return p


NRC_TRAIN_BUFFER_SIZE = 2 * 65536   # shared::trainBufferSize (neural_radiance_caching_shared.h:8-9)
NRC_TRAINING_DATA_PER_FRAME = 65536
NRC_INVALID_VERTEX = 0x007FFFFF     # shared::invalidVertexDataIndex
(NRC_STATE_NUM_TRAINING_DATA, NRC_STATE_TILE_SIZE, NRC_STATE_OFFSET_UNBIASED_TILE, NRC_STATE_OFFSET_TRAINING_PATH,
 NRC_STATE_TARGET_MIN, NRC_STATE_TARGET_MAX, NRC_STATE_TARGET_AVG, NRC_STATE_NUM_INFERENCE_QUERIES) = 0, 2, 6, 7, 8, 11, 20, 26


def nrc_num_suffixes(width: int, height: int) -> int:
    return ((width + 3) // 4) * ((height + 3) // 4)


def nrc_query_capacity(width: int, height: int) -> int:
    return (width * height + nrc_num_suffixes(width, height) + 127) // 128 * 128


REGIR_SLOTS_PER_CELL = 512  # shared::kNumLightSlotsPerCell


def linear_buffer_layout(buffer_id: int, width: int, height: int, params=None):
    """(numpy dtype, columns, rows) of the NRC / ReGIR buffers, which are linear rather than image shaped"""
    n = width * height
    if buffer_id == BUF_PRESAMPLED_LIGHTS:
        return (np.uint32, 12, 128 * 1024)
    if buffer_id == BUF_PRESAMPLE_RNG:
        return (np.uint64, 1, 128 * 1024)
    if BUF_REGIR_SLOTS <= buffer_id <= BUF_REGIR_NUM_ACTIVE_CELLS:
        dim = [int(d) for d in params.regirGridDim] if params is not None else [32, 8, 32]
        if 0 in dim:
            dim = [32, 8, 32]
        cells = dim[0] * dim[1] * dim[2]
        return {BUF_REGIR_SLOTS: (np.uint32, 16, cells * REGIR_SLOTS_PER_CELL),
                BUF_REGIR_SLOT_RNG: (np.uint64, 1, cells * REGIR_SLOTS_PER_CELL),
                BUF_REGIR_CELL_ACCESSES: (np.uint32, 1, cells), BUF_REGIR_LAST_ACCESS: (np.uint32, 1, cells),
                BUF_REGIR_NUM_ACTIVE_CELLS: (np.uint32, 1, 2)}[buffer_id]
    return {
        BUF_NRC_INFERENCE_QUERY: (np.float32, 14, nrc_query_capacity(width, height)),
        BUF_NRC_TERMINAL_INFO: (np.uint32, 4, n),
        BUF_NRC_INFERRED_RADIANCE: (np.float32, 3, nrc_query_capacity(width, height)),
        BUF_NRC_FRAME_CONTRIBUTION: (np.float32, 3, n),
        BUF_NRC_TRAIN_QUERY: (np.float32, 14, NRC_TRAIN_BUFFER_SIZE),
        BUF_NRC_TRAIN_TARGET: (np.float32, 3, NRC_TRAIN_BUFFER_SIZE),
        BUF_NRC_TRAIN_VERTEX_INFO: (np.uint32, 4, NRC_TRAIN_BUFFER_SIZE),
        BUF_NRC_TRAIN_SUFFIX_TERMINAL: (np.uint32, 1, nrc_num_suffixes(width, height)),
        BUF_NRC_STATE: (np.uint32, 1, 32),
    }.get(buffer_id)


def scene_aabb(scene):
    """world-space bounds of every instanced vertex (stands in for scene.initialSceneAabb, which the reference host
    accumulates from transformed group boxes, neural_radiance_caching_main.cpp:1096)"""
    cached = getattr(scene, "_aabb_cache", None)
    if cached is not None:
        return cached
    lo = np.full(3, np.inf, dtype=np.float32)
    hi = np.full(3, -np.inf, dtype=np.float32)
    for inst in scene.instances:
        m = np.asarray(inst.transform, dtype=np.float32).reshape(3, 4)
        for slot in inst.mesh_slots:
            v = np.asarray(scene.meshes[slot].positions, dtype=np.float32).reshape(-1, 3)
            w = (v @ m[:, :3].T + m[:, 3]).astype(np.float32)
            lo = np.minimum(lo, w.min(axis=0))
            hi = np.maximum(hi, w.max(axis=0))
    scene._aabb_cache = ([float(x) for x in lo], [float(x) for x in hi])
    return scene._aabb_cache


OP_LIGHT_DIST, OP_GBUFFER, OP_RESTIR, OP_PEER_PUSH_ROWS, OP_PEER_SIGNAL, OP_PEER_WAIT = 0, 1, 2, 3, 4, 5


class GfxBatchOp(C.Structure):
    _fields_ = [("op", c_u32), ("a", c_u32), ("b", c_u32), ("c", c_u32), ("d", c_u32), ("e", c_u32), ("pad", c_u32 * 2),
                ("params", GfxFrameParams)]


class GfxStripFrame(C.Structure):
    _fields_ = [(n, c_u32) for n in ("frameIndex", "numSpatialPasses", "unbiased", "temporal", "y0", "y1", "halo", "rank", "world",
                                     "usePeer", "peerSeq")]


_DECLS = {
    "gfx_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "gfx_ctx_destroy": (None, [C.c_void_p]),
    "gfx_last_error_string": (C.c_char_p, [C.c_void_p]),
    "gfx_synchronize": (C.c_int, [C.c_void_p, C.c_void_p]),
    "gfx_kernel_launch_count": (C.c_uint64, [C.c_void_p]),
    "gfx_scene_upload": (C.c_int, [C.c_void_p, C.POINTER(GfxSceneDesc)]),
    "gfx_scene_update_instances": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxInstanceDesc), c_u32]),
    "gfx_bvh_build": (C.c_int, [C.c_void_p, C.c_void_p, c_u32]),
    "gfx_bvh_info": (C.c_int, [C.c_void_p, C.POINTER(GfxBvhInfo)]),
    "gfx_bvh_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfx_bvh_import": (C.c_int, [C.c_void_p, C.c_void_p, c_u32, C.c_void_p, c_u32, C.c_void_p, c_u32]),
    "gfx_trace_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.c_void_p, C.c_int]),
    "gfx_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.c_void_p, C.c_int]),
    "gfx_light_dist_build": (C.c_int, [C.c_void_p, C.c_void_p, c_u32]),
    "gfx_framebuffer_allgather": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.c_void_p]),
    "gfx_framebuffer_allgatherv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(c_u32), c_u32, C.c_void_p]),
    "gfx_restir_strip_frame": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), C.POINTER(GfxStripFrame)]),
    "gfx_launch_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxBatchOp), c_u32]),
    "gfx_light_pick_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.c_void_p, C.c_void_p]),
    "gfx_env_light_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, c_u32, C.c_void_p]),
    "gfx_light_dist_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(c_f)]),
    "gfx_frame_create": (C.c_int, [C.c_void_p, c_u32, c_u32]),
    "gfx_rng_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "gfx_restir_setup_neighbor_table": (C.c_int, [C.c_void_p]),
    "gfx_buffer_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, c_u32, C.c_void_p, C.c_size_t]),
    "gfx_buffer_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, c_u32, C.c_void_p, C.c_size_t]),
    "gfx_buffer_device_ptr": (C.c_void_p, [C.c_void_p, C.c_int, c_u32, C.POINTER(C.c_size_t)]),
    "gfx_stats_read": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_int]),
    "gfx_gbuffer_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams)]),
    "gfx_restir_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), C.c_int]),
    "gfx_svgf_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), C.c_int, c_u32]),
    "gfx_pathtrace_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), C.c_int]),
    "gfx_timing_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "gfx_timing_read": (C.c_int, [C.c_void_p, C.c_void_p, c_u32, C.POINTER(c_u32)]),
    "gfx_present_launch": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxPresentParams)]),
    "gfx_peer_export": (C.c_int, [C.c_void_p, C.c_int, c_u32, C.c_void_p]),
    "gfx_peer_open": (C.c_int, [C.c_void_p, c_u32, C.c_int, c_u32, C.c_void_p]),
    "gfx_peer_push_rows": (C.c_int, [C.c_void_p, C.c_void_p, c_u32, C.c_int, c_u32, c_u32, c_u32]),
    "gfx_peer_signal": (C.c_int, [C.c_void_p, C.c_void_p, c_u32, c_u32, c_u32]),
    "gfx_peer_wait": (C.c_int, [C.c_void_p, C.c_void_p, c_u32, c_u32]),
    "gfx_peer_status": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(c_u32)]),
    "gfx_peer_close": (C.c_int, [C.c_void_p]),
    "gfx_regir_build_cells": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), c_u32, C.c_int]),
    "gfx_regir_update_access": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), c_u32]),
    "gfx_nrc_preprocess": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams), c_u32, c_u32, C.c_int]),
    "gfx_nrc_frame_infer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "gfx_nrc_shard": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "gfx_nrc_frame_infer_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, c_u32]),
    "gfx_nrc_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams)]),
    "gfx_nrc_propagate": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams)]),
    "gfx_nrc_shuffle": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(GfxFrameParams)]),
    "gfx_nrc_frame_train": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]),
    "gfx_nrc_create": (C.c_int, [C.c_void_p, c_u32, c_f, C.POINTER(C.c_void_p)]),
    "gfx_nrc_destroy": (None, [C.c_void_p]),
    "gfx_nrc_infer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_u32]),
    "gfx_nrc_train": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.POINTER(c_f)]),
    "gfx_nrc_reset": (C.c_int, [C.c_void_p, c_u32]),
    "gfx_nrc_read": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    "gfx_nrc_encode_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, c_u32, C.c_void_p]),
    "gfx_nrc_keep_gradients": (C.c_int, [C.c_void_p, C.c_int]),
    "gfx_nrc_get_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "gfx_nrc_set_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "gfx_nrc_num_params": (c_u32, [C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_DECLS.keys())


def load_library(path: str | None = None) -> C.CDLL:
    """Load libgfxb200.so and attach prototypes.  Raises OSError if the CUDA extension has not been
    built (python -c 'import __graft_entry__ as g; g.build()') — there is no fallback path."""
    path = path or os.environ.get("GFXB200_LIB") or LIB_PATH  # GFXB200_LIB: another build of the library, e.g. to compare two commits
    if not os.path.exists(path):
        raise OSError(f"{path} not found: build the CUDA extension first (__graft_entry__.build()); "
                      "gfxexp_b200 has no CPU fallback")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _DECLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib
