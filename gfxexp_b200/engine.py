"""Host-side mirror of the reference's per-app frame loops, on top of the C ABI.

`Context` is a thin, loud wrapper over libgfxb200.so (every non-zero status raises GfxError with
gfx_last_error_string).  `ReSTIRRenderer.render_frame` issues the launch sequence of
restir_di/restir_di_main.cpp:2245-2421 (updateASs once, setupLightInstDistribution, gBuffer launch,
performInitialAndTemporalRIS, numSpatialReusePasses x performSpatialRIS with ping-pong reservoirs,
shading).  There is no CPU path here: without the CUDA library nothing runs.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import abi


class GfxError(RuntimeError):
    pass


class Context:
    def __init__(self, device: int = 0, lib: Optional[C.CDLL] = None):
        self.lib = lib or abi.load_library()
        h = C.c_void_p()
        rc = self.lib.gfx_ctx_create(device, C.byref(h))
        if rc != 0:
            raise GfxError(f"gfx_ctx_create(device={device}) failed with status {rc} "
                           "(-2 = no sm_100 device; this library has no CPU fallback)")
        self.h = h
        self.device = device
        self.width = self.height = 0
        self._scene_arrays = None

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.gfx_last_error_string(self.h)
            raise GfxError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "h", None):
            self.lib.gfx_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self, stream=None):
        self._check(self.lib.gfx_synchronize(self.h, stream), "gfx_synchronize")

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.gfx_kernel_launch_count(self.h))

    # -- scene / BVH ------------------------------------------------------------------------
    def upload_scene(self, scene):
        self._scene_arrays = abi.SceneArrays(scene)
        self._check(self.lib.gfx_scene_upload(self.h, C.byref(self._scene_arrays.desc)), "gfx_scene_upload")

    def update_instances(self, instance_descs, stream=None):
        """per-frame instance update (InstanceController::update): new transforms, curToPrevTransform, normal matrices;
        follow with build_bvh (GFX_BVH_BUILD_FAST for per-frame rebuilds) and build_light_distributions"""
        self._check(self.lib.gfx_scene_update_instances(self.h, stream, instance_descs, len(instance_descs)),
                    "gfx_scene_update_instances")

    def build_bvh(self, flags: int = 0, stream=None):
        self._check(self.lib.gfx_bvh_build(self.h, stream, flags), "gfx_bvh_build")

    def bvh_info(self) -> abi.GfxBvhInfo:
        info = abi.GfxBvhInfo()
        self._check(self.lib.gfx_bvh_info(self.h, C.byref(info)), "gfx_bvh_info")
        return info

    def export_bvh(self):
        info = self.bvh_info()
        nodes = np.zeros(info.numNodes, dtype=abi.NODE_DTYPE)
        refs = np.zeros(info.numPrimRefs, dtype=np.uint32)
        tris = np.zeros(info.numTriangles, dtype=abi.TRI_DTYPE)
        self._check(self.lib.gfx_bvh_export(self.h, nodes.ctypes.data, refs.ctypes.data, tris.ctypes.data),
                    "gfx_bvh_export")
        return nodes, refs, tris

    def import_bvh(self, nodes, refs, tris):
        nodes = np.ascontiguousarray(nodes)
        refs = np.ascontiguousarray(refs)
        tris = np.ascontiguousarray(tris)
        self._check(self.lib.gfx_bvh_import(self.h, nodes.ctypes.data, nodes.shape[0], refs.ctypes.data,
                                            refs.shape[0], tris.ctypes.data, tris.shape[0]), "gfx_bvh_import")

    def trace(self, rays: np.ndarray, mode: int = abi.TRACE_CLOSEST, stream=None) -> np.ndarray:
        rays = np.ascontiguousarray(rays)
        assert rays.dtype == abi.RAY_DTYPE
        hits = np.zeros(rays.shape[0], dtype=abi.HIT_DTYPE)
        self._check(self.lib.gfx_trace(self.h, stream, rays.ctypes.data, rays.shape[0], hits.ctypes.data, mode),
                    "gfx_trace")
        self.synchronize(stream)
        return hits

    def trace_device(self, d_rays: int, num_rays: int, d_hits: int, mode: int = abi.TRACE_CLOSEST, stream=None):
        self._check(self.lib.gfx_trace_device(self.h, stream, d_rays, num_rays, d_hits, mode), "gfx_trace_device")

    def build_light_distributions(self, buffer_index: int = 0, stream=None):
        self._check(self.lib.gfx_light_dist_build(self.h, stream, buffer_index), "gfx_light_dist_build")

    def light_dist(self):
        n = len(self._scene_arrays.scene.instances)
        w = np.zeros(n, dtype=np.float32)
        cdf = np.zeros(n, dtype=np.float32)
        integ = C.c_float()
        self._check(self.lib.gfx_light_dist_export(self.h, w.ctypes.data, cdf.ctypes.data, C.byref(integ)),
                    "gfx_light_dist_export")
        return w, cdf, integ.value

    # -- frame state --------------------------------------------------------------------------
    def create_frame(self, width: int, height: int, seed: int = 591842031321323413):
        self._check(self.lib.gfx_frame_create(self.h, width, height), "gfx_frame_create")
        self.width, self.height = width, height
        self._check(self.lib.gfx_rng_seed(self.h, seed), "gfx_rng_seed")
        self._check(self.lib.gfx_restir_setup_neighbor_table(self.h), "gfx_restir_setup_neighbor_table")

    def download(self, buffer_id: int, index: int = 0, out: Optional[np.ndarray] = None, stream=None) -> np.ndarray:
        dtype, comps, planes = abi.BUFFER_LAYOUT[buffer_id]
        count = planes * self.height * self.width * comps
        arr = out if out is not None else np.empty(count, dtype=dtype)
        self._check(self.lib.gfx_buffer_download(self.h, stream, buffer_id, index, arr.ctypes.data, arr.nbytes),
                    "gfx_buffer_download")
        if out is not None:
            return out
        if planes > 1:
            return arr.reshape(planes, self.height, self.width, comps)
        return arr.reshape(self.height, self.width, comps) if comps > 1 else arr.reshape(self.height, self.width)

    def upload(self, buffer_id: int, index: int, data: np.ndarray, stream=None):
        data = np.ascontiguousarray(data)
        self._check(self.lib.gfx_buffer_upload(self.h, stream, buffer_id, index, data.ctypes.data, data.nbytes),
                    "gfx_buffer_upload")

    def device_ptr(self, buffer_id: int, index: int = 0):
        nbytes = C.c_size_t()
        p = self.lib.gfx_buffer_device_ptr(self.h, buffer_id, index, C.byref(nbytes))
        return p, nbytes.value

    def read_stats(self, reset: bool = True, stream=None):
        out = (C.c_uint64 * 4)()
        self._check(self.lib.gfx_stats_read(self.h, stream, out, 1 if reset else 0), "gfx_stats_read")
        return [int(v) for v in out]

    def timing_enable(self, on: bool = True):
        self._check(self.lib.gfx_timing_enable(self.h, 1 if on else 0), "gfx_timing_enable")

    def timing_read(self) -> dict:
        """{kernel label: (total ms, launches)} since the last read; CUDA events around every kernel launch"""
        buf = (abi.GfxKernelTiming * 64)()
        n = abi.c_u32()
        self._check(self.lib.gfx_timing_read(self.h, buf, 64, C.byref(n)), "gfx_timing_read")
        return {buf[i].label.decode(): (float(buf[i].totalMs), int(buf[i].launches)) for i in range(n.value)}

    # -- multi-GPU peer exchange (csrc/peer.cu) ---------------------------------------------------
    def peer_export(self, buffer_id: int, index: int = 0) -> bytes:
        h = C.create_string_buffer(64)
        self._check(self.lib.gfx_peer_export(self.h, buffer_id, index, h), "gfx_peer_export")
        return h.raw

    def peer_open(self, link: int, buffer_id: int, index: int, handle: bytes):
        self._check(self.lib.gfx_peer_open(self.h, link, buffer_id, index, C.create_string_buffer(handle, 64)), "gfx_peer_open")

    def peer_timed_out(self, stream=None) -> bool:
        v = abi.c_u32()
        self._check(self.lib.gfx_peer_status(self.h, stream, C.byref(v)), "gfx_peer_status")
        return v.value != 0

    # -- launches -------------------------------------------------------------------------------
    def gbuffer(self, params, stream=None):
        self._check(self.lib.gfx_gbuffer_launch(self.h, stream, C.byref(params)), "gfx_gbuffer_launch")

    def restir(self, params, pass_id: int, stream=None):
        self._check(self.lib.gfx_restir_launch(self.h, stream, C.byref(params), pass_id), "gfx_restir_launch")

    def present(self, source_buffer: int = abi.BUF_BEAUTY_ACCUM, source_index: int = 0, mode: int = abi.PRESENT_COLOR,
                flags: int = abi.PRESENT_TONE_MAP | abi.PRESENT_SRGB_GAMMA, brightness_scale: float = 1.0,
                alpha_override: float = 1.0, stream=None) -> np.ndarray:
        """accumulation buffer -> tone-mapped, sRGB-encoded RGBA8 [H, W] uint32 (R | G << 8 | B << 16 | A << 24), the
        packing of the reference's saveImage(path, w, h, const uint32_t*)"""
        pp = abi.GfxPresentParams(source_buffer, source_index, mode, flags, brightness_scale, alpha_override)
        self._check(self.lib.gfx_present_launch(self.h, stream, C.byref(pp)), "gfx_present_launch")
        return self.download(abi.BUF_PRESENT_RGBA8)

    def pathtrace(self, params, variant: int = abi.PT_BASELINE, stream=None):
        """one sample per pixel of the path tracer (path_tracing_main.cpp:1780-1789) from the current G-buffer"""
        self._check(self.lib.gfx_pathtrace_launch(self.h, stream, C.byref(params), variant), "gfx_pathtrace_launch")

    def svgf(self, params, pass_id: int, stage: int = 0, stream=None):
        self._check(self.lib.gfx_svgf_launch(self.h, stream, C.byref(params), pass_id, stage), "gfx_svgf_launch")

    # -- NRC frame (neural_radiance_caching_main.cpp:2270-2368) -------------------------------------
    def download_linear(self, buffer_id: int, index: int = 0, stream=None, params=None) -> np.ndarray:
        """NRC / ReGIR buffers (GFX_BUF_NRC_*, GFX_BUF_REGIR_*) as [rows, cols]"""
        dtype, cols, rows = abi.linear_buffer_layout(buffer_id, self.width, self.height, params)
        arr = np.empty((rows, cols), dtype=dtype)
        self._check(self.lib.gfx_buffer_download(self.h, stream, buffer_id, index, arr.ctypes.data, arr.nbytes),
                    "gfx_buffer_download")
        return arr

    # -- ReGIR (regir_main.cpp:2033-2068) -----------------------------------------------------------
    def regir_build_cells(self, params, frame_index: int, temporal: bool, stream=None):
        self._check(self.lib.gfx_regir_build_cells(self.h, stream, C.byref(params), frame_index & 0xFFFFFFFF, 1 if temporal else 0),
                    "gfx_regir_build_cells")

    def regir_update_access(self, params, frame_index: int, stream=None):
        self._check(self.lib.gfx_regir_update_access(self.h, stream, C.byref(params), frame_index & 0xFFFFFFFF),
                    "gfx_regir_update_access")

    def regir_frame(self, params, frame_index: int, temporal: bool = True, stream=None):
        """one ReGIR frame (regir_main.cpp:2022-2068): G-buffer, cell reservoirs (+ temporal reuse after the first
        frame of a sequence), path tracing with reservoir-based NEE, last-access bookkeeping"""
        params.frameIndex = frame_index
        params.bufferIndex = frame_index % 2
        self.gbuffer(params, stream)
        self.regir_build_cells(params, frame_index, temporal and frame_index > 0, stream)
        self.pathtrace(params, abi.PT_REGIR, stream)
        self.regir_update_access(params, frame_index, stream)

    def nrc_preprocess(self, params, offset_unbiased_tile: int, offset_training_path: int, new_sequence: bool, stream=None):
        self._check(self.lib.gfx_nrc_preprocess(self.h, stream, C.byref(params), offset_unbiased_tile & 0xFFFFFFFF,
                                                offset_training_path & 0xFFFFFFFF, 1 if new_sequence else 0),
                    "gfx_nrc_preprocess")

    def nrc_frame_infer(self, net: "NeuralRadianceCache", stream=None):
        self._check(self.lib.gfx_nrc_frame_infer(self.h, net.h, stream), "gfx_nrc_frame_infer")

    def nrc_accumulate(self, params, stream=None):
        self._check(self.lib.gfx_nrc_accumulate(self.h, stream, C.byref(params)), "gfx_nrc_accumulate")

    def nrc_propagate(self, params, stream=None):
        self._check(self.lib.gfx_nrc_propagate(self.h, stream, C.byref(params)), "gfx_nrc_propagate")

    def nrc_shuffle(self, params, stream=None):
        self._check(self.lib.gfx_nrc_shuffle(self.h, stream, C.byref(params)), "gfx_nrc_shuffle")

    def nrc_frame_train(self, net: "NeuralRadianceCache", want_loss: bool = False, stream=None):
        loss = C.c_float()
        self._check(self.lib.gfx_nrc_frame_train(self.h, net.h, stream, C.byref(loss) if want_loss else None),
                    "gfx_nrc_frame_train")
        return loss.value if want_loss else None

    def nrc_frame(self, net: "NeuralRadianceCache", params, frame_index: int, offsets, train: bool = True,
                  want_loss: bool = False, stream=None):
        """One frame of neural_radiance_caching_main.cpp:2256-2368 with useNRC: G-buffer, preprocessNRC, pathTraceNRC,
        infer, accumulate and (when training) propagate, shuffle, 4 training steps.  `offsets` are the two
        perFrameRng() draws of :2273-2275.  Everything is enqueued on `stream`; nothing synchronises with the host
        unless the loss is requested."""
        params.frameIndex = frame_index
        params.bufferIndex = frame_index % 2
        self.gbuffer(params, stream)
        self.nrc_preprocess(params, offsets[0], offsets[1], frame_index == 0, stream)
        self.pathtrace(params, abi.PT_NRC, stream)
        self.nrc_frame_infer(net, stream)
        self.nrc_accumulate(params, stream)
        if train:
            self.nrc_propagate(params, stream)
            self.nrc_shuffle(params, stream)
            return self.nrc_frame_train(net, want_loss, stream)
        return None


class NeuralRadianceCache:
    """Mirror of the reference's NeuralRadianceCache facade (neural_radiance_caching/network_interface.h:14-28):
    initialize -> __init__, infer, train, finalize -> close.  Device buffers are torch CUDA tensors or raw
    device pointers (queries: float[numData, 14] row per query; predictions/targets: float[numData, 3])."""

    def __init__(self, ctx: "Context", num_hidden_layers: int = 2, learning_rate: float = 1e-2):
        self.ctx = ctx
        h = C.c_void_p()
        ctx._check(ctx.lib.gfx_nrc_create(ctx.h, num_hidden_layers, learning_rate, C.byref(h)), "gfx_nrc_create")
        self.h = h
        self.num_params = int(ctx.lib.gfx_nrc_num_params(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.ctx.lib.gfx_nrc_destroy(self.h)
            self.h = None

    def set_params(self, params_f16: np.ndarray):
        p = np.ascontiguousarray(params_f16, dtype=np.float16)
        self.ctx._check(self.ctx.lib.gfx_nrc_set_params(self.h, p.ctypes.data, p.nbytes), "gfx_nrc_set_params")

    def get_params(self) -> np.ndarray:
        out = np.empty(self.num_params, dtype=np.float16)
        self.ctx._check(self.ctx.lib.gfx_nrc_get_params(self.h, out.ctypes.data, out.nbytes), "gfx_nrc_get_params")
        return out

    def encode(self, queries, num_data: int, stream=None) -> np.ndarray:
        """test hook: the encoded network input [num_data][64] float16 as the inference kernels produce it"""
        import torch
        out = torch.empty((num_data, 64), dtype=torch.float16, device="cuda")
        self.ctx._check(self.ctx.lib.gfx_nrc_encode_debug(self.h, stream, self._ptr(queries), num_data, out.data_ptr()),
                        "gfx_nrc_encode_debug")
        torch.cuda.synchronize()
        return out.cpu().numpy()

    def reset(self, seed: int = 1337):
        """re-initialise like a fresh tcnn::Trainer with this seed (gfx_nrc_create does it with 1337, the reference's)"""
        self.ctx._check(self.ctx.lib.gfx_nrc_reset(self.h, seed), "gfx_nrc_reset")

    def keep_gradients(self, on: bool = True):
        self.ctx._check(self.ctx.lib.gfx_nrc_keep_gradients(self.h, 1 if on else 0), "gfx_nrc_keep_gradients")

    def read(self, which: int) -> np.ndarray:
        """abi.NRC_READ_MASTER / _GRADIENTS -> float32[num_params]; _TRAINING / _INFERENCE -> float16[num_params]"""
        dtype = np.float32 if which in (abi.NRC_READ_MASTER, abi.NRC_READ_GRADIENTS) else np.float16
        out = np.empty(self.num_params, dtype=dtype)
        self.ctx._check(self.ctx.lib.gfx_nrc_read(self.h, which, out.ctypes.data, out.nbytes), "gfx_nrc_read")
        return out

    @staticmethod
    def _ptr(t):
        return t if isinstance(t, int) else t.data_ptr()

    def infer(self, queries, predictions, num_data: int, stream=None):
        self.ctx._check(self.ctx.lib.gfx_nrc_infer(self.h, stream, self._ptr(queries), self._ptr(predictions), num_data),
                        "gfx_nrc_infer")

    def train(self, queries, targets, num_data: int, want_loss: bool = False, stream=None):
        loss = C.c_float()
        self.ctx._check(self.ctx.lib.gfx_nrc_train(self.h, stream, self._ptr(queries), self._ptr(targets), num_data,
                                                   C.byref(loss) if want_loss else None), "gfx_nrc_train")
        return loss.value if want_loss else None


def primary_rays(params, width: int, height: int) -> np.ndarray:
    """pinhole primary rays of setupGBuffers (optix_gbuffer_kernels.cu:21-27; SURVEY.md A.4): dir = normalize(orientation *
    (vw (0.5 - x), vh (0.5 - y), 1)), x = (ix + 0.5) / W - for gfx_trace statistics and tools (the G-buffer kernel generates its
    own rays on the device)"""
    cam = params.camera
    ori = np.asarray(cam.orientation[:], dtype=np.float32).reshape(3, 3)
    vh = np.float32(2.0 * np.tan(np.float32(cam.fovY) * np.float32(0.5)))
    vw = np.float32(cam.aspect) * vh
    x = (np.arange(width, dtype=np.float32) + np.float32(0.5)) / np.float32(width)
    y = (np.arange(height, dtype=np.float32) + np.float32(0.5)) / np.float32(height)
    d = np.stack(np.broadcast_arrays((vw * (np.float32(0.5) - x))[None, :], (vh * (np.float32(0.5) - y))[:, None],
                                     np.ones((height, width), dtype=np.float32)), axis=-1).astype(np.float32)
    d = d @ ori.T
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    rays = np.zeros(width * height, dtype=abi.RAY_DTYPE)
    rays["org"] = np.asarray(cam.position[:], dtype=np.float32)
    rays["dir"] = d.reshape(-1, 3)
    rays["tmax"] = np.float32(3.402823466e+38)
    return rays


def random_nrc_params(num_params: int, num_matrix_weights: int, seed: int = 1337, grid_amplitude: float = 1e-4) -> np.ndarray:
    """Xavier-uniform MLP matrices and U(-a, a) hash-grid entries (tcnn: gpu_matrix.h initialize_xavier_uniform,
    grid.h:1267-1272), from a numpy stream (the reference's pcg32 stream is not reproduced)."""
    rng = np.random.default_rng(seed)
    p = np.empty(num_params, dtype=np.float32)
    bound = np.sqrt(6.0 / (64 + 64))
    p[:num_matrix_weights] = rng.uniform(-bound, bound, num_matrix_weights)
    p[num_matrix_weights:] = rng.uniform(-grid_amplitude, grid_amplitude, num_params - num_matrix_weights)
    return p.astype(np.float16)


def restir_frame_passes(params, frame_index: int, num_spatial_passes: int = 1, temporal: bool = True,
                        unbiased: bool = False):
    """The launch list of one ReSTIR DI frame (restir_di_main.cpp:2321-2421).  Yields
    (kind, pass_id) with `params` mutated in place exactly as the host mutates plp between launches."""
    params.frameIndex = frame_index
    params.bufferIndex = frame_index % 2
    params.useUnbiasedEstimator = 1 if unbiased else 0
    # enableTemporalReuse is the renderer *config* flag; the first frame of a sequence only selects the
    # performInitialRIS entry point (restir_di_main.cpp:2378-2383) and resets the flow buffer (:2340)
    params.enableTemporalReuse = 1 if temporal else 0
    params.enableSpatialReuse = 1 if num_spatial_passes > 0 else 0
    new_sequence = frame_index == 0
    params.resetFlowBuffer = 1 if new_sequence else 0
    yield ("gbuffer", -1)
    # curReservoirIndex = (lastReservoirIndex + 1) % 2, starts so that frame 0 writes reservoir 0
    base = (frame_index * (1 + num_spatial_passes)) % 2
    params.currentReservoirIndex = base
    if params.enableTemporalReuse and not new_sequence:
        yield ("restir", abi.RESTIR_INITIAL_AND_TEMPORAL_UNBIASED if unbiased else abi.RESTIR_INITIAL_AND_TEMPORAL_BIASED)
    else:
        yield ("restir", abi.RESTIR_INITIAL_RIS)
    cur = base
    for s in range(num_spatial_passes):
        params.currentReservoirIndex = cur
        params.spatialNeighborBaseIndex = (frame_index * num_spatial_passes * max(params.numSpatialNeighbors, 1)
                                           + s * params.numSpatialNeighbors) % 1024
        yield ("restir", abi.RESTIR_SPATIAL_UNBIASED if unbiased else abi.RESTIR_SPATIAL_BIASED)
        cur = (cur + 1) % 2
    params.currentReservoirIndex = cur
    yield ("restir", abi.RESTIR_SHADING)


def restir_rearch_frame_passes(params, frame_index: int, temporal: bool = True, spatial: bool = True, unbiased: bool = False):
    """The launch list of one frame of the rearchitected ReSTIR renderer (restir_di_main.cpp:2321-2366, 2423-2493).  Yields
    (kind, pass_id) with `params` mutated in place as the host mutates plp: reservoirs ping-pong once per frame,
    spatialNeighborBaseIndex advances by one, and the first frame of a sequence selects the entry points without reuse
    (here: enableTemporalReuse / enableSpatialReuse = 0 for the launches of that frame)."""
    params.frameIndex = frame_index
    params.bufferIndex = frame_index % 2
    params.useUnbiasedEstimator = 1 if unbiased else 0
    new_sequence = frame_index == 0
    params.resetFlowBuffer = 1 if new_sequence else 0
    params.currentReservoirIndex = frame_index % 2          # (lastReservoirIndex + 1) % 2
    params.spatialNeighborBaseIndex = frame_index           # ++lastSpatialNeighborBaseIndex per frame
    yield ("gbuffer", None)
    yield ("restir", abi.RESTIR_PRESAMPLE_LIGHTS)
    yield ("restir", abi.RESTIR_PER_PIXEL_RIS)
    params.enableTemporalReuse = 1 if (temporal and not new_sequence) else 0
    params.enableSpatialReuse = 1 if (spatial and not new_sequence) else 0
    yield ("restir", abi.RESTIR_TRACE_SHADOW_RAYS)
    yield ("restir", abi.RESTIR_SHADE_AND_RESAMPLE)
    params.enableTemporalReuse = 1 if temporal else 0
    params.enableSpatialReuse = 1 if spatial else 0


def svgf_frame_passes(params, frame_index: int, num_filtering_stages: int = 5):
    """The launch list of the SVGF part of a frame (svgf/svgf_main.cpp:2118-2172): temporal accumulation of
    the demodulated lighting, variance estimate, 5 a-trous stages, background fill, albedo modulation + TAA.
    Yields (pass_id, stage); sets the first-frame flag exactly like the host (`isFirstFrame`)."""
    if frame_index == 0:
        params.svgfFlags |= abi.SVGF_IS_FIRST_FRAME
    else:
        params.svgfFlags &= ~abi.SVGF_IS_FIRST_FRAME
    yield (abi.SVGF_TEMPORAL_ACCUMULATE, 0)
    yield (abi.SVGF_ESTIMATE_VARIANCE, 0)
    for stage in range(num_filtering_stages):
        yield (abi.SVGF_ATROUS, stage)
    yield (abi.SVGF_FILL_BACKGROUND, num_filtering_stages)
    yield (abi.SVGF_MODULATE_TAA, num_filtering_stages)


class ReSTIRRenderer:
    """Config-2 style frame driver (OriginalReSTIRBiased by default)."""

    def __init__(self, ctx: Context, scene, width: int, height: int, num_spatial_passes: int = 1,
                 unbiased: bool = False):
        self.ctx = ctx
        self.scene = scene
        self.params = abi.default_frame_params(scene, width, height)
        self.num_spatial_passes = num_spatial_passes
        self.unbiased = unbiased
        self.frame_index = 0

    def render_frame(self, stream=None):
        self.ctx.build_light_distributions(self.frame_index % 2, stream)
        for kind, pass_id in restir_frame_passes(self.params, self.frame_index, self.num_spatial_passes,
                                                 True, self.unbiased):
            if kind == "gbuffer":
                self.ctx.gbuffer(self.params, stream)
            else:
                self.ctx.restir(self.params, pass_id, stream)
        self.frame_index += 1
