#!/usr/bin/env python
"""bench.py — the hot path's headline benchmark (BASELINE.json: Mrays/s and fps at 1920x1080, 1 spp).

A "step" is one ReSTIR DI frame of config 2 (BASELINE.json configs[1]): Bistro-exterior-class
synthetic scene (~2.87 M triangles, 1 106 instances, 20 050 emissive triangles), 1920x1080, 1 spp,
32 initial candidates, temporal reuse, 1 spatial pass x 4 neighbours, shading
= setupLightInstDistribution + setupGBuffers + performInitialAndTemporalRISBiased +
  performSpatialRISBiased + shading (restir_di/restir_di_main.cpp:2303-2421).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (C ABI)
  python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU
                                                           # (oracle port; oracle/_ref is unbuildable)

--steps K sets the frames of every timed loop.  --dump-outputs DIR writes what the timed path computed in its last step, the
1920x1080 RGBA float32 beauty framebuffer, to DIR/beauty.npy; the scene, the camera and the per-frame seeds are fixed, so two
builds run with the same arguments can be compared output for output.

One JSON line on stdout (rank 0).  `value` = rays traced by the whole job per second with
everything resident in HBM; `e2e` = the same through the C ABI with per-frame host->device uploads
(instance table + parameter blocks from pinned memory) and the device->host read of the beauty
framebuffer inside the timed region; `roofline` = the dominant kernel against the measured HBM
peak; `cpu_baseline` = the oracle on the host cores on a bounded sample of the same frame.  At N = 1 the
line also carries the rest of BASELINE.json's metric, measured in the same process on the same scene:
`nrc` (inference / training ms, TFLOP/s, fraction of the measured sustained bf16 tensor peak),
`north_star_frame` (ReSTIR DI + NRC in one 1080p frame: ms, fps) and `svgf` (config 4: ms per frame,
algorithmic GB/s, fraction of the measured HBM peak).  At every N the line carries `config5`: BASELINE.json's fifth
config - ReSTIR DI + NRC in one 3840x2160 frame, strips over the N ranks, the NRC half sharded with its training
data kept identical to one GPU (gfx_nrc_shard) - with ms, fps, Mrays/s and rank 0's per-kernel times.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WIDTH, HEIGHT = 1920, 1080
METRIC = "Mrays/s at 1920x1080 1spp (ReSTIR DI frame: 32 candidates, temporal + 1x4 spatial reuse)"
WORKLOAD = "restir_di config 2: bistro_class synthetic scene 1920x1080 1spp, 32 candidates, temporal + 1x4 spatial reuse"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_tensor_peak():
    """sustained bf16 TFLOP/s (a kernel timed inside a long step), else the recipe's fallback"""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md).  nvidia-smi needs a few hundred
    ms to produce its first line, longer than a 20-frame region, so the process is started once, early, and keeps logging
    with timestamps; mark() / summary() select the lines that fall inside a region (or, if the region was shorter than the
    sampling period, the lines nearest to it, flagged in `window`)."""

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []   # (host time of arrival, parsed fields)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def start(self):
        self.t0 = time.perf_counter()

    def stop(self):
        """summary of the region [start(), now]"""
        t1 = time.perf_counter()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)  # let the line that covers the end of the region arrive
        inside = [ln for t, ln in self.lines if self.t0 <= t <= t1 + 0.06]
        window = "inside the timed region"
        if not inside:
            near = sorted(self.lines, key=lambda tl: min(abs(tl[0] - self.t0), abs(tl[0] - t1)))[:3]
            inside = [ln for _, ln in near]
            window = "nearest samples (region shorter than the 50 ms sampling period)"
        sm, smmax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in inside:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smmax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smmax) if smmax else None,
                "samples": len(sm), "reasons": sorted(reasons), "window": window}

    def close(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
# (profiles/r02_summary.md): RIS candidate kernel (ris_r02), visibility trace (trace_r02)
NCU_DRAM_TRAFFIC = {"ris_candidates": 273.2e6, "trace_visibility": 87.6e6}
# what actually bounds the dominant kernel (same capture): issue slots at ~15 of 32 lanes, then the L1 data pipe - not HBM
NCU_NOTE = {"ris_candidates": {"capture": "gpurun_out/ris_r02.ncu-rep (profiles/r02_summary.md section 2)",
                               "l1tex_data_pipe_lsu_wavefronts_pct_of_peak": 73.7, "l1_load_wavefronts_per_launch": 104.8e6,
                               "issue_active_pct": 54.4, "warps_active_pct": 46.4, "lanes_per_instruction": 19.7,
                               "reading": "not an HBM kernel: per candidate a 32-byte guide entry and up to 128 bytes of a light record are "
                                          "gathered per lane (94 % L2 hits) and 30 % of the candidates get an IEEE-exact BSDF evaluation; "
                                          "bound by the L1 data pipe's wavefront rate (74 %) and instruction issue (54 %) at 46 % "
                                          "occupancy; DRAM traffic 273 MB against 249 MB algorithmic"}}


def frame_launches(ctx, params, frame_index, num_spatial_passes, timers=None):
    """Issue one frame; with `timers` (dict name -> list of (start, end) events) bracket every launch."""
    from gfxexp_b200 import engine
    import torch

    def timed(name, fn):
        if timers is None:
            fn()
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        timers.setdefault(name, []).append((a, b))

    timed("light_dist", lambda: ctx.build_light_distributions(frame_index % 2))
    names = {0: "initial_ris", 1: "initial_temporal_ris", 2: "initial_temporal_ris_unbiased", 3: "spatial_ris",
             4: "spatial_ris_unbiased", 5: "shading"}
    for kind, pass_id in engine.restir_frame_passes(params, frame_index, num_spatial_passes):
        if kind == "gbuffer":
            timed("gbuffer", lambda: ctx.gbuffer(params))
        else:
            timed(names[pass_id], lambda pid=pass_id: ctx.restir(params, pid))


def traversal_stats(ctx, rays, mode):
    """mean (internal nodes, triangles tested) per ray from the stats variant of the trace kernel."""
    from gfxexp_b200 import abi
    hits = ctx.trace(rays, mode | abi.TRACE_STATS)
    packed = hits["instUserData"]
    return float((packed & 0xFFFF).mean()), float((packed >> 16).mean())


def cpu_reference_step(O, oframe, params, rows, halo, num_spatial_passes, threads):
    """The reference algorithm (oracle port) on a bounded sample: a full-width strip of `rows` rows
    (+halo rows for the per-pixel passes feeding the spatial gather).  Returns seconds per pass kind."""
    from gfxexp_b200 import abi, engine
    H = oframe.H
    y0 = (H - rows) // 2
    t = {}
    for kind, pass_id in engine.restir_frame_passes(params, 0, num_spatial_passes):
        needs_halo = kind == "gbuffer" or pass_id in (abi.RESTIR_INITIAL_RIS, abi.RESTIR_INITIAL_AND_TEMPORAL_BIASED)
        lo = max(0, y0 - (halo if needs_halo else 0))
        hi = min(H, y0 + rows + (halo if needs_halo else 0))
        params.tileOriginY, params.tileRows = lo, hi - lo
        t0 = time.perf_counter()
        if kind == "gbuffer":
            oframe.gbuffer(params, threads)
        else:
            oframe.restir(params, pass_id, threads)
        dt = time.perf_counter() - t0
        name = "gbuffer" if kind == "gbuffer" else str(pass_id)
        # scale this pass to a full frame by the rows it actually processed
        t[name] = t.get(name, 0.0) + dt * (H / (hi - lo))
    params.tileOriginY, params.tileRows = 0, 0
    return t


def tcnn_reference_timing():
    """The reference's own NRC kernels (tiny-cuda-nn built from /root/reference into oracle/_ref/libtcnn_nrc.so, see
    oracle/ref_tcnn) timed on this GPU: ms per inference of a 1080p frame's queries and per 16 384-sample training step."""
    path = os.path.join(ROOT, "oracle", "_ref", "libtcnn_nrc.so")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/libtcnn_nrc.so not built"}
    try:
        lib = C.CDLL(path)
        vp, u32 = C.c_void_p, C.c_uint32
        lib.tcnn_nrc_create.argtypes = [u32, u32, C.c_float, C.POINTER(vp)]
        lib.tcnn_nrc_time_infer.argtypes = [vp, vp, u32, u32, u32, C.POINTER(C.c_float)]
        lib.tcnn_nrc_time_train.argtypes = [vp, vp, vp, u32, u32, u32, C.POINTER(C.c_float)]
        lib.tcnn_nrc_destroy.argtypes = [vp]
        h = vp()
        if lib.tcnn_nrc_create(1, 2, 1e-2, C.byref(h)) != 0:
            return {"unavailable": "tcnn_nrc_create failed (no GPU?)"}
        rng = np.random.default_rng(0)
        n = ((WIDTH * HEIGHT + WIDTH * HEIGHT // 48 + 127) // 128) * 128
        q = rng.uniform(0, 1, size=(n, 14)).astype(np.float32)
        ms_inf, ms_tr = C.c_float(), C.c_float()
        assert lib.tcnn_nrc_time_infer(h, q.ctypes.data, n, 3, 10, C.byref(ms_inf)) == 0
        nt = 16384
        tq, tt = q[:nt].copy(), rng.uniform(0, 1, size=(nt, 3)).astype(np.float32)
        assert lib.tcnn_nrc_time_train(h, tq.ctypes.data, tt.ctypes.data, nt, 3, 20, C.byref(ms_tr)) == 0
        lib.tcnn_nrc_destroy(h)
        return {"kind": "reference (tiny-cuda-nn kernel_grid + kernel_one_blob_soa + kernel_mlp_fused, unmodified, sm_100a build)",
                "infer_queries": n, "infer_ms": ms_inf.value, "infer_tflops": 18432.0 * n / ms_inf.value / 1e9,
                "train_samples": nt, "train_step_ms": ms_tr.value, "train_tflops": 55296.0 * nt / ms_tr.value / 1e9}
    except (OSError, AssertionError) as e:
        return {"unavailable": f"{type(e).__name__}: {e}"}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the renderer of oracle/_ref is unbuildable) on the host
    cores.  A step is the bounded sample itself - a full-width strip of --cpu-rows rows through every pass of the frame - and
    `value` is the rays the oracle really traced in it per second; nothing is extrapolated into the timed numbers."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gfxexp_b200 import abi, scenes
    from tests import oracle_lib as O
    threads = os.cpu_count() or 1
    scene = scenes.bistro_class_scene()
    oscene = O.OracleScene(scene)
    oframe = O.OracleFrame(oscene, WIDTH, HEIGHT)
    params = abi.default_frame_params(scene, WIDTH, HEIGHT)
    rows, halo = args.cpu_rows, 24
    times, rays, full_frame_s = [], [], []
    for it in range(args.warmup + args.steps):
        O.rays_traced(reset=True)
        t0 = time.perf_counter()
        t = cpu_reference_step(O, oframe, params, rows, halo, 1, threads)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
            rays.append(O.rays_traced(reset=True))
            full_frame_s.append(sum(t.values()))
    step_s = float(np.mean(times))
    value = float(np.mean(rays)) / step_s / 1e6
    sample = (f"{rows}-row full-width strip (+{halo}-row halo for the per-pixel passes feeding the spatial gather) of the 1920x1080 "
              f"frame through all passes = one step; value = rays the oracle traced in the strip / its wall time")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "triangles": scene.num_triangles, "instances": len(scene.instances),
                   "emissive_triangles": scene.num_emissive_triangles,
                   "rays_per_step": float(np.mean(rays)), "rows_per_step": rows,
                   "full_frame_ms_extrapolated_by_rows": float(np.mean(full_frame_s)) * 1e3,
                   "fps_extrapolated_by_rows": 1.0 / float(np.mean(full_frame_s)),
                   "parallelism": f"{threads} host threads (OpenMP over pixels)",
                   "bvh": "bvh::buildGeometryBVH<8> restatement (SBVH, budget .3), build %.1f s single-thread" % oscene.build_seconds},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "nrc_reference": tcnn_reference_timing(),
    }
    emit_line(line)


def measure_nrc_and_svgf(ctx, scene, args):
    """NRC MLP TFLOP/s (the second half of BASELINE.json's metric), the north-star frame (ReSTIR DI + NRC at 1080p) and SVGF
    (config 4), on the config-2 scene, CUDA events on the launching stream, inputs resident.  NRC numbers come from the
    frames themselves: the inference batch is the frame's pad128(W*H + #tiles) queries, training is the 4 x 16 384 shuffled
    records, after a warm-up that lets the tile-size controller and the cache settle."""
    import torch
    from gfxexp_b200 import abi, engine
    px = WIDTH * HEIGHT
    hbm_peak, hbm_src = measured_peaks()
    tpeak, tsrc = measured_tensor_peak()
    out = {}
    # ---- north-star frame: one G-buffer, ReSTIR DI passes, NRC path tracing + inference + 4 training steps
    pc = abi.default_frame_params(scene, WIDTH, HEIGHT)
    net = engine.NeuralRadianceCache(ctx, 2, 1e-2)
    rng = np.random.default_rng(0)

    # the same driver as the multi-GPU runs, with one rank: the four training steps of frame f run on a second stream under
    # the G-buffer / ReSTIR passes of frame f + 1 (gfxexp_b200/multigpu.py enable_nrc)
    from gfxexp_b200 import multigpu
    driver = multigpu.StripDriver(ctx, pc, WIDTH, HEIGHT, 0, 1)
    driver.enable_nrc(net)

    def combined_frame(f):
        pc.numAccumFrames = f
        driver.render_restir_nrc_frame(f, [int(rng.integers(0, 2 ** 32)) for _ in range(2)])

    n_warm, n_frames = 16, args.steps
    for f in range(n_warm):
        combined_frame(f)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for f in range(n_warm, n_warm + n_frames):
        combined_frame(f)
    driver.wait_training()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n_frames
    out["north_star_frame"] = {"what": "ReSTIR DI (32 candidates, temporal + 1x4 spatial) + NRC (path tracing with cache "
                                       "termination, inference, 4 training steps) in one frame, one G-buffer, 1920x1080, 1 GPU; "
                                       "the training steps of frame f overlap the ReSTIR passes of frame f + 1",
                               "ms": ms, "fps": 1e3 / ms, "target_fps": 60.0, "frames_timed": n_frames}
    # per-kernel times of the same frames (events inside the library)
    driver.wait_training()
    driver.train_stream = None  # kernel times in stream order: no training kernel waits behind another stream's blocks
    ctx.timing_enable(True)
    ctx.timing_read()
    reps = 6
    for f in range(n_warm + n_frames, n_warm + n_frames + reps):
        combined_frame(f)
    timing = ctx.timing_read()
    ctx.timing_enable(False)
    per_frame = {k: v[0] / reps for k, v in timing.items()}
    st = ctx.download_linear(abi.BUF_NRC_STATE)[:, 0]
    nq = int(st[abi.NRC_STATE_NUM_INFERENCE_QUERIES])
    infer_ms = sum(per_frame.get(k, 0.0) for k in ("nrc_pack_positions", "nrc_grid_encode", "nrc_infer"))
    train_ms = sum(per_frame.get(k, 0.0) for k in ("nrc_train_prep_weights", "nrc_train_fwd_bwd", "nrc_adam_ema"))
    mlp_ms = per_frame.get("nrc_infer", 0.0)
    out["nrc"] = {"infer_queries": nq, "infer_ms": infer_ms, "infer_tflops": 18432.0 * nq / infer_ms / 1e9,
                  "tensor_frac": 18432.0 * nq / infer_ms / 1e9 / tpeak,
                  "infer_kernels_ms": {k: per_frame.get(k, 0.0) for k in ("nrc_pack_positions", "nrc_grid_encode", "nrc_infer")},
                  "mlp_kernel_tflops": 18432.0 * nq / mlp_ms / 1e9 if mlp_ms else None,
                  "mlp_kernel_tensor_frac": 18432.0 * nq / mlp_ms / 1e9 / tpeak if mlp_ms else None,
                  "train_samples": 65536, "train_ms": train_ms, "train_tflops": 55296.0 * 65536 / train_ms / 1e9,
                  "train_tensor_frac": 55296.0 * 65536 / train_ms / 1e9 / tpeak,
                  "flop_per_query": 18432, "flop_per_training_sample": 55296, "dtype": "f16 operands, f32 accumulate (tcgen05)",
                  "peak": tpeak, "peak_source": tsrc,
                  "frame_kernels_ms": {k: round(v, 4) for k, v in sorted(per_frame.items(), key=lambda kv: -kv[1])}}
    net.close()
    # ---- SVGF (config 4) on the ReSTIR DI output
    ren = engine.ReSTIRRenderer(ctx, scene, WIDTH, HEIGHT)
    svgf_ms = []
    for f in range(3 + args.steps):  # the first three frames warm up
        ren.render_frame()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for pass_id, stage in engine.svgf_frame_passes(ren.params, f):
            ctx.svgf(ren.params, pass_id, stage)
        b.record()
        svgf_ms.append((a, b))
    torch.cuda.synchronize()
    sms = float(np.mean([a.elapsed_time(b) for a, b in svgf_ms[3:]]))
    out["svgf"] = {"what": "temporal accumulation + variance + 5 a-trous stages + background + modulate/TAA on the ReSTIR DI "
                           "frame, 1920x1080", "ms": sms, "algorithmic_bytes_per_px": 456,
                   "GBps": 456.0 * px / sms / 1e6, "frac": 456.0 * px / sms / 1e6 / hbm_peak, "peak": hbm_peak, "peak_source": hbm_src}
    return out


def measure_config5(scene, args, rank, world, local_rank):
    """BASELINE.json config 5: ReSTIR DI + NRC combined, 3840x2160, screen strips across the ranks, one all-gather of the
    composited framebuffer.  All ranks call this.  The DI half exchanges seam rows as at 1080p; the NRC half traces and infers
    its rows, numbers the training vertices over the whole frame (one word per rank and path-tracing round all-gathered),
    merges the records with one integer all-reduce and trains replicated (gfx_nrc_shard, include/gfxb200.h).  A context of
    its own: the 1080p frame of the headline stays untouched."""
    import torch
    import torch.distributed as dist
    from gfxexp_b200 import abi, engine, multigpu
    W5, H5 = 3840, 2160
    if H5 % world:
        return None
    ctx = engine.Context(local_rank)
    ctx.upload_scene(scene)
    ctx.build_bvh()
    ctx.create_frame(W5, H5)
    p = abi.default_frame_params(scene, W5, H5)
    net = engine.NeuralRadianceCache(ctx, 2, 1e-2)
    boundaries = None
    if os.environ.get("GFX_MULTIGPU_BALANCED_STRIPS") == "1":
        boundaries = multigpu.StripDriver.cost_balanced_boundaries(ctx, p, W5, H5, world)
    driver = multigpu.StripDriver(ctx, p, W5, H5, rank, world, boundaries=boundaries)
    driver.enable_nrc(net)
    rng = np.random.default_rng(5)
    frame = 0

    def one_frame():
        nonlocal frame
        p.numAccumFrames = frame
        driver.render_restir_nrc_frame(frame, [int(rng.integers(0, 2 ** 32)) for _ in range(2)])
        frame += 1

    for _ in range(12):  # the tile-size controller and the cache settle
        one_frame()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    driver.check_peers()
    ctx.read_stats(reset=True)
    n_frames = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_frames):
        one_frame()
    driver.wait_training()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    driver.check_peers()
    ms = e0.elapsed_time(e1)
    rays = float(ctx.read_stats(reset=True)[0])
    lo_h, hi_h = max(0, driver.y0 - driver.halo), min(H5, driver.y1 + driver.halo)
    rays -= ((driver.y0 - lo_h) + (hi_h - driver.y1)) * W5 * n_frames  # recomputed G-buffer halo rows are not throughput
    st = ctx.download_linear(abi.BUF_NRC_STATE)[:, 0]
    # where the strip's frame goes: per-kernel CUDA events inside the library (this rank's launches; collectives and peer
    # waits are the remainder against `ms`)
    driver.wait_training()
    driver.train_stream = None  # kernel times in stream order
    ctx.timing_enable(True)
    ctx.timing_read()
    reps = 6
    for _ in range(reps):
        one_frame()
    torch.cuda.synchronize()
    timing = ctx.timing_read()
    ctx.timing_enable(False)
    per_frame = {k: round(v[0] / reps, 4) for k, v in sorted(timing.items(), key=lambda kv: -kv[1][0])}
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        r = torch.tensor([rays], device="cuda", dtype=torch.float64)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        rays = float(r.item())
    out = {"what": "ReSTIR DI (32 candidates, temporal + 1x4 spatial) + NRC (path tracing with cache termination, inference, "
                   "4 training steps) in one 3840x2160 frame, %s on %d GPU(s), framebuffer all-gathered" % (
                       "cost-balanced strips at rows %s" % driver.boundaries if boundaries is not None else "strips of %d rows" % (H5 // world), world),
           "n_gpus": world, "ms": ms / n_frames, "fps": 1e3 * n_frames / ms, "Mrays_per_s": rays / (ms * 1e-3) / 1e6,
           "rays_per_pixel": rays / n_frames / (W5 * H5), "frames_timed": n_frames,
           "training_records_last_frame": int(st[abi.NRC_STATE_NUM_TRAINING_DATA + (frame - 1) % 2]),
           "tile_size": [int(st[abi.NRC_STATE_TILE_SIZE + 2 * ((frame - 1) % 2)]), int(st[abi.NRC_STATE_TILE_SIZE + 2 * ((frame - 1) % 2) + 1])],
           "nrc": "inference sharded by strip, training replicated on all ranks (weights bit-identical, tests/test_gpu_multigpu.py)",
           "rank0_kernels_ms": per_frame, "rank0_kernels_sum_ms": round(sum(per_frame.values()), 4)}
    net.close()
    if driver.comm is not None:
        driver.comm.close()
    ctx.close()
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from gfxexp_b200 import abi, engine, scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    sampler = ClockSampler(local_rank)  # started now: nvidia-smi takes a while to deliver its first line
    scene = scenes.bistro_class_scene()
    ctx = engine.Context(local_rank)
    t0 = time.perf_counter()
    ctx.upload_scene(scene)
    ctx.synchronize()
    upload_s = time.perf_counter() - t0
    # BVH build: once untimed (allocations), then timed
    ctx.build_bvh()
    ctx.synchronize()
    t0 = time.perf_counter()
    ctx.build_bvh()
    ctx.synchronize()
    bvh_build_ms = (time.perf_counter() - t0) * 1e3
    info = ctx.bvh_info()
    ctx.create_frame(WIDTH, HEIGHT)
    params = abi.default_frame_params(scene, WIDTH, HEIGHT)
    nsp = 1

    if world > 1:
        from gfxexp_b200 import multigpu
        # seam rows travel as one-sided pushes over NVLink peer memory; GFX_MULTIGPU_NCCL=1 selects NCCL send/recv (A/B)
        # GFX_MULTIGPU_BALANCED_STRIPS=1 (A/B): strip boundaries that equalise the geometry-hit pixels per strip instead of the
        # rows.  Measured at N = 8 and rejected as the default: 1.298 ms against 1.147 ms with equal rows (config 5: 5.95 against
        # 5.86 ms) - hit counts do not predict a strip's cost in this view (profiles/r02_summary.md section 7)
        boundaries = None
        if os.environ.get("GFX_MULTIGPU_BALANCED_STRIPS") == "1":
            boundaries = multigpu.StripDriver.cost_balanced_boundaries(ctx, params, WIDTH, HEIGHT, world)
        driver = multigpu.StripDriver(ctx, params, WIDTH, HEIGHT, rank, world, peer=os.environ.get("GFX_MULTIGPU_NCCL") != "1",
                                      boundaries=boundaries)
        if boundaries is not None:
            driver.use_raw_communicator()  # gfx_framebuffer_allgatherv: one NCCL group launch for the unequal strips
    else:
        driver = None

    def one_frame(fi, timers=None):
        if driver is not None:
            driver.render_frame(fi, nsp)
        else:
            frame_launches(ctx, params, fi, nsp, timers)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if driver is not None:
            driver.check_peers()  # a seam wait that timed out would mean stale rows inside the region just timed

    frame = 0
    for _ in range(max(args.warmup, 3)):
        one_frame(frame)
        frame += 1
    barrier()
    ctx.read_stats(reset=True)
    launches0 = ctx.kernel_launches

    # ---- timed region 1: everything resident in HBM -------------------------------------------
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        one_frame(frame)
        frame += 1
    ev1.record()
    barrier()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    rays = ctx.read_stats(reset=True)[0]
    # --dump-outputs: what the timed path computed in its last step, the beauty framebuffer a caller of the frame receives
    # (at N > 1 the composited frame every rank holds after the all-gather)
    last_beauty = None
    if args.dump_outputs and rank == 0:
        last_beauty = (driver.composited.cpu().numpy().reshape(HEIGHT, WIDTH, 4) if driver is not None
                       else ctx.download(abi.BUF_BEAUTY_ACCUM))
    # the G-buffer halo rows a rank recomputes for the spatial pass are redundant work, not throughput: their primary rays
    # are not counted (so `value` at N > 1 is the same frame's rays as at N = 1, over a shorter time)
    halo_rays_per_frame = 0
    if driver is not None:
        lo_h, hi_h = max(0, driver.y0 - driver.halo), min(HEIGHT, driver.y1 + driver.halo)
        halo_rays_per_frame = ((driver.y0 - lo_h) + (hi_h - driver.y1)) * WIDTH
        rays -= halo_rays_per_frame * args.steps
    launches = ctx.kernel_launches - launches0
    if world > 1:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        r = torch.tensor([rays], device="cuda", dtype=torch.float64)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        rays = float(r.item())
    ms_per_step = ms_total / args.steps
    value = rays / (ms_total * 1e-3) / 1e6
    rays_per_px = rays / args.steps / (WIDTH * HEIGHT)

    # ---- timed region 2: end to end through the C ABI with host buffers ---------------------------
    # The host receives every frame (the reference displays every frame; with double-buffered StreamChain<2> launches,
    # common_host.h:144-195, frame N+1 is recorded while N executes).  Same here: the beauty rows are snapshotted on the
    # render stream (device-to-device) and drained to pinned host memory on a copy stream while the next frame renders;
    # the timed region ends with a full synchronisation, so all K results have arrived.
    sa = ctx._scene_arrays
    inst_bytes = C.sizeof(abi.GfxInstanceDesc) * len(scene.instances)
    param_bytes = C.sizeof(abi.GfxFrameParams) * (3 + nsp)
    rows_lo, rows_hi = (driver.y0, driver.y1) if driver is not None else (0, HEIGHT)
    nrows = rows_hi - rows_lo
    pinned = [torch.empty((nrows, WIDTH, 4), dtype=torch.float32, pin_memory=True) for _ in range(2)]
    staging = [torch.empty((nrows, WIDTH, 4), dtype=torch.float32, device="cuda") for _ in range(2)]
    render_stream = torch.cuda.default_stream()
    copy_stream = torch.cuda.Stream()
    snap_ready = [torch.cuda.Event() for _ in range(2)]
    copy_done = [torch.cuda.Event() for _ in range(2)]
    for e in copy_done:
        e.record(copy_stream)
    cudart = C.CDLL("libcudart.so.12") if os.path.exists("/usr/local/cuda/lib64/libcudart.so.12") else C.CDLL("libcudart.so")
    cudart.cudaMemcpyAsync.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    strip_bytes = nrows * WIDTH * 16

    def one_frame_e2e(fi):
        # host -> device: the instance table (InstanceController::update re-uploads it every frame,
        # common/common_host.h:798-856) + the per-launch parameter blocks; device -> host: the beauty
        # framebuffer rows this rank owns.
        ctx._check(ctx.lib.gfx_scene_update_instances(ctx.h, None, sa.instances, len(scene.instances)),
                   "gfx_scene_update_instances")
        one_frame(fi)
        slot = fi % 2
        p, nbytes = ctx.device_ptr(abi.BUF_BEAUTY_ACCUM, 0)
        render_stream.wait_event(copy_done[slot])           # the previous drain of this slot has finished
        rc = cudart.cudaMemcpyAsync(C.c_void_p(staging[slot].data_ptr()), C.c_void_p(p + rows_lo * WIDTH * 16),
                                    C.c_size_t(strip_bytes), 3, C.c_void_p(render_stream.cuda_stream))
        assert rc == 0
        snap_ready[slot].record(render_stream)
        copy_stream.wait_event(snap_ready[slot])
        rc = cudart.cudaMemcpyAsync(C.c_void_p(pinned[slot].data_ptr()), C.c_void_p(staging[slot].data_ptr()),
                                    C.c_size_t(strip_bytes), 2, C.c_void_p(copy_stream.cuda_stream))
        assert rc == 0
        copy_done[slot].record(copy_stream)

    one_frame_e2e(frame)
    frame += 1
    barrier()
    ctx.read_stats(reset=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        one_frame_e2e(frame)
        frame += 1
    for e in copy_done:                      # the timed region ends when the last frame has reached the host
        render_stream.wait_event(e)
    ev1.record()
    barrier()
    e2e_ms = ev0.elapsed_time(ev1)
    sampler.close()
    e2e_rays = ctx.read_stats(reset=True)[0] - halo_rays_per_frame * args.steps
    if world > 1:
        t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        r = torch.tensor([e2e_rays], device="cuda", dtype=torch.float64)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        e2e_rays = float(r.item())
    e2e_value = e2e_rays / (e2e_ms * 1e-3) / 1e6
    copy_stream.synchronize()
    assert float(pinned[(frame - 1) % 2][..., 3].min()) == 1.0  # the last frame really arrived (alpha plane)
    d2h_bytes = (rows_hi - rows_lo) * WIDTH * 16

    config5 = None if args.headline_only else measure_config5(scene, args, rank, world, local_rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel breakdown + roofline of the dominant kernel (rank 0, single-GPU launches) ------
    roofline = None
    breakdown = {}
    if driver is None:
        # every kernel launch bracketed by CUDA events on its stream inside the library (gfx_timing_enable)
        ctx.timing_enable(True)
        ctx.timing_read()
        for _ in range(args.steps):
            frame_launches(ctx, params, frame, nsp, None)
            frame += 1
        timing = ctx.timing_read()
        ctx.timing_enable(False)
        breakdown = {k: ms / n for k, (ms, n) in timing.items()}                 # ms per launch
        launches_per_frame = {k: n / args.steps for k, (ms, n) in timing.items()}
        dominant = max(breakdown, key=breakdown.get)
        # traversal statistics of this BVH for the rays the dominant kernel traces
        prim = engine.primary_rays(params, WIDTH, HEIGHT)[:: 7]
        n_int_p, n_tri_p = traversal_stats(ctx, prim, abi.TRACE_CLOSEST)
        gb2 = ctx.download(abi.BUF_GBUFFER2, params.bufferIndex).view(np.float32)
        gb0 = ctx.download(abi.BUF_GBUFFER0, params.bufferIndex)
        res = ctx.download(abi.BUF_RESERVOIR, params.currentReservoirIndex).view(np.float32)
        hit = gb0[..., 0] != 0xFFFFFFFF
        org = gb2[..., :3][hit][::7]
        tgt = res[1][..., :3][hit][::7]
        d = tgt - org
        dist_ = np.linalg.norm(d, axis=1)
        ok = dist_ > 1e-3
        sh = np.zeros(int(ok.sum()), dtype=abi.RAY_DTYPE)
        sh["org"] = org[ok] + 1e-3 * (d[ok] / dist_[ok, None])
        sh["dir"] = d[ok] / dist_[ok, None]
        sh["tmax"] = dist_[ok] * 0.9999
        n_int_s, n_tri_s = traversal_stats(ctx, sh, abi.TRACE_ANY)
        px = WIDTH * HEIGHT
        trav_primary = 80 * n_int_p + 52 * n_tri_p + 64
        trav_shadow = 80 * n_int_s + 52 * n_tri_s + 64
        # algorithmic bytes per pixel, SURVEY.md §8(d): struct sizes of the reference + traversal counters
        # per launch; the wavefront trace kernel serves ~0.94 (initial) / ~0.94 (shading) rays per pixel
        rays_vis = (rays_per_px - 1.0) / 2.0
        # HBM-side: compulsory bytes per pixel with perfect on-chip reuse (SURVEY.md 8d); a ray is 32 B in + 32 B out.
        # L2-side: what a launch additionally pulls through L2 - BVH nodes / triangles per ray (the BVH, 188 MB, is re-read by
        # every ray that visits a node), light records per RIS candidate (32 B guide entry + up to 128 B record).
        alg = {
            "gbuffer": 56 + 32 + 3 * 48 + 16 + 64,
            "ris_candidates": 120,
            "ris_resolve_temporal": 112 + 9,
            "ris_megakernel": 120 + 112 + 64,
            "trace_visibility": rays_vis * 64,
            "spatial_ris": 592,
            "shading_rays": 104 + 36,
            "shading": 120,
            "shading_megakernel": 120 + 64,
        }
        l2_side = {
            "gbuffer": trav_primary - 64,
            "ris_candidates": 32 * (32 + 0.5 * 64 + 0.35 * 96),
            "ris_megakernel": trav_shadow - 64,
            "trace_visibility": rays_vis * (trav_shadow - 64),
            "shading_megakernel": trav_shadow - 64,
        }
        hbm_peak, peak_src = measured_peaks()
        bytes_per_launch = alg.get(dominant, 0) * px
        achieved = bytes_per_launch / (breakdown[dominant] * 1e-3) / 1e9
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": NCU_DRAM_TRAFFIC.get(dominant), "traffic_source": "ncu --set full, profiles/r02_summary.md", "ncu": NCU_NOTE.get(dominant), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": bytes_per_launch, "ms_per_launch": breakdown[dominant],
                    "traversal": {"primary_nodes_per_ray": n_int_p, "primary_tris_per_ray": n_tri_p,
                                  "shadow_nodes_per_ray": n_int_s, "shadow_tris_per_ray": n_tri_s},
                    "per_kernel": {k: {"ms_per_launch": breakdown[k], "launches_per_frame": launches_per_frame[k],
                                       "hbm_GBps": alg.get(k, 0) * px / (breakdown[k] * 1e-3) / 1e9,
                                       "hbm_frac": alg.get(k, 0) * px / (breakdown[k] * 1e-3) / 1e9 / hbm_peak,
                                       "l2_side_GBps": l2_side.get(k, 0) * px / (breakdown[k] * 1e-3) / 1e9}
                                   for k in breakdown},
                    "frame": {"algorithmic_bytes": 1032 * px + 64 * rays_per_px * px, "hbm_GBps": (1032 + 64 * rays_per_px) * px / (ms_per_step * 1e-3) / 1e9,
                              "hbm_frac": (1032 + 64 * rays_per_px) * px / (ms_per_step * 1e-3) / 1e9 / hbm_peak}}

    # ---- the rest of BASELINE.json's metric, same process / scene / clocks (rank 0, N = 1) ----------------------------
    extras = {}
    if driver is None and not args.headline_only:
        extras = measure_nrc_and_svgf(ctx, scene, args)

    # ---- CPU baseline: the oracle on the host cores, bounded sample (rank 0, N=1 only) -------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        from tests import oracle_lib as O
        threads = os.cpu_count() or 1
        oscene = O.OracleScene(scene)
        oframe = O.OracleFrame(oscene, WIDTH, HEIGHT)
        cparams = abi.default_frame_params(scene, WIDTH, HEIGHT)
        t = cpu_reference_step(O, oframe, cparams, args.cpu_rows, 24, nsp, threads)
        frame_s = sum(t.values())
        cpu_baseline = {"value": rays_per_px * WIDTH * HEIGHT / frame_s / 1e6, "unit": "Mrays/s", "cores": threads,
                        "kind": "port", "fps": 1.0 / frame_s, "bvh_build_s_single_thread": oscene.build_seconds,
                        "sample": f"{args.cpu_rows}-row full-width strip (+24-row halo for the per-pixel passes) of the "
                                  f"1920x1080 frame per pass, scaled to the full frame by rows; rays counted as the "
                                  f"GPU's {rays_per_px:.3f} rays/px"}

    line = {
        "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "fps": 1e3 / ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "triangles": info.numTriangles, "bvh_nodes": info.numNodes, "instances": len(scene.instances),
                   "emissive_triangles": scene.num_emissive_triangles, "rays_per_pixel": rays_per_px,
                   "l2": "inputs larger than L2 (BVH %.0f MB + %.0f MB of per-pixel state per frame)" % (
                       (info.numTriangles * 52 + info.numNodes * 80) / 1e6, WIDTH * HEIGHT * 400 / 1e6),
                   "parallelism": ("screen strips x%d %s (24-row G-buffer halo recomputed per seam, its rays not counted), seam rows by %s, "
                                   "beauty strips all-gathered with NCCL" % (
                       world, ("of equal work, rows %s" % driver.boundaries) if not driver.rows else "of equal height",
                       "one-sided NVLink peer-memory pushes" if driver.backend.peer_ready else "NCCL send/recv"))
                   if world > 1 else "1 GPU",
                   "bvh_build_ms": bvh_build_ms, "scene_upload_s": upload_s},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_ms / args.steps, "fps": 1e3 * args.steps / e2e_ms,
                "h2d_bytes_per_step": inst_bytes + param_bytes, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": launches,
    }
    if roofline is not None:
        line["roofline"] = roofline
    line.update(extras)
    if config5 is not None:
        line["config5"] = config5
    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    if last_beauty is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "beauty.npy"), np.ascontiguousarray(last_beauty, dtype=np.float32))
    emit_line(line)
    if world > 1:
        dist.destroy_process_group()


_RESULT_FD = None


def claim_stdout():
    """stdout carries ONE JSON line.  Libraries print there too (NCCL announces its version through C stdio when a communicator
    is created), so fd 1 is pointed at stderr for the whole run and the result line goes to the original stdout."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="gfxb200", choices=["gfxb200", "reference"])
    ap.add_argument("--cpu-rows", type=int, default=48, help="rows of the CPU-baseline strip sample")
    ap.add_argument("--rays-per-px", type=float, default=2.883, help="--impl reference: rays per pixel (GPU-counted)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the NRC / north-star / SVGF measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the beauty framebuffer of the last timed frame to DIR/beauty.npy (float32 [H, W, 4])")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "gfxb200":
        ap.error("--dump-outputs writes the CUDA path's frame: --impl gfxb200 only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
