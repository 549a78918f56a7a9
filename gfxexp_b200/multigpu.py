"""Screen-strip sharding of a ReSTIR DI frame across the GPUs of one box (SURVEY.md §8e).

Rank r owns the contiguous rows [r*H/N, (r+1)*H/N).  Scene, BVH and light tables are replicated; every
rank allocates full-frame buffers and addresses rows globally, so exchanged rows land at their own
offsets.  Per frame:

  1. G-buffer for the owned rows plus `halo` rows on each side (stateless, recomputed instead of sent)
  2. initial(+temporal) RIS on the owned rows                                    - no communication
  3. exchange of the reservoir + reservoir-info halo rows with the neighbour ranks (the spatial pass
     gathers within `spatialNeighborRadius` pixels, restir_di_main.cpp:2069; default 20).  On GPUs this is a
     one-sided push over NVLink peer memory: each rank's kernels store its seam rows into the neighbour's
     buffers and raise a sequence flag there (csrc/peer.cu, inside gfx_restir_strip_frame); without peer links
     (NCCL, or the gloo/CPU arm) `exchange_halo` uses send/recv.
  4. spatial RIS pass(es) on the owned rows (halo exchange again after every pass that feeds another)
  5. shading on the owned rows, exchange of the final reservoir halo (next frame's temporal reuse)
  6. all-gather of the composited beauty strips: the one mandatory collective

What a rank can read across a seam is `halo` rows, so the driver refuses configurations that would read further:
`spatialNeighborRadius` must not exceed `halo`, and the temporal pass - which follows the motion vector to the previous frame's
G-buffer and reservoirs (optix_restir_di_kernels.cu:150-153) - is only valid while no pixel moves by more than `halo` rows per
frame: a moving camera (or animated instances) needs `max_motion_rows` stated by the caller (<= halo), and a frame whose camera
differs from the previous one is rejected without it.  A stalled neighbour (k_peerWait's time-out, csrc/peer.cu) is detected by
`check_peers()`, which the driver calls every `check_every` frames and callers call before trusting a timed region.

The driver is backend-agnostic: `GpuBackend` drives libgfxb200 with NCCL on the device pointers,
`tests/test_multigpu_cpu.py` drives the CPU oracle through the same code with gloo, which is how the
host-side sharding logic is verified bit-for-bit against a single-process render.
"""
from __future__ import annotations

from typing import List, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import abi, engine


class _DevicePtr:
    """Zero-copy torch view of a raw device pointer through __cuda_array_interface__."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class NcclComm:
    """A raw ncclComm_t over the ranks of the default torch.distributed group, created with ctypes on the NCCL the process has
    loaded - what a C++ host has from nccl.h.  The library takes it for the collectives it issues itself
    (gfx_framebuffer_allgather, the sharded NRC frame of gfx_nrc_shard).  The unique id travels through torch.distributed."""

    def __init__(self, rank: int, world: int):
        import ctypes as C

        class UniqueId(C.Structure):  # ncclUniqueId, passed by value
            _fields_ = [("internal", C.c_byte * 128)]
        self.lib = C.CDLL("libnccl.so.2")  # the soname resolves to the copy torch has loaded
        uid = UniqueId()
        if rank == 0 and self.lib.ncclGetUniqueId(C.byref(uid)) != 0:
            raise RuntimeError("ncclGetUniqueId failed")
        ids = [bytes(uid)]
        dist.broadcast_object_list(ids, src=0)
        C.memmove(C.byref(uid), ids[0], 128)
        self.handle = C.c_void_p()
        self.lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, UniqueId, C.c_int]
        # NCCL announces its version on stdout at the first ncclCommInitRank of a process (NCCL_DEBUG=VERSION/WARN); hosts
        # that own stdout (bench.py prints ONE JSON line) get it on stderr instead
        import os
        import sys
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            rc = self.lib.ncclCommInitRank(C.byref(self.handle), world, uid, rank)
            C.CDLL(None).fflush(None)  # NCCL writes through C stdio: empty its buffer while fd 1 still points at stderr
        finally:
            os.dup2(saved, 1)
            os.close(saved)
        if rc != 0:
            raise RuntimeError("ncclCommInitRank failed")
        self.lib.ncclCommDestroy.argtypes = [C.c_void_p]

    def close(self):
        if self.handle:
            self.lib.ncclCommDestroy(self.handle)
            self.handle = None


class GpuBackend:
    """Launches go through gfx_launch_batch: the driver's calls are recorded into one array of GfxBatchOp records per frame and
    handed to the library in ONE call (flush) - at 8 GPUs a strip frame is ~35 launches in ~1.3 ms of GPU time, and a Python /
    ctypes round trip per launch made the host the bottleneck."""
    MAX_OPS = 128

    def __init__(self, ctx: engine.Context):
        self.ctx = ctx
        self._views = {}
        self._ops = (abi.GfxBatchOp * self.MAX_OPS)()
        self._n = 0

    def _record(self, op, a=0, b=0, c=0, d=0, e=0, params=None):
        if self._n == self.MAX_OPS:
            self.flush()
        o = self._ops[self._n]
        o.op, o.a, o.b, o.c, o.d, o.e = op, a, b, c, d, e
        if params is not None:
            import ctypes as C
            C.memmove(C.addressof(o.params), C.addressof(params), C.sizeof(abi.GfxFrameParams))
        self._n += 1

    def flush(self):
        if self._n:
            n, self._n = self._n, 0
            self.ctx._check(self.ctx.lib.gfx_launch_batch(self.ctx.h, None, self._ops, n), "gfx_launch_batch")

    def light_dist(self, frame_index: int):
        self._record(abi.OP_LIGHT_DIST, frame_index % 2)

    def gbuffer(self, params):
        self._record(abi.OP_GBUFFER, params=params)

    def restir(self, params, pass_id: int):
        self._record(abi.OP_RESTIR, pass_id, params=params)

    def tensor(self, buffer_id: int, index: int = 0) -> torch.Tensor:
        key = (buffer_id, index)
        if key not in self._views:
            ptr, nbytes = self.ctx.device_ptr(buffer_id, index)
            self._views[key] = torch.as_tensor(_DevicePtr(ptr, nbytes), device=f"cuda:{self.ctx.device}")
        return self._views[key]

    def new_tensor(self, numel: int) -> torch.Tensor:
        return torch.empty(numel, dtype=torch.float32, device=f"cuda:{self.ctx.device}")

    # -- one-sided seam exchange over peer memory -------------------------------------------------------
    PEER_BUFFERS = [(abi.BUF_RESERVOIR, 0), (abi.BUF_RESERVOIR, 1), (abi.BUF_RESERVOIR_INFO, 0), (abi.BUF_RESERVOIR_INFO, 1)]

    def enable_peer(self, rank: int, world: int):
        """Exchange IPC handles with the neighbour ranks (all ranks must call this; one all_gather_object)."""
        mine = {"flags": self.ctx.peer_export(abi.BUF_PEER_FLAGS, 0)}
        for b, i in self.PEER_BUFFERS:
            mine[(b, i)] = self.ctx.peer_export(b, i)
        everyone = [None] * world
        dist.all_gather_object(everyone, mine)
        for link, other in ((0, rank - 1), (1, rank + 1)):
            if 0 <= other < world:
                self.ctx.peer_open(link, abi.BUF_PEER_FLAGS, 0, everyone[other]["flags"])
                for b, i in self.PEER_BUFFERS:
                    self.ctx.peer_open(link, b, i, everyone[other][(b, i)])
        self.peer_ready = True
        self.peer_seq = 0

    peer_ready = False
    peer_seq = 0


def balanced_boundaries(row_cost, world: int, min_rows: int, align: int = 8) -> List[int]:
    """Rows [b[r], b[r + 1]) for rank r such that the strips carry about equal cost under the given per-row cost estimate.
    Boundaries are multiples of `align` (the 8x8 light-subset tiles of the rearchitected renderer) and every strip
    keeps at least `min_rows` rows (the halo: a seam exchange only reaches the adjacent rank)."""
    cost = np.asarray(row_cost, dtype=np.float64)
    H = cost.shape[0]
    cum = np.concatenate([[0.0], np.cumsum(cost)])
    min_rows = max(min_rows, align)
    b = [0]
    for r in range(1, world):
        target = cum[-1] * r / world
        y = int(np.searchsorted(cum, target))
        y = int(round(y / align)) * align
        lo = b[-1] + min_rows
        hi = H - (world - r) * min_rows
        lo = (lo + align - 1) // align * align
        hi = hi // align * align
        if lo > hi:
            raise ValueError(f"{H} rows cannot be split into {world} strips of at least {min_rows} rows")
        b.append(min(max(y, lo), hi))
    b.append(H)
    return b


class StripDriver:
    def __init__(self, backend_or_ctx, params, width: int, height: int, rank: int, world: int, halo: int = 24,
                 peer: bool = True, max_motion_rows: int = 0, check_every: int = 0, boundaries: Optional[List[int]] = None):
        self.backend = GpuBackend(backend_or_ctx) if isinstance(backend_or_ctx, engine.Context) else backend_or_ctx
        self.params = params
        self.W, self.H = width, height
        self.rank, self.world = rank, world
        self.halo = halo
        if boundaries is None:
            rows = (height + world - 1) // world
            if rows * world != height:
                raise ValueError(f"height {height} must be divisible by the number of ranks {world} (or pass `boundaries`)")
            boundaries = [r * rows for r in range(world)] + [height]
        boundaries = [int(v) for v in boundaries]
        if len(boundaries) != world + 1 or boundaries[0] != 0 or boundaries[-1] != height or any(
                boundaries[r + 1] <= boundaries[r] for r in range(world)):
            raise ValueError(f"boundaries {boundaries}: need {world + 1} increasing rows from 0 to {height}")
        self.boundaries = boundaries
        self.y0, self.y1 = boundaries[rank], boundaries[rank + 1]
        heights = [boundaries[r + 1] - boundaries[r] for r in range(world)]
        self.rows = heights[0] if len(set(heights)) == 1 else 0  # 0: strips of unequal height (all-gather-v)
        rows = min(heights)
        if world > 1 and rows < halo:
            raise ValueError(f"{rows} rows per rank < halo {halo}: the seam exchange only reaches the adjacent rank")
        if params.enableJittering:
            raise ValueError("strip sharding recomputes G-buffer halo rows; sub-pixel jitter would double-advance their RNG")
        if world > 1 and params.spatialNeighborRadius > halo:
            raise ValueError(f"spatialNeighborRadius {params.spatialNeighborRadius} > halo {halo}: the spatial pass would read "
                             "rows that are neither owned nor exchanged")
        if max_motion_rows > halo:
            raise ValueError(f"max_motion_rows {max_motion_rows} > halo {halo}: temporal reuse would read unexchanged rows")
        self.max_motion_rows = max_motion_rows
        self.check_every = check_every
        self.frames_rendered = 0
        self._strip = abi.GfxStripFrame()
        self._strip.y0, self._strip.y1, self._strip.halo = self.y0, self.y1, halo
        self._strip.rank, self._strip.world, self._strip.usePeer = rank, world, 1
        self.composited = self.backend.new_tensor(width * height * 4)
        if world > 1 and isinstance(self.backend, GpuBackend) and peer:
            self.backend.enable_peer(rank, world)

    # -- helpers --------------------------------------------------------------------------------------
    def _tile(self, lo: int, hi: int):
        self.params.tileOriginY, self.params.tileRows = lo, hi - lo

    def _row_slices(self, buffer_id: int, index: int, lo: int, hi: int) -> List[torch.Tensor]:
        """Views of rows [lo, hi) of every plane of a frame buffer."""
        _, comps, planes = abi.BUFFER_LAYOUT[buffer_id]
        words = comps * (2 if buffer_id == abi.BUF_RNG else 1)
        t = self.backend.tensor(buffer_id, index)
        plane = self.W * self.H * words
        return [t[p * plane + lo * self.W * words: p * plane + hi * self.W * words] for p in range(planes)]

    def exchange_halo(self, buffers):
        """Neighbour exchange of `halo` seam rows for the given [(buffer_id, index)] list."""
        if self.world == 1:
            return
        if hasattr(self.backend, "flush"):
            self.backend.flush()  # the recorded launches must be in the stream before the send/recv
        ops = []
        for buffer_id, index in buffers:
            if self.rank > 0:  # my top rows go up, their bottom rows come down
                up = self.rank - 1
                for s in self._row_slices(buffer_id, index, self.y0, min(self.y0 + self.halo, self.y1)):
                    ops.append(dist.P2POp(dist.isend, s, up))
                for s in self._row_slices(buffer_id, index, max(self.y0 - self.halo, 0), self.y0):
                    ops.append(dist.P2POp(dist.irecv, s, up))
            if self.rank < self.world - 1:
                down = self.rank + 1
                for s in self._row_slices(buffer_id, index, max(self.y1 - self.halo, self.y0), self.y1):
                    ops.append(dist.P2POp(dist.isend, s, down))
                for s in self._row_slices(buffer_id, index, self.y1, min(self.y1 + self.halo, self.H)):
                    ops.append(dist.P2POp(dist.irecv, s, down))
        if ops:
            for work in dist.batch_isend_irecv(ops):
                work.wait()

    def check_peers(self):
        """raises if a seam wait timed out since the last check (a stalled neighbour: rows of this frame may be stale)"""
        if self.world > 1 and getattr(self.backend, "peer_ready", False):
            if self.backend.ctx.peer_timed_out():
                raise RuntimeError(f"rank {self.rank}: a peer seam wait timed out (csrc/peer.cu k_peerWait): frames since the "
                                   "last check may contain stale seam rows")

    @staticmethod
    def _camera_moved(p) -> bool:
        import ctypes as C
        return bytes(C.string_at(C.addressof(p.camera), C.sizeof(p.camera))) != bytes(C.string_at(C.addressof(p.prevCamera), C.sizeof(p.prevCamera)))

    # -- ReSTIR DI + NRC in one frame (BASELINE config 5) ---------------------------------------------------
    def use_raw_communicator(self):
        """collectives through the library on a raw ncclComm_t (gfx_framebuffer_allgather[v]) instead of torch.distributed"""
        if self.world > 1 and getattr(self, "comm", None) is None:
            self.comm = NcclComm(self.rank, self.world)

    @staticmethod
    def cost_balanced_boundaries(ctx: "engine.Context", params, width: int, height: int, world: int, halo: int = 24,
                                 sky_cost: float = 0.15) -> List[int]:
        """Strip boundaries from the view itself: one full-frame G-buffer pass on this rank (every rank holds the whole scene and
        computes the same, deterministic, answer - no communication), cost of a row = its pixels that hit geometry + `sky_cost`
        per pixel (a miss pixel still costs its primary ray and a write in the shading pass).  An experiment, not the default:
        on the bistro-class view at 8 GPUs this estimate made the frame SLOWER than equal rows (1.298 vs 1.147 ms) - the rows near
        the horizon, with long rays through many buildings, cost more per hit pixel than the foreground."""
        if world == 1:
            return [0, height]
        saved = (params.tileOriginY, params.tileRows)
        params.tileOriginY, params.tileRows = 0, 0
        ctx.gbuffer(params)
        params.tileOriginY, params.tileRows = saved
        ctx.synchronize()
        gb0 = ctx.download(abi.BUF_GBUFFER0, params.bufferIndex)
        hits = (gb0[..., 0] != 0xFFFFFFFF).sum(axis=1).astype(np.float64)
        return balanced_boundaries(hits + sky_cost * width, world, halo)

    def enable_nrc(self, net: "engine.NeuralRadianceCache", overlap_training: bool = True):
        """Shard the NRC half of the frame over the ranks (gfx_nrc_shard): every rank path-traces and infers its rows, the
        training vertices are numbered over the whole frame, the records are merged, training runs replicated.
        overlap_training: the four training steps of frame f (a latency chain of small launches, replicated on every rank) run
        on a second stream under the G-buffer / ReSTIR DI passes of frame f + 1; the next inference waits for them, so the
        results are the same bits as in stream order."""
        if (self.y0 * self.W) % 128 or (self.W * self.H) % 128:
            raise ValueError("NRC strips must start on a multiple of 128 pixels (the inference tile)")
        self.net = net
        self.comm = getattr(self, "comm", None)
        self.train_stream = torch.cuda.Stream(device=f"cuda:{self.backend.ctx.device}") if overlap_training else None
        self.trained = None
        ctx = self.backend.ctx
        if self.world > 1:
            self.use_raw_communicator()
            ctx._check(ctx.lib.gfx_nrc_shard(ctx.h, self.comm.handle, self.rank, self.world), "gfx_nrc_shard")

    def render_restir_nrc_frame(self, frame_index: int, offsets, num_spatial_passes: int = 1, unbiased: bool = False,
                                train: bool = True):
        """ReSTIR DI passes (as render_frame) then the NRC frame of engine.Context.nrc_frame on the same G-buffer, both on this
        rank's rows; `offsets` are the two perFrameRng() draws (identical on all ranks).  One all-gather of the beauty strips
        at the end."""
        ctx, p = self.backend.ctx, self.params
        self.render_frame(frame_index, num_spatial_passes, unbiased, composite=False)
        self._tile(self.y0, self.y1)
        ctx.nrc_preprocess(p, offsets[0], offsets[1], frame_index == 0)
        ctx.pathtrace(p, abi.PT_NRC)
        self.wait_training()  # the weights of the previous frame's training steps; its shuffled records may be overwritten
        if self.world > 1:
            ctx._check(ctx.lib.gfx_nrc_frame_infer_rows(ctx.h, self.net.h, None, self.y0, self.y1), "gfx_nrc_frame_infer_rows")
        else:
            ctx.nrc_frame_infer(self.net)
        ctx.nrc_accumulate(p)
        if train:
            ctx.nrc_propagate(p)
            ctx.nrc_shuffle(p)
            if self.train_stream is not None:
                shuffled = torch.cuda.Event()
                shuffled.record()
                self.train_stream.wait_event(shuffled)
                ctx.nrc_frame_train(self.net, stream=self.train_stream.cuda_stream)
                self.trained = torch.cuda.Event()
                self.trained.record(self.train_stream)
            else:
                ctx.nrc_frame_train(self.net)
        self._finish_frame()

    def wait_training(self):
        """make the current stream wait for the training steps still running on the side stream (call before timing stops
        or before reading the weights)"""
        if getattr(self, "trained", None) is not None:
            torch.cuda.current_stream().wait_event(self.trained)
            self.trained = None

    # -- one frame ------------------------------------------------------------------------------------
    def render_frame(self, frame_index: int, num_spatial_passes: int = 1, unbiased: bool = False, composite: bool = True):
        p = self.params
        b = self.backend
        if self.world > 1 and frame_index > 0 and p.enableTemporalReuse and self.max_motion_rows == 0 and self._camera_moved(p):
            raise ValueError("the camera moved between frames: temporal reuse follows motion vectors across strip seams, state "
                             "max_motion_rows (<= halo) when constructing the StripDriver")
        if isinstance(b, GpuBackend) and (self.world == 1 or b.peer_ready):
            # the whole strip frame - ~35 launches incl. the one-sided seam exchanges - in ONE library call
            # (gfx_restir_strip_frame, csrc/api.cu: the same launch list as below, in C++)
            st = self._strip
            st.frameIndex, st.numSpatialPasses, st.unbiased, st.temporal = frame_index, num_spatial_passes, int(unbiased), 1
            st.peerSeq = b.peer_seq
            b.ctx._check(b.ctx.lib.gfx_restir_strip_frame(b.ctx.h, None, p, st), "gfx_restir_strip_frame")
            b.peer_seq = st.peerSeq
            if composite:
                self._finish_frame()
            return
        b.light_dist(frame_index)
        lo_h, hi_h = max(0, self.y0 - self.halo), min(self.H, self.y1 + self.halo)
        spatial_seen = 0
        # the generator mutates `p` between launches exactly like the reference host mutates plp
        for kind, pass_id in engine.restir_frame_passes(p, frame_index, num_spatial_passes, True, unbiased):
            if kind == "gbuffer":
                self._tile(lo_h, hi_h)
                b.gbuffer(p)
            elif pass_id in (abi.RESTIR_INITIAL_RIS, abi.RESTIR_INITIAL_AND_TEMPORAL_BIASED,
                             abi.RESTIR_INITIAL_AND_TEMPORAL_UNBIASED):
                self._tile(self.y0, self.y1)
                b.restir(p, pass_id)
                if num_spatial_passes > 0:
                    cur = p.currentReservoirIndex
                    self.exchange_halo([(abi.BUF_RESERVOIR, cur), (abi.BUF_RESERVOIR_INFO, cur)])
            elif pass_id in (abi.RESTIR_SPATIAL_BIASED, abi.RESTIR_SPATIAL_UNBIASED):
                self._tile(self.y0, self.y1)
                b.restir(p, pass_id)
                spatial_seen += 1
                dst = (p.currentReservoirIndex + 1) % 2
                if spatial_seen < num_spatial_passes:
                    self.exchange_halo([(abi.BUF_RESERVOIR, dst), (abi.BUF_RESERVOIR_INFO, dst)])
            else:  # shading
                self._tile(self.y0, self.y1)
                b.restir(p, pass_id)
                # final reservoirs of the seam rows: next frame's temporal reuse may look across the seam
                cur = p.currentReservoirIndex
                self.exchange_halo([(abi.BUF_RESERVOIR, cur), (abi.BUF_RESERVOIR_INFO, cur)])
        self._tile(0, 0)
        if hasattr(b, "flush"):
            b.flush()
        if composite:
            self._finish_frame()

    def _finish_frame(self):
        p = self.params
        if self.world > 1 and getattr(self, "comm", None) is not None:
            # the library's own collective on the host's communicator (the same one the sharded NRC frame uses)
            ctx = self.backend.ctx
            if self.rows:
                ctx._check(ctx.lib.gfx_framebuffer_allgather(ctx.h, self.comm.handle, None, self.rows, self.composited.data_ptr()),
                           "gfx_framebuffer_allgather")
            else:
                import ctypes as C
                starts = (C.c_uint32 * (self.world + 1))(*self.boundaries)
                ctx._check(ctx.lib.gfx_framebuffer_allgatherv(ctx.h, self.comm.handle, None, starts, self.world,
                                                              self.composited.data_ptr()), "gfx_framebuffer_allgatherv")
        elif self.world > 1 and self.rows:
            strip = self._row_slices(abi.BUF_BEAUTY_ACCUM, 0, self.y0, self.y1)[0]
            dist.all_gather_into_tensor(self.composited, strip.contiguous())
        elif self.world > 1:  # strips of unequal height without a raw communicator: one broadcast per strip
            words = self.W * 4
            mine = self._row_slices(abi.BUF_BEAUTY_ACCUM, 0, self.y0, self.y1)[0]
            self.composited[self.y0 * words: self.y1 * words].copy_(mine)
            for r in range(self.world):
                dist.broadcast(self.composited[self.boundaries[r] * words: self.boundaries[r + 1] * words], src=r)
        elif isinstance(self.backend, GpuBackend):
            self.composited = self.backend.tensor(abi.BUF_BEAUTY_ACCUM, 0)  # one rank: the beauty buffer is the frame
        else:
            self.composited.copy_(self.backend.tensor(abi.BUF_BEAUTY_ACCUM, 0))
        p.tileOriginY, p.tileRows = 0, 0
        self.frames_rendered += 1
        if self.check_every and self.frames_rendered % self.check_every == 0:
            self.check_peers()
