// trace.cu — wavefront ray tracing: persistent threads pulling rays from SoA queues.
//
// Entry points
//  * traceRays            bvh::traverse<8> (common/bvh_builder.cpp:1653-1663) for a batch of 32-byte ray
//                         records -> 32-byte shared::HitObject records (common/common_shared.h:1065-1078);
//  * traceVisibilityQueue the visibility rays of the ReSTIR passes (restir_di_shared.h:559-582 + the AH program
//                         optix_restir_di_kernels.cu:5-8): rays were appended to the frame's queue by the
//                         producing kernel with warp-ballot compaction, results land in a per-pixel byte.
//
// The kernel itself (persistent threads with warp-ballot refill) lives in wavefront.cuh.
#include "wavefront.cuh"
#include "context.h"

namespace gfx {

struct HitWriter { // GfxHitObject records, indexed by ray
    const uint2* geomToInstMesh;
    uint4* hits;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        const Hit &h = st.best;
        const bool isHit = h.storageIndex != 0xFFFFFFFFu;
        // STATS: instUserData = internal nodes visited | triangles tested << 16 (bvh::TraversalStatistics)
        const uint32_t userData = STATS ? (min(h.statNodes, 0xFFFFu) | (min(h.statTris, 0xFFFFu) << 16)) : 0u;
        if (ANY_HIT) {
            // visibility payload: dist = 0 when occluded, tmax otherwise (the AH program writes 0.0f)
            hits[2 * (size_t)ray] = make_uint4(__float_as_uint(isHit ? 0.0f : st.tmax), 0xFFFFFFFFu, userData, 0xFFFFFFFFu);
            hits[2 * (size_t)ray + 1] = make_uint4(isHit ? 0u : 0xFFFFFFFFu, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u);
            return;
        }
        const uint32_t inst = isHit && geomToInstMesh ? __ldg(geomToInstMesh + h.geomIndex).x : 0xFFFFFFFFu;
        const float bcA = 1.0f - (h.bcB + h.bcC);
        hits[2 * (size_t)ray] = make_uint4(__float_as_uint(h.dist), inst, userData, h.geomIndex);
        hits[2 * (size_t)ray + 1] = isHit
            ? make_uint4(h.primIndex, __float_as_uint(bcA), __float_as_uint(h.bcB), __float_as_uint(h.bcC))
            : make_uint4(0xFFFFFFFFu, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u);
    }
};

struct VisibilityWriter { // one byte per pixel that asked
    const uint32_t* rayPixel;
    uint8_t* visibility;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        visibility[__ldg(rayPixel + ray)] = st.best.storageIndex == 0xFFFFFFFFu ? 1 : 0;
    }
};

int traceRays(gfx_ctx* ctx, cudaStream_t stream, const GfxRay* dRays, uint32_t numRays, GfxHitObject* dHits, int mode) {
    if (numRays == 0)
        return GFX_OK;
    const DevScene dev = ctx->devScene();
    const float4* r = reinterpret_cast<const float4*>(dRays);
    HitWriter w{ dev.geomToInstMesh, reinterpret_cast<uint4*>(dHits) };
    uint32_t* counter = ctx->traceFetchCounter;
    GFX_CUDA(ctx, cudaMemsetAsync(counter, 0, 4, stream));
    const int grid = min(wavefrontGrid(), (int)((numRays + 127) / 128));
    GFX_TIMED(ctx, stream, "trace_batch");
    switch (mode) {
    case GFX_TRACE_CLOSEST: k_traceWavefront<false, false><<<grid, 128, 0, stream>>>(dev.bvh, r, nullptr, numRays, counter, w); break;
    case GFX_TRACE_ANY: k_traceWavefront<true, false><<<grid, 128, 0, stream>>>(dev.bvh, r, nullptr, numRays, counter, w); break;
    case GFX_TRACE_CLOSEST | GFX_TRACE_STATS: k_traceWavefront<false, true><<<grid, 128, 0, stream>>>(dev.bvh, r, nullptr, numRays, counter, w); break;
    case GFX_TRACE_ANY | GFX_TRACE_STATS: k_traceWavefront<true, true><<<grid, 128, 0, stream>>>(dev.bvh, r, nullptr, numRays, counter, w); break;
    default:
        ctx->setError("gfx_trace: unknown mode");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

int resetVisibilityQueue(gfx_ctx* ctx, cudaStream_t stream) {
    GFX_CUDA(ctx, cudaMemsetAsync(ctx->frame.rayCounters, 0, 8, stream));
    return GFX_OK;
}

int traceVisibilityQueue(gfx_ctx* ctx, cudaStream_t stream) {
    const DevScene dev = ctx->devScene();
    const FrameState &F = ctx->frame;
    VisibilityWriter w{ F.rayPixel, F.visibility };
    GFX_TIMED(ctx, stream, "trace_visibility");
    // ReSTIR visibility rays mostly reach their light: postponed leaf tests win 10 % over immediate ones
    k_traceWavefrontDeferred<true, false><<<wavefrontGrid(), 128, 0, stream>>>(dev.bvh, F.rayQueue, F.rayCounters, 0u, F.rayCounters + 1, w);
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

} // namespace gfx
