// pathtrace.cu — the unidirectional path tracer as a wavefront pipeline on sm_100a.
//
// Replaces pathTracing.optixPipeline.launch(W, H, 1) (path_tracing/path_tracing_main.cpp:1780-1789) and its
// programs pathTrace_rayGen_generic / pathTrace_closestHit_generic / miss / performNextEventEstimation
// (path_tracing/gpu_kernels/optix_pathtracing_kernels.cu:18-71, 73-216, 218-300, 310-341) with
// computeSurfacePoint<> (path_tracing/path_tracing_shared.h:484-621); compile-time switches as in :12-16
// (area sampling, implicit + explicit light sampling, MIS).
//
// OptiX runs this as a per-pixel megakernel that recurses into closest-hit programs.  Here a path is a
// record in HBM and one frame is
//     k_ptFirstHit                          shade the G-buffer hit: emission, NEE (shadow ray request), BSDF sample
//     for pathLength = 2 .. maxPathLength
//         k_traceWavefront<any>             shadow rays of the previous vertex; the writer adds the unoccluded
//                                           NEE contribution to the path's radiance (keeps the reference's
//                                           summation order: NEE of vertex k before the emission of vertex k+1)
//         k_traceWavefront<closest>         extension rays -> (geometry, primitive, barycentrics) per queue slot
//         k_ptBounce                        closest-hit program on the compacted queue of live paths
//     k_ptAccumulate                        running mean into the beauty buffer
// Queues are compacted with one atomic per warp (ballot), each round has its own counters (one memset per
// frame) and the trace kernel is the persistent-thread kernel of wavefront.cuh, so lanes that finish early or
// whose path died do not idle.  Per-path state: rng (frame.rng), alpha|prevDirPDensity and radiance as two
// float4 planes indexed by pixel.  The RNG draw order of every pixel is the reference's.
#include "pathtrace.cuh"

namespace gfx {

// One path vertex: NEE + next direction.  The ReGIR variant (regir/gpu_kernels/optix_pathtracing_kernels.cu) draws its
// light sample from the cell reservoirs and runs the length limit and a Russian roulette of the ray-generation
// loop *before* the extension ray is traced (:254-263, `if constexpr (useReGIR || ...)`), in addition to the
// roulette of the closest-hit program.
template <bool REGIR>
GFX_D void shadeVertexVariant(const DevScene &s, const DevRegir &rg, const DevFrameParams &p, const f3 &positionInWorld,
                              const f3 &vOutLocal, const ReferenceFrame &shadingFrame, const BSDF &bsdf, PCG32RNG &rng, f3 alpha,
                              uint32_t pathLength, f3* radiance, VertexOutput* out) {
    if (REGIR) {
        neeRegir(s, rg, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, radiance, out);
        sampleNextDirection(vOutLocal, shadingFrame, bsdf, rng, alpha, out);
        if (out->wantExtension) {
            if (pathLength + 1 >= p.maxPathLength) {
                out->wantExtension = false;
            }
            else {
                const float continueProb = fminf(sRGB_calcLuminance(out->alpha) / sRGB_calcLuminance(f3(1.0f)), 1.0f);
                if (rng.getFloat0cTo1o() >= continueProb)
                    out->wantExtension = false;
                else
                    out->alpha /= continueProb;
            }
        }
    }
    else {
        shadeVertex(s, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, radiance, out);
    }
}

// pathTrace_rayGen_generic up to the path extension loop (:73-160)
template <bool REGIR>
__global__ void __launch_bounds__(64, kBounceMinBlocks) k_ptFirstHit(DevScene s, DevFrame f, DevFrameParams p, DevPathState ps, DevRegir rg) {
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    const uint32_t lane = (threadIdx.x + threadIdx.y * blockDim.x) & 31u;
    const bool inside = x < f.W && y < p.y1;
    const uint32_t pix = inside ? y * f.W + x : 0u;

    bool alive = false;
    f3 positionInWorld(0.0f);
    VertexOutput v;
    v.wantShadow = v.wantExtension = false;
    if (inside) {
        const uint4 gb0 = f.gb0[p.bufferIndex][pix];
        f3 radiance(0.001f, 0.001f, 0.001f);
        if (gb0.x != 0xFFFFFFFFu) {
            const DevInstance* inst = s.instances + gb0.x;
            const DevMesh mesh = s.meshes[gb0.y];
            const float bcB = decodeBarycentric((uint16_t)(gb0.w & 0xFFFFu));
            const float bcC = decodeBarycentric((uint16_t)(gb0.w >> 16));
            SurfacePoint sp;
            computeSurfacePointFromGBuffer(s, inst, mesh, gb0.z, bcB, bcC, &sp);

            const f3 alpha(1.0f);
            PCG32RNG rng{ f.rng[pix] };
            const GfxMaterialDesc* mat = s.materials + mesh.materialSlot;
            const f3 vOut = normalize(p.camera.position - sp.positionInWorld);
            const float frontHit = dot(vOut, sp.geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
            positionInWorld = offsetRayOrigin(sp.positionInWorld, frontHit * sp.geometricNormalInWorld);
            const ReferenceFrame shadingFrame(sp.shadingNormalInWorld, sp.texCoord0DirInWorld);
            const f3 vOutLocal = shadingFrame.toLocal(vOut);

            radiance = f3(0.0f);
            if (vOutLocal.z > 0 && mat->hasEmittance)
                radiance += alpha * f3(mat->emittance[0], mat->emittance[1], mat->emittance[2]) / kPi;
            const BSDF bsdf = setupBsdfAtHit(s, mesh, gb0.z, bcB, bcC);
            shadeVertexVariant<REGIR>(s, rg, p, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, 1u, &radiance, &v);
            f.rng[pix] = rng.state;
            ps.alphaPdf[pix] = make_float4(v.alpha.x, v.alpha.y, v.alpha.z, v.dirPDensity);
            alive = true;
        }
        else if (s.env.enabled) { // :200-207: the environment seen directly; the miss program left (u, v) in the barycentrics
            radiance = s.env.powerCoeff * envFetch(s.env, decodeBarycentric((uint16_t)(gb0.w & 0xFFFFu)), decodeBarycentric((uint16_t)(gb0.w >> 16)));
        }
        ps.radiance[pix] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
    }
    emitRays(s, ps, ps.counters, 0u, lane, pix, positionInWorld, v, alive);
}

// pathTrace_closestHit_generic (:218-300) + the bookkeeping of the path extension loop (:161-194) for the
// compacted queue of live paths; `round` = pathLength - 2 selects the queue parity and the counters.
template <bool REGIR>
__global__ void __launch_bounds__(64, kBounceMinBlocks) k_ptBounce(DevScene s, DevFrame f, DevFrameParams p, DevPathState ps, DevRegir rg, uint32_t round,
                                                 uint32_t maxLengthTerminate) {
    const uint32_t curQueue = round & 1u, nextQueue = curQueue ^ 1u;
    const uint32_t* roundCounters = ps.counters + 4 * round;
    uint32_t* nextCounters = ps.counters + 4 * (round + 1);
    const uint32_t count = roundCounters[0];
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warpsPerGrid = gridDim.x * (blockDim.x >> 5);
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const float initImportance = sRGB_calcLuminance(f3(1.0f));

    for (uint32_t base = warp * 32u; base < count; base += warpsPerGrid * 32u) {
        const uint32_t slot = base + lane;
        bool alive = false;
        uint32_t pix = 0;
        f3 positionInWorld(0.0f);
        VertexOutput v;
        v.wantShadow = v.wantExtension = false;
        if (slot < count) {
            const uint4 hit = ps.extHits[slot];
            if (hit.y != 0xFFFFFFFFu) { // miss program: no environment light, the path ends
                pix = ps.extPixel[curQueue][slot];
                const float4 r0 = ps.extRays[curQueue][2 * (size_t)slot];
                const float4 r1 = ps.extRays[curQueue][2 * (size_t)slot + 1];
                const f3 rayOrigin(r0.x, r0.y, r0.z), rayDir(r1.x, r1.y, r1.z);
                const float4 ap = ps.alphaPdf[pix];
                f3 alpha(ap.x, ap.y, ap.z);
                const float prevDirPDensity = ap.w;
                const float4 rad = ps.radiance[pix];
                f3 radiance(rad.x, rad.y, rad.z);
                PCG32RNG rng{ f.rng[pix] };

                const uint2 im = __ldg(s.geomToInstMesh + hit.x);
                const DevInstance* inst = s.instances + im.x;
                const DevMesh mesh = s.meshes[im.y];
                SurfacePoint sp;
                computeSurfacePointAtHit(s, inst, mesh, hit.y, __uint_as_float(hit.z), __uint_as_float(hit.w), &sp);
                if (REGIR) // regir's closest-hit program never computes it (uninitialised in the reference): defined as 0
                    sp.hypAreaPDensity = 0.0f;
                const GfxMaterialDesc* mat = s.materials + mesh.materialSlot;

                const f3 vOut = normalize(-rayDir);
                const float frontHit = dot(vOut, sp.geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
                const ReferenceFrame shadingFrame(sp.shadingNormalInWorld, sp.texCoord0DirInWorld);
                positionInWorld = offsetRayOrigin(sp.positionInWorld, frontHit * sp.geometricNormalInWorld);
                const f3 vOutLocal = shadingFrame.toLocal(vOut);

                // implicit light sampling, MIS against the hypothetical NEE density (:262-275)
                if (vOutLocal.z > 0 && mat->hasEmittance) {
                    const f3 emittance(mat->emittance[0], mat->emittance[1], mat->emittance[2]);
                    const float dist2 = sqLength(positionInWorld - rayOrigin);
                    const float lightPDensity = sp.hypAreaPDensity * dist2 / vOutLocal.z;
                    const float bsdfPDensity = prevDirPDensity;
                    const float misWeight = pow2f(bsdfPDensity) / (pow2f(bsdfPDensity) + pow2f(lightPDensity));
                    radiance += alpha * emittance * (misWeight / kPi);
                }

                // Russian roulette (:277-281)
                const float continueProb = fminf(sRGB_calcLuminance(alpha) / initImportance, 1.0f);
                if (!(rng.getFloat0cTo1o() >= continueProb || maxLengthTerminate)) {
                    alpha /= continueProb;
                    const BSDF bsdf = setupBsdfAtHit(s, mesh, hit.y, __uint_as_float(hit.z), __uint_as_float(hit.w));
                    shadeVertexVariant<REGIR>(s, rg, p, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, round + 2, &radiance, &v);
                    ps.alphaPdf[pix] = make_float4(v.alpha.x, v.alpha.y, v.alpha.z, v.dirPDensity);
                    alive = true;
                }
                f.rng[pix] = rng.state;
                ps.radiance[pix] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
            }
            else if (!REGIR && s.env.enabled) { // miss program (:310-341); the ReGIR ray type's miss program is empty
                const uint32_t missPix = ps.extPixel[curQueue][slot];
                const float4 r1 = ps.extRays[curQueue][2 * (size_t)slot + 1];
                const float4 ap = ps.alphaPdf[missPix];
                const f3 implicit = evaluateEnvLightOnMiss(s, f3(r1.x, r1.y, r1.z), ap.w, false);
                float4 rad = ps.radiance[missPix];
                const f3 add = f3(ap.x, ap.y, ap.z) * implicit;
                rad.x += add.x; rad.y += add.y; rad.z += add.z;
                ps.radiance[missPix] = rad;
            }
        }
        emitRays(s, ps, nextCounters, nextQueue, lane, pix, positionInWorld, v, alive);
    }
}

// ray-gen epilogue (:202-215)
__global__ void __launch_bounds__(256) k_ptAccumulate(DevFrame f, DevFrameParams p, DevPathState ps) {
    const uint32_t n = (p.y1 - p.y0) * f.W;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const size_t pix = (size_t)p.y0 * f.W + i;
    const float4 rad = ps.radiance[pix];
    const f3 contribution(rad.x, rad.y, rad.z);
    f3 prevColorResult(0.0f);
    if (p.numAccumFrames > 0) {
        const float4 b = f.beauty[pix];
        prevColorResult = f3(b.x, b.y, b.z);
    }
    const float curWeight = 1.0f / (1 + p.numAccumFrames);
    const f3 colorResult = (1 - curWeight) * prevColorResult + curWeight * contribution;
    f.beauty[pix] = make_float4(colorResult.x, colorResult.y, colorResult.z, 1.0f);
}

int ensurePathTraceBuffers(gfx_ctx* ctx) {
    FrameState &F = ctx->frame;
    const size_t n = (size_t)F.W * F.H;
    if (F.ptAlphaPdf)
        return GFX_OK;
    GFX_CUDA(ctx, cudaMalloc(&F.ptAlphaPdf, n * 16));
    GFX_CUDA(ctx, cudaMalloc(&F.ptRadiance, n * 16));
    for (int i = 0; i < 2; ++i) {
        GFX_CUDA(ctx, cudaMalloc(&F.ptExtRays[i], n * 32));
        GFX_CUDA(ctx, cudaMalloc(&F.ptExtPixel[i], n * 4));
    }
    GFX_CUDA(ctx, cudaMalloc(&F.ptExtHits, n * 16));
    GFX_CUDA(ctx, cudaMalloc(&F.ptShadowPending, n * 16));
    GFX_CUDA(ctx, cudaMalloc(&F.ptCounters, (kMaxPathRounds + 1) * 16));
    return GFX_OK;
}

DevPathState makePathState(const gfx_ctx* ctx) {
    const FrameState &F = ctx->frame;
    DevPathState ps;
    ps.alphaPdf = F.ptAlphaPdf;
    ps.radiance = F.ptRadiance;
    for (int i = 0; i < 2; ++i) {
        ps.extRays[i] = F.ptExtRays[i];
        ps.extPixel[i] = F.ptExtPixel[i];
    }
    ps.extHits = F.ptExtHits;
    ps.shadowRays = F.rayQueue;
    ps.shadowPixel = F.rayPixel;
    ps.shadowPending = F.ptShadowPending;
    ps.counters = F.ptCounters;
    return ps;
}

int launchPathTrace(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params, int variant) {
    if (variant == GFX_PT_NRC)
        return launchPathTraceNrc(ctx, stream, params);
    if (variant != GFX_PT_BASELINE && variant != GFX_PT_REGIR) {
        ctx->setError("gfx_pathtrace_launch: unknown variant");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    const bool regir = variant == GFX_PT_REGIR;
    if (regir && !ctx->frame.regir.created) {
        ctx->setError("gfx_pathtrace_launch(GFX_PT_REGIR): call gfx_regir_build_cells first");
        return GFX_ERR_NOT_READY;
    }
    const int rc = ensurePathTraceBuffers(ctx);
    if (rc != GFX_OK)
        return rc;
    FrameState &F = ctx->frame;
    DevFrameParams p = makeDevParams(ctx, params);
    if (p.y1 <= p.y0)
        return GFX_OK;
    p.maxPathLength = params->maxPathLength ? params->maxPathLength : 5u; // 0 = the hosts' default
    const DevScene s = ctx->devScene(params);
    const DevFrame f = ctx->devFrame();
    const DevPathState ps = makePathState(ctx);
    DevRegir rg = {};
    if (regir)
        rg = makeDevRegir(ctx, params);

    const uint32_t maxPathLength = p.maxPathLength;
    const uint32_t numRounds = min(max(maxPathLength, 2u) - 1u, kMaxPathRounds); // pathLength = 2 .. maxPathLength
    GFX_CUDA(ctx, cudaMemsetAsync(F.ptCounters, 0, (kMaxPathRounds + 1) * 16, stream));

    const dim3 block(8, 8);
    const dim3 grid((F.W + 7) / 8, (p.y1 - p.y0 + 7) / 8);
    { GFX_TIMED(ctx, stream, "pt_first_hit");
    if (regir)
        k_ptFirstHit<true><<<grid, block, 0, stream>>>(s, f, p, ps, rg);
    else
        k_ptFirstHit<false><<<grid, block, 0, stream>>>(s, f, p, ps, rg); }
    ctx->launches++;
    const int traceGrid = wavefrontGrid();
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    const ShadowAccumulateWriter shadowWriter{ ps.shadowPixel, ps.shadowPending, ps.radiance };
    const ExtensionHitWriter extWriter{ ps.extHits };
    for (uint32_t round = 0; round < numRounds; ++round) {
        uint32_t* c = F.ptCounters + 4 * round;
        { GFX_TIMED(ctx, stream, "pt_trace_shadow"); k_traceWavefront<true, false><<<traceGrid, 128, 0, stream>>>(s.bvh, ps.shadowRays, c + 2, 0u, c + 3, shadowWriter); }
        { GFX_TIMED(ctx, stream, "pt_trace_extension"); k_traceWavefront<false, false><<<traceGrid, 128, 0, stream>>>(s.bvh, ps.extRays[round & 1], c + 0, 0u, c + 1, extWriter); }
        const uint32_t maxLengthTerminate = (round + 2 >= maxPathLength || round + 1 == numRounds) ? 1u : 0u;
        GFX_TIMED(ctx, stream, "pt_bounce");
        if (regir)
            k_ptBounce<true><<<sms * 16, 64, 0, stream>>>(s, f, p, ps, rg, round, maxLengthTerminate);
        else
            k_ptBounce<false><<<sms * 16, 64, 0, stream>>>(s, f, p, ps, rg, round, maxLengthTerminate);
        ctx->launches += 3;
    }
    // the last round requests no rays (maxLengthTerminate), nothing is left in flight
    const uint32_t numPixels = (p.y1 - p.y0) * F.W;
    { GFX_TIMED(ctx, stream, "pt_accumulate"); k_ptAccumulate<<<(numPixels + 255) / 256, 256, 0, stream>>>(f, p, ps); }
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

} // namespace gfx
