// pathtrace.cuh — the pieces every wavefront path tracer of this library shares (pathtrace.cu: path_tracing's
// pathTraceBaseline; nrc_pathtrace.cu: neural_radiance_caching's pathTraceNRC): surface-point reconstruction
// (computeSurfacePoint<>, path_tracing_shared.h:484-621 and its copies in the other *_shared.h), the vertex
// shading step = next event estimation + BSDF sampling (optix_pathtracing_kernels.cu:18-71, 136-146, 283-299),
// compacted ray queues and the writers of the persistent trace kernel.
#pragma once
#include "wavefront.cuh"
#include "lighting.cuh"
#include "context.h"

namespace gfx {

constexpr uint32_t kMaxPathRounds = 64;
// occupancy of the first-hit / bounce kernels: 16 blocks of 64 threads per SM = 64 registers (measured against the 88-128
// ptxas picks unconstrained: path-tracer bounce 0.44 -> 0.37 ms, NRC bounce 0.58 -> 0.53 ms; profiles/r02_summary.md)
constexpr int kBounceMinBlocks = 16;

struct DevPathState {
    float4* alphaPdf;      // per pixel: alpha.rgb, prevDirPDensity
    float4* radiance;      // per pixel: contribution.rgb
    float4* extRays[2];    // per slot: (org, tmin) (dir, tmax)
    uint32_t* extPixel[2]; // per slot: pixel index
    uint4* extHits;        // per slot: geomIndex, primIndex, bcB, bcC
    float4* shadowRays;    // per slot
    uint32_t* shadowPixel; // per slot
    float4* shadowPending; // per slot: alpha * NEE value if unoccluded, w = scale (misWeight / areaPDensity)
    uint32_t* counters;    // per round: extCount, extFetch, shadowCount, shadowFetch
};

DevPathState makePathState(const gfx_ctx* ctx); // pathtrace.cu

struct SurfacePoint {
    f3 positionInWorld, shadingNormalInWorld, texCoord0DirInWorld, geometricNormalInWorld;
    float hypAreaPDensity;
};

struct TriangleVertices {
    f3 pA, pB, pC, nA, nB, nC, tA, tB, tC;
};
GFX_D TriangleVertices fetchTriangle(const DevScene &s, const DevMesh &mesh, uint32_t primIndex) {
    const uint4 tri = __ldg(s.triangles + mesh.triBase + primIndex);
    const float4* vA = s.vertices + 3 * (size_t)(mesh.vertexBase + tri.x);
    const float4* vB = s.vertices + 3 * (size_t)(mesh.vertexBase + tri.y);
    const float4* vC = s.vertices + 3 * (size_t)(mesh.vertexBase + tri.z);
    const float4 a0 = __ldg(vA), a1 = __ldg(vA + 1), a2 = __ldg(vA + 2);
    const float4 b0 = __ldg(vB), b1 = __ldg(vB + 1), b2 = __ldg(vB + 2);
    const float4 c0 = __ldg(vC), c1 = __ldg(vC + 1), c2 = __ldg(vC + 2);
    TriangleVertices t;
    t.pA = f3(a0.x, a0.y, a0.z); t.pB = f3(b0.x, b0.y, b0.z); t.pC = f3(c0.x, c0.y, c0.z);
    t.nA = f3(a1.x, a1.y, a1.z); t.nB = f3(b1.x, b1.y, b1.z); t.nC = f3(c1.x, c1.y, c1.z);
    t.tA = f3(a2.x, a2.y, a2.z); t.tB = f3(b2.x, b2.y, b2.z); t.tC = f3(c2.x, c2.y, c2.z);
    return t;
}

// the BSDF at a hit of the path tracers (bsdf.setup(mat, texCoord, 0.0f), optix_pathtracing_kernels.cu:120-121, 283-284): the
// texture coordinate bcA tcA + bcB tcB + bcC tcC (path_tracing_shared.h:497, 601) is only interpolated in a textured scene, out of line
static __device__ __noinline__ BSDF setupBsdfTexturedAtHit(const GfxMaterialDesc* materials, const uint4* materialTextures, const uint4* texTable,
                                                           const float4* texPool, const uint4* triangles, const float4* vertices,
                                                           uint32_t triBase, uint32_t vertexBase, uint32_t matSlot, uint32_t primIndex,
                                                           float bcB, float bcC) {
    const uint4 tri = __ldg(triangles + triBase + primIndex);
    const float4* vA = vertices + 3 * (size_t)(vertexBase + tri.x);
    const float4* vB = vertices + 3 * (size_t)(vertexBase + tri.y);
    const float4* vC = vertices + 3 * (size_t)(vertexBase + tri.z);
    const float bcA = 1 - (bcB + bcC);
    const f2 texCoord = bcA * f2(__ldg(vA).w, __ldg(vA + 1).w) + bcB * f2(__ldg(vB).w, __ldg(vB + 1).w) + bcC * f2(__ldg(vC).w, __ldg(vC + 1).w);
    return setupBsdfTextured(materials, materialTextures, texTable, texPool, matSlot, texCoord.x, texCoord.y);
}
GFX_D BSDF setupBsdfAtHit(const DevScene &s, const DevMesh &mesh, uint32_t primIndex, float bcB, float bcC) {
    if (s.materialTextures)
        return setupBsdfTexturedAtHit(s.materials, s.materialTextures, s.texTable, s.texPool, s.triangles, s.vertices, mesh.triBase,
                                      mesh.vertexBase, mesh.materialSlot, primIndex, bcB, bcC);
    const GfxMaterialDesc* m = s.materials + mesh.materialSlot;
    BSDF b;
    b.setup(m->bsdfType, m->p0, m->p1, m->p2);
    return b;
}

// path_tracing_shared.h:582-621 (first hit, from GBuffer0's quantised barycentrics)
GFX_D void computeSurfacePointFromGBuffer(const DevScene &s, const DevInstance* inst, const DevMesh &mesh,
                                          uint32_t primIndex, float bcB, float bcC, SurfacePoint* sp) {
    const TriangleVertices t = fetchTriangle(s, mesh, primIndex);
    const float bcA = 1 - (bcB + bcC);
    const f3 positionInObj = bcA * t.pA + bcB * t.pB + bcC * t.pC;
    sp->positionInWorld = xfmPoint(inst->transform, positionInObj);
    sp->geometricNormalInWorld = normalize(mul3x3(inst->normalMatrix, cross(t.pB - t.pA, t.pC - t.pA)));
    const f3 shadingNormalInObj = bcA * t.nA + bcB * t.nB + bcC * t.nC;
    const f3 texCoord0DirInObj = bcA * t.tA + bcB * t.tB + bcC * t.tC;
    sp->shadingNormalInWorld = normalize(mul3x3(inst->normalMatrix, shadingNormalInObj));
    sp->texCoord0DirInWorld = xfmVector(inst->transform, texCoord0DirInObj);
    sp->texCoord0DirInWorld = normalize(
        sp->texCoord0DirInWorld - dot(sp->shadingNormalInWorld, sp->texCoord0DirInWorld) * sp->shadingNormalInWorld);
    if (!allFinite(sp->shadingNormalInWorld)) {
        sp->geometricNormalInWorld = f3(0, 0, 1);
        sp->shadingNormalInWorld = f3(0, 0, 1);
        sp->texCoord0DirInWorld = f3(1, 0, 0);
    }
    if (!allFinite(sp->texCoord0DirInWorld)) {
        f3 bitangent;
        makeCoordinateSystem(sp->shadingNormalInWorld, &sp->texCoord0DirInWorld, &bitangent);
    }
    sp->hypAreaPDensity = 0.0f;
}

// path_tracing_shared.h:484-580 with computeHypotheticalAreaPDensity = true, useSolidAngleSampling = false
GFX_D void computeSurfacePointAtHit(const DevScene &s, const DevInstance* inst, const DevMesh &mesh,
                                    uint32_t primIndex, float bcB, float bcC, SurfacePoint* sp) {
    const TriangleVertices t = fetchTriangle(s, mesh, primIndex);
    const f3 pA = xfmPoint(inst->transform, t.pA);
    const f3 pB = xfmPoint(inst->transform, t.pB);
    const f3 pC = xfmPoint(inst->transform, t.pC);
    const float bcA = 1 - (bcB + bcC);

    sp->positionInWorld = bcA * pA + bcB * pB + bcC * pC;
    const f3 shadingNormalInObj = bcA * t.nA + bcB * t.nB + bcC * t.nC;
    const f3 texCoord0DirInObj = bcA * t.tA + bcB * t.tB + bcC * t.tC;

    sp->geometricNormalInWorld = cross(pB - pA, pC - pA);
    const float area = 0.5f * length(sp->geometricNormalInWorld);
    sp->geometricNormalInWorld = sp->geometricNormalInWorld / (2 * area);

    sp->shadingNormalInWorld = normalize(mul3x3(inst->normalMatrix, shadingNormalInObj));
    sp->texCoord0DirInWorld = normalize(xfmVector(inst->transform, texCoord0DirInObj));
    if (!allFinite(sp->shadingNormalInWorld)) {
        sp->shadingNormalInWorld = f3(0, 0, 1);
        sp->texCoord0DirInWorld = f3(1, 0, 0);
    }
    if (!allFinite(sp->texCoord0DirInWorld)) {
        f3 bitangent;
        makeCoordinateSystem(sp->shadingNormalInWorld, &sp->texCoord0DirInWorld, &bitangent);
    }

    // hypothetical density with which explicit light sampling would have produced this point (:535-575)
    float lightProb = 1.0f;
    if (s.env.enabled) // path_tracing_shared.h:540-541
        lightProb *= (1 - kProbToSampleEnvLight);
    const float instImportance = inst->geomIntegral;
    lightProb *= (pow2f(inst->uniformScale) * instImportance) / __ldg(s.instIntegral);
    lightProb *= mesh.primIntegral / instImportance;
    if (!isfinite(lightProb)) {
        sp->hypAreaPDensity = 0.0f;
        return;
    }
    lightProb *= mesh.primIntegral == 0.0f ? 0.0f : __ldg(s.primWeights + mesh.triBase + primIndex) / mesh.primIntegral;
    sp->hypAreaPDensity = lightProb / area;
}

// one slot of a compacted queue per requesting lane; one atomic per warp
GFX_D uint32_t allocQueueSlot(uint32_t* counter, bool want, uint32_t lane) {
    const uint32_t mask = __ballot_sync(0xFFFFFFFFu, want);
    if (mask == 0)
        return 0;
    const int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if ((int)lane == leader)
        base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    return base + __popc(mask & ((1u << lane) - 1u));
}

// The part of a path vertex both programs share: next event estimation (optix_pathtracing_kernels.cu:18-71)
// and BSDF sampling of the next direction (:136-146 / :283-299).  Rays are only requested here.
struct VertexOutput {
    bool wantShadow, wantExtension;
    f3 shadowDir;
    float shadowTmax;
    float4 pending;
    f3 nextDir;
    f3 alpha;
    float dirPDensity;
    // for the NRC training records: the NEE estimate without the path throughput (directContNEE) as it is if no
    // shadow ray was requested or the ray turns out occluded, and as it is if the ray turns out unoccluded
    f3 directContNEE, neeUnoccluded;
    f3 localThroughput;
};

GFX_D void neeBaseline(const DevScene &s, const f3 &positionInWorld, const f3 &vOutLocal, const ReferenceFrame &shadingFrame,
                       const BSDF &bsdf, PCG32RNG &rng, const f3 &alpha, f3* radiance, VertexOutput* out) {
    out->wantShadow = false;
    out->directContNEE = f3(0.0f);
    out->neeUnoccluded = f3(0.0f);
    float uLight = rng.getFloat0cTo1o();
    float probToSampleCurLightType;
    const bool selectEnvLight = chooseEnvForNee(s, &uLight, &probToSampleCurLightType); // :25-42
    const float u0 = rng.getFloat0cTo1o();
    const float u1 = rng.getFloat0cTo1o();
    LightSample lightSample;
    float areaPDensity = 0.0f;
    if (selectEnvLight)
        sampleEnvLight(s, u0, u1, &lightSample, &areaPDensity);
    else
        sampleLight(s, uLight, u0, u1, &lightSample, &areaPDensity);
    areaPDensity *= probToSampleCurLightType;
    if (areaPDensity > 0.0f) {
        f3 shadowRay = lightSample.atInfinity ? lightSample.position : (lightSample.position - positionInWorld);
        const float dist2 = sqLength(shadowRay);
        float dist = sqrtf(dist2);
        shadowRay /= dist;
        const f3 vInLocal = shadingFrame.toLocal(shadowRay);
        const float lpCos = fabsf(dot(shadowRay, lightSample.normal));
        float bsdfPDensity = bsdf.evaluatePDF(vOutLocal, vInLocal) * lpCos / dist2;
        if (!isfinite(bsdfPDensity))
            bsdfPDensity = 0.0f;
        const float lightPDensity = areaPDensity;
        const float misWeight = pow2f(lightPDensity) / (pow2f(bsdfPDensity) + pow2f(lightPDensity));
        const float scale = misWeight / areaPDensity;
        // performDirectLighting<.., true> = visibility * value; the ray is only needed when value != 0
        const f3 value = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample);
        const f3 nee = value * scale;
        const f3 unoccluded = alpha * nee;
        out->neeUnoccluded = nee;
        if (value.x == 0.0f && value.y == 0.0f && value.z == 0.0f) {
            *radiance += unoccluded; // 0 (or NaN for a non-finite scale) whatever the visibility
            out->directContNEE = nee;
        }
        else {
            out->directContNEE = f3(0.0f) * scale;
            out->wantShadow = true;
            out->shadowDir = shadowRay;
            if (lightSample.atInfinity) // performDirectLighting<.., true>: the environment is 1e+10 away
                dist = 1e+10f;
            out->shadowTmax = dist * 0.9999f;
            out->pending = make_float4(unoccluded.x, unoccluded.y, unoccluded.z, scale);
        }
    }
}

GFX_D void sampleNextDirection(const f3 &vOutLocal, const ReferenceFrame &shadingFrame, const BSDF &bsdf, PCG32RNG &rng, f3 alpha,
                               VertexOutput* out) {
    f3 vInLocal;
    float dirPDensity;
    const float uDir0 = rng.getFloat0cTo1o();
    const float uDir1 = rng.getFloat0cTo1o();
    out->localThroughput = bsdf.sampleThroughput(vOutLocal, uDir0, uDir1, &vInLocal, &dirPDensity);
    alpha *= out->localThroughput;
    out->nextDir = shadingFrame.fromLocal(vInLocal);
    out->alpha = alpha;
    out->dirPDensity = dirPDensity;
    // the path extension loop (:161-165) stops on an invalid sample before tracing anything
    out->wantExtension = dirPDensity > 0.0f && isfinite(dirPDensity);
}

GFX_D void shadeVertex(const DevScene &s, const f3 &positionInWorld, const f3 &vOutLocal, const ReferenceFrame &shadingFrame,
                       const BSDF &bsdf, PCG32RNG &rng, f3 alpha, f3* radiance, VertexOutput* out) {
    neeBaseline(s, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, radiance, out);
    sampleNextDirection(vOutLocal, shadingFrame, bsdf, rng, alpha, out);
}

// ---- ReGIR (regir.cu builds the cell reservoirs; the path tracer resamples them) -------------------------
constexpr uint32_t kNumLightSlotsPerCell = 512; // regir_shared.h:7

struct DevRegir {
    float4* slots[2];            // one 64-byte record per light slot, see GFX_BUF_REGIR_SLOTS
    unsigned long long* slotRngs;
    uint32_t* perCellNumAccesses;
    uint32_t* lastAccessFrameIndices;
    uint32_t* numActiveCells;    // [2]
    uint32_t dimX, dimY, dimZ, numCells;
    f3 gridOrigin, gridCellSize;
    uint32_t log2NumCandidatesPerLightSlot, log2NumCandidatesPerCell, enableCellRandomization, bufferIndex;
};
DevRegir makeDevRegir(const gfx_ctx* ctx, const GfxFrameParams* p); // regir.cu

// regir_shared.h:731-742; the float -> uint32 conversion saturates like cvt.rzi.u32.f32
GFX_D uint32_t calcCellLinearIndex(const DevRegir &rg, const f3 &positionInWorld) {
    const f3 relPos = positionInWorld - rg.gridOrigin;
    const uint32_t ix = min(dm_f2uint(relPos.x / rg.gridCellSize.x), rg.dimX - 1);
    const uint32_t iy = min(dm_f2uint(relPos.y / rg.gridCellSize.y), rg.dimY - 1);
    const uint32_t iz = min(dm_f2uint(relPos.z / rg.gridCellSize.z), rg.dimZ - 1);
    return iz * rg.dimX * rg.dimY + iy * rg.dimX + ix;
}

// sampleFromCell + performNextEventEstimation<true> (regir/gpu_kernels/optix_pathtracing_kernels.cu:18-101)
GFX_D void neeRegir(const DevScene &s, const DevRegir &rg, const f3 &positionInWorld, const f3 &vOutLocal,
                    const ReferenceFrame &shadingFrame, const BSDF &bsdf, PCG32RNG &rng, const f3 &alpha, f3* radiance,
                    VertexOutput* out) {
    out->wantShadow = false;
    out->directContNEE = f3(0.0f);
    out->neeUnoccluded = f3(0.0f);
    f3 randomOffset(0.0f);
    if (rg.enableCellRandomization) {
        const float o0 = -0.5f + rng.getFloat0cTo1o();
        const float o1 = -0.5f + rng.getFloat0cTo1o();
        const float o2 = -0.5f + rng.getFloat0cTo1o();
        randomOffset = rg.gridCellSize * f3(o0, o1, o2);
    }
    const uint32_t cellLinearIndex = calcCellLinearIndex(rg, positionInWorld + randomOffset);
    const uint32_t resStartIndex = kNumLightSlotsPerCell * cellLinearIndex;
    { // atomicAdd(&perCellNumAccesses[cell], 1u), aggregated over the lanes of the warp that touch the same cell
        const uint32_t peers = __match_any_sync(__activemask(), cellLinearIndex);
        if ((threadIdx.x + threadIdx.y * blockDim.x) % 32 == (uint32_t)(__ffs(peers) - 1))
            atomicAdd(rg.perCellNumAccesses + cellLinearIndex, (uint32_t)__popc(peers));
    }

    const uint32_t numResampling = 1u << rg.log2NumCandidatesPerCell;
    float sumWeights = 0.0f;
    uint32_t combinedStreamLength = 0;
    f3 selectedContribution(0.0f), selectedPosition(0.0f);
    uint32_t selectedAtInfinity = 0;
    float selectedTargetPDensity = 0.0f;
    const float4* slots = rg.slots[rg.bufferIndex];
    for (uint32_t i = 0; i < numResampling; ++i) {
        // mapPrimarySampleToDiscrete (common_shared.h:140-150)
        const uint32_t lightSlotIdx = resStartIndex + min(dm_f2uint(rng.getFloat0cTo1o() * kNumLightSlotsPerCell), kNumLightSlotsPerCell - 1);
        const float4* rec = slots + 4 * (size_t)lightSlotIdx;
        const float4 r0 = rec[0], r1 = rec[1], r2 = rec[2];
        const uint32_t m = __float_as_uint(r1.w);
        const uint32_t streamLength = m & 0x7FFFFFFFu;
        combinedStreamLength += streamLength;
        const float recPDFEstimate = r2.w;
        if (recPDFEstimate == 0.0f)
            continue;
        LightSample ls;
        ls.emittance = f3(r0.x, r0.y, r0.z);
        ls.position = f3(r1.x, r1.y, r1.z);
        ls.normal = f3(r2.x, r2.y, r2.z);
        ls.atInfinity = m >> 31;
        const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, ls);
        const float targetPDensity = convertToWeight(cont);
        const float weight = targetPDensity * recPDFEstimate * streamLength;
        // Reservoir::update
        sumWeights += weight;
        if (rng.getFloat0cTo1o() < weight / sumWeights) {
            selectedContribution = cont;
            selectedPosition = ls.position;
            selectedAtInfinity = ls.atInfinity;
            selectedTargetPDensity = targetPDensity;
        }
    }
    const float weightForEstimate = 1.0f / combinedStreamLength;
    float recProbDensityEstimate = weightForEstimate * sumWeights / selectedTargetPDensity;
    if (!isfinite(recProbDensityEstimate))
        recProbDensityEstimate = 0.0f;
    if (recProbDensityEstimate > 0.0f) {
        // ret = unshadowedContribution * (visibility * recProbDensityEstimate)
        const f3 cont = selectedContribution;
        const f3 nee = cont * (1.0f * recProbDensityEstimate);
        const f3 unoccluded = alpha * nee;
        out->neeUnoccluded = nee;
        if (cont.x == 0.0f && cont.y == 0.0f && cont.z == 0.0f) {
            *radiance += unoccluded;
            out->directContNEE = nee;
        }
        else {
            // evaluateVisibility (regir_shared.h:544-566); an environment sample is a direction, 1e+10 away
            f3 shadowRayDir = selectedAtInfinity ? selectedPosition : (selectedPosition - positionInWorld);
            float dist = sqrtf(sqLength(shadowRayDir));
            shadowRayDir /= dist;
            if (selectedAtInfinity)
                dist = 1e+10f;
            out->directContNEE = cont * (0.0f * recProbDensityEstimate);
            out->wantShadow = true;
            out->shadowDir = shadowRayDir;
            out->shadowTmax = dist * 0.9999f;
            out->pending = make_float4(unoccluded.x, unoccluded.y, unoccluded.z, (cont.x + cont.y + cont.z) * 0.0f);
        }
    }
}

GFX_D void emitRays(const DevScene &s, const DevPathState &ps, uint32_t* roundCounters, uint32_t nextQueue, uint32_t lane,
                    uint32_t pix, const f3 &positionInWorld, const VertexOutput &v, bool alive) {
    const bool wantShadow = alive && v.wantShadow;
    const bool wantExt = alive && v.wantExtension;
    const uint32_t shadowSlot = allocQueueSlot(roundCounters + 2, wantShadow, lane);
    const uint32_t extSlot = allocQueueSlot(roundCounters + 0, wantExt, lane);
    if (wantShadow) {
        ps.shadowRays[2 * (size_t)shadowSlot] = make_float4(positionInWorld.x, positionInWorld.y, positionInWorld.z, 0.0f);
        ps.shadowRays[2 * (size_t)shadowSlot + 1] = make_float4(v.shadowDir.x, v.shadowDir.y, v.shadowDir.z, v.shadowTmax);
        ps.shadowPixel[shadowSlot] = pix;
        ps.shadowPending[shadowSlot] = v.pending;
    }
    if (wantExt) {
        ps.extRays[nextQueue][2 * (size_t)extSlot] = make_float4(positionInWorld.x, positionInWorld.y, positionInWorld.z, 0.0f);
        ps.extRays[nextQueue][2 * (size_t)extSlot + 1] = make_float4(v.nextDir.x, v.nextDir.y, v.nextDir.z, 3.402823466e+38f);
        ps.extPixel[nextQueue][extSlot] = pix;
    }
    // ray statistics (frame.stats[0]): one atomic per warp
    const uint32_t n = __popc(__ballot_sync(0xFFFFFFFFu, wantShadow)) + __popc(__ballot_sync(0xFFFFFFFFu, wantExt));
    if (lane == 0 && n)
        atomicAdd(s.rayCounter, (unsigned long long)n);
}

struct ExtensionHitWriter { // closest hit -> what the closest-hit program reads from OptiX (HitPointParameter::get)
    uint4* hits;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        const Hit &h = st.best;
        const bool isHit = h.storageIndex != 0xFFFFFFFFu;
        hits[ray] = make_uint4(h.geomIndex, isHit ? h.primIndex : 0xFFFFFFFFu, __float_as_uint(h.bcB), __float_as_uint(h.bcC));
    }
};

struct ShadowAccumulateWriter { // visibility * (alpha * f * Le * G * misWeight / p) of performNextEventEstimation
    const uint32_t* shadowPixel;
    const float4* pending;
    float4* radiance;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        const float4 c = pending[ray];
        const bool unoccluded = st.best.storageIndex == 0xFFFFFFFFu;
        if (!unoccluded && isfinite(c.w))
            return; // alpha * (0 * scale) = 0
        float4* dst = radiance + shadowPixel[ray]; // at most one shadow ray per path and round: no race
        float4 r = *dst;
        if (unoccluded) {
            r.x += c.x; r.y += c.y; r.z += c.z;
        }
        else {
            const float nan = __int_as_float(0x7FC00000);
            r.x += nan; r.y += nan; r.z += nan;
        }
        *dst = r;
    }
};

} // namespace gfx
