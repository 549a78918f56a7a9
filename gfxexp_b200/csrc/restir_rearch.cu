// restir_rearch.cu — the "rearchitected" ReSTIR DI renderer as sm_100a kernels.
//
// Replaces kernelPerformLightPreSampling / kernelPerformPerPixelRIS (restir_di/gpu_kernels/per_pixel_ris.cu:6-40,
// 44-128) and restirRearch.optixPipeline.launch with the entry points traceShadowRays[With…Reuse{Biased,Unbiased}]
// and shadeAndResample[With…Reuse] (restir_di/gpu_kernels/optix_restir_di_rearch_kernels.cu:14-225, 263-400,
// 402-664; launch sites restir_di/restir_di_main.cpp:2423-2493).
//
// * Presampled lights are 48-byte records (PreSampledLight 44 B padded): three aligned 16-byte loads per candidate;
//   the whole table (128 x 1024 x 48 B = 6.3 MB) stays in the 126 MB L2 and a tile's 1024-entry subset (48 KB) is
//   shared by the 64 pixels of the tile.
// * traceShadowRays is split request -> trace -> (bits land by atomicOr): the request kernel evaluates the
//   heuristics, the reused visibility bits and up to 3 (biased) / 7 (unbiased) shadow rays per pixel, each tagged with
//   the SampleVisibility bits it answers (the unbiased program traces the temporal / spatiotemporal sample from the
//   current point twice, :81-83 + :98-100 and :177-179 + :194-196; one ray answers both bits here); the
//   persistent-thread kernel of wavefront.cuh traces the compacted queue.
// * shadeAndResample is a per-pixel kernel without rays.
#include "restir_common.cuh"
#include "wavefront.cuh"
#include <random>
#include <vector>

namespace gfx {

constexpr uint32_t kNumLightSubsets = 128;  // restir_di_shared.h:8
constexpr uint32_t kLightSubsetSize = 1024; // restir_di_shared.h:9
constexpr uint32_t kNumPreSampledLights = kNumLightSubsets * kLightSubsetSize;

enum : uint32_t { // SampleVisibility (restir_di_shared.h:146-164)
    SV_NEW = 1u << 0, SV_NEW_ON_T = 1u << 1, SV_NEW_ON_ST = 1u << 2,
    SV_T_PASSED = 1u << 3, SV_T = 1u << 4, SV_T_ON_CUR = 1u << 5, SV_T_ON_ST = 1u << 6,
    SV_ST_PASSED = 1u << 7, SV_ST = 1u << 8, SV_ST_ON_CUR = 1u << 9, SV_ST_ON_T = 1u << 10,
    SV_SELECTED = 1u << 11
};

struct DevRearch {
    float4* preSampledLights;        // 3 x float4 per entry
    unsigned long long* rngs;
    uint32_t* sampleVis[2];
    float4* rays;                    // 2 x float4 per ray
    uint32_t* rayPixel;
    uint32_t* rayMask;
    uint32_t* counters;              // [0] queued, [1] fetched
};

static DevRearch makeDevRearch(const gfx_ctx* ctx) {
    const FrameState::Rearch &R = ctx->frame.rearch;
    DevRearch d;
    d.preSampledLights = R.preSampledLights;
    d.rngs = R.rngs;
    d.sampleVis[0] = R.sampleVis[0];
    d.sampleVis[1] = R.sampleVis[1];
    d.rays = R.rays;
    d.rayPixel = R.rayPixel;
    d.rayMask = R.rayMask;
    d.counters = R.counters;
    return d;
}

int ensureRearch(gfx_ctx* ctx, uint32_t raysPerPixel) {
    FrameState &F = ctx->frame;
    FrameState::Rearch &R = F.rearch;
    const size_t n = (size_t)F.W * F.H;
    if (!R.created) {
        GFX_CUDA(ctx, cudaMalloc(&R.preSampledLights, (size_t)kNumPreSampledLights * 48));
        GFX_CUDA(ctx, cudaMemset(R.preSampledLights, 0, (size_t)kNumPreSampledLights * 48));
        GFX_CUDA(ctx, cudaMalloc(&R.rngs, (size_t)kNumPreSampledLights * 8));
        std::vector<unsigned long long> states(kNumPreSampledLights);
        std::mt19937_64 rngSeed(894213312210ull); // restir_di_main.cpp:1217
        for (auto &st : states)
            st = rngSeed();
        GFX_CUDA(ctx, cudaMemcpy(R.rngs, states.data(), states.size() * 8, cudaMemcpyHostToDevice));
        for (int i = 0; i < 2; ++i) {
            GFX_CUDA(ctx, cudaMalloc(&R.sampleVis[i], n * 4));
            GFX_CUDA(ctx, cudaMemset(R.sampleVis[i], 0, n * 4));
        }
        GFX_CUDA(ctx, cudaMalloc(&R.counters, 16));
        R.created = true;
    }
    if (raysPerPixel > R.raysPerPixel) {
        cudaFree(R.rays); cudaFree(R.rayPixel); cudaFree(R.rayMask);
        R.rays = nullptr; R.rayPixel = nullptr; R.rayMask = nullptr;
        GFX_CUDA(ctx, cudaMalloc(&R.rays, n * raysPerPixel * 32));
        GFX_CUDA(ctx, cudaMalloc(&R.rayPixel, n * raysPerPixel * 4));
        GFX_CUDA(ctx, cudaMalloc(&R.rayMask, n * raysPerPixel * 4));
        R.raysPerPixel = raysPerPixel;
    }
    return GFX_OK;
}

// per_pixel_ris.cu:6-40
__global__ void __launch_bounds__(128) k_presampleLights(DevScene s, DevRearch r) {
    const uint32_t linearThreadIndex = blockDim.x * blockIdx.x + threadIdx.x;
    if (linearThreadIndex >= kNumPreSampledLights)
        return;
    PCG32RNG rng{ r.rngs[linearThreadIndex] };
    LightSample ls = emptyLightSample();
    float areaPDensity = 0.0f;
    // :12-28: with an environment light the first probToSampleEnvLight * lightSubsetSize lights of every subset sample it
    float probToSampleCurLightType = 1.0f;
    bool sampleEnv = false;
    if (s.env.enabled) {
        if (__ldg(s.instIntegral) > 0.0f) {
            const uint32_t indexInSubset = linearThreadIndex % kLightSubsetSize;
            sampleEnv = indexInSubset < kProbToSampleEnvLight * kLightSubsetSize;
            probToSampleCurLightType = sampleEnv ? kProbToSampleEnvLight : (1 - kProbToSampleEnvLight);
        }
        else {
            sampleEnv = true;
        }
    }
    const float ul = rng.getFloat0cTo1o();
    const float u0 = rng.getFloat0cTo1o();
    const float u1 = rng.getFloat0cTo1o();
    if (sampleEnv)
        sampleEnvLight(s, u0, u1, &ls, &areaPDensity);
    else
        sampleLight(s, ul, u0, u1, &ls, &areaPDensity);
    areaPDensity *= probToSampleCurLightType;
    r.rngs[linearThreadIndex] = rng.state;
    float4* o = r.preSampledLights + 3 * (size_t)linearThreadIndex;
    o[0] = make_float4(ls.emittance.x, ls.emittance.y, ls.emittance.z, areaPDensity);
    o[1] = make_float4(ls.position.x, ls.position.y, ls.position.z, __uint_as_float(ls.atInfinity));
    o[2] = make_float4(ls.normal.x, ls.normal.y, ls.normal.z, 0.0f);
}

struct RearchShadingPoint {
    f3 positionInWorld, vOutLocal;
    ReferenceFrame shadingFrame;
    BSDF bsdf;
};
// the prologue of performPerPixelRIS / shadeAndResample and computeMISWeight's neighbour reconstruction
GFX_D RearchShadingPoint reconstructShadingPoint(const DevScene &s, const DevFrame &f, uint32_t bufIdx, size_t pix, const f3 &cameraPosition) {
    const float4 g2 = f.gb2[bufIdx][pix];
    const uint4 g3 = f.gb3[bufIdx][pix];
    RearchShadingPoint sp;
    const f3 positionInWorld(g2.x, g2.y, g2.z);
    const f3 geometricNormalInWorld = decodeVector(__float_as_uint(g2.w));
    const f3 vOut = normalize(cameraPosition - positionInWorld);
    const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
    sp.positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);
    sp.shadingFrame = ReferenceFrame(decodeVector(g3.x), decodeVector(g3.y));
    sp.vOutLocal = sp.shadingFrame.toLocal(vOut);
    sp.bsdf = setupBsdf(s, g3.w, decodeTexCoords(g3.z));
    return sp;
}

GFX_D LightSample loadPreSampled(const float4* table, uint32_t index, float* areaPDensity) {
    const float4* e = table + 3 * (size_t)index;
    const float4 a = __ldg(e), b = __ldg(e + 1), c = __ldg(e + 2);
    LightSample ls;
    ls.emittance = f3(a.x, a.y, a.z);
    *areaPDensity = a.w;
    ls.position = f3(b.x, b.y, b.z);
    ls.atInfinity = __float_as_uint(b.w);
    ls.normal = f3(c.x, c.y, c.z);
    return ls;
}

// per_pixel_ris.cu:44-128; one block = one 8x8 tile (shared::tileSizeX/Y)
__global__ void __launch_bounds__(64) k_perPixelRIS(DevScene s, DevFrame f, DevFrameParams p, DevRearch r) {
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    const bool inside = x < f.W && y < p.y1;
    const size_t pix = inside ? (size_t)y * f.W + x : 0;
    const uint32_t curBufIdx = p.bufferIndex;

    PCG32RNG rng{ inside ? f.rng[pix] : 0ull };
    __shared__ uint32_t sm_perTileLightSubsetIndex;
    if (threadIdx.x == 0 && threadIdx.y == 0) // the tile origin is always inside the image
        sm_perTileLightSubsetIndex = min(dm_f2uint(rng.getFloat0cTo1o() * kNumLightSubsets), kNumLightSubsets - 1);
    __syncthreads();
    if (!inside)
        return;
    const float4* lightSubSet = r.preSampledLights + 3 * (size_t)sm_perTileLightSubsetIndex * kLightSubsetSize;

    if (f.gb0[curBufIdx][pix].x == 0xFFFFFFFFu)
        return;
    const RearchShadingPoint sp = reconstructShadingPoint(s, f, curBufIdx, pix, p.camera.position);

    const uint32_t curResIndex = p.currentReservoirIndex;
    float sumWeights = 0.0f;
    uint32_t selected = 0xFFFFFFFFu;
    float selectedTargetDensity = 0.0f;
    const uint32_t numCandidates = 1u << p.log2NumCandidateSamples;
    for (uint32_t i = 0; i < numCandidates; ++i) {
        const uint32_t lightIndex = min(dm_f2uint(rng.getFloat0cTo1o() * kLightSubsetSize), kLightSubsetSize - 1);
        float areaPDensity;
        const LightSample ls = loadPreSampled(lightSubSet, lightIndex, &areaPDensity);
        const f3 cont = performDirectLighting<false>(s, sp.positionInWorld, sp.vOutLocal, sp.shadingFrame, sp.bsdf, ls);
        if (cont.x == 0.0f && cont.y == 0.0f && cont.z == 0.0f && areaPDensity > 0.0f) {
            (void)rng.getFloat0cTo1o(); // weight 0: the reservoir keeps its sample, the draw is still consumed
            continue;
        }
        const float targetDensity = convertToWeight(cont);
        const float weight = targetDensity / areaPDensity;
        const float u = rng.getFloat0cTo1o();
        sumWeights += weight;
        if (u < weight / sumWeights) {
            selected = lightIndex;
            selectedTargetDensity = targetDensity;
        }
    }
    Reservoir reservoir;
    reservoir.initialize(emptyLightSample());
    if (selected != 0xFFFFFFFFu) {
        float unused;
        reservoir.sample = loadPreSampled(lightSubSet, selected, &unused);
    }
    reservoir.sumWeights = sumWeights;
    reservoir.streamLength = numCandidates;

    float recPDFEstimate = reservoir.sumWeights / (selectedTargetDensity * reservoir.streamLength);
    if (!isfinite(recPDFEstimate)) {
        recPDFEstimate = 0.0f;
        selectedTargetDensity = 0.0f;
    }
    f.rng[pix] = rng.state;
    storeReservoir(f, curResIndex, pix, reservoir);
    f.reservoirInfo[curResIndex][pix] = make_float2(recPDFEstimate, selectedTargetDensity);
}

GFX_D void temporalNeighborCoord(const DevFrame &f, uint32_t curBufIdx, size_t pix, uint32_t x, uint32_t y, int* nbx, int* nby) {
    const float2 gb1 = f.gb1[curBufIdx][pix];
    *nbx = dm_f2int(x + 0.5f - gb1.x);
    *nby = dm_f2int(y + 0.5f - gb1.y);
}
GFX_D void spatialNeighborCoord(const DevFrame &f, const DevFrameParams &p, uint32_t x, uint32_t y, PCG32RNG &rng, int* nbx, int* nby,
                                float* deltaX, float* deltaY) {
    float radius = p.spatialNeighborRadius;
    if (p.useLowDiscrepancyNeighbors) {
        const uint32_t deltaIndex = p.spatialNeighborBaseIndex + 5 * x + 7 * y;
        const float2 delta = __ldg(f.neighborDeltas + deltaIndex % 1024);
        *deltaX = radius * delta.x;
        *deltaY = radius * delta.y;
    }
    else {
        radius *= sqrtf(rng.getFloat0cTo1o());
        const float angle = 2 * kPi * rng.getFloat0cTo1o();
        float sa, ca;
        dm_sincos(angle, &sa, &ca);
        *deltaX = radius * ca;
        *deltaY = radius * sa;
    }
    *nbx = dm_f2int(x + 0.5f + *deltaX);
    *nby = dm_f2int(y + 0.5f + *deltaY);
}

struct ShadowRequest {
    bool want;
    f3 org;
    LightSample ls;
    uint32_t mask;
};
GFX_D void enqueueShadow(const DevScene &s, const DevRearch &r, uint32_t lane, uint32_t pix, const ShadowRequest &q) {
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, q.want);
    if (ballot == 0)
        return;
    const int leader = __ffs(ballot) - 1;
    uint32_t base = 0;
    if ((int)lane == leader) {
        base = atomicAdd(r.counters, (uint32_t)__popc(ballot));
        atomicAdd(s.rayCounter, (unsigned long long)__popc(ballot));
    }
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    if (q.want) {
        const uint32_t slot = base + __popc(ballot & ((1u << lane) - 1u));
        RayRequest rr;
        visibilityRay(q.org, q.ls, pix, &rr);
        r.rays[2 * (size_t)slot] = make_float4(rr.org.x, rr.org.y, rr.org.z, 0.0f);
        r.rays[2 * (size_t)slot + 1] = make_float4(rr.dir.x, rr.dir.y, rr.dir.z, rr.tmax);
        r.rayPixel[slot] = pix;
        r.rayMask[slot] = q.mask;
    }
}

// traceShadowRays<T,S,U> (optix_restir_di_rearch_kernels.cu:14-225): everything but the traversal
template <bool withTemporalRIS, bool withSpatialRIS, bool useUnbiasedEstimator>
__global__ void __launch_bounds__(64) k_shadowRayRequests(DevScene s, DevFrame f, DevFrameParams p, DevRearch r) {
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    const uint32_t lane = (threadIdx.x + threadIdx.y * blockDim.x) & 31u;
    const bool inside = x < f.W && y < p.y1;
    const uint32_t pix = inside ? y * f.W + x : 0u;
    const uint32_t curBufIdx = p.bufferIndex, prevBufIdx = (curBufIdx + 1) % 2;
    const uint32_t curResIndex = p.currentReservoirIndex, prevResIndex = (curResIndex + 1) % 2;

    // up to 7 rays: new | temporal (+onCurrent) | new on temporal | spatiotemporal (+onCurrent) | new on spatiotemporal |
    //               temporal on spatiotemporal | spatiotemporal on temporal
    ShadowRequest q[7];
#pragma unroll
    for (int i = 0; i < 7; ++i)
        q[i].want = false;

    const bool active = inside && f.gb0[curBufIdx][pix].x != 0xFFFFFFFFu;
    if (active) {
        const float4 g2 = f.gb2[curBufIdx][pix];
        const uint4 g3 = f.gb3[curBufIdx][pix];
        f3 positionInWorld(g2.x, g2.y, g2.z);
        const f3 geometricNormalInWorld = decodeVector(__float_as_uint(g2.w));
        const f3 shadingNormalInWorld = decodeVector(g3.x);
        const f3 vOut = p.camera.position - positionInWorld;
        const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
        positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);
        const float dist = length(vOut);

        auto neighborOrigin = [&](size_t nbPix) {
            const float4 n2 = f.gb2[prevBufIdx][nbPix];
            const f3 nbPositionInWorld(n2.x, n2.y, n2.z);
            const f3 nbGeometricNormalInWorld = decodeVector(__float_as_uint(n2.w));
            const f3 nbVOut = p.prevCamera.position - nbPositionInWorld;
            const float nbFrontHit = dot(nbVOut, nbGeometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
            return offsetRayOrigin(nbPositionInWorld, nbFrontHit * nbGeometricNormalInWorld);
        };

        uint32_t sampleVis = 0;
        LightSample newSample;
        bool newSampleIsValid;
        {
            const Reservoir reservoir = loadReservoir(f, curResIndex, pix);
            newSample = reservoir.sample;
            newSampleIsValid = reservoir.sumWeights > 0.0f;
            if (newSampleIsValid) {
                q[0].want = true; q[0].org = positionInWorld; q[0].ls = newSample; q[0].mask = SV_NEW;
            }
        }

        int tNbX = 0, tNbY = 0;
        f3 tNbPositionInWorld(0.0f);
        bool temporalSampleIsValid = false;
        LightSample temporalSample = emptyLightSample();
        if (withTemporalRIS) {
            temporalNeighborCoord(f, curBufIdx, pix, x, y, &tNbX, &tNbY);
            if (testNeighbor<true>(f, p.camera, prevBufIdx, tNbX, tNbY, dist, shadingNormalInWorld))
                sampleVis |= SV_T_PASSED;
            if (sampleVis & SV_T_PASSED) {
                const size_t nbPix = (size_t)tNbY * f.W + tNbX;
                if (p.reuseVisibilityForTemporal && !useUnbiasedEstimator) {
                    if (r.sampleVis[prevBufIdx][nbPix] & SV_SELECTED)
                        sampleVis |= SV_T;
                }
                else {
                    const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
                    temporalSample = neighbor.sample;
                    temporalSampleIsValid = neighbor.sumWeights > 0.0f;
                    if (temporalSampleIsValid) {
                        q[1].want = true; q[1].org = positionInWorld; q[1].ls = temporalSample;
                        q[1].mask = SV_T | (useUnbiasedEstimator ? SV_T_ON_CUR : 0u);
                    }
                }
                if (useUnbiasedEstimator) {
                    tNbPositionInWorld = neighborOrigin(nbPix);
                    if (newSampleIsValid) {
                        q[2].want = true; q[2].org = tNbPositionInWorld; q[2].ls = newSample; q[2].mask = SV_NEW_ON_T;
                    }
                }
            }
        }

        int stNbX = 0, stNbY = 0;
        f3 stNbPositionInWorld(0.0f);
        bool spatiotemporalSampleIsValid = false;
        LightSample spatiotemporalSample = emptyLightSample();
        if (withSpatialRIS) {
            float deltaX, deltaY;
            PCG32RNG rng{ f.rng[pix] }; // the advanced state is not stored (:148-150)
            spatialNeighborCoord(f, p, x, y, rng, &stNbX, &stNbY, &deltaX, &deltaY);
            bool passed = testNeighbor<true>(f, p.camera, prevBufIdx, stNbX, stNbY, dist, shadingNormalInWorld);
            passed = passed && (stNbX != (int)x || stNbY != (int)y);
            if (passed) {
                sampleVis |= SV_ST_PASSED;
                const size_t nbPix = (size_t)stNbY * f.W + stNbX;
                bool reused = false;
                if (p.reuseVisibilityForSpatiotemporal && !useUnbiasedEstimator) {
                    const float threshold2 = pow2f(p.radiusThresholdForSpatialVisReuse);
                    const float dist2 = pow2f(deltaX) + pow2f(deltaY);
                    reused = dist2 < threshold2;
                }
                if (reused) {
                    if (r.sampleVis[prevBufIdx][nbPix] & SV_SELECTED)
                        sampleVis |= SV_ST;
                }
                else {
                    const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
                    spatiotemporalSample = neighbor.sample;
                    spatiotemporalSampleIsValid = neighbor.sumWeights > 0.0f;
                    if (spatiotemporalSampleIsValid) {
                        q[3].want = true; q[3].org = positionInWorld; q[3].ls = spatiotemporalSample;
                        q[3].mask = SV_ST | (useUnbiasedEstimator ? SV_ST_ON_CUR : 0u);
                    }
                }
                if (useUnbiasedEstimator) {
                    stNbPositionInWorld = neighborOrigin(nbPix);
                    if (newSampleIsValid) {
                        q[4].want = true; q[4].org = stNbPositionInWorld; q[4].ls = newSample; q[4].mask = SV_NEW_ON_ST;
                    }
                }
            }
        }

        if (useUnbiasedEstimator && withTemporalRIS && withSpatialRIS) {
            if ((sampleVis & SV_T_PASSED) && (sampleVis & SV_ST_PASSED)) {
                if (temporalSampleIsValid) {
                    q[5].want = true; q[5].org = stNbPositionInWorld; q[5].ls = temporalSample; q[5].mask = SV_T_ON_ST;
                }
                if (spatiotemporalSampleIsValid) {
                    q[6].want = true; q[6].org = tNbPositionInWorld; q[6].ls = spatiotemporalSample; q[6].mask = SV_ST_ON_T;
                }
            }
        }
        r.sampleVis[curBufIdx][pix] = sampleVis; // the visibility bits are OR-ed in by the trace kernel
    }

    enqueueShadow(s, r, lane, pix, q[0]);
    if (withTemporalRIS) {
        enqueueShadow(s, r, lane, pix, q[1]);
        if (useUnbiasedEstimator)
            enqueueShadow(s, r, lane, pix, q[2]);
    }
    if (withSpatialRIS) {
        enqueueShadow(s, r, lane, pix, q[3]);
        if (useUnbiasedEstimator)
            enqueueShadow(s, r, lane, pix, q[4]);
    }
    if (useUnbiasedEstimator && withTemporalRIS && withSpatialRIS) {
        enqueueShadow(s, r, lane, pix, q[5]);
        enqueueShadow(s, r, lane, pix, q[6]);
    }
}

struct SampleVisibilityWriter {
    const uint32_t* rayPixel;
    const uint32_t* rayMask;
    uint32_t* sampleVis;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        if (st.best.storageIndex == 0xFFFFFFFFu)
            atomicOr(sampleVis + __ldg(rayPixel + ray), __ldg(rayMask + ray));
    }
};

enum class SampleType { New = 0, Temporal, Spatiotemporal };

// optix_restir_di_rearch_kernels.cu:263-400 with useMIS_RIS = true
template <SampleType sampleType, bool withTemporalRIS, bool withSpatialRIS>
GFX_D float computeMISWeight(const DevScene &s, const DevFrame &f, const DevFrameParams &p, uint32_t prevBufIdx, uint32_t prevResIndex,
                             uint32_t maxPrevStreamLength, uint32_t sampleVis, uint32_t selfStreamLength, const RearchShadingPoint &sp,
                             int tNbX, int tNbY, int stNbX, int stNbY, uint32_t streamLength, const LightSample &lightSample,
                             float sampleTargetDensity) {
    const float numMisWeight = sampleTargetDensity;
    float denomMisWeight = numMisWeight * streamLength;

    if (sampleType != SampleType::New) {
        const f3 cont = performDirectLighting<false>(s, sp.positionInWorld, sp.vOutLocal, sp.shadingFrame, sp.bsdf, lightSample);
        float targetDensity = convertToWeight(cont);
        if (p.useUnbiasedEstimator)
            targetDensity *= sampleType == SampleType::Temporal ? ((sampleVis & SV_T_ON_CUR) ? 1 : 0) : ((sampleVis & SV_ST_ON_CUR) ? 1 : 0);
        denomMisWeight += targetDensity * selfStreamLength;
    }
    if (sampleType != SampleType::Temporal && withTemporalRIS) {
        if (sampleVis & SV_T_PASSED) {
            const size_t nbPix = (size_t)tNbY * f.W + tNbX;
            const RearchShadingPoint nb = reconstructShadingPoint(s, f, prevBufIdx, nbPix, p.prevCamera.position);
            const f3 cont = performDirectLighting<false>(s, nb.positionInWorld, nb.vOutLocal, nb.shadingFrame, nb.bsdf, lightSample);
            float nbTargetDensity = convertToWeight(cont);
            if (p.useUnbiasedEstimator)
                nbTargetDensity *= sampleType == SampleType::New ? ((sampleVis & SV_NEW_ON_T) ? 1 : 0) : ((sampleVis & SV_ST_ON_T) ? 1 : 0);
            const uint32_t nbM = __float_as_uint(f.reservoir[prevResIndex][(size_t)f.W * f.H + nbPix].w) & 0x7FFFFFFFu;
            const uint32_t nbStreamLength = min(nbM, maxPrevStreamLength);
            denomMisWeight += nbTargetDensity * nbStreamLength;
        }
    }
    if (sampleType != SampleType::Spatiotemporal && withSpatialRIS) {
        if (sampleVis & SV_ST_PASSED) {
            const size_t nbPix = (size_t)stNbY * f.W + stNbX;
            const RearchShadingPoint nb = reconstructShadingPoint(s, f, prevBufIdx, nbPix, p.prevCamera.position);
            const f3 cont = performDirectLighting<false>(s, nb.positionInWorld, nb.vOutLocal, nb.shadingFrame, nb.bsdf, lightSample);
            float nbTargetDensity = convertToWeight(cont);
            if (p.useUnbiasedEstimator)
                nbTargetDensity *= sampleType == SampleType::New ? ((sampleVis & SV_NEW_ON_ST) ? 1 : 0) : ((sampleVis & SV_T_ON_ST) ? 1 : 0);
            const uint32_t nbM = __float_as_uint(f.reservoir[prevResIndex][(size_t)f.W * f.H + nbPix].w) & 0x7FFFFFFFu;
            const uint32_t nbStreamLength = min(nbM, maxPrevStreamLength);
            denomMisWeight += nbTargetDensity * nbStreamLength;
        }
    }
    return numMisWeight / denomMisWeight;
}

// optix_restir_di_rearch_kernels.cu:402-664
template <bool withTemporalRIS, bool withSpatialRIS>
__global__ void __launch_bounds__(64) k_shadeAndResample(DevScene s, DevFrame f, DevFrameParams p, DevRearch r) {
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    if (x >= f.W || y >= p.y1)
        return;
    const size_t pix = (size_t)y * f.W + x;
    const uint32_t curBufIdx = p.bufferIndex, prevBufIdx = (curBufIdx + 1) % 2;
    const uint32_t curResIndex = p.currentReservoirIndex, prevResIndex = (curResIndex + 1) % 2;
    const uint4 gb0 = f.gb0[curBufIdx][pix];
    const uint4 gb3 = f.gb3[curBufIdx][pix];

    f3 contribution(0.01f, 0.01f, 0.01f);
    if (gb0.x != 0xFFFFFFFFu) {
        PCG32RNG rng{ f.rng[pix] };
        int tNbX = 0, tNbY = 0, stNbX = 0, stNbY = 0;
        if (withTemporalRIS)
            temporalNeighborCoord(f, curBufIdx, pix, x, y, &tNbX, &tNbY);
        if (withSpatialRIS) {
            float deltaX, deltaY;
            spatialNeighborCoord(f, p, x, y, rng, &stNbX, &stNbY, &deltaX, &deltaY);
        }
        const RearchShadingPoint sp = reconstructShadingPoint(s, f, curBufIdx, pix, p.camera.position);
        const GfxMaterialDesc* mat = s.materials + gb3.w;

        contribution = f3(0.0f);
        if (sp.vOutLocal.z > 0) {
            f3 emittance(0.0f);
            if (mat->hasEmittance)
                emittance = f3(mat->emittance[0], mat->emittance[1], mat->emittance[2]);
            contribution += emittance / kPi;
        }

        uint32_t sampleVis = r.sampleVis[curBufIdx][pix];
        float selectedTargetDensity = 0.0f;
        Reservoir combinedReservoir;
        uint32_t combinedStreamLength = 0;
        combinedReservoir.initialize(emptyLightSample());
        f3 directCont(0.0f);
        float selectedMisWeight = 0.0f;

        const Reservoir selfRes = loadReservoir(f, curResIndex, pix);
        const float2 selfResInfo = f.reservoirInfo[curResIndex][pix];
        const uint32_t selfStreamLength = selfRes.streamLength;
        const uint32_t maxPrevStreamLength = 20 * selfStreamLength;

        // new sample of the current pixel
        {
            if (selfResInfo.x > 0.0f && (sampleVis & SV_NEW)) {
                const LightSample lightSample = selfRes.sample;
                const f3 cont = performDirectLighting<false>(s, sp.positionInWorld, sp.vOutLocal, sp.shadingFrame, sp.bsdf, lightSample);
                const float targetDensity = convertToWeight(cont);
                float misWeight;
                if (withTemporalRIS || withSpatialRIS)
                    misWeight = computeMISWeight<SampleType::New, withTemporalRIS, withSpatialRIS>(
                        s, f, p, prevBufIdx, prevResIndex, maxPrevStreamLength, sampleVis, selfStreamLength, sp,
                        tNbX, tNbY, stNbX, stNbY, selfStreamLength, lightSample, selfResInfo.y);
                else
                    misWeight = 1.0f / selfStreamLength;
                directCont += (misWeight * selfResInfo.x * selfStreamLength) * cont;
                combinedReservoir = selfRes;
                selectedTargetDensity = targetDensity;
                selectedMisWeight = misWeight;
                sampleVis |= SV_SELECTED; // selectedSample = newSample (set in this branch)
            }
            combinedStreamLength = selfStreamLength;
        }

        if (withTemporalRIS) {
            if (sampleVis & SV_T_PASSED) {
                const size_t nbPix = (size_t)tNbY * f.W + tNbX;
                const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
                const float2 neighborInfo = f.reservoirInfo[prevResIndex][nbPix];
                const uint32_t nbStreamLength = min(neighbor.streamLength, maxPrevStreamLength);
                if (neighborInfo.x > 0.0f) {
                    const LightSample nbLightSample = neighbor.sample;
                    const f3 cont = performDirectLighting<false>(s, sp.positionInWorld, sp.vOutLocal, sp.shadingFrame, sp.bsdf, nbLightSample);
                    const float targetDensity = convertToWeight(cont);
                    const float misWeight = computeMISWeight<SampleType::Temporal, withTemporalRIS, withSpatialRIS>(
                        s, f, p, prevBufIdx, prevResIndex, maxPrevStreamLength, sampleVis, selfStreamLength, sp,
                        tNbX, tNbY, stNbX, stNbY, nbStreamLength, nbLightSample, neighborInfo.y);
                    const float weight = targetDensity * neighborInfo.x * nbStreamLength;
                    const uint32_t visBit = (sampleVis & SV_T) ? 1u : 0u;
                    directCont += (visBit * misWeight * neighborInfo.x * nbStreamLength) * cont;
                    if (combinedReservoir.update(nbLightSample, weight, rng.getFloat0cTo1o())) {
                        selectedTargetDensity = targetDensity;
                        selectedMisWeight = misWeight;
                        sampleVis = visBit ? (sampleVis | SV_SELECTED) : (sampleVis & ~SV_SELECTED);
                    }
                }
                combinedStreamLength += nbStreamLength;
            }
        }
        if (withSpatialRIS) {
            if (sampleVis & SV_ST_PASSED) {
                const size_t nbPix = (size_t)stNbY * f.W + stNbX;
                const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
                const float2 neighborInfo = f.reservoirInfo[prevResIndex][nbPix];
                const uint32_t nbStreamLength = min(neighbor.streamLength, maxPrevStreamLength);
                if (neighborInfo.x > 0.0f) {
                    const LightSample nbLightSample = neighbor.sample;
                    const f3 cont = performDirectLighting<false>(s, sp.positionInWorld, sp.vOutLocal, sp.shadingFrame, sp.bsdf, nbLightSample);
                    const float targetDensity = convertToWeight(cont);
                    const float misWeight = computeMISWeight<SampleType::Spatiotemporal, withTemporalRIS, withSpatialRIS>(
                        s, f, p, prevBufIdx, prevResIndex, maxPrevStreamLength, sampleVis, selfStreamLength, sp,
                        tNbX, tNbY, stNbX, stNbY, nbStreamLength, nbLightSample, neighborInfo.y);
                    const float weight = targetDensity * neighborInfo.x * nbStreamLength;
                    const uint32_t visBit = (sampleVis & SV_ST) ? 1u : 0u;
                    directCont += (visBit * misWeight * neighborInfo.x * nbStreamLength) * cont;
                    if (combinedReservoir.update(nbLightSample, weight, rng.getFloat0cTo1o())) {
                        selectedTargetDensity = targetDensity;
                        selectedMisWeight = misWeight;
                        sampleVis = visBit ? (sampleVis | SV_SELECTED) : (sampleVis & ~SV_SELECTED);
                    }
                }
                combinedStreamLength += nbStreamLength;
            }
        }

        combinedReservoir.streamLength = combinedStreamLength;
        contribution += directCont;

        float recPDFEstimate = selectedMisWeight * combinedReservoir.sumWeights / selectedTargetDensity;
        if (!isfinite(recPDFEstimate) || (p.reuseVisibility && !(sampleVis & SV_SELECTED))) {
            recPDFEstimate = 0.0f;
            selectedTargetDensity = 0.0f;
        }
        r.sampleVis[curBufIdx][pix] = sampleVis;
        storeReservoir(f, curResIndex, pix, combinedReservoir);
        f.reservoirInfo[curResIndex][pix] = make_float2(recPDFEstimate, selectedTargetDensity);
        f.rng[pix] = rng.state;
    }
    else if (s.env.enabled) { // optix_restir_di_rearch_kernels.cu:648-656: the environment seen directly
        const f2 texCoord = decodeTexCoords(gb3.z);
        contribution = s.env.powerCoeff * envFetch(s.env, texCoord.x, texCoord.y);
    }

    f3 prevColorResult(0.0f);
    if (p.numAccumFrames > 0) {
        const float4 pb = f.beauty[pix];
        prevColorResult = f3(pb.x, pb.y, pb.z);
    }
    const float curWeight = 1.0f / (1 + p.numAccumFrames);
    const f3 colorResult = (1 - curWeight) * prevColorResult + curWeight * contribution;
    f.beauty[pix] = make_float4(colorResult.x, colorResult.y, colorResult.z, 1.0f);
}

int launchReSTIRRearch(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params, int pass) {
    DevFrameParams p = makeDevParams(ctx, params);
    if (p.y1 <= p.y0)
        return GFX_OK;
    if (p.y0 % 8 != 0) {
        ctx->setError("rearchitected ReSTIR: tileOriginY must be a multiple of the 8x8 light-subset tile");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    if (p.log2NumCandidateSamples > 15)
        return GFX_ERR_INVALID_ARGUMENT;
    const bool T = params->enableTemporalReuse != 0, S = params->enableSpatialReuse != 0, U = params->useUnbiasedEstimator != 0;
    const int rc = ensureRearch(ctx, pass == GFX_RESTIR_TRACE_SHADOW_RAYS ? (U ? 7u : 3u) : 0u);
    if (rc != GFX_OK)
        return rc;
    const dim3 block(8, 8);
    const dim3 grid((ctx->frame.W + 7) / 8, (p.y1 - p.y0 + 7) / 8);
    const DevScene s = ctx->devScene(params);
    const DevFrame f = ctx->devFrame();
    const DevRearch r = makeDevRearch(ctx);
    switch (pass) {
    case GFX_RESTIR_PRESAMPLE_LIGHTS: {
        GFX_TIMED(ctx, stream, "rearch_presample_lights");
        k_presampleLights<<<kNumPreSampledLights / 128, 128, 0, stream>>>(s, r);
        ctx->launches++;
    } break;
    case GFX_RESTIR_PER_PIXEL_RIS: {
        GFX_TIMED(ctx, stream, "rearch_per_pixel_ris");
        k_perPixelRIS<<<grid, block, 0, stream>>>(s, f, p, r);
        ctx->launches++;
    } break;
    case GFX_RESTIR_TRACE_SHADOW_RAYS: {
        GFX_CUDA(ctx, cudaMemsetAsync(r.counters, 0, 8, stream));
        {
            GFX_TIMED(ctx, stream, "rearch_shadow_requests");
            if (!T && !S) k_shadowRayRequests<false, false, false><<<grid, block, 0, stream>>>(s, f, p, r);
            else if (T && !S && !U) k_shadowRayRequests<true, false, false><<<grid, block, 0, stream>>>(s, f, p, r);
            else if (!T && S && !U) k_shadowRayRequests<false, true, false><<<grid, block, 0, stream>>>(s, f, p, r);
            else if (T && S && !U) k_shadowRayRequests<true, true, false><<<grid, block, 0, stream>>>(s, f, p, r);
            else if (T && !S && U) k_shadowRayRequests<true, false, true><<<grid, block, 0, stream>>>(s, f, p, r);
            else if (!T && S && U) k_shadowRayRequests<false, true, true><<<grid, block, 0, stream>>>(s, f, p, r);
            else k_shadowRayRequests<true, true, true><<<grid, block, 0, stream>>>(s, f, p, r);
        }
        {
            GFX_TIMED(ctx, stream, "rearch_trace_shadow");
            const SampleVisibilityWriter w{ r.rayPixel, r.rayMask, r.sampleVis[p.bufferIndex] };
            // postponed leaf tests: 1.84 -> 1.60 ms biased, 6.21 -> 5.29 ms unbiased on config 2 against immediate ones
            k_traceWavefrontDeferred<true, false><<<wavefrontGrid(), 128, 0, stream>>>(s.bvh, r.rays, r.counters, 0u, r.counters + 1, w);
        }
        ctx->launches += 2;
    } break;
    case GFX_RESTIR_SHADE_AND_RESAMPLE: {
        GFX_TIMED(ctx, stream, "rearch_shade_and_resample");
        if (!T && !S) k_shadeAndResample<false, false><<<grid, block, 0, stream>>>(s, f, p, r);
        else if (T && !S) k_shadeAndResample<true, false><<<grid, block, 0, stream>>>(s, f, p, r);
        else if (!T && S) k_shadeAndResample<false, true><<<grid, block, 0, stream>>>(s, f, p, r);
        else k_shadeAndResample<true, true><<<grid, block, 0, stream>>>(s, f, p, r);
        ctx->launches++;
    } break;
    default:
        ctx->setError("gfx_restir_launch: unknown pass");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

} // namespace gfx
