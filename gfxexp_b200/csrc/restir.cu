// restir.cu — ReSTIR DI passes as sm_100a kernels.
//
// Replaces restir.optixPipeline.launch(W, H, 1) with the ray-generation entry points
// performInitialRIS / performInitialAndTemporalRIS{Biased,Unbiased} / performSpatialRIS{Biased,
// Unbiased} / shading (restir_di/gpu_kernels/optix_restir_di_kernels.cu:14-287, 303-547, 559-637;
// launch sites restir_di/restir_di_main.cpp:2378-2421) and the helpers they share
// (sampleLight<false> restir_di_shared.h:320-516, performDirectLighting :518-557,
// evaluateVisibility :559-582, testNeighbor :747-771).  Visibility rays run through the inline
// any-hit traversal of traverse.cuh instead of optixTrace + the AH program.
//
// Per-pixel state is SoA: reservoirs are three float4 planes (Le|sumW, pos|M, n|-) so a pixel's own
// reservoir is three coalesced 16-byte loads; neighbour gathers hit the same planes through L2.
// RNG draw order per pixel is the reference's (SURVEY.md Appendix A.3).
#include "restir_common.cuh"

namespace gfx {

// PHASE 0: the whole program in one kernel (megakernel form of the reference), for frames without visibility reuse.
// PHASE 1: candidates + recPDF, the visibility ray is only *requested* (wavefront form).
// PHASE 2: applies the answered visibility, then the temporal merge.
//
// PHASE 1 without an environment light runs the candidate loop in two phases (kRisTwoPhase); PHASE 0 and frames with an
// environment light, whose candidates choose their light type by index, run it in lock step.
// ncu on the lock-step loop (round 2, profiles/r02_summary.md):
// ~70 % of the candidates are dark and leave after the staged light fetch, so everything after the bounding-sphere test - 74 %
// of the kernel's issue slots - ran with 9-16 of 32 lanes.  Phase A walks all 2^n candidates in lock step but only draws ul,
// picks the light and tests its bounding sphere (the other three draws of a candidate are skipped with the LCG's 4-step
// jump), leaving per lane a bit mask of survivors and their keys in shared memory.  Phase B is a per-lane loop over the
// lane's own survivors, in candidate order: the PCG32 state at the candidate is rebuilt from the jump table, u0 / u1 / u
// are drawn, and the candidate runs steps 1-2 of the light fetch, the BSDF and the reservoir update exactly as in the
// lock-step loop.  A warp then iterates max-over-lanes(#survivors) ~ 20 times instead of 32, with the expensive part at
// ~70 % instead of 30 % lane utilisation; each pixel still sees the reference's sequence of Reservoir::update calls
// (restir_di_shared.h:118-125) and draws, so results are bit-identical.
constexpr uint32_t kRisMaxCandidates = 32; // the two-phase loop keeps one key per candidate and thread in shared memory
template <int PHASE, bool ENV>
constexpr bool kRisTwoPhase = PHASE == 1 && !ENV;

template <bool withTemporalRIS, bool useUnbiasedEstimator, int PHASE, bool ENV>
GFX_D bool risPixel(const DevScene &s, const DevFrame &f, const DevFrameParams &p, RayRequest* request, uint32_t* candidateKeys) {
    // optix_restir_di_kernels.cu:14-287
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    if (x >= f.W || y >= p.y1)
        return false;
    const size_t pix = (size_t)y * f.W + x;
    const uint32_t curBufIdx = p.bufferIndex;

    const uint4 gb0 = f.gb0[curBufIdx][pix];
    if (gb0.x == 0xFFFFFFFFu)
        return false;
    const float4 gb2 = f.gb2[curBufIdx][pix];
    const uint4 gb3 = f.gb3[curBufIdx][pix];

    f3 positionInWorld(gb2.x, gb2.y, gb2.z);
    const f3 geometricNormalInWorld = decodeVector(__float_as_uint(gb2.w));

    PCG32RNG rng{ f.rng[pix] };

    f3 vOut = p.camera.position - positionInWorld;
    const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
    positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);
    const float dist = length(vOut);
    vOut /= dist;

    const f3 shadingNormalInWorld = decodeVector(gb3.x);
    const f3 shadingTangentInWorld = decodeVector(gb3.y);
    const ReferenceFrame shadingFrame(shadingNormalInWorld, shadingTangentInWorld);
    const f3 vOutLocal = shadingFrame.toLocal(vOut);
    const BSDF bsdf = setupBsdf(s, gb3.w, decodeTexCoords(gb3.z));

    const uint32_t curResIndex = p.currentReservoirIndex;
    Reservoir reservoir;
    reservoir.initialize(emptyLightSample());

    float selectedTargetDensity = 0.0f;
    float recPDFEstimate = 0.0f;
    if (PHASE != 2) {
    const uint32_t numCandidates = 1u << p.log2NumCandidateSamples;
    // Streaming RIS (:66-123).  Reservoir::update (restir_di_shared.h:118-125) is spelled out: instead of
    // copying the 10-float LightSample on every acceptance, the three primary sample values that
    // generated it are kept and the winner is re-generated once after the loop (sampleLight is a pure
    // function of (ul, u0, u1)), which is bit-identical and frees registers in the hot loop.
    float selUl = 0.0f, selU0 = 0.0f, selU1 = 0.0f;
    bool hasSelection = false;
    bool selEnv = false; // ENV: the selected candidate came from the environment map
    float sumWeights = 0.0f;
    if (kRisTwoPhase<PHASE, ENV> && numCandidates <= kRisMaxCandidates) {
        uint32_t* myKeys = candidateKeys + (threadIdx.x + threadIdx.y * blockDim.x); // [candidate][64 threads]
        const uint64_t state0 = rng.state;
        // ---- phase A: ul, light pick, bounding sphere
        // (two candidates per trip so that two guide reads are in flight: the loop is a chain of dependent L2 round trips)
        uint32_t survivors = 0;
        for (uint32_t i = 0; i < numCandidates; i += 2) {
            const float ulA = pcg32Float(rng.state);
            rng.state = rng.state * kPcg32Jump4.mul[1] + kPcg32Jump4.add[1]; // the candidate's four draws
            const float ulB = pcg32Float(rng.state);
            const F8 gA = pickGuideFetch(s, ulA);
            const F8 gB = pickGuideFetch(s, ulB);
            const uint32_t codeA = classifyLight(s, ulA, gA, positionInWorld, shadingNormalInWorld, vOutLocal.z);
            myKeys[i * 64] = codeA;
            survivors |= codeA != kLightDark ? (1u << i) : 0u;
            if (i + 1 < numCandidates) {
                rng.state = rng.state * kPcg32Jump4.mul[1] + kPcg32Jump4.add[1];
                const uint32_t codeB = classifyLight(s, ulB, gB, positionInWorld, shadingNormalInWorld, vOutLocal.z);
                myKeys[(i + 1) * 64] = codeB;
                survivors |= codeB != kLightDark ? (2u << i) : 0u;
            }
        }
        // ---- phase B: this lane's survivors, in candidate order
        uint32_t selIdx = 0;
        while (survivors) {
            const uint32_t i = (uint32_t)__ffs((int)survivors) - 1u;
            survivors &= survivors - 1u;
            const uint32_t code = myKeys[i * 64];
            uint64_t st = state0 * __ldg(&kPcg32Jump4.mul[i]) + __ldg(&kPcg32Jump4.add[i]); // state before the candidate's ul
            st = st * 6364136223846793005ULL + 1;
            const float u0 = pcg32Float(st);
            st = st * 6364136223846793005ULL + 1;
            const float u1 = pcg32Float(st);
            st = st * 6364136223846793005ULL + 1;
            LightSample lightSample = emptyLightSample();
            float probDensity;
            if (finishLightSample(s, code, u0, u1, positionInWorld, shadingNormalInWorld, vOutLocal.z, &lightSample, &probDensity))
                continue;
            const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample);
            const bool deadCont = cont.x == 0.0f && cont.y == 0.0f && cont.z == 0.0f;
            if (deadCont && probDensity > 0.0f)
                continue;
            const float targetDensity = convertToWeight(cont);
            const float weight = targetDensity / probDensity;
            const float u = pcg32Float(st);
            sumWeights += weight;
            if (u < weight / sumWeights) {
                selIdx = i;
                hasSelection = true;
                selectedTargetDensity = targetDensity;
            }
        }
        if (hasSelection) { // the winner's three primary sample values, from the stream position of its candidate
            uint64_t st = state0 * __ldg(&kPcg32Jump4.mul[selIdx]) + __ldg(&kPcg32Jump4.add[selIdx]);
            selUl = pcg32Float(st);
            st = st * 6364136223846793005ULL + 1;
            selU0 = pcg32Float(st);
            st = st * 6364136223846793005ULL + 1;
            selU1 = pcg32Float(st);
        }
    }
    else {
    for (uint32_t i = 0; i < numCandidates; ++i) {
        float ul = rng.getFloat0cTo1o();
        float probToSampleCurLightType = 1.0f;
        // with an environment light the first probToSampleEnvLight * numCandidates candidates sample it (:72-90)
        bool sampleEnv = false;
        if (ENV)
            sampleEnv = chooseEnvForCandidate(s, i, numCandidates, &ul, &probToSampleCurLightType);
        LightSample lightSample = emptyLightSample();
        float probDensity;
        const float u0 = rng.getFloat0cTo1o();
        const float u1 = rng.getFloat0cTo1o();
        if (ENV && sampleEnv) {
            sampleEnvLight(s, u0, u1, &lightSample, &probDensity);
        }
        // staged fetch of the light triangle: certainly-dark candidates stop early (their contribution is exactly
        // RGB(0): the reservoir is untouched and only the acceptance draw is consumed, as in the dead path below)
        else if (sampleLightUnlessDark(s, ul, u0, u1, positionInWorld, shadingNormalInWorld, vOutLocal.z, &lightSample, &probDensity)) {
            (void)rng.getFloat0cTo1o();
            continue;
        }
        probDensity *= probToSampleCurLightType;
        // Dead candidates (light faces away, or lies below the shading horizon: ~70 % of them) contribute exactly
        // RGB(0) (performDirectLighting returns RGB(0) before any arithmetic when lpCos <= 0, and the BRDFs
        // return RGB(0) when vGiven.z * vSampled.z <= 0), so weight = +0 / probDensity = +0 and the reservoir
        // is untouched: skip the three IEEE divisions, which would all take the 0/x slow path.
        const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample);
        const bool deadCont = cont.x == 0.0f && cont.y == 0.0f && cont.z == 0.0f;
        if (deadCont && probDensity > 0.0f) {
            (void)rng.getFloat0cTo1o();
            continue;
        }
        const float targetDensity = convertToWeight(cont);
        const float weight = targetDensity / probDensity;
        const float u = rng.getFloat0cTo1o();
        sumWeights += weight;
        if (u < weight / sumWeights) {
            selUl = ul;
            selU0 = u0;
            selU1 = u1;
            selEnv = ENV && sampleEnv;
            hasSelection = true;
            selectedTargetDensity = targetDensity;
        }
    }
    }
    if (hasSelection) {
        float unusedDensity;
        if (ENV && selEnv)
            sampleEnvLight(s, selU0, selU1, &reservoir.sample, &unusedDensity);
        else
            sampleLight(s, selUl, selU0, selU1, &reservoir.sample, &unusedDensity);
    }
    reservoir.sumWeights = sumWeights;
    reservoir.streamLength = numCandidates;

    recPDFEstimate = reservoir.sumWeights / (selectedTargetDensity * reservoir.streamLength);
    if (!isfinite(recPDFEstimate)) {
        recPDFEstimate = 0.0f;
        selectedTargetDensity = 0.0f;
    }
    }
    else { // PHASE 2: pick up where phase 1 stopped
        reservoir = loadReservoir(f, curResIndex, pix);
        const float2 info = f.reservoirInfo[curResIndex][pix];
        recPDFEstimate = info.x;
        selectedTargetDensity = info.y;
    }

    if (p.reuseVisibility && selectedTargetDensity > 0.0f) {
        if (PHASE == 1) {
            visibilityRay(positionInWorld, reservoir.sample, (uint32_t)pix, request);
            f.rng[pix] = rng.state;
            storeReservoir(f, curResIndex, pix, reservoir);
            f.reservoirInfo[curResIndex][pix] = make_float2(recPDFEstimate, selectedTargetDensity);
            return true;
        }
        const bool visible = PHASE == 2 ? (f.visibility[pix] != 0) : evaluateVisibility(s, positionInWorld, reservoir.sample);
        if (!visible) {
            recPDFEstimate = 0.0f;
            selectedTargetDensity = 0.0f;
        }
    }
    if (PHASE == 1) {
        f.rng[pix] = rng.state;
        storeReservoir(f, curResIndex, pix, reservoir);
        f.reservoirInfo[curResIndex][pix] = make_float2(recPDFEstimate, selectedTargetDensity);
        return false;
    }

    if (withTemporalRIS) {
        const uint32_t prevBufIdx = (curBufIdx + 1) % 2;
        const uint32_t prevResIndex = (curResIndex + 1) % 2;

        bool neighborIsSelected = false;
        const uint32_t selfStreamLength = reservoir.streamLength;
        if (recPDFEstimate == 0.0f)
            reservoir.initialize(emptyLightSample());
        uint32_t combinedStreamLength = selfStreamLength;
        const uint32_t maxPrevStreamLength = 20 * selfStreamLength;

        const float2 gb1 = f.gb1[curBufIdx][pix];
        const int nbx = dm_f2int(x + 0.5f - gb1.x);
        const int nby = dm_f2int(y + 0.5f - gb1.y);

        const bool acceptedNeighbor = testNeighbor<!useUnbiasedEstimator>(f, p.camera, prevBufIdx, nbx, nby, dist, shadingNormalInWorld);
        if (acceptedNeighbor) {
            const size_t nbPix = (size_t)nby * f.W + nbx;
            const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
            const float2 neighborInfo = f.reservoirInfo[prevResIndex][nbPix];
            const LightSample nbLightSample = neighbor.sample;
            const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, nbLightSample);
            const float targetDensity = convertToWeight(cont);
            const uint32_t nbStreamLength = min(neighbor.streamLength, maxPrevStreamLength);
            const float weight = targetDensity * neighborInfo.x * nbStreamLength;
            if (reservoir.update(nbLightSample, weight, rng.getFloat0cTo1o())) {
                selectedTargetDensity = targetDensity;
                if (useUnbiasedEstimator)
                    neighborIsSelected = true;
            }
            combinedStreamLength += nbStreamLength;
        }
        reservoir.streamLength = combinedStreamLength;

        float weightForEstimate;
        if (useUnbiasedEstimator) { // :192-266, useMIS_RIS = true
            const LightSample selectedLightSample = reservoir.sample;
            float numWeight, denomWeight;
            {
                const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, selectedLightSample);
                const float targetDensityForSelf = convertToWeight(cont);
                numWeight = targetDensityForSelf;
                denomWeight = targetDensityForSelf * selfStreamLength;
            }
            if (acceptedNeighbor) {
                const size_t nbPix = (size_t)nby * f.W + nbx;
                const float4 nbGb2 = f.gb2[prevBufIdx][nbPix];
                const uint4 nbGb3 = f.gb3[prevBufIdx][nbPix];
                f3 nbPositionInWorld(nbGb2.x, nbGb2.y, nbGb2.z);
                const f3 nbGeometricNormalInWorld = decodeVector(__float_as_uint(nbGb2.w));
                const f3 nbVOut = normalize(p.prevCamera.position - nbPositionInWorld);
                const float nbFrontHit = dot(nbVOut, nbGeometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
                nbPositionInWorld = offsetRayOrigin(nbPositionInWorld, nbFrontHit * nbGeometricNormalInWorld);
                const BSDF nbBsdf = setupBsdf(s, nbGb3.w, decodeTexCoords(nbGb3.z));
                const ReferenceFrame nbShadingFrame(decodeVector(nbGb3.x), decodeVector(nbGb3.y));
                const f3 nbVOutLocal = nbShadingFrame.toLocal(nbVOut);
                const Reservoir neighbor = loadReservoir(f, prevResIndex, nbPix);
                const f3 cont = performDirectLighting<false>(s, nbPositionInWorld, nbVOutLocal, nbShadingFrame, nbBsdf, selectedLightSample);
                const float nbTargetDensity = convertToWeight(cont);
                const uint32_t nbStreamLength = min(neighbor.streamLength, maxPrevStreamLength);
                denomWeight += nbTargetDensity * nbStreamLength;
                if (neighborIsSelected)
                    numWeight = nbTargetDensity;
            }
            weightForEstimate = numWeight / denomWeight;
        }
        else {
            weightForEstimate = 1.0f / reservoir.streamLength;
        }

        recPDFEstimate = weightForEstimate * reservoir.sumWeights / selectedTargetDensity;
        if (!isfinite(recPDFEstimate)) {
            recPDFEstimate = 0.0f;
            selectedTargetDensity = 0.0f;
        }
    }

    f.rng[pix] = rng.state;
    storeReservoir(f, curResIndex, pix, reservoir);
    f.reservoirInfo[curResIndex][pix] = make_float2(recPDFEstimate, selectedTargetDensity);
    return false;
}

constexpr int kRisMinBlocks = 16; // 64 registers: measured 1.49 ms against 1.80 ms at the 84 registers ptxas picks unconstrained (profiles/r02_summary.md)
template <bool withTemporalRIS, bool useUnbiasedEstimator, int PHASE, bool ENV = false>
__global__ void __launch_bounds__(64, kRisMinBlocks) k_initialAndTemporalRIS(DevScene s, DevFrame f, DevFrameParams p) {
    RayRequest request;
    uint32_t* candidateKeys = nullptr;
    if constexpr (kRisTwoPhase<PHASE, ENV>) {
        __shared__ uint32_t keys[kRisMaxCandidates * 64]; // [candidate][thread of the 8x8 block]
        candidateKeys = keys;
    }
    const bool want = risPixel<withTemporalRIS, useUnbiasedEstimator, PHASE, ENV>(s, f, p, &request, candidateKeys);
    if (PHASE == 1)
        enqueueRay(f, s.rayCounter, want, request);
}

// ---------------------------------------------------------------------------------------------
GFX_D void neighborCoord(const DevFrame &f, const DevFrameParams &p, uint32_t x, uint32_t y, int nIdx, PCG32RNG &rng,
                         int* nbx, int* nby) { // optix_restir_di_kernels.cu:356-371
    float radius = p.spatialNeighborRadius;
    float deltaX, deltaY;
    if (p.useLowDiscrepancyNeighbors) {
        const float2 delta = __ldg(f.neighborDeltas + ((p.spatialNeighborBaseIndex + nIdx) % 1024));
        deltaX = radius * delta.x;
        deltaY = radius * delta.y;
    }
    else {
        radius *= sqrtf(rng.getFloat0cTo1o());
        const float angle = 2 * kPi * rng.getFloat0cTo1o();
        float sa, ca;
        dm_sincos(angle, &sa, &ca);
        deltaX = radius * ca;
        deltaY = radius * sa;
    }
    *nbx = dm_f2int(x + 0.5f + deltaX);
    *nby = dm_f2int(y + 0.5f + deltaY);
}

template <bool useUnbiasedEstimator>
__global__ void __launch_bounds__(64) k_spatialRIS(DevScene s, DevFrame f, DevFrameParams p) {
    // optix_restir_di_kernels.cu:303-547
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    if (x >= f.W || y >= p.y1)
        return;
    const size_t pix = (size_t)y * f.W + x;
    const uint32_t bufIdx = p.bufferIndex;

    const uint4 gb0 = f.gb0[bufIdx][pix];
    if (gb0.x == 0xFFFFFFFFu)
        return;
    const float4 gb2 = f.gb2[bufIdx][pix];
    const uint4 gb3 = f.gb3[bufIdx][pix];

    f3 positionInWorld(gb2.x, gb2.y, gb2.z);
    const f3 geometricNormalInWorld = decodeVector(__float_as_uint(gb2.w));
    PCG32RNG rng{ f.rng[pix] };

    f3 vOut = p.camera.position - positionInWorld;
    const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
    positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);
    const float dist = length(vOut);
    vOut /= dist;

    const ReferenceFrame shadingFrame(decodeVector(gb3.x), decodeVector(gb3.y));
    const f3 vOutLocal = shadingFrame.toLocal(vOut);
    const BSDF bsdf = setupBsdf(s, gb3.w, decodeTexCoords(gb3.z));

    const uint32_t srcResIndex = p.currentReservoirIndex;
    const uint32_t dstResIndex = (srcResIndex + 1) % 2;

    Reservoir combinedReservoir;
    combinedReservoir.initialize(emptyLightSample());
    float selectedTargetDensity = 0.0f;
    int32_t selectedNeighborIndex = -1;

    const Reservoir self = loadReservoir(f, srcResIndex, pix);
    const float2 selfResInfo = f.reservoirInfo[srcResIndex][pix];
    if (selfResInfo.x > 0.0f) {
        combinedReservoir = self;
        selectedTargetDensity = selfResInfo.y;
    }
    uint32_t combinedStreamLength = self.streamLength;

    for (int nIdx = 0; nIdx < (int)p.numSpatialNeighbors; ++nIdx) {
        int nbx, nby;
        neighborCoord(f, p, x, y, nIdx, rng, &nbx, &nby);
        const bool acceptedNeighbor =
            testNeighbor<!useUnbiasedEstimator>(f, p.camera, bufIdx, nbx, nby, dist, shadingFrame.normal)
            && (nbx != (int)x || nby != (int)y);
        if (acceptedNeighbor) {
            const size_t nbPix = (size_t)nby * f.W + nbx;
            const Reservoir neighbor = loadReservoir(f, srcResIndex, nbPix);
            const float2 neighborInfo = f.reservoirInfo[srcResIndex][nbPix];
            const LightSample nbLightSample = neighbor.sample;
            const f3 cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, nbLightSample);
            const float targetDensity = convertToWeight(cont);
            const uint32_t nbStreamLength = neighbor.streamLength;
            const float weight = targetDensity * neighborInfo.x * nbStreamLength;
            if (combinedReservoir.update(nbLightSample, weight, rng.getFloat0cTo1o())) {
                selectedTargetDensity = targetDensity;
                if (useUnbiasedEstimator)
                    selectedNeighborIndex = nIdx;
            }
            combinedStreamLength += nbStreamLength;
        }
    }
    combinedReservoir.streamLength = combinedStreamLength;

    float weightForEstimate = 0.0f;
    if (useUnbiasedEstimator) { // :414-529
        if (selectedTargetDensity > 0.0f) {
            const LightSample selectedLightSample = combinedReservoir.sample;
            float numWeight, denomWeight;
            bool visibility = true;
            {
                f3 cont;
                if (p.reuseVisibility)
                    cont = performDirectLighting<true>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, selectedLightSample);
                else
                    cont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, selectedLightSample);
                const float targetDensityForSelf = convertToWeight(cont);
                if (p.reuseVisibility)
                    visibility = targetDensityForSelf > 0.0f;
                numWeight = targetDensityForSelf;
                denomWeight = targetDensityForSelf * self.streamLength;
            }
            for (int nIdx = 0; nIdx < (int)p.numSpatialNeighbors; ++nIdx) {
                int nbx, nby;
                neighborCoord(f, p, x, y, nIdx, rng, &nbx, &nby);
                const bool acceptedNeighbor =
                    (nbx >= 0 && nbx < (int)f.W && nby >= 0 && nby < (int)f.H) && (nbx != (int)x || nby != (int)y);
                if (acceptedNeighbor) {
                    const size_t nbPix = (size_t)nby * f.W + nbx;
                    if (f.gb0[bufIdx][nbPix].x == 0xFFFFFFFFu)
                        continue;
                    const float4 nbGb2 = f.gb2[bufIdx][nbPix];
                    const uint4 nbGb3 = f.gb3[bufIdx][nbPix];
                    f3 nbPositionInWorld(nbGb2.x, nbGb2.y, nbGb2.z);
                    const f3 nbGeometricNormalInWorld = decodeVector(__float_as_uint(nbGb2.w));
                    const f3 nbVOut = normalize(p.prevCamera.position - nbPositionInWorld);
                    const float nbFrontHit = dot(nbVOut, nbGeometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
                    nbPositionInWorld = offsetRayOrigin(nbPositionInWorld, nbFrontHit * nbGeometricNormalInWorld);
                    const BSDF nbBsdf = setupBsdf(s, nbGb3.w, decodeTexCoords(nbGb3.z));
                    const ReferenceFrame nbShadingFrame(decodeVector(nbGb3.x), decodeVector(nbGb3.y));
                    const f3 nbVOutLocal = nbShadingFrame.toLocal(nbVOut);
                    const Reservoir neighbor = loadReservoir(f, srcResIndex, nbPix);
                    f3 cont;
                    if (p.reuseVisibility)
                        cont = performDirectLighting<true>(s, nbPositionInWorld, nbVOutLocal, nbShadingFrame, nbBsdf, selectedLightSample);
                    else
                        cont = performDirectLighting<false>(s, nbPositionInWorld, nbVOutLocal, nbShadingFrame, nbBsdf, selectedLightSample);
                    const float nbTargetDensity = convertToWeight(cont);
                    const uint32_t nbStreamLength = neighbor.streamLength;
                    denomWeight += nbTargetDensity * nbStreamLength;
                    if (nIdx == selectedNeighborIndex)
                        numWeight = nbTargetDensity;
                }
            }
            weightForEstimate = numWeight / denomWeight;
            if (p.reuseVisibility && !visibility)
                weightForEstimate = 0.0f;
        }
    }
    else {
        weightForEstimate = 1.0f / combinedReservoir.streamLength;
    }

    float recPDFEstimate = weightForEstimate * combinedReservoir.sumWeights / selectedTargetDensity;
    float targetDensityOut = selectedTargetDensity;
    if (!isfinite(recPDFEstimate)) {
        recPDFEstimate = 0.0f;
        targetDensityOut = 0.0f;
    }

    f.rng[pix] = rng.state;
    storeReservoir(f, dstResIndex, pix, combinedReservoir);
    f.reservoirInfo[dstResIndex][pix] = make_float2(recPDFEstimate, targetDensityOut);
}

// ---------------------------------------------------------------------------------------------
// wavefront form of `shading`: phase 1 only requests the shadow ray of the surviving sample
__global__ void __launch_bounds__(64) k_shadingRays(DevScene s, DevFrame f, DevFrameParams p) {
    RayRequest request;
    bool want = false;
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    if (x < f.W && y < p.y1) {
        const size_t pix = (size_t)y * f.W + x;
        const uint32_t bufIdx = p.bufferIndex;
        if (f.gb0[bufIdx][pix].x != 0xFFFFFFFFu) {
            const float2 reservoirInfo = f.reservoirInfo[p.currentReservoirIndex][pix];
            const float recPDFEstimate = reservoirInfo.x;
            if (recPDFEstimate > 0 && isfinite(recPDFEstimate)) {
                const float4 gb2 = f.gb2[bufIdx][pix];
                f3 positionInWorld(gb2.x, gb2.y, gb2.z);
                const f3 geometricNormalInWorld = decodeVector(__float_as_uint(gb2.w));
                const f3 vOut = normalize(p.camera.position - positionInWorld);
                const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
                positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);
                const Reservoir reservoir = loadReservoir(f, p.currentReservoirIndex, pix);
                visibilityRay(positionInWorld, reservoir.sample, (uint32_t)pix, &request);
                want = true;
            }
        }
    }
    enqueueRay(f, s.rayCounter, want, request);
}

template <bool QUEUED_VISIBILITY>
__global__ void __launch_bounds__(64) k_shading(DevScene s, DevFrame f, DevFrameParams p) {
    // optix_restir_di_kernels.cu:559-637
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    if (x >= f.W || y >= p.y1)
        return;
    const size_t pix = (size_t)y * f.W + x;
    const uint32_t bufIdx = p.bufferIndex;
    const uint4 gb0 = f.gb0[bufIdx][pix];
    const uint4 gb3 = f.gb3[bufIdx][pix];

    f3 contribution(0.01f, 0.01f, 0.01f);
    if (gb0.x != 0xFFFFFFFFu) {
        const float4 gb2 = f.gb2[bufIdx][pix];
        f3 positionInWorld(gb2.x, gb2.y, gb2.z);
        const f3 geometricNormalInWorld = decodeVector(__float_as_uint(gb2.w));
        const f3 vOut = normalize(p.camera.position - positionInWorld);
        const float frontHit = dot(vOut, geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
        positionInWorld = offsetRayOrigin(positionInWorld, frontHit * geometricNormalInWorld);

        const ReferenceFrame shadingFrame(decodeVector(gb3.x), decodeVector(gb3.y));
        const f3 vOutLocal = shadingFrame.toLocal(vOut);
        const GfxMaterialDesc* mat = s.materials + gb3.w;
        const BSDF bsdf = setupBsdf(s, gb3.w, decodeTexCoords(gb3.z));

        const uint32_t curResIndex = p.currentReservoirIndex;
        const Reservoir reservoir = loadReservoir(f, curResIndex, pix);
        const float2 reservoirInfo = f.reservoirInfo[curResIndex][pix];

        contribution = f3(0.0f);
        if (vOutLocal.z > 0) {
            f3 emittance(0.0f);
            if (mat->hasEmittance)
                emittance = f3(mat->emittance[0], mat->emittance[1], mat->emittance[2]);
            contribution += emittance / kPi;
        }

        const LightSample lightSample = reservoir.sample;
        f3 directCont(0.0f);
        const float recPDFEstimate = reservoirInfo.x;
        if (recPDFEstimate > 0 && isfinite(recPDFEstimate)) {
            const bool visDone = p.reuseVisibility &&
                (!p.enableTemporalReuse || (p.enableSpatialReuse && p.useUnbiasedEstimator));
            if (visDone)
                directCont = performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample);
            else if (QUEUED_VISIBILITY) // performDirectLighting<true> with the answer of the wavefront trace
                directCont = f.visibility[pix] ? performDirectLighting<false>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample)
                                               : f3(0.0f);
            else
                directCont = performDirectLighting<true>(s, positionInWorld, vOutLocal, shadingFrame, bsdf, lightSample);
        }
        contribution += recPDFEstimate * directCont;
    }
    else if (s.env.enabled) { // :620-629: the environment seen directly; the miss program left (u, v) in the texture coordinates
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

int launchReSTIR(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params, int pass) {
    const DevFrameParams p = makeDevParams(ctx, params);
    if (p.y1 <= p.y0)
        return GFX_OK;
    if (p.log2NumCandidateSamples > 15 || p.numSpatialNeighbors > 15)
        return GFX_ERR_INVALID_ARGUMENT; // 4-bit fields in the reference (restir_di_shared.h:258-259)
    const dim3 block(8, 8);
    const dim3 grid((ctx->frame.W + 7) / 8, (p.y1 - p.y0 + 7) / 8);
    const DevScene s = ctx->devScene(params);
    const DevFrame f = ctx->devFrame();
    // with visibility reuse the RIS pass is a wavefront: request rays -> persistent-thread trace -> resolve; without it
    // there is no ray to trace and one kernel does the pass
#define RIS_LAUNCH(T, U) \
    if (p.reuseVisibility) { \
        int rc_ = resetVisibilityQueue(ctx, stream); if (rc_) return rc_; \
        { GFX_TIMED(ctx, stream, "ris_candidates"); \
          if (s.env.enabled) k_initialAndTemporalRIS<T, U, 1, true><<<grid, block, 0, stream>>>(s, f, p); \
          else k_initialAndTemporalRIS<T, U, 1><<<grid, block, 0, stream>>>(s, f, p); } ctx->launches++; \
        rc_ = traceVisibilityQueue(ctx, stream); if (rc_) return rc_; \
        { GFX_TIMED(ctx, stream, "ris_resolve_temporal"); k_initialAndTemporalRIS<T, U, 2><<<grid, block, 0, stream>>>(s, f, p); } \
    } else { \
        { GFX_TIMED(ctx, stream, "ris_megakernel"); \
          if (s.env.enabled) k_initialAndTemporalRIS<T, U, 0, true><<<grid, block, 0, stream>>>(s, f, p); \
          else k_initialAndTemporalRIS<T, U, 0><<<grid, block, 0, stream>>>(s, f, p); } \
    }
    switch (pass) {
    case GFX_RESTIR_INITIAL_RIS: RIS_LAUNCH(false, false); break;
    case GFX_RESTIR_INITIAL_AND_TEMPORAL_BIASED: RIS_LAUNCH(true, false); break;
    case GFX_RESTIR_INITIAL_AND_TEMPORAL_UNBIASED: RIS_LAUNCH(true, true); break;
    case GFX_RESTIR_SPATIAL_BIASED: { GFX_TIMED(ctx, stream, "spatial_ris"); k_spatialRIS<false><<<grid, block, 0, stream>>>(s, f, p); } break;
    case GFX_RESTIR_SPATIAL_UNBIASED: { GFX_TIMED(ctx, stream, "spatial_ris_unbiased"); k_spatialRIS<true><<<grid, block, 0, stream>>>(s, f, p); } break;
    case GFX_RESTIR_SHADING: {
        const bool visDone = p.reuseVisibility && (!p.enableTemporalReuse || (p.enableSpatialReuse && p.useUnbiasedEstimator));
        if (!visDone) {
            int rc_ = resetVisibilityQueue(ctx, stream); if (rc_) return rc_;
            { GFX_TIMED(ctx, stream, "shading_rays"); k_shadingRays<<<grid, block, 0, stream>>>(s, f, p); } ctx->launches++;
            rc_ = traceVisibilityQueue(ctx, stream); if (rc_) return rc_;
            { GFX_TIMED(ctx, stream, "shading"); k_shading<true><<<grid, block, 0, stream>>>(s, f, p); }
        }
        else {
            { GFX_TIMED(ctx, stream, "shading_megakernel"); k_shading<false><<<grid, block, 0, stream>>>(s, f, p); }
        }
        break;
    }
    default:
        ctx->setError("gfx_restir_launch: unknown pass");
        return GFX_ERR_INVALID_ARGUMENT;
    }
#undef RIS_LAUNCH
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

} // namespace gfx
