// lighting.cuh — light sampling and direct-lighting helpers shared by the ReSTIR, ReGIR and path-tracing kernels.
//
// sampleLight<false> (restir_di/restir_di_shared.h:320-516; identical copies live in path_tracing_shared.h:220-482,
// regir_shared.h, neural_radiance_caching_shared.h, svgf_shared.h), performDirectLighting (:518-557),
// evaluateVisibility (:559-582).  Visibility rays run through the inline any-hit traversal of traverse.cuh
// (fused kernels) or are queued for trace.cu's persistent kernel (wavefront kernels).
#pragma once
#include "traverse.cuh"
#include "shading.cuh"

namespace gfx {

struct LightSample { // restir_di_shared.h:89-96
    f3 emittance, position, normal;
    uint32_t atInfinity;
};
GFX_D LightSample emptyLightSample() {
    LightSample s;
    s.emittance = f3(0.0f);
    s.position = f3(0.0f);
    s.normal = f3(0.0f);
    s.atInfinity = 0;
    return s;
}

GFX_D float convertToWeight(const f3 &c) { return (c.x + c.y + c.z) / 3; } // restir_di_shared.h:82-85

// last index with cdf[idx] <= u: the power-of-two stepping search of
// DiscreteDistribution1DTemplate::sample (common_shared.h:226-232)
GFX_D uint32_t searchCdf(const float* __restrict__ cdf, uint32_t numValues, float u) {
    int idx = 0;
    for (int d = (int)(nextPowerOf2(numValues) >> 1); d >= 1; d >>= 1) {
        if (idx + d >= (int)numValues)
            continue;
        if (__ldg(cdf + idx + d) <= u)
            idx += d;
    }
    return (uint32_t)idx;
}
// the same search seeded by a guide table (scene.cuh): exact, 1-3 loads instead of log2(n)
GFX_D uint32_t guidedSearchCdf(const float* __restrict__ cdf, const uint32_t* __restrict__ guide, uint32_t guideSize,
                               float u01, float u) {
    const uint32_t b = min(dm_f2uint(u01 * (float)guideSize), guideSize - 1);
    uint32_t idx = __ldg(guide + b);
    const uint32_t hi = __ldg(guide + b + 1);
    while (idx < hi && __ldg(cdf + idx + 1) <= u)
        ++idx;
    return idx;
}
GFX_D float remapCdf(const float* __restrict__ cdf, uint32_t numValues, float integral, uint32_t idx, float u) {
    // common_shared.h:235-241
    const float lCDF = __ldg(cdf + idx);
    float rCDF = integral;
    if (idx < numValues - 1)
        rCDF = __ldg(cdf + idx + 1);
    return (u - lCDF) / (rCDF - lCDF);
}

// sm_100's 256-bit read-only load (LDG.E.256): one L1 tag lookup for 32 bytes.  volatile: ptxas would otherwise hoist the
// later stages' loads of sampleLightUnlessDark above the dark tests (it did, ncu round 2: all nine record loads were issued by
// every survivor of the sphere test), which is exactly the traffic the staging is there to avoid.
struct F8 { float4 lo, hi; };
GFX_D F8 ldg256(const float4* p) {
    F8 r;
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.lo.x), "=f"(r.lo.y), "=f"(r.lo.z), "=f"(r.lo.w), "=f"(r.hi.x), "=f"(r.hi.y), "=f"(r.hi.z), "=f"(r.hi.w)
                 : "l"(p));
    return r;
}
GFX_D float ldg32v(const float* p) {
    float r;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// the normal matrix of an instance out of the compact table (scene.cuh): one 256-bit load + one scalar
GFX_D f3 applyNormalMatrix(const DevScene &s, uint32_t instSlot, const f3 &n) {
    const float4* mp = s.normalMats + (size_t)kNormalMatStride * instSlot;
    const F8 a = ldg256(mp);
    const float m[9] = { a.lo.x, a.lo.y, a.lo.z, a.lo.w, a.hi.x, a.hi.y, a.hi.z, a.hi.w, ldg32v(reinterpret_cast<const float*>(mp + 2)) };
    return mul3x3(m, n);
}

// The three DiscreteDistribution1D::sample calls of sampleLight (instance, geometry instance, primitive;
// restir_di_shared.h:356-409, common_shared.h:209-246) spelled out; weights[idx] / integral comes from the pre-divided prob
// tables.  This is the DEFINITION of the light pick; the kernels use its flattened form (pickLightTriangle below), which
// lights.cu derives from it.  Returns a key: the index of the light record, or kPickNone | position for sampleLight's
// probability-0 early outs (distinct positions give distinct keys, so that equal keys at two values of ul mean "same piece").
GFX_D uint32_t chainPickLightTriangle(const DevScene &s, float ul, float* lightProbOut) {
    float lightProb = 1.0f;

    // instance
    const float instIntegral = __ldg(s.instIntegral);
    float u = ul * instIntegral;
    const uint32_t instSlot = guidedSearchCdf(s.instCdf, s.instGuide, kInstGuideSize, ul, u);
    const float uGeomInst = remapCdf(s.instCdf, s.numInstances, instIntegral, instSlot, u);
    const float instProb = __ldg(s.instProb + instSlot);
    lightProb *= instProb;
    const DevInstance* inst = s.instances + instSlot;
    if (instProb == 0.0f)
        return kPickNone | 0x20000000u | instSlot;

    // geometry instance
    const uint32_t firstMeshSlot = inst->firstMeshSlot, numMeshSlots = inst->numMeshSlots;
    const float geomIntegral = inst->geomIntegral;
    u = uGeomInst * geomIntegral;
    const uint32_t geomInstIndexInInst = searchCdf(s.geomCdf + firstMeshSlot, numMeshSlots, u);
    const float uPrim = remapCdf(s.geomCdf + firstMeshSlot, numMeshSlots, geomIntegral, geomInstIndexInInst, u);
    const float geomInstProb = __ldg(s.geomProb + firstMeshSlot + geomInstIndexInInst);
    const uint32_t geomInstSlot = __ldg(s.instanceMeshSlots + firstMeshSlot + geomInstIndexInInst);
    lightProb *= geomInstProb;
    if (geomInstProb == 0.0f)
        return kPickNone | (firstMeshSlot + geomInstIndexInInst);

    // primitive
    const DevMesh* mesh = s.meshes + geomInstSlot;
    const uint32_t triBase = mesh->triBase;
    u = uPrim * mesh->primIntegral;
    const uint32_t primIndex = guidedSearchCdf(s.primCdf + triBase, s.primGuide + (size_t)geomInstSlot * (kPrimGuideSize + 1),
                                               kPrimGuideSize, uPrim, u);
    const float primProb = __ldg(s.primProb + triBase + primIndex);
    lightProb *= primProb;

    *lightProbOut = lightProb;
    const uint32_t base = __ldg(s.lightTriBase + inst->geomBase + geomInstIndexInInst);
    if (base == 0xFFFFFFFFu) // a geometry without an emitter: only reachable when every weight is 0 (0 / 0 probabilities)
        return kPickNone | 0x10000000u | (firstMeshSlot + geomInstIndexInInst);
    return base + primIndex;
}

// The flattened pick (scene.cuh, lights.cu): the piece that contains ul - its key and the head of its light record (cull
// sphere, area density, instance slot), which for a pure bucket arrives with the guide entry itself.
struct LightPick {
    uint32_t key;      // light record index, or kPickNone set
    float4 sphere;     // centre, radius (< 0: do not cull)
    float density;     // lightProb * recArea
    uint32_t instSlot;
};
GFX_D F8 pickGuideFetch(const DevScene &s, float ul) { // the guide entry of ul's bucket (issue early, resolve later)
    const uint32_t b = min(dm_f2uint(ul * (float)kPickGuideSize), kPickGuideSize - 1); // exact: a power-of-two product, floored
    return ldg256(s.pickGuide + 2 * (size_t)b);
}
GFX_D LightPick pickLightFromGuide(const DevScene &s, float ul, const F8 &g) {
    LightPick r;
    const uint32_t head = __float_as_uint(g.lo.x);
    if (head & kPickPure) {
        r.key = head & ~kPickPure;
        r.sphere = make_float4(g.lo.y, g.lo.z, g.lo.w, g.hi.x);
        r.density = g.hi.y;
        r.instSlot = __float_as_uint(g.hi.z);
        return r;
    }
    const uint32_t ulBits = __float_as_uint(ul);
    uint32_t idx = head;
    uint2 piece = __ldg(s.pickPieces + idx);
    for (;;) {
        const uint2 next = __ldg(s.pickPieces + idx + 1);
        if (next.x > ulBits)
            break;
        piece = next;
        ++idx;
    }
    r.key = piece.y;
    r.sphere = make_float4(0.0f, 0.0f, 0.0f, -1.0f);
    r.density = 0.0f;
    r.instSlot = 0;
    if (!(r.key & kPickNone)) {
        const F8 h0 = ldg256(s.lightTris + kLightTriStride * (size_t)r.key);
        r.sphere = h0.lo;
        r.density = h0.hi.x;
        r.instSlot = __float_as_uint(h0.hi.y);
    }
    return r;
}
GFX_D LightPick pickLight(const DevScene &s, float ul) { return pickLightFromGuide(s, ul, pickGuideFetch(s, ul)); }
GFX_D uint32_t pickLightTriangle(const DevScene &s, float ul) { return pickLight(s, ul).key; }

// A Low-Distortion Map Between Triangle and Square (restir_di_shared.h:485-498)
GFX_D void squareToTriangle(float u0, float u1, float* bcA, float* bcB, float* bcC) {
    float a = 0.5f * u0;
    float b = 0.5f * u1;
    const float offset = b - a;
    if (offset > 0)
        b += offset;
    else
        a -= offset;
    *bcA = a;
    *bcB = b;
    *bcC = 1 - (a + b);
}

GFX_D void sampleLight(const DevScene &s, float ul, float u0, float u1, LightSample* lightSample, float* areaPDensity) {
    // restir_di_shared.h:320-516 with sampleEnvLight = false, useSolidAngleSampling = false; the triangle operands come
    // from the light records (lights.cu), produced by the reference's own expressions, so the result is bit-identical.
    const LightPick pick = pickLight(s, ul);
    if (pick.key & kPickNone) {
        *areaPDensity = 0.0f;
        return;
    }
    const float4* e = s.lightTris + kLightTriStride * (size_t)pick.key;
    const F8 h1 = ldg256(e + 2), h2 = ldg256(e + 4), h3 = ldg256(e + 6);
    const f3 pA(h1.lo.x, h1.lo.y, h1.lo.z), pB(h1.lo.w, h1.hi.x, h1.hi.y), pC(h1.hi.z, h1.hi.w, h2.lo.x);
    const f3 nA(h2.lo.y, h2.lo.z, h2.lo.w), nB(h2.hi.x, h2.hi.y, h2.hi.z), nC(h2.hi.w, h3.lo.x, h3.lo.y);
    float bcA, bcB, bcC;
    squareToTriangle(u0, u1, &bcA, &bcB, &bcC);

    *areaPDensity = pick.density;

    lightSample->position = bcA * pA + bcB * pB + bcC * pC;
    lightSample->atInfinity = 0;
    lightSample->normal = bcA * nA + bcB * nB + bcC * nC;
    lightSample->normal = normalize(applyNormalMatrix(s, pick.instSlot, lightSample->normal));
    lightSample->emittance = f3(h3.lo.z, h3.lo.w, h3.hi.x);
}

// ---- environment light ---------------------------------------------------------------------------------------------
// RegularConstantContinuousDistribution1D::sample / evaluatePDF (common_shared.h:316-348, CDF variant)
GFX_D float regularSample(const float* __restrict__ PDF, const float* __restrict__ CDF, uint32_t numValues, float u, float* probDensity) {
    int idx = 0;
    for (int d = (int)(nextPowerOf2(numValues) >> 1); d >= 1; d >>= 1) {
        if (idx + d >= (int)numValues)
            continue;
        if (__ldg(CDF + idx + d) <= u)
            idx += d;
    }
    const float lo = __ldg(CDF + idx);
    const float t = (u - lo) / (__ldg(CDF + idx + 1) - lo);
    *probDensity = __ldg(PDF + idx);
    return (idx + t) / numValues;
}
GFX_D uint32_t mapPrimarySampleToDiscrete(float u01, uint32_t numValues) { // common_shared.h:142-152
    return min(dm_f2uint(u01 * numValues), numValues - 1);
}
// RegularConstantContinuousDistribution2D::sample / evaluatePDF (:371-383)
GFX_D void envSample(const DevEnvLight &e, float u0, float u1, float* d0, float* d1, float* probDensity) {
    float topPDF;
    *d1 = regularSample(e.topPdf, e.topCdf, e.H, u1, &topPDF);
    const uint32_t row = mapPrimarySampleToDiscrete(*d1, e.H);
    *d0 = regularSample(e.pdf + (size_t)row * e.W, e.cdf + (size_t)row * (e.W + 1), e.W, u0, probDensity);
    *probDensity *= topPDF;
}
GFX_D float envEvaluatePDF(const DevEnvLight &e, float d0, float d1) {
    const uint32_t row = mapPrimarySampleToDiscrete(d1, e.H);
    const uint32_t col = min(e.W - 1, dm_f2uint(d0 * e.W));
    return __ldg(e.topPdf + min(e.H - 1, dm_f2uint(d1 * e.H))) * __ldg(e.pdf + (size_t)row * e.W + col);
}
// tex2DLod<float4>(envLightTexture, u, v, 0).xyz with the reference's sampler (common_host.cpp:2664-2669: linear filter, clamp
// addressing, normalised coordinates) in software: the texture unit's arithmetic - xB = u W - 0.5, i = floor(xB), the fraction
// kept with 8 fractional bits, the four texels blended - spelled out in fp32
// (the three heavier functions are out of line and take the 56-byte descriptor by value: kernels that never meet an environment
// light keep their register budget and no kernel parameter has its address taken)
static __device__ __noinline__ f3 envFetchOutOfLine(DevEnvLight e, float u, float v) {
    const float xB = u * e.W - 0.5f, yB = v * e.H - 0.5f;
    const float fx = floorf(xB), fy = floorf(yB);
    const float a = floorf((xB - fx) * 256.0f + 0.5f) * (1.0f / 256.0f);
    const float b = floorf((yB - fy) * 256.0f + 0.5f) * (1.0f / 256.0f);
    const uint32_t x0 = dm_f2uint(fminf(fmaxf(fx, 0.0f), (float)(e.W - 1))), x1 = dm_f2uint(fminf(fmaxf(fx + 1.0f, 0.0f), (float)(e.W - 1)));
    const uint32_t y0 = dm_f2uint(fminf(fmaxf(fy, 0.0f), (float)(e.H - 1))), y1 = dm_f2uint(fminf(fmaxf(fy + 1.0f, 0.0f), (float)(e.H - 1)));
    const float4 t00 = __ldg(e.texels + (size_t)y0 * e.W + x0), t10 = __ldg(e.texels + (size_t)y0 * e.W + x1);
    const float4 t01 = __ldg(e.texels + (size_t)y1 * e.W + x0), t11 = __ldg(e.texels + (size_t)y1 * e.W + x1);
    const float w00 = (1 - a) * (1 - b), w10 = a * (1 - b), w01 = (1 - a) * b, w11 = a * b;
    return w00 * f3(t00.x, t00.y, t00.z) + w10 * f3(t10.x, t10.y, t10.z) + w01 * f3(t01.x, t01.y, t01.z) + w11 * f3(t11.x, t11.y, t11.z);
}
GFX_D f3 envFetch(const DevEnvLight &e, float u, float v) { return envFetchOutOfLine(e, u, v); }
// sampleLight with sampleEnvLight = true (restir_di_shared.h:330-364)
struct EnvLightSample {
    LightSample sample;
    float areaPDensity;
};
static __device__ __noinline__ EnvLightSample sampleEnvLightOutOfLine(DevEnvLight env, float u0, float u1) {
    EnvLightSample out;
    LightSample* lightSample = &out.sample;
    float* areaPDensity = &out.areaPDensity;
    float u, v, uvPDF;
    envSample(env, u0, u1, &u, &v, &uvPDF);
    const float phi = 2 * kPi * u;
    const float theta = kPi * v;
    float posPhi = phi - env.rotation;
    posPhi = posPhi - floorf(posPhi / (2 * kPi)) * 2 * kPi;
    const f3 direction = fromPolarYUp(posPhi, theta);
    lightSample->position = direction;
    lightSample->atInfinity = 1;
    lightSample->normal = -direction;
    lightSample->emittance = f3(0.0f);
    const float sinTheta = dm_sin(theta);
    if (sinTheta == 0.0f) {
        *areaPDensity = 0.0f;
        return out;
    }
    *areaPDensity = uvPDF / (2 * kPi * kPi * sinTheta);
    f3 emittance(kPi * env.powerCoeff);
    emittance *= envFetchOutOfLine(env, u, v);
    lightSample->emittance = emittance;
    return out;
}
GFX_D void sampleEnvLight(const DevScene &s, float u0, float u1, LightSample* lightSample, float* areaPDensity) {
    const EnvLightSample r = sampleEnvLightOutOfLine(s.env, u0, u1);
    *lightSample = r.sample;
    *areaPDensity = r.areaPDensity;
}
// the choice between the environment and the emitters that the streaming-RIS loops make for candidate i of n
// (optix_restir_di_kernels.cu:72-90, build_cell_reservoirs.cu:120-139): returns sampleEnvLight, remaps ul
GFX_D bool chooseEnvForCandidate(const DevScene &s, uint32_t i, uint32_t numCandidates, float* ul, float* probToSampleCurLightType) {
    *probToSampleCurLightType = 1.0f;
    if (!s.env.enabled)
        return false;
    if (!(__ldg(s.instIntegral) > 0.0f))
        return true;
    const float prob = fminf(fmaxf(kProbToSampleEnvLight * numCandidates - i, 0.0f), 1.0f);
    if (*ul < prob) {
        *probToSampleCurLightType = kProbToSampleEnvLight;
        *ul = *ul / prob;
        return true;
    }
    *probToSampleCurLightType = 1.0f - kProbToSampleEnvLight;
    *ul = (*ul - prob) / (1 - prob);
    return false;
}
// the path tracers' choice per next-event estimation (optix_pathtracing_kernels.cu:27-42)
GFX_D bool chooseEnvForNee(const DevScene &s, float* uLight, float* probToSampleCurLightType) {
    *probToSampleCurLightType = 1.0f;
    if (!s.env.enabled)
        return false;
    if (!(__ldg(s.instIntegral) > 0.0f))
        return true;
    if (*uLight < kProbToSampleEnvLight) {
        *probToSampleCurLightType = kProbToSampleEnvLight;
        *uLight /= *probToSampleCurLightType;
        return true;
    }
    *probToSampleCurLightType = 1.0f - kProbToSampleEnvLight;
    *uLight = (*uLight - kProbToSampleEnvLight) / *probToSampleCurLightType;
    return false;
}
// the miss programs of the path tracers (optix_pathtracing_kernels.cu:310-341; neural_radiance_caching/...:625-650, which
// multiplies by probToSampleEnvLight unconditionally): luminance x MIS weight of the environment along rayDir
static __device__ __noinline__ f3 evaluateEnvLightOnMissOutOfLine(DevEnvLight env, f3 rayDirIn, float prevDirPDensity, float probToSampleEnv) {
    const f3 rayDir = normalize(rayDirIn);
    float posPhi, theta;
    toPolarYUp(rayDir, &posPhi, &theta);
    float phi = posPhi + env.rotation;
    phi = phi - floorf(phi / (2 * kPi)) * 2 * kPi;
    const float tu = phi / (2 * kPi), tv = theta / kPi;
    const f3 luminance = env.powerCoeff * envFetchOutOfLine(env, tu, tv);
    const float uvPDF = envEvaluatePDF(env, tu, tv);
    const float hypAreaPDensity = uvPDF / (2 * kPi * kPi * dm_sin(theta));
    const float lightPDensity = probToSampleEnv * hypAreaPDensity;
    const float bsdfPDensity = prevDirPDensity;
    const float misWeight = pow2f(bsdfPDensity) / (pow2f(bsdfPDensity) + pow2f(lightPDensity));
    return luminance * misWeight;
}
GFX_D f3 evaluateEnvLightOnMiss(const DevScene &s, const f3 &rayDir, float prevDirPDensity, bool nrcVariant) {
    const float probToSampleEnv = (nrcVariant || __ldg(s.instIntegral) > 0.0f) ? kProbToSampleEnvLight : 1.0f;
    return evaluateEnvLightOnMissOutOfLine(s.env, rayDir, prevDirPDensity, probToSampleEnv);
}

// sampleLight for the RIS candidate loop, fetching the 128-byte light record in steps and stopping as soon as the candidate is
// certain to contribute RGB(0) to this shading point.  ncu: the candidate kernel is bound by the L1 data pipe's wavefront rate
// (every lane reads a different light, so every load instruction of the sampling chain is up to 32 wavefronts) and by issue
// slots; ~70 % of the candidates are dark (65 % lie below the shading horizon).
//   step 0: the bounding sphere of the light triangle - it arrived with the pick (guide entry).  Wholly below the shading
//           horizon -> dark, no further load;
//   step 1: the three vertices (2 x 256 bits) -> sample position.  Below the shading horizon (the BRDFs return RGB(0) when
//           vGiven.z * vSampled.z <= 0)?  -> dark;
//   step 2: the vertex normals, the emittance (256 bits) and the instance's normal matrix (256 + 32 bits) -> un-normalised light
//           normal.  Facing away (lpCos <= 0)? -> dark; otherwise the normalisation: the full sample.
// The tests run on un-normalised vectors with a relative margin of 1e-3 on the cosine (the sphere test with twice that, so
// that every sample point of the triangle would pass the per-sample test too; tests/cpp/sphere_cull_check.cpp) - three orders
// of magnitude above the rounding of the exact evaluation - so borderline samples go on to the exact path and no decision ever
// differs from performDirectLighting's; NaNs and a zero distance fail the comparisons and also go on.  Returns true for "dark"
// (then *areaPDensity is positive); otherwise the outputs are sampleLight's, bit for bit.
GFX_D bool sampleLightUnlessDark(const DevScene &s, float ul, float u0, float u1, const f3 &shadingPoint,
                                 const f3 &shadingNormal, float vOutLocalZ, LightSample* lightSample, float* areaPDensity) {
    const LightPick pick = pickLight(s, ul);
    if (pick.key & kPickNone) {
        *areaPDensity = 0.0f;
        return false;
    }
    {   // step 0: the whole triangle lies below the shading horizon if its bounding sphere does:
        //   -dot(q - p, n) sgn >= t - r |n|  and  |q - p| <= |c - p| + r   for every q in the sphere
        // (radius >= 0 also says that the selection density of this light is a positive finite number)
        const f3 dc = f3(pick.sphere.x, pick.sphere.y, pick.sphere.z) - shadingPoint;
        const float r = pick.sphere.w;
        const float t = -(dot(dc, shadingNormal) * vOutLocalZ);          // > 0: centre on the far side of the surface
        const float margin = t - 1.001f * r * fabsf(vOutLocalZ);
        if (r >= 0.0f && margin > 0.0f && margin * margin > 8e-6f * (sqLength(dc) + r * r) * (vOutLocalZ * vOutLocalZ)) {
            *areaPDensity = 1.0f; // any positive number: the caller only asks whether the density is positive
            return true;
        }
    }
    const float4* e = s.lightTris + kLightTriStride * (size_t)pick.key;
    const F8 h1 = ldg256(e + 2), h2 = ldg256(e + 4);
    const f3 pA(h1.lo.x, h1.lo.y, h1.lo.z), pB(h1.lo.w, h1.hi.x, h1.hi.y), pC(h1.hi.z, h1.hi.w, h2.lo.x);
    float bcA, bcB, bcC;
    squareToTriangle(u0, u1, &bcA, &bcB, &bcC);
    const float density = pick.density;
    *areaPDensity = density;
    const f3 position = bcA * pA + bcB * pB + bcC * pC;

    const float k = 1e-6f; // (1e-3)^2
    const f3 d = position - shadingPoint;
    const float dd = sqLength(d);
    const float b = dot(d, shadingNormal) * vOutLocalZ; // < 0: light and viewer on opposite sides of the surface
    if (density > 0.0f && b < 0.0f && b * b > k * dd * (vOutLocalZ * vOutLocalZ))
        return true;

    const F8 h3 = ldg256(e + 6);
    const f3 nA(h2.lo.y, h2.lo.z, h2.lo.w), nB(h2.hi.x, h2.hi.y, h2.hi.z), nC(h2.hi.w, h3.lo.x, h3.lo.y);
    f3 normal = bcA * nA + bcB * nB + bcC * nC;
    normal = applyNormalMatrix(s, pick.instSlot, normal);
    const float a = dot(d, normal); // > 0: the emitter faces away from the shading point
    if (density > 0.0f && a > 0.0f && a * a > k * dd * sqLength(normal))
        return true;

    lightSample->position = position;
    lightSample->atInfinity = 0;
    lightSample->normal = normalize(normal);
    lightSample->emittance = f3(h3.lo.z, h3.lo.w, h3.hi.x);
    return false;
}

// sampleLightUnlessDark in two halves for the two-phase candidate loop of the ReSTIR initial pass (restir.cu):
//   classifyLight    the pick and step 0 (bounding sphere) -> kLightDark, or the light's key with bit 31 = "the dark tests may
//                    be used" (the selection density is a positive finite number; otherwise the exact path decides);
//   finishLightSample steps 1 and 2 from the key alone (density and instance slot come from the record's H3 copy).
constexpr uint32_t kLightDark = 0xFFFFFFFFu;
constexpr uint32_t kLightCullable = 0x80000000u;
GFX_D uint32_t classifyLight(const DevScene &s, float ul, const F8 &guideEntry, const f3 &shadingPoint, const f3 &shadingNormal,
                             float vOutLocalZ) {
    const LightPick pick = pickLightFromGuide(s, ul, guideEntry);
    if (pick.key & kPickNone)
        return kPickNone; // every "no light" key is the same to the caller
    const f3 dc = f3(pick.sphere.x, pick.sphere.y, pick.sphere.z) - shadingPoint;
    const float r = pick.sphere.w;
    const float t = -(dot(dc, shadingNormal) * vOutLocalZ);
    const float margin = t - 1.001f * r * fabsf(vOutLocalZ);
    if (r >= 0.0f && margin > 0.0f && margin * margin > 8e-6f * (sqLength(dc) + r * r) * (vOutLocalZ * vOutLocalZ))
        return kLightDark;
    return pick.key | (r >= 0.0f ? kLightCullable : 0u);
}
// returns true for "dark"; otherwise *lightSample / *areaPDensity are sampleLight's, bit for bit
GFX_D bool finishLightSample(const DevScene &s, uint32_t code, float u0, float u1, const f3 &shadingPoint, const f3 &shadingNormal,
                             float vOutLocalZ, LightSample* lightSample, float* areaPDensity) {
    if (code & kPickNone) {
        *areaPDensity = 0.0f;
        return false;
    }
    const bool cullable = (code & kLightCullable) != 0; // implies density > 0
    const float4* e = s.lightTris + kLightTriStride * (size_t)(code & 0x3FFFFFFFu);
    const F8 h1 = ldg256(e + 2), h2 = ldg256(e + 4);
    const f3 pA(h1.lo.x, h1.lo.y, h1.lo.z), pB(h1.lo.w, h1.hi.x, h1.hi.y), pC(h1.hi.z, h1.hi.w, h2.lo.x);
    float bcA, bcB, bcC;
    squareToTriangle(u0, u1, &bcA, &bcB, &bcC);
    const f3 position = bcA * pA + bcB * pB + bcC * pC;

    const float k = 1e-6f; // (1e-3)^2
    const f3 d = position - shadingPoint;
    const float dd = sqLength(d);
    const float b = dot(d, shadingNormal) * vOutLocalZ; // < 0: light and viewer on opposite sides of the surface
    if (cullable && b < 0.0f && b * b > k * dd * (vOutLocalZ * vOutLocalZ)) {
        *areaPDensity = 1.0f;
        return true;
    }
    const F8 h3 = ldg256(e + 6);
    const float density = h3.hi.z;
    *areaPDensity = density;
    const f3 nA(h2.lo.y, h2.lo.z, h2.lo.w), nB(h2.hi.x, h2.hi.y, h2.hi.z), nC(h2.hi.w, h3.lo.x, h3.lo.y);
    f3 normal = bcA * nA + bcB * nB + bcC * nC;
    normal = applyNormalMatrix(s, __float_as_uint(h3.hi.w), normal);
    const float a = dot(d, normal); // > 0: the emitter faces away from the shading point
    if (cullable && a > 0.0f && a * a > k * dd * sqLength(normal))
        return true;

    lightSample->position = position;
    lightSample->atInfinity = 0;
    lightSample->normal = normalize(normal);
    lightSample->emittance = f3(h3.lo.z, h3.lo.w, h3.hi.x);
    return false;
}

GFX_D bool traceVisibility(const DevScene &s, const f3 &org, const f3 &dir, float tmax) {
    // ray statistics: one atomic per warp per call site (lanes currently active here)
    const uint32_t active = __activemask();
    if ((threadIdx.x + threadIdx.y * blockDim.x) % 32 == (uint32_t)(__ffs(active) - 1))
        atomicAdd(s.rayCounter, (unsigned long long)__popc(active));
    const Hit h = traverseBvh<true>(s.bvh, org, dir, 0.0f, tmax);
    return h.storageIndex == 0xFFFFFFFFu;
}

GFX_D bool evaluateVisibility(const DevScene &s, const f3 &shadingPoint, const LightSample &ls) { // :559-582
    f3 shadowRayDir = ls.atInfinity ? ls.position : (ls.position - shadingPoint);
    const float dist2 = sqLength(shadowRayDir);
    float dist = sqrtf(dist2);
    shadowRayDir /= dist;
    if (ls.atInfinity)
        dist = 1e+10f;
    return traceVisibility(s, shadingPoint, shadowRayDir, dist * 0.9999f);
}

template <bool withVisibility>
GFX_D f3 performDirectLighting(const DevScene &s, const f3 &shadingPoint, const f3 &vOutLocal,
                               const ReferenceFrame &shadingFrame, const BSDF &bsdf, const LightSample &ls) { // :518-557
    f3 shadowRayDir = ls.atInfinity ? ls.position : (ls.position - shadingPoint);
    const float dist2 = sqLength(shadowRayDir);
    float dist = sqrtf(dist2);
    shadowRayDir /= dist;
    const f3 shadowRayDirLocal = shadingFrame.toLocal(shadowRayDir);

    const float lpCos = dot(-shadowRayDir, ls.normal);
    const float spCos = shadowRayDirLocal.z;

    float visibility = 1.0f;
    if (withVisibility) {
        if (ls.atInfinity)
            dist = 1e+10f;
        if (!traceVisibility(s, shadingPoint, shadowRayDir, dist * 0.9999f))
            visibility = 0.0f;
    }

    if (visibility > 0 && lpCos > 0) {
        const f3 Le = ls.emittance / kPi;
        const f3 fsValue = bsdf.evaluate(vOutLocal, shadowRayDirLocal);
        const float G = lpCos * fabsf(spCos) / dist2;
        return fsValue * Le * G;
    }
    return f3(0.0f);
}

// tex2DLod<float4>(materialTexture, u, v, 0) with the reference's material samplers (common_host.cpp:1462-1481: linear filter,
// repeat addressing) in software: u -> frac(u), xB = frac(u) W - 0.5, i = floor(xB) and i + 1 wrapped modulo W, the fraction kept
// with 8 fractional bits, the four texels blended in fp32 (the same arithmetic as envFetch, other addressing mode)
static __device__ __noinline__ float4 textureFetchRepeat(const float4* texels, uint32_t W, uint32_t H, float u, float v) {
    const float xB = (u - floorf(u)) * W - 0.5f, yB = (v - floorf(v)) * H - 0.5f;
    const float fx = floorf(xB), fy = floorf(yB);
    const float a = floorf((xB - fx) * 256.0f + 0.5f) * (1.0f / 256.0f);
    const float b = floorf((yB - fy) * 256.0f + 0.5f) * (1.0f / 256.0f);
    const int ix = dm_f2int(fx), iy = dm_f2int(fy); // -1 .. W - 1
    const uint32_t x0 = ix < 0 ? W - 1 : (uint32_t)ix, x1 = (uint32_t)(ix + 1) >= W ? 0u : (uint32_t)(ix + 1);
    const uint32_t y0 = iy < 0 ? H - 1 : (uint32_t)iy, y1 = (uint32_t)(iy + 1) >= H ? 0u : (uint32_t)(iy + 1);
    const float4 t00 = __ldg(texels + (size_t)y0 * W + x0), t10 = __ldg(texels + (size_t)y0 * W + x1);
    const float4 t01 = __ldg(texels + (size_t)y1 * W + x0), t11 = __ldg(texels + (size_t)y1 * W + x1);
    const float w00 = (1 - a) * (1 - b), w10 = a * (1 - b), w01 = (1 - a) * b, w11 = a * b;
    return make_float4(w00 * t00.x + w10 * t10.x + w01 * t01.x + w11 * t11.x, w00 * t00.y + w10 * t10.y + w01 * t01.y + w11 * t11.y,
                       w00 * t00.z + w10 * t10.z + w01 * t01.z + w11 * t11.z, w00 * t00.w + w10 * t10.w + w01 * t01.w + w11 * t11.w);
}
// BSDF::setup(mat, texCoord, 0.0f) (common_device.cuh:376-385, 778-826): the material's constants, or its image textures at
// texCoord.  The textured form is out of line (and takes the tables as plain pointers): a scene without image textures runs
// exactly the code it ran before they existed.
static __device__ __noinline__ BSDF setupBsdfTextured(const GfxMaterialDesc* materials, const uint4* materialTextures, const uint4* texTable,
                                                      const float4* texPool, uint32_t matSlot, float tu, float tv) {
    const GfxMaterialDesc* m = materials + matSlot;
    const uint4 tex = __ldg(materialTextures + matSlot);
    float p0[3] = { m->p0[0], m->p0[1], m->p0[2] }, p1[3] = { m->p1[0], m->p1[1], m->p1[2] }, p2 = m->p2;
    if (tex.x != 0xFFFFFFFFu) {
        const uint4 d = __ldg(texTable + tex.x);
        const float4 t = textureFetchRepeat(texPool + d.x, d.y, d.z, tu, tv);
        p0[0] = t.x; p0[1] = t.y; p0[2] = t.z;
    }
    if (tex.y != 0xFFFFFFFFu) {
        const uint4 d = __ldg(texTable + tex.y);
        const float4 t = textureFetchRepeat(texPool + d.x, d.y, d.z, tu, tv);
        p1[0] = t.x; p1[1] = t.y; p1[2] = t.z;
    }
    if (tex.z != 0xFFFFFFFFu) {
        const uint4 d = __ldg(texTable + tex.z);
        p2 = textureFetchRepeat(texPool + d.x, d.y, d.z, tu, tv).x;
    }
    BSDF b;
    b.setup(m->bsdfType, p0, p1, p2);
    return b;
}
GFX_D BSDF setupBsdf(const DevScene &s, uint32_t matSlot, const f2 &texCoord) {
    if (s.materialTextures)
        return setupBsdfTextured(s.materials, s.materialTextures, s.texTable, s.texPool, matSlot, texCoord.x, texCoord.y);
    const GfxMaterialDesc* m = s.materials + matSlot;
    BSDF b;
    b.setup(m->bsdfType, m->p0, m->p1, m->p2);
    return b;
}

} // namespace gfx
