// bvh_build.cu — GPU LBVH builder emitting the reference's wide-BVH format.
//
// Stands where Scene::updateASs -> optixAccelBuild stands (common/common_host.h:1027-1100,
// utils/optix_util.cpp:1776,2799) and where the CPU bvh::buildGeometryBVH<8>
// (common/bvh_builder.cpp:656-1125) stands for the software path.  Output is bit-compatible with
// shared::CompressedInternalNode_T<8> / TriangleStorage / PrimitiveReference
// (common/common_shared.h:757-917,1012-1025), so the reference traverser can walk it.
//
// Pipeline (all on the device, one stream):
//   1 flatten      : world-space TriangleStorage per (instance, mesh, prim) + AABB + scene bounds
//   2 morton       : 63-bit Morton key of the AABB centre
//   3 sort         : cub::DeviceRadixSort (key, triangle id)
//   4 hierarchy    : default: PLOC (Meister & Bittner 2018) - parallel locally-ordered agglomerative clustering of the
//                    Morton-ordered leaves (each cluster merges with its mutual nearest neighbour, by surface area of
//                    the union, within +-16 positions; compaction; repeat) = a SAH-quality binary tree;
//                    GFX_BVH_BUILD_FAST: Karras 2012 binary radix tree over the sorted keys + bottom-up refit with
//                    per-node arrival counters (5.1 ms for 2.87 M triangles, ~40 % more node visits per ray)
//   5 collapse     : level-synchronous top-down collapse of the binary tree into 8-wide nodes
//                    (largest-surface-area child is opened first, like the reference's task loop
//                    :777-800), leaves of <= maxLeaf triangles (default 2), conservative 8-bit quantisation.
#include "scene.cuh"
#include "context.h"
#include <cub/cub.cuh>

namespace gfx {

__device__ __forceinline__ uint32_t orderedFromFloat(float f) {
    const uint32_t u = __float_as_uint(f);
    return u ^ (u < 0x80000000u ? 0x80000000u : 0xFFFFFFFFu);
}
__device__ __forceinline__ float floatFromOrdered(uint32_t u) {
    return __uint_as_float(u ^ (u >= 0x80000000u ? 0x80000000u : 0xFFFFFFFFu));
}

// ---- 1. flatten -----------------------------------------------------------------------------
__global__ void k_flatten(DevScene scene, const uint32_t* __restrict__ geomTriOffsets, uint32_t numGeoms,
                          uint32_t numTris, float4* __restrict__ tris, float4* __restrict__ triLo,
                          float4* __restrict__ triHi, uint32_t* __restrict__ sceneBounds /*6 ordered uints*/) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    f3 lo(INFINITY), hi(-INFINITY);
    if (t < numTris) {
        // geometry of this triangle: largest g with geomTriOffsets[g] <= t  (extractGeomAndPrimIndex,
        // common/bvh_builder.cpp:680-692)
        uint32_t g = 0;
        for (uint32_t d = 1u << (31 - __clz(max(numGeoms, 1u))); d >= 1; d >>= 1) {
            if (g + d < numGeoms && __ldg(geomTriOffsets + g + d) <= t)
                g += d;
        }
        const uint32_t prim = t - __ldg(geomTriOffsets + g);
        const uint2 im = __ldg(scene.geomToInstMesh + g);
        const DevInstance* inst = scene.instances + im.x;
        const DevMesh mesh = scene.meshes[im.y];
        const uint4 tri = __ldg(scene.triangles + mesh.triBase + prim);
        const float4 a = __ldg(scene.vertices + 3 * (size_t)(mesh.vertexBase + tri.x));
        const float4 b = __ldg(scene.vertices + 3 * (size_t)(mesh.vertexBase + tri.y));
        const float4 c = __ldg(scene.vertices + 3 * (size_t)(mesh.vertexBase + tri.z));
        // calcTriangleVertices: preTransform * p (common/bvh_builder.cpp:176-209)
        const f3 pA = xfmPoint(inst->transform, f3(a.x, a.y, a.z));
        const f3 pB = xfmPoint(inst->transform, f3(b.x, b.y, b.z));
        const f3 pC = xfmPoint(inst->transform, f3(c.x, c.y, c.z));
        tris[3 * (size_t)t + 0] = make_float4(pA.x, pA.y, pA.z, pB.x);
        tris[3 * (size_t)t + 1] = make_float4(pB.y, pB.z, pC.x, pC.y);
        tris[3 * (size_t)t + 2] = make_float4(pC.z, __uint_as_float(g), __uint_as_float(prim), 0.0f);
        lo = min3(min3(pA, pB), pC);
        hi = max3(max3(pA, pB), pC);
        triLo[t] = make_float4(lo.x, lo.y, lo.z, 0.0f);
        triHi[t] = make_float4(hi.x, hi.y, hi.z, 0.0f);
    }
    // block reduction of the scene bounds, then 6 atomics per block
    typedef cub::BlockReduce<float, 256> BR;
    __shared__ typename BR::TempStorage tmp;
    float v;
    v = BR(tmp).Reduce(lo.x, cub::Min()); __syncthreads(); if (threadIdx.x == 0) atomicMin(sceneBounds + 0, orderedFromFloat(v));
    v = BR(tmp).Reduce(lo.y, cub::Min()); __syncthreads(); if (threadIdx.x == 0) atomicMin(sceneBounds + 1, orderedFromFloat(v));
    v = BR(tmp).Reduce(lo.z, cub::Min()); __syncthreads(); if (threadIdx.x == 0) atomicMin(sceneBounds + 2, orderedFromFloat(v));
    v = BR(tmp).Reduce(hi.x, cub::Max()); __syncthreads(); if (threadIdx.x == 0) atomicMax(sceneBounds + 3, orderedFromFloat(v));
    v = BR(tmp).Reduce(hi.y, cub::Max()); __syncthreads(); if (threadIdx.x == 0) atomicMax(sceneBounds + 4, orderedFromFloat(v));
    v = BR(tmp).Reduce(hi.z, cub::Max()); __syncthreads(); if (threadIdx.x == 0) atomicMax(sceneBounds + 5, orderedFromFloat(v));
}

// ---- 2. morton ------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t expandBits21(uint64_t v) {
    v &= 0x1FFFFFull;
    v = (v | v << 32) & 0x1F00000000FFFFull;
    v = (v | v << 16) & 0x1F0000FF0000FFull;
    v = (v | v << 8) & 0x100F00F00F00F00Full;
    v = (v | v << 4) & 0x10C30C30C30C30C3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}
__global__ void k_morton(uint32_t numTris, const float4* __restrict__ triLo, const float4* __restrict__ triHi,
                         const uint32_t* __restrict__ sceneBounds, uint64_t* __restrict__ keys, uint32_t* __restrict__ ids) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= numTris)
        return;
    const f3 smin(floatFromOrdered(sceneBounds[0]), floatFromOrdered(sceneBounds[1]), floatFromOrdered(sceneBounds[2]));
    const f3 smax(floatFromOrdered(sceneBounds[3]), floatFromOrdered(sceneBounds[4]), floatFromOrdered(sceneBounds[5]));
    const float4 lo = triLo[t], hi = triHi[t];
    const f3 c(0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z));
    const f3 ext = smax - smin;
    const float sx = ext.x > 0 ? 2097151.0f / ext.x : 0.0f;
    const float sy = ext.y > 0 ? 2097151.0f / ext.y : 0.0f;
    const float sz = ext.z > 0 ? 2097151.0f / ext.z : 0.0f;
    const uint64_t qx = (uint64_t)fminf(fmaxf((c.x - smin.x) * sx, 0.0f), 2097151.0f);
    const uint64_t qy = (uint64_t)fminf(fmaxf((c.y - smin.y) * sy, 0.0f), 2097151.0f);
    const uint64_t qz = (uint64_t)fminf(fmaxf((c.z - smin.z) * sz, 0.0f), 2097151.0f);
    keys[t] = (expandBits21(qx) << 2) | (expandBits21(qy) << 1) | expandBits21(qz);
    ids[t] = t;
}

// ---- 4. Karras hierarchy --------------------------------------------------------------------
__device__ __forceinline__ int deltaKey(const uint64_t* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n)
        return -1;
    const uint64_t a = keys[i], b = keys[j];
    if (a == b)
        return 64 + __clz((uint32_t)i ^ (uint32_t)j);
    return __clzll((long long)(a ^ b));
}
// children are encoded as index | 0x80000000 for leaves
__global__ void k_hierarchy(int n, const uint64_t* __restrict__ keys, uint32_t* __restrict__ childL,
                            uint32_t* __restrict__ childR, uint32_t* __restrict__ rangeFirst,
                            uint32_t* __restrict__ rangeLast, uint32_t* __restrict__ parentOfInternal,
                            uint32_t* __restrict__ parentOfLeaf) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1)
        return;
    const int d = (deltaKey(keys, n, i, i + 1) - deltaKey(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    const int deltaMin = deltaKey(keys, n, i, i - d);
    int lmax = 2;
    while (deltaKey(keys, n, i, i + lmax * d) > deltaMin)
        lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (deltaKey(keys, n, i, i + (l + t) * d) > deltaMin)
            l += t;
    const int j = i + l * d;
    const int deltaNode = deltaKey(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) / 2;; t = (t + 1) / 2) {
        if (deltaKey(keys, n, i, i + (s + t) * d) > deltaNode)
            s += t;
        if (t == 1)
            break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int first = min(i, j), last = max(i, j);
    const uint32_t left = (first == gamma) ? ((uint32_t)gamma | 0x80000000u) : (uint32_t)gamma;
    const uint32_t right = (last == gamma + 1) ? ((uint32_t)(gamma + 1) | 0x80000000u) : (uint32_t)(gamma + 1);
    childL[i] = left;
    childR[i] = right;
    rangeFirst[i] = (uint32_t)(last - first + 1); // number of triangles below node i
    rangeLast[i] = (uint32_t)last;
    if (left & 0x80000000u) parentOfLeaf[gamma] = (uint32_t)i; else parentOfInternal[gamma] = (uint32_t)i;
    if (right & 0x80000000u) parentOfLeaf[gamma + 1] = (uint32_t)i; else parentOfInternal[gamma + 1] = (uint32_t)i;
    if (i == 0)
        parentOfInternal[0] = 0xFFFFFFFFu;
}

// ---- 5. refit -------------------------------------------------------------------------------
// binary node boxes: internal i -> boxLo/Hi[i], leaf j -> boxLo/Hi[(n-1)+j]
__global__ void k_refit(int n, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ triLo,
                        const float4* __restrict__ triHi, const uint32_t* __restrict__ childL,
                        const uint32_t* __restrict__ childR, const uint32_t* __restrict__ parentOfInternal,
                        const uint32_t* __restrict__ parentOfLeaf, uint32_t* __restrict__ counters,
                        float4* boxLo, float4* boxHi) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n)
        return;
    const uint32_t tid = sortedIds[j];
    boxLo[(n - 1) + j] = triLo[tid];
    boxHi[(n - 1) + j] = triHi[tid];
    if (n == 1)
        return;
    __threadfence();
    uint32_t p = parentOfLeaf[j];
    while (p != 0xFFFFFFFFu) {
        if (atomicAdd(counters + p, 1u) == 0u)
            return; // the sibling subtree is not done yet
        __threadfence();
        const uint32_t l = childL[p], r = childR[p];
        const uint32_t li = (l & 0x80000000u) ? (uint32_t)(n - 1) + (l & 0x7FFFFFFFu) : l;
        const uint32_t ri = (r & 0x80000000u) ? (uint32_t)(n - 1) + (r & 0x7FFFFFFFu) : r;
        const volatile float4* vlo = boxLo;
        const volatile float4* vhi = boxHi;
        const float4 a = make_float4(vlo[li].x, vlo[li].y, vlo[li].z, 0), b = make_float4(vlo[ri].x, vlo[ri].y, vlo[ri].z, 0);
        const float4 c = make_float4(vhi[li].x, vhi[li].y, vhi[li].z, 0), d = make_float4(vhi[ri].x, vhi[ri].y, vhi[ri].z, 0);
        boxLo[p] = make_float4(fminf(a.x, b.x), fminf(a.y, b.y), fminf(a.z, b.z), 0.0f);
        boxHi[p] = make_float4(fmaxf(c.x, d.x), fmaxf(c.y, d.y), fmaxf(c.z, d.z), 0.0f);
        __threadfence();
        p = parentOfInternal[p];
    }
}

// ---- 6. collapse ----------------------------------------------------------------------------
struct CollapseArgs {
    int n;                   // triangles
    uint32_t maxLeaf;
    const uint32_t* childL;
    const uint32_t* childR;
    const uint32_t* count;   // triangles below an internal node
    const float4* boxLo;
    const float4* boxHi;
    const uint32_t* sortedIds;
    uint4* nodes;            // output, 5 x uint4 per node
    uint32_t* primRefs;      // output
    uint32_t* counters;      // [0] nodes allocated, [1] primRefs allocated, [2] next-queue size
    const uint2* queueIn;    // (wide node index, binary node ref)
    uint2* queueOut;
    uint32_t queueInSize;
};

__device__ __forceinline__ uint32_t refCount(const CollapseArgs &a, uint32_t ref) {
    return (ref & 0x80000000u) ? 1u : a.count[ref];
}
__device__ __forceinline__ uint32_t refBoxIndex(const CollapseArgs &a, uint32_t ref) {
    return (ref & 0x80000000u) ? (uint32_t)(a.n - 1) + (ref & 0x7FFFFFFFu) : ref;
}

__global__ void k_collapse(CollapseArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.queueInSize)
        return;
    const uint2 item = a.queueIn[i];
    const uint32_t wide = item.x;
    const uint32_t root = item.y;

    uint32_t ch[8];
    float area[8];
    bool leafSized[8]; // child becomes a leaf of this wide node (<= maxLeaf triangles)
    int nc = 0;
    auto pushChild = [&](uint32_t ref) {
        const uint32_t bi = refBoxIndex(a, ref);
        const float4 lo = a.boxLo[bi], hi = a.boxHi[bi];
        const float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
        ch[nc] = ref;
        leafSized[nc] = refCount(a, ref) <= a.maxLeaf;
        area[nc] = dx * dy + dy * dz + dz * dx;
        ++nc;
    };
    auto openChild = [&](int k) { // replace child k in place by its left half, append the right half
        const uint32_t ref = ch[k];
        const int saved = nc;
        nc = k;
        pushChild(a.childL[ref]);
        nc = saved;
        pushChild(a.childR[ref]);
    };
    if (refCount(a, root) <= a.maxLeaf && (root & 0x80000000u)) {
        pushChild(root);
    }
    else {
        pushChild(a.childL[root]);
        pushChild(a.childR[root]);
        // phase 1: open the largest-area subtree that is too big for a leaf (the reference's task loop
        // picks the largest-surface-area splittable child the same way, bvh_builder.cpp:785-800)
        while (nc < 8) {
            int best = -1;
            float bestArea = -1.0f;
            for (int k = 0; k < nc; ++k)
                if (!leafSized[k] && area[k] > bestArea) {
                    bestArea = area[k];
                    best = k;
                }
            if (best < 0)
                break;
            openChild(best);
        }
        // phase 2: spare slots are used to split multi-triangle leaves (tighter boxes, fewer triangle
        // tests per ray, fuller nodes)
        while (nc < 8) {
            int best = -1;
            float bestArea = -1.0f;
            for (int k = 0; k < nc; ++k)
                if (leafSized[k] && !(ch[k] & 0x80000000u) && area[k] > bestArea) {
                    bestArea = area[k];
                    best = k;
                }
            if (best < 0)
                break;
            openChild(best);
        }
    }

    // classify + allocate
    uint32_t numInt = 0, numLeafPrims = 0;
    for (int k = 0; k < nc; ++k) {
        if (!leafSized[k]) ++numInt;
        else numLeafPrims += refCount(a, ch[k]);
    }
    const uint32_t nodeBase = numInt ? atomicAdd(a.counters + 0, numInt) : 0xFFFFFFFFu;
    const uint32_t primBase = numLeafPrims ? atomicAdd(a.counters + 1, numLeafPrims) : 0xFFFFFFFFu;
    const uint32_t queueBase = numInt ? atomicAdd(a.counters + 2, numInt) : 0u;

    // quantisation frame (setQuantizationAabb, common_shared.h:814-830) from the exact node box,
    // with the exponent bumped until origin + 255 * scale covers the box in float arithmetic.
    const uint32_t rbi = refBoxIndex(a, root);
    const float4 nlo = a.boxLo[rbi], nhi = a.boxHi[rbi];
    const float org[3] = { nlo.x, nlo.y, nlo.z };
    const float mx[3] = { nhi.x, nhi.y, nhi.z };
    uint32_t expo[3];
    float scale[3], recScale[3];
    for (int d = 0; d < 3; ++d) {
        const float dd = (mx[d] - org[d]) * (1.0f / 255.0f);
        const uint32_t us = __float_as_uint(dd);
        uint32_t e = (us >> 23) + ((us & 0x7FFFFFu) ? 1u : 0u);
        while (e < 254u && org[d] + 255.0f * __uint_as_float(e << 23) < mx[d])
            ++e;
        expo[d] = e;
        scale[d] = __uint_as_float(e << 23);
        recScale[d] = scale[d] != 0.0f ? 1.0f / scale[d] : 0.0f;
    }

    uint32_t qmin[3][2] = { { 0, 0 }, { 0, 0 }, { 0, 0 } }; // [axis][word]: 8 bytes as two uint32
    uint32_t qmax[3][2] = { { 0, 0 }, { 0, 0 }, { 0, 0 } };
    uint32_t metas[2] = { 0, 0 };
    uint32_t internalMask = 0;
    uint32_t nthInt = 0, leafOffset = 0;
    for (int k = 0; k < 8; ++k) {
        const int w = k >> 2, sh = 8 * (k & 3);
        if (k >= nc) { // setInvalidChildBox (common_shared.h:852-860)
            for (int d = 0; d < 3; ++d) {
                qmin[d][w] |= 255u << sh;
            }
            continue;
        }
        const uint32_t ref = ch[k];
        const uint32_t bi = refBoxIndex(a, ref);
        const float4 lo4 = a.boxLo[bi], hi4 = a.boxHi[bi];
        const float lo[3] = { lo4.x, lo4.y, lo4.z }, hi[3] = { hi4.x, hi4.y, hi4.z };
        for (int d = 0; d < 3; ++d) {
            // setChildAabb (common_shared.h:839-851) + a fix-up so that the *decoded* box
            // (origin + q * scale, rounded) always contains the child box
            int q0 = (int)dm_f2uint((lo[d] - org[d]) * recScale[d]);
            q0 = min(q0, 255);
            while (q0 > 0 && org[d] + (float)q0 * scale[d] > lo[d])
                --q0;
            int q1 = (int)min(dm_f2uint((hi[d] - org[d]) * recScale[d]) + 1u, 255u);
            while (q1 < 255 && org[d] + (float)q1 * scale[d] < hi[d])
                ++q1;
            qmin[d][w] |= (uint32_t)q0 << sh;
            qmax[d][w] |= (uint32_t)q1 << sh;
        }
        if (!leafSized[k]) {
            internalMask |= 1u << k;
            a.queueOut[queueBase + nthInt] = make_uint2(nodeBase + nthInt, ref);
            ++nthInt;
        }
        else {
            metas[w] |= leafOffset << sh;
            // the triangles of the subtree, left to right (<= maxLeaf of them)
            const uint32_t total = refCount(a, ref);
            uint32_t stack[32];
            int sp = 0;
            uint32_t written = 0;
            stack[sp++] = ref;
            while (sp > 0) {
                const uint32_t r = stack[--sp];
                if (r & 0x80000000u) {
                    a.primRefs[primBase + leafOffset + written] = a.sortedIds[r & 0x7FFFFFFFu] | (written + 1 == total ? 0x80000000u : 0u);
                    ++written;
                }
                else {
                    stack[sp++] = a.childR[r];
                    stack[sp++] = a.childL[r];
                }
            }
            leafOffset += total;
        }
    }

    uint4* np = a.nodes + 5 * (size_t)wide;
    np[0] = make_uint4(__float_as_uint(org[0]), __float_as_uint(org[1]), __float_as_uint(org[2]),
                       expo[0] | (expo[1] << 8) | (expo[2] << 16) | (internalMask << 24));
    np[1] = make_uint4(nodeBase, primBase, metas[0], metas[1]);
    np[2] = make_uint4(qmin[0][0], qmin[0][1], qmin[1][0], qmin[1][1]);
    np[3] = make_uint4(qmin[2][0], qmin[2][1], qmax[0][0], qmax[0][1]);
    np[4] = make_uint4(qmax[1][0], qmax[1][1], qmax[2][0], qmax[2][1]);
}

// ---- 4'. PLOC ------------------------------------------------------------------------------
constexpr int kPlocMaxRadius = 64;
constexpr int kPlocBlock = 256;

__global__ void k_plocInit(int n, const uint32_t* __restrict__ sortedIds, const float4* __restrict__ triLo,
                           const float4* __restrict__ triHi, uint32_t* __restrict__ clusters, float4* boxLo, float4* boxHi) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n)
        return;
    const uint32_t tid = sortedIds[j];
    boxLo[(n - 1) + j] = triLo[tid];
    boxHi[(n - 1) + j] = triHi[tid];
    clusters[j] = (uint32_t)j | 0x80000000u;
}

// nearest[i] = the cluster within +-radius positions whose union with cluster i has the smallest surface area;
// ties are broken on (min(i,j), max(i,j)) so that the globally best pair is always mutual and every pass merges
__global__ void __launch_bounds__(kPlocBlock) k_plocNearest(int m, int n, int kPlocRadius, const uint32_t* __restrict__ clusters,
                                                            const float4* __restrict__ boxLo, const float4* __restrict__ boxHi,
                                                            uint32_t* __restrict__ nearest) {
    __shared__ float sLo[kPlocBlock + 2 * kPlocMaxRadius][3];
    __shared__ float sHi[kPlocBlock + 2 * kPlocMaxRadius][3];
    const int blockStart = blockIdx.x * kPlocBlock;
    for (int t = threadIdx.x; t < kPlocBlock + 2 * kPlocRadius; t += kPlocBlock) {
        const int idx = blockStart - kPlocRadius + t;
        float4 lo = make_float4(0, 0, 0, 0), hi = lo;
        if (idx >= 0 && idx < m) {
            const uint32_t ref = clusters[idx];
            const uint32_t bi = (ref & 0x80000000u) ? (uint32_t)(n - 1) + (ref & 0x7FFFFFFFu) : ref;
            lo = boxLo[bi];
            hi = boxHi[bi];
        }
        sLo[t][0] = lo.x; sLo[t][1] = lo.y; sLo[t][2] = lo.z;
        sHi[t][0] = hi.x; sHi[t][1] = hi.y; sHi[t][2] = hi.z;
    }
    __syncthreads();
    const int i = blockStart + threadIdx.x;
    if (i >= m)
        return;
    const int li = threadIdx.x + kPlocRadius;
    const float ax = sLo[li][0], ay = sLo[li][1], az = sLo[li][2];
    const float bx = sHi[li][0], by = sHi[li][1], bz = sHi[li][2];
    float bestArea = 3.402823466e+38f;
    int best = -1;
    for (int d = -kPlocRadius; d <= kPlocRadius; ++d) {
        const int j = i + d;
        if (d == 0 || j < 0 || j >= m)
            continue;
        const int lj = li + d;
        const float dx = fmaxf(bx, sHi[lj][0]) - fminf(ax, sLo[lj][0]);
        const float dy = fmaxf(by, sHi[lj][1]) - fminf(ay, sLo[lj][1]);
        const float dz = fmaxf(bz, sHi[lj][2]) - fminf(az, sLo[lj][2]);
        const float area = dx * dy + dy * dz + dz * dx;
        bool better = area < bestArea;
        if (area == bestArea && best >= 0) {
            const int a0 = min(i, j), a1 = max(i, j), b0 = min(i, best), b1 = max(i, best);
            better = a0 < b0 || (a0 == b0 && a1 < b1);
        }
        if (better) {
            bestArea = area;
            best = j;
        }
    }
    nearest[i] = (uint32_t)best;
}

__global__ void k_plocMerge(int m, int n, const uint32_t* __restrict__ clusters, const uint32_t* __restrict__ nearest,
                            uint32_t* __restrict__ childL, uint32_t* __restrict__ childR, uint32_t* __restrict__ count,
                            float4* boxLo, float4* boxHi, uint32_t* __restrict__ nodeCounter, uint32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m)
        return;
    const uint32_t j = nearest[i];
    const uint32_t self = clusters[i];
    if (j >= (uint32_t)m || nearest[j] != (uint32_t)i) {
        out[i] = self;
        return;
    }
    if ((uint32_t)i > j) {
        out[i] = 0xFFFFFFFFu; // absorbed by its partner
        return;
    }
    const uint32_t other = clusters[j];
    const uint32_t node = atomicAdd(nodeCounter, 1u);
    const uint32_t bi = (self & 0x80000000u) ? (uint32_t)(n - 1) + (self & 0x7FFFFFFFu) : self;
    const uint32_t bj = (other & 0x80000000u) ? (uint32_t)(n - 1) + (other & 0x7FFFFFFFu) : other;
    const float4 alo = boxLo[bi], ahi = boxHi[bi], blo = boxLo[bj], bhi = boxHi[bj];
    childL[node] = self;
    childR[node] = other;
    count[node] = ((self & 0x80000000u) ? 1u : count[self]) + ((other & 0x80000000u) ? 1u : count[other]);
    boxLo[node] = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.0f);
    boxHi[node] = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.0f);
    out[i] = node;
}

// ---- 4''. binned SAH, top-down ----------------------------------------------------------------
// Default hierarchy for static scenes.  Level-synchronous: every open node of a level is split by ONE thread block
// (1024 threads for nodes above kSahBigNode triangles, 64 below), which
//   1. reduces the node's AABB and the bounds of its triangle centroids,
//   2. bins the centroids into 16 bins on each axis (shared-memory atomics on order-preserving integer images of the
//      float bounds, so the result does not depend on the order of the atomics),
//   3. evaluates the 3 x 15 split planes with the surface-area heuristic  A_L N_L + A_R N_R  (Wald 2007),
//   4. partitions its slice of the triangle order stably (ballot ranks + running offsets) and opens two children.
// The reference builds its hierarchy with the same heuristic on the CPU (bvh_builder.cpp:656-1125, binned object
// splits + spatial splits); the 8-wide collapse below is shared with the other two hierarchies.
constexpr uint32_t kSahBins = 16;
constexpr uint32_t kSahBigNode = 4096;
// Above this a node is split by MANY blocks (k_sahHuge*): in round 1 the first five levels - one 1024-thread block per node,
// i.e. one SM for the root's 2.87 M triangles - took 45 of the builder's 65 ms.
constexpr uint32_t kSahHugeNode = 131072;
constexpr uint32_t kSahHugeChunk = 8192;  // triangles per block of the multi-block passes

struct SahArgs {
    uint32_t n;
    const float4* triLo;
    const float4* triHi;
    uint32_t* order;      // triangle ids, partitioned in place level by level
    uint32_t* scratch;
    uint32_t* childL;
    uint32_t* childR;
    uint32_t* count;
    float4* boxLo;
    float4* boxHi;
    uint32_t* counters;   // [0] next small-list size, [1] next big-list size, [2] internal nodes allocated, [3] next huge-list size
    const uint4* listIn;  // (node, start, end, -)
    uint4* smallOut;
    uint4* bigOut;
    uint4* hugeOut;
    uint32_t listSize;
};

// where a child slice goes next: one-triangle leaves are references, everything else gets a node index and a work record
__device__ __forceinline__ uint32_t sahEmitChild(const SahArgs &a, uint32_t first, uint32_t last) {
    const uint32_t cnum = last - first;
    if (cnum == 1)
        return 0x80000000u | first;
    const uint32_t idx = atomicAdd(a.counters + 2, 1u);
    const uint4 out = make_uint4(idx, first, last, 0u);
    if (cnum > kSahHugeNode)
        a.hugeOut[atomicAdd(a.counters + 3, 1u)] = out;
    else if (cnum > kSahBigNode)
        a.bigOut[atomicAdd(a.counters + 1, 1u)] = out;
    else
        a.smallOut[atomicAdd(a.counters + 0, 1u)] = out;
    return idx;
}

template <uint32_t BLOCK>
__global__ void __launch_bounds__(BLOCK) k_sahSplit(SahArgs a) {
    constexpr uint32_t WARPS = BLOCK / 32;
    __shared__ uint32_t sBoundsLo[2][3], sBoundsHi[2][3];            // [0] AABB, [1] centroid bounds (ordered ints)
    // one private copy of the bins per warp keeps the shared-memory atomics of a 1024-thread block from serialising on
    // 16 addresses; copy 0 receives the reduction
    __shared__ uint32_t sBinLo[WARPS][3][kSahBins][3], sBinHi[WARPS][3][kSahBins][3], sBinCount[WARPS][3][kSahBins];
    __shared__ float sAxisCost[3];
    __shared__ uint32_t sAxisPlane[3], sAxisLeft[3];
    __shared__ uint32_t sSplitAxis, sSplitPlane, sNumLeft;
    __shared__ uint32_t sWarpL[WARPS], sWarpR[WARPS];
    __shared__ uint32_t sRunL, sRunR;

    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint4 rec = a.listIn[blockIdx.x];
    const uint32_t node = rec.x, start = rec.y, end = rec.z;
    const uint32_t num = end - start;

    if (tid < 3) {
        sBoundsLo[0][tid] = sBoundsLo[1][tid] = 0xFFFFFFFFu;
        sBoundsHi[0][tid] = sBoundsHi[1][tid] = 0u;
    }
    for (uint32_t i = tid; i < WARPS * 3 * kSahBins * 3; i += BLOCK) {
        (&sBinLo[0][0][0][0])[i] = 0xFFFFFFFFu;
        (&sBinHi[0][0][0][0])[i] = 0u;
    }
    for (uint32_t i = tid; i < WARPS * 3 * kSahBins; i += BLOCK)
        (&sBinCount[0][0][0])[i] = 0u;
    __syncthreads();

    // 1. bounds
    {
        float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
        float clo[3] = { INFINITY, INFINITY, INFINITY }, chi[3] = { -INFINITY, -INFINITY, -INFINITY };
        for (uint32_t i = start + tid; i < end; i += BLOCK) {
            const uint32_t t = a.order[i];
            const float4 l = a.triLo[t], h = a.triHi[t];
            const float bl[3] = { l.x, l.y, l.z }, bh[3] = { h.x, h.y, h.z };
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                const float c = 0.5f * bl[d] + 0.5f * bh[d];
                lo[d] = fminf(lo[d], bl[d]); hi[d] = fmaxf(hi[d], bh[d]);
                clo[d] = fminf(clo[d], c); chi[d] = fmaxf(chi[d], c);
            }
        }
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            for (int off = 16; off > 0; off >>= 1) {
                lo[d] = fminf(lo[d], __shfl_xor_sync(0xFFFFFFFFu, lo[d], off));
                hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xFFFFFFFFu, hi[d], off));
                clo[d] = fminf(clo[d], __shfl_xor_sync(0xFFFFFFFFu, clo[d], off));
                chi[d] = fmaxf(chi[d], __shfl_xor_sync(0xFFFFFFFFu, chi[d], off));
            }
            if (lane == 0) {
                atomicMin(&sBoundsLo[0][d], orderedFromFloat(lo[d]));
                atomicMax(&sBoundsHi[0][d], orderedFromFloat(hi[d]));
                atomicMin(&sBoundsLo[1][d], orderedFromFloat(clo[d]));
                atomicMax(&sBoundsHi[1][d], orderedFromFloat(chi[d]));
            }
        }
    }
    __syncthreads();
    float cLo[3], binScale[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        cLo[d] = floatFromOrdered(sBoundsLo[1][d]);
        const float ext = floatFromOrdered(sBoundsHi[1][d]) - cLo[d];
        binScale[d] = ext > 0.0f ? (float)kSahBins / ext : 0.0f;
    }
    if (tid == 0) {
        a.boxLo[node] = make_float4(floatFromOrdered(sBoundsLo[0][0]), floatFromOrdered(sBoundsLo[0][1]), floatFromOrdered(sBoundsLo[0][2]), 0.0f);
        a.boxHi[node] = make_float4(floatFromOrdered(sBoundsHi[0][0]), floatFromOrdered(sBoundsHi[0][1]), floatFromOrdered(sBoundsHi[0][2]), 0.0f);
        a.count[node] = num;
    }
    auto binOf = [&](float c, int d) -> uint32_t {
        const float f = (c - cLo[d]) * binScale[d];
        const uint32_t b = (uint32_t)fmaxf(f, 0.0f);
        return b < kSahBins - 1 ? b : kSahBins - 1;
    };

    // 2. binning.  Each thread walks a contiguous run of the slice: neighbours in the (initially Morton) order fall
    // into the same bin, so a strided assignment would make all lanes of a warp hit one address per atomic.
    const uint32_t perThread = (num + BLOCK - 1) / BLOCK;
    const uint32_t runBegin = min(end, start + tid * perThread), runEnd = min(end, runBegin + perThread);
    for (uint32_t i = runBegin; i < runEnd; ++i) {
        const uint32_t t = a.order[i];
        const float4 l = a.triLo[t], h = a.triHi[t];
        const float bl[3] = { l.x, l.y, l.z }, bh[3] = { h.x, h.y, h.z };
        const uint32_t ol[3] = { orderedFromFloat(l.x), orderedFromFloat(l.y), orderedFromFloat(l.z) };
        const uint32_t oh[3] = { orderedFromFloat(h.x), orderedFromFloat(h.y), orderedFromFloat(h.z) };
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const uint32_t b = binOf(0.5f * bl[d] + 0.5f * bh[d], d);
            atomicAdd(&sBinCount[warp][d][b], 1u);
#pragma unroll
            for (int e = 0; e < 3; ++e) {
                atomicMin(&sBinLo[warp][d][b][e], ol[e]);
                atomicMax(&sBinHi[warp][d][b][e], oh[e]);
            }
        }
    }
    __syncthreads();
    if (WARPS > 1) {
        for (uint32_t i = tid; i < 3 * kSahBins * 3; i += BLOCK) {
            uint32_t lo = 0xFFFFFFFFu, hi = 0u;
            for (uint32_t w = 0; w < WARPS; ++w) {
                lo = min(lo, (&sBinLo[w][0][0][0])[i]);
                hi = max(hi, (&sBinHi[w][0][0][0])[i]);
            }
            (&sBinLo[0][0][0][0])[i] = lo;
            (&sBinHi[0][0][0][0])[i] = hi;
        }
        for (uint32_t i = tid; i < 3 * kSahBins; i += BLOCK) {
            uint32_t c = 0;
            for (uint32_t w = 0; w < WARPS; ++w)
                c += (&sBinCount[w][0][0])[i];
            (&sBinCount[0][0][0])[i] = c;
        }
        __syncthreads();
    }

    // 3. plane evaluation, one thread per axis
    if (tid < 3) {
        const int d = (int)tid;
        float rightArea[kSahBins];
        uint32_t rightCount[kSahBins];
        float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
        uint32_t cnt = 0;
        for (int b = (int)kSahBins - 1; b >= 1; --b) {
            if (sBinCount[0][d][b]) {
                for (int e = 0; e < 3; ++e) {
                    lo[e] = fminf(lo[e], floatFromOrdered(sBinLo[0][d][b][e]));
                    hi[e] = fmaxf(hi[e], floatFromOrdered(sBinHi[0][d][b][e]));
                }
                cnt += sBinCount[0][d][b];
            }
            const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
            rightArea[b] = cnt ? ex * ey + ey * ez + ez * ex : 0.0f;
            rightCount[b] = cnt;
        }
        for (int e = 0; e < 3; ++e) { lo[e] = INFINITY; hi[e] = -INFINITY; }
        cnt = 0;
        float bestCost = INFINITY;
        uint32_t bestPlane = 0, bestLeft = 0;
        for (int b = 0; b < (int)kSahBins - 1; ++b) { // plane b+1: bins 0..b left
            if (sBinCount[0][d][b]) {
                for (int e = 0; e < 3; ++e) {
                    lo[e] = fminf(lo[e], floatFromOrdered(sBinLo[0][d][b][e]));
                    hi[e] = fmaxf(hi[e], floatFromOrdered(sBinHi[0][d][b][e]));
                }
                cnt += sBinCount[0][d][b];
            }
            if (cnt == 0 || rightCount[b + 1] == 0)
                continue;
            const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
            const float cost = (ex * ey + ey * ez + ez * ex) * (float)cnt + rightArea[b + 1] * (float)rightCount[b + 1];
            if (cost < bestCost) {
                bestCost = cost;
                bestPlane = (uint32_t)b + 1;
                bestLeft = cnt;
            }
        }
        sAxisCost[d] = bestCost;
        sAxisPlane[d] = bestPlane;
        sAxisLeft[d] = bestLeft;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t axis = 0;
        if (sAxisCost[1] < sAxisCost[axis]) axis = 1;
        if (sAxisCost[2] < sAxisCost[axis]) axis = 2;
        sSplitAxis = axis;
        sSplitPlane = sAxisPlane[axis];       // 0: all centroids coincide -> split the slice in the middle
        sNumLeft = sAxisPlane[axis] ? sAxisLeft[axis] : num / 2;
        sRunL = 0;
        sRunR = 0;
    }
    __syncthreads();
    const uint32_t axis = sSplitAxis, plane = sSplitPlane, numLeft = sNumLeft;

    // 4. stable partition through the scratch buffer
    if (plane) {
        for (uint32_t base = start; base < end; base += BLOCK) {
            const uint32_t i = base + tid;
            const bool valid = i < end;
            uint32_t t = 0;
            bool left = false;
            if (valid) {
                t = a.order[i];
                const float4 l = a.triLo[t], h = a.triHi[t];
                const float c = axis == 0 ? 0.5f * l.x + 0.5f * h.x : axis == 1 ? 0.5f * l.y + 0.5f * h.y : 0.5f * l.z + 0.5f * h.z;
                left = binOf(c, (int)axis) < plane;
            }
            const uint32_t ballotL = __ballot_sync(0xFFFFFFFFu, valid && left);
            const uint32_t ballotR = __ballot_sync(0xFFFFFFFFu, valid && !left);
            if (lane == 0) {
                sWarpL[warp] = __popc(ballotL);
                sWarpR[warp] = __popc(ballotR);
            }
            __syncthreads();
            uint32_t offL = sRunL, offR = sRunR, totL = 0, totR = 0;
            for (uint32_t w = 0; w < WARPS; ++w) {
                if (w < warp) { offL += sWarpL[w]; offR += sWarpR[w]; }
                totL += sWarpL[w]; totR += sWarpR[w];
            }
            if (valid) {
                const uint32_t lt = (1u << lane) - 1u;
                if (left)
                    a.scratch[start + offL + __popc(ballotL & lt)] = t;
                else
                    a.scratch[start + numLeft + offR + __popc(ballotR & lt)] = t;
            }
            __syncthreads();
            if (tid == 0) {
                sRunL += totL;
                sRunR += totR;
            }
            __syncthreads();
        }
        for (uint32_t i = start + tid; i < end; i += BLOCK)
            a.order[i] = a.scratch[i];
    }

    // 5. children
    if (tid == 0) {
        a.childL[node] = sahEmitChild(a, start, start + numLeft);
        a.childR[node] = sahEmitChild(a, start + numLeft, end);
    }
}

// ---- the same split for huge nodes, spread over many blocks ------------------------------------------------------------
// Per node one SahHugeNode record in global memory; bounds and bins are min / max / count over order-preserving integer images,
// so the merged result - hence the chosen plane - does not depend on how the triangles are spread over blocks, and the
// partition is stable (per-block left / right counts, a scan per node, then a scatter with those offsets): the tree is the
// one k_sahSplit would build.
struct SahHugeNode {
    uint32_t boundsLo[2][3], boundsHi[2][3];   // [0] AABB, [1] centroid bounds
    uint32_t binLo[3][kSahBins][3], binHi[3][kSahBins][3], binCount[3][kSahBins];
    uint32_t splitAxis, splitPlane, numLeft, firstBlock;
};
struct SahHugeArgs {
    SahArgs a;
    SahHugeNode* nodes;     // one per entry of a.listIn
    uint32_t* blockLeft;    // per block: triangles of its chunk that go left; then the block's left offset
    uint32_t* blockRight;   // per block: right offset
};
// block -> (list entry, chunk) by walking the (short) list
__device__ __forceinline__ bool sahHugeLocate(const SahArgs &a, uint32_t block, uint32_t* entry, uint32_t* chunkBegin, uint32_t* chunkEnd) {
    uint32_t first = 0;
    for (uint32_t e = 0; e < a.listSize; ++e) {
        const uint4 rec = a.listIn[e];
        const uint32_t blocks = (rec.z - rec.y + kSahHugeChunk - 1) / kSahHugeChunk;
        if (block < first + blocks) {
            *entry = e;
            *chunkBegin = rec.y + (block - first) * kSahHugeChunk;
            *chunkEnd = min(rec.z, *chunkBegin + kSahHugeChunk);
            return true;
        }
        first += blocks;
    }
    return false;
}
__global__ void k_sahHugeInit(SahHugeArgs h) {
    SahHugeNode &N = h.nodes[blockIdx.x];
    uint32_t* w = reinterpret_cast<uint32_t*>(&N);
    for (uint32_t i = threadIdx.x; i < sizeof(SahHugeNode) / 4; i += blockDim.x)
        w[i] = 0u;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < 6; i += blockDim.x)
        (&N.boundsLo[0][0])[i] = 0xFFFFFFFFu;
    for (uint32_t i = threadIdx.x; i < 3 * kSahBins * 3; i += blockDim.x)
        (&N.binLo[0][0][0])[i] = 0xFFFFFFFFu;
    if (threadIdx.x == 0) { // first block of this node in the level's block numbering
        uint32_t first = 0;
        for (uint32_t e = 0; e < blockIdx.x; ++e)
            first += (h.a.listIn[e].z - h.a.listIn[e].y + kSahHugeChunk - 1) / kSahHugeChunk;
        N.firstBlock = first;
    }
}
__global__ void __launch_bounds__(1024) k_sahHugeBounds(SahHugeArgs h) {
    uint32_t entry, begin, end;
    if (!sahHugeLocate(h.a, blockIdx.x, &entry, &begin, &end))
        return;
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    float clo[3] = { INFINITY, INFINITY, INFINITY }, chi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (uint32_t i = begin + threadIdx.x; i < end; i += blockDim.x) {
        const uint32_t t = h.a.order[i];
        const float4 l = h.a.triLo[t], u = h.a.triHi[t];
        const float bl[3] = { l.x, l.y, l.z }, bh[3] = { u.x, u.y, u.z };
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float c = 0.5f * bl[d] + 0.5f * bh[d];
            lo[d] = fminf(lo[d], bl[d]); hi[d] = fmaxf(hi[d], bh[d]);
            clo[d] = fminf(clo[d], c); chi[d] = fmaxf(chi[d], c);
        }
    }
    SahHugeNode &N = h.nodes[entry];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        for (int off = 16; off > 0; off >>= 1) {
            lo[d] = fminf(lo[d], __shfl_xor_sync(0xFFFFFFFFu, lo[d], off));
            hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xFFFFFFFFu, hi[d], off));
            clo[d] = fminf(clo[d], __shfl_xor_sync(0xFFFFFFFFu, clo[d], off));
            chi[d] = fmaxf(chi[d], __shfl_xor_sync(0xFFFFFFFFu, chi[d], off));
        }
        if ((threadIdx.x & 31u) == 0) {
            atomicMin(&N.boundsLo[0][d], orderedFromFloat(lo[d]));
            atomicMax(&N.boundsHi[0][d], orderedFromFloat(hi[d]));
            atomicMin(&N.boundsLo[1][d], orderedFromFloat(clo[d]));
            atomicMax(&N.boundsHi[1][d], orderedFromFloat(chi[d]));
        }
    }
}
struct SahBinning { // centroid -> bin, exactly k_sahSplit's
    float cLo[3], binScale[3];
    __device__ __forceinline__ SahBinning(const uint32_t (*boundsLo)[3], const uint32_t (*boundsHi)[3]) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            cLo[d] = floatFromOrdered(boundsLo[1][d]);
            const float ext = floatFromOrdered(boundsHi[1][d]) - cLo[d];
            binScale[d] = ext > 0.0f ? (float)kSahBins / ext : 0.0f;
        }
    }
    __device__ __forceinline__ uint32_t binOf(float c, int d) const {
        const float f = (c - cLo[d]) * binScale[d];
        const uint32_t b = (uint32_t)fmaxf(f, 0.0f);
        return b < kSahBins - 1 ? b : kSahBins - 1;
    }
};
__global__ void __launch_bounds__(1024) k_sahHugeBin(SahHugeArgs h) {
    constexpr uint32_t WARPS = 32;
    __shared__ uint32_t sBinLo[WARPS][3][kSahBins][3], sBinHi[WARPS][3][kSahBins][3], sBinCount[WARPS][3][kSahBins];
    uint32_t entry, begin, end;
    if (!sahHugeLocate(h.a, blockIdx.x, &entry, &begin, &end))
        return;
    SahHugeNode &N = h.nodes[entry];
    const uint32_t tid = threadIdx.x, warp = tid >> 5;
    for (uint32_t i = tid; i < WARPS * 3 * kSahBins * 3; i += 1024) {
        (&sBinLo[0][0][0][0])[i] = 0xFFFFFFFFu;
        (&sBinHi[0][0][0][0])[i] = 0u;
    }
    for (uint32_t i = tid; i < WARPS * 3 * kSahBins; i += 1024)
        (&sBinCount[0][0][0])[i] = 0u;
    __syncthreads();
    const SahBinning binning(N.boundsLo, N.boundsHi);
    const uint32_t num = end - begin, perThread = (num + 1023) / 1024;
    const uint32_t runBegin = min(end, begin + tid * perThread), runEnd = min(end, runBegin + perThread);
    for (uint32_t i = runBegin; i < runEnd; ++i) {
        const uint32_t t = h.a.order[i];
        const float4 l = h.a.triLo[t], u = h.a.triHi[t];
        const float bl[3] = { l.x, l.y, l.z }, bh[3] = { u.x, u.y, u.z };
        const uint32_t ol[3] = { orderedFromFloat(l.x), orderedFromFloat(l.y), orderedFromFloat(l.z) };
        const uint32_t oh[3] = { orderedFromFloat(u.x), orderedFromFloat(u.y), orderedFromFloat(u.z) };
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const uint32_t b = binning.binOf(0.5f * bl[d] + 0.5f * bh[d], d);
            atomicAdd(&sBinCount[warp][d][b], 1u);
#pragma unroll
            for (int e = 0; e < 3; ++e) {
                atomicMin(&sBinLo[warp][d][b][e], ol[e]);
                atomicMax(&sBinHi[warp][d][b][e], oh[e]);
            }
        }
    }
    __syncthreads();
    for (uint32_t i = tid; i < 3 * kSahBins * 3; i += 1024) {
        uint32_t lo = 0xFFFFFFFFu, hi = 0u;
        for (uint32_t w = 0; w < WARPS; ++w) {
            lo = min(lo, (&sBinLo[w][0][0][0])[i]);
            hi = max(hi, (&sBinHi[w][0][0][0])[i]);
        }
        if (lo != 0xFFFFFFFFu)
            atomicMin(&N.binLo[0][0][0] + i, lo);
        if (hi != 0u)
            atomicMax(&N.binHi[0][0][0] + i, hi);
    }
    for (uint32_t i = tid; i < 3 * kSahBins; i += 1024) {
        uint32_t c = 0;
        for (uint32_t w = 0; w < WARPS; ++w)
            c += (&sBinCount[w][0][0])[i];
        if (c)
            atomicAdd(&N.binCount[0][0] + i, c);
    }
}
// plane evaluation (k_sahSplit step 3) and the node's box, one block of 32 threads per node
__global__ void k_sahHugeEval(SahHugeArgs h) {
    __shared__ float sAxisCost[3];
    __shared__ uint32_t sAxisPlane[3], sAxisLeft[3];
    SahHugeNode &N = h.nodes[blockIdx.x];
    const uint4 rec = h.a.listIn[blockIdx.x];
    const uint32_t node = rec.x, num = rec.z - rec.y;
    const uint32_t tid = threadIdx.x;
    if (tid < 3) {
        const int d = (int)tid;
        float rightArea[kSahBins];
        uint32_t rightCount[kSahBins];
        float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
        uint32_t cnt = 0;
        for (int b = (int)kSahBins - 1; b >= 1; --b) {
            if (N.binCount[d][b]) {
                for (int e = 0; e < 3; ++e) {
                    lo[e] = fminf(lo[e], floatFromOrdered(N.binLo[d][b][e]));
                    hi[e] = fmaxf(hi[e], floatFromOrdered(N.binHi[d][b][e]));
                }
                cnt += N.binCount[d][b];
            }
            const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
            rightArea[b] = cnt ? ex * ey + ey * ez + ez * ex : 0.0f;
            rightCount[b] = cnt;
        }
        for (int e = 0; e < 3; ++e) { lo[e] = INFINITY; hi[e] = -INFINITY; }
        cnt = 0;
        float bestCost = INFINITY;
        uint32_t bestPlane = 0, bestLeft = 0;
        for (int b = 0; b < (int)kSahBins - 1; ++b) {
            if (N.binCount[d][b]) {
                for (int e = 0; e < 3; ++e) {
                    lo[e] = fminf(lo[e], floatFromOrdered(N.binLo[d][b][e]));
                    hi[e] = fmaxf(hi[e], floatFromOrdered(N.binHi[d][b][e]));
                }
                cnt += N.binCount[d][b];
            }
            if (cnt == 0 || rightCount[b + 1] == 0)
                continue;
            const float ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
            const float cost = (ex * ey + ey * ez + ez * ex) * (float)cnt + rightArea[b + 1] * (float)rightCount[b + 1];
            if (cost < bestCost) {
                bestCost = cost;
                bestPlane = (uint32_t)b + 1;
                bestLeft = cnt;
            }
        }
        sAxisCost[d] = bestCost;
        sAxisPlane[d] = bestPlane;
        sAxisLeft[d] = bestLeft;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t axis = 0;
        if (sAxisCost[1] < sAxisCost[axis]) axis = 1;
        if (sAxisCost[2] < sAxisCost[axis]) axis = 2;
        N.splitAxis = axis;
        N.splitPlane = sAxisPlane[axis];
        N.numLeft = sAxisPlane[axis] ? sAxisLeft[axis] : num / 2;
        h.a.boxLo[node] = make_float4(floatFromOrdered(N.boundsLo[0][0]), floatFromOrdered(N.boundsLo[0][1]), floatFromOrdered(N.boundsLo[0][2]), 0.0f);
        h.a.boxHi[node] = make_float4(floatFromOrdered(N.boundsHi[0][0]), floatFromOrdered(N.boundsHi[0][1]), floatFromOrdered(N.boundsHi[0][2]), 0.0f);
        h.a.count[node] = num;
    }
}
__device__ __forceinline__ bool sahHugeGoesLeft(const SahHugeArgs &h, const SahHugeNode &N, const SahBinning &binning, uint32_t t) {
    const float4 l = h.a.triLo[t], u = h.a.triHi[t];
    const uint32_t axis = N.splitAxis;
    const float c = axis == 0 ? 0.5f * l.x + 0.5f * u.x : axis == 1 ? 0.5f * l.y + 0.5f * u.y : 0.5f * l.z + 0.5f * u.z;
    return binning.binOf(c, (int)axis) < N.splitPlane;
}
__global__ void __launch_bounds__(1024) k_sahHugeCount(SahHugeArgs h) {
    __shared__ uint32_t sLeft;
    uint32_t entry, begin, end;
    if (!sahHugeLocate(h.a, blockIdx.x, &entry, &begin, &end))
        return;
    const SahHugeNode &N = h.nodes[entry];
    if (threadIdx.x == 0)
        sLeft = 0;
    __syncthreads();
    uint32_t left = 0;
    if (N.splitPlane) {
        const SahBinning binning(N.boundsLo, N.boundsHi);
        for (uint32_t i = begin + threadIdx.x; i < end; i += blockDim.x)
            left += sahHugeGoesLeft(h, N, binning, h.a.order[i]) ? 1u : 0u;
    }
    for (int off = 16; off > 0; off >>= 1)
        left += __shfl_xor_sync(0xFFFFFFFFu, left, off);
    if ((threadIdx.x & 31u) == 0 && left)
        atomicAdd(&sLeft, left);
    __syncthreads();
    if (threadIdx.x == 0)
        h.blockLeft[blockIdx.x] = sLeft;
}
// per node: block offsets of the stable partition, and the two children
__global__ void k_sahHugeOffsets(SahHugeArgs h) {
    if (threadIdx.x != 0)
        return;
    const SahHugeNode &N = h.nodes[blockIdx.x];
    const uint4 rec = h.a.listIn[blockIdx.x];
    const uint32_t blocks = (rec.z - rec.y + kSahHugeChunk - 1) / kSahHugeChunk;
    uint32_t offL = 0, offR = 0;
    for (uint32_t b = 0; b < blocks; ++b) {
        const uint32_t chunk = min(kSahHugeChunk, rec.z - rec.y - b * kSahHugeChunk);
        const uint32_t left = h.blockLeft[N.firstBlock + b];
        h.blockLeft[N.firstBlock + b] = offL;
        h.blockRight[N.firstBlock + b] = offR;
        offL += left;
        offR += chunk - left;
    }
    h.a.childL[rec.x] = sahEmitChild(h.a, rec.y, rec.y + N.numLeft);
    h.a.childR[rec.x] = sahEmitChild(h.a, rec.y + N.numLeft, rec.z);
}
__global__ void __launch_bounds__(1024) k_sahHugeScatter(SahHugeArgs h) {
    constexpr uint32_t WARPS = 32;
    __shared__ uint32_t sWarpL[WARPS], sWarpR[WARPS];
    __shared__ uint32_t sRunL, sRunR;
    uint32_t entry, begin, end;
    if (!sahHugeLocate(h.a, blockIdx.x, &entry, &begin, &end))
        return;
    const SahHugeNode &N = h.nodes[entry];
    if (!N.splitPlane)
        return; // all centroids coincide: the slice is cut in the middle as it stands
    const uint4 rec = h.a.listIn[entry];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const SahBinning binning(N.boundsLo, N.boundsHi);
    if (tid == 0) {
        sRunL = h.blockLeft[blockIdx.x];
        sRunR = h.blockRight[blockIdx.x];
    }
    __syncthreads();
    for (uint32_t base = begin; base < end; base += 1024) {
        const uint32_t i = base + tid;
        const bool valid = i < end;
        uint32_t t = 0;
        bool left = false;
        if (valid) {
            t = h.a.order[i];
            left = sahHugeGoesLeft(h, N, binning, t);
        }
        const uint32_t ballotL = __ballot_sync(0xFFFFFFFFu, valid && left);
        const uint32_t ballotR = __ballot_sync(0xFFFFFFFFu, valid && !left);
        if (lane == 0) {
            sWarpL[warp] = __popc(ballotL);
            sWarpR[warp] = __popc(ballotR);
        }
        __syncthreads();
        uint32_t offL = sRunL, offR = sRunR, totL = 0, totR = 0;
        for (uint32_t w = 0; w < WARPS; ++w) {
            if (w < warp) { offL += sWarpL[w]; offR += sWarpR[w]; }
            totL += sWarpL[w]; totR += sWarpR[w];
        }
        if (valid) {
            const uint32_t lt = (1u << lane) - 1u;
            if (left)
                h.a.scratch[rec.y + offL + __popc(ballotL & lt)] = t;
            else
                h.a.scratch[rec.y + N.numLeft + offR + __popc(ballotR & lt)] = t;
        }
        __syncthreads();
        if (tid == 0) {
            sRunL += totL;
            sRunR += totR;
        }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(1024) k_sahHugeCopyBack(SahHugeArgs h) {
    uint32_t entry, begin, end;
    if (!sahHugeLocate(h.a, blockIdx.x, &entry, &begin, &end))
        return;
    if (!h.nodes[entry].splitPlane)
        return;
    for (uint32_t i = begin + threadIdx.x; i < end; i += blockDim.x)
        h.a.order[i] = h.a.scratch[i];
}

// leaf boxes in their final order
__global__ void k_sahLeafBoxes(int n, const uint32_t* __restrict__ order, const float4* __restrict__ triLo,
                               const float4* __restrict__ triHi, float4* boxLo, float4* boxHi) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n)
        return;
    const uint32_t t = order[j];
    boxLo[(n - 1) + j] = triLo[t];
    boxHi[(n - 1) + j] = triHi[t];
}

struct PlocValid {
    __device__ __forceinline__ bool operator()(const uint32_t &v) const { return v != 0xFFFFFFFFu; }
};

__global__ void k_initBounds(uint32_t* sceneBounds) {
    if (threadIdx.x < 3) sceneBounds[threadIdx.x] = 0xFFFFFFFFu;
    else if (threadIdx.x < 6) sceneBounds[threadIdx.x] = 0u;
}

// ---------------------------------------------------------------------------------------------
int buildBvh(gfx_ctx* ctx, cudaStream_t stream, uint32_t flags) {
    SceneState &S = ctx->scene;
    const uint32_t n = S.numFlatTris;
    uint32_t maxLeaf = flags & 0xFFu;
    if (maxLeaf == 0) maxLeaf = 2; // measured on config 2: 2-3 triangles per leaf trace fastest (tools/bvh_quality.py --sweep)
    if (maxLeaf > 31) maxLeaf = 31;

    BvhState &B = ctx->bvh;
    // Output arrays and scratch are kept between builds of the same triangle count (per-frame rebuilds of an animated scene:
    // ~30 cudaMalloc / cudaFree pairs per build were a third of the rebuild time in round 1); anything else re-allocates.
    if (B.builtForTris != n) {
        B.release();
        B.builtForTris = 0;
    }
    B.ready = false;
    B.numTris = n;
    if (n == 0) {
        B.numNodes = 0;
        B.numPrimRefs = 0;
        return GFX_OK;
    }
    // scratch, carved out of one arena
    float4 *triLo, *triHi, *boxLo, *boxHi;
    uint64_t *keys, *keysSorted;
    uint32_t *ids, *idsSorted, *childL, *childR, *rangeFirst, *rangeLast, *parentI, *parentL, *arrive, *counters;
    uint2 *queueA, *queueB;
    uint4 *bigListStore[2], *hugeListStore[2];
    void *tmp, *selTmp, *hugeNodeStore;
    uint32_t* hugeBlockStore;
    const uint32_t bigCapacity = n / kSahBigNode + 2, hugeCapacity = n / kSahHugeNode + 2;
    const uint32_t hugeMaxBlocks = n / kSahHugeChunk + hugeCapacity + 1;
    size_t tmpBytes = 0, selBytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmpBytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                    (uint32_t*)nullptr, (int)n, 0, 63, stream);
    cub::DeviceSelect::If(nullptr, selBytes, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, PlocValid(), stream);
    {
        size_t offset = 0;
        auto take = [&](size_t bytes) { const size_t at = offset; offset += (bytes + 255) & ~(size_t)255; return at; };
        const size_t oTriLo = take((size_t)n * 16), oTriHi = take((size_t)n * 16), oBoxLo = take((size_t)2 * n * 16), oBoxHi = take((size_t)2 * n * 16);
        const size_t oKeys = take((size_t)n * 8), oKeysSorted = take((size_t)n * 8), oIds = take((size_t)n * 4), oIdsSorted = take((size_t)n * 4);
        const size_t oChildL = take((size_t)n * 4), oChildR = take((size_t)n * 4), oRangeFirst = take((size_t)n * 4), oRangeLast = take((size_t)n * 4);
        const size_t oParentI = take((size_t)n * 4), oParentL = take((size_t)n * 4), oArrive = take((size_t)n * 4), oCounters = take(16);
        const size_t oQueueA = take((size_t)n * 8), oQueueB = take((size_t)n * 8);
        const size_t oBig0 = take((size_t)bigCapacity * 16), oBig1 = take((size_t)bigCapacity * 16);
        const size_t oHuge0 = take((size_t)hugeCapacity * 16), oHuge1 = take((size_t)hugeCapacity * 16);
        const size_t oHugeNodes = take((size_t)hugeCapacity * sizeof(SahHugeNode)), oHugeBlocks = take((size_t)hugeMaxBlocks * 8);
        const size_t oTmp = take(tmpBytes), oSel = take(selBytes);
        if (offset > B.scratchBytes) {
            cudaFree(B.scratch);
            B.scratch = nullptr;
            B.scratchBytes = 0;
            GFX_CUDA(ctx, cudaMalloc(&B.scratch, offset));
            B.scratchBytes = offset;
        }
        uint8_t* base = reinterpret_cast<uint8_t*>(B.scratch);
        triLo = reinterpret_cast<float4*>(base + oTriLo); triHi = reinterpret_cast<float4*>(base + oTriHi);
        boxLo = reinterpret_cast<float4*>(base + oBoxLo); boxHi = reinterpret_cast<float4*>(base + oBoxHi);
        keys = reinterpret_cast<uint64_t*>(base + oKeys); keysSorted = reinterpret_cast<uint64_t*>(base + oKeysSorted);
        ids = reinterpret_cast<uint32_t*>(base + oIds); idsSorted = reinterpret_cast<uint32_t*>(base + oIdsSorted);
        childL = reinterpret_cast<uint32_t*>(base + oChildL); childR = reinterpret_cast<uint32_t*>(base + oChildR);
        rangeFirst = reinterpret_cast<uint32_t*>(base + oRangeFirst); rangeLast = reinterpret_cast<uint32_t*>(base + oRangeLast);
        parentI = reinterpret_cast<uint32_t*>(base + oParentI); parentL = reinterpret_cast<uint32_t*>(base + oParentL);
        arrive = reinterpret_cast<uint32_t*>(base + oArrive); counters = reinterpret_cast<uint32_t*>(base + oCounters);
        queueA = reinterpret_cast<uint2*>(base + oQueueA); queueB = reinterpret_cast<uint2*>(base + oQueueB);
        bigListStore[0] = reinterpret_cast<uint4*>(base + oBig0); bigListStore[1] = reinterpret_cast<uint4*>(base + oBig1);
        hugeListStore[0] = reinterpret_cast<uint4*>(base + oHuge0); hugeListStore[1] = reinterpret_cast<uint4*>(base + oHuge1);
        hugeNodeStore = base + oHugeNodes;
        hugeBlockStore = reinterpret_cast<uint32_t*>(base + oHugeBlocks);
        tmp = base + oTmp; selTmp = base + oSel;
    }
    if (B.builtForTris != n) {
        GFX_CUDA(ctx, cudaMalloc(&B.tris, (size_t)n * 48));
        GFX_CUDA(ctx, cudaMalloc(&B.primRefs, (size_t)n * 4));
        // every wide node has >= 2 children except a degenerate root, so #nodes <= n
        GFX_CUDA(ctx, cudaMalloc(&B.nodes, (size_t)max(n, 1u) * 80));
        GFX_CUDA(ctx, cudaMalloc(&B.sceneBounds, 6 * 4));
        B.builtForTris = n;
    }

    const DevScene dev = ctx->devScene();
    const uint32_t blocks = (n + 255) / 256;
    k_initBounds<<<1, 32, 0, stream>>>(B.sceneBounds); ctx->launches++;
    k_flatten<<<blocks, 256, 0, stream>>>(dev, S.geomTriOffsets, S.numGeoms, n, B.tris, triLo, triHi, B.sceneBounds); ctx->launches++;
    k_morton<<<blocks, 256, 0, stream>>>(n, triLo, triHi, B.sceneBounds, keys, ids); ctx->launches++;

    cub::DeviceRadixSort::SortPairs(tmp, tmpBytes, keys, keysSorted, ids, idsSorted, (int)n, 0, 63, stream); ctx->launches += 8;

    uint32_t rootRef = n == 1 ? 0x80000000u : 0u;
    const bool fast = (flags & GFX_BVH_BUILD_FAST) != 0;
    if (fast || n < 3) {
        GFX_CUDA(ctx, cudaMemsetAsync(arrive, 0, (size_t)n * 4, stream));
        if (n > 1) {
            // rangeFirst receives the triangle count of each node (the collapse needs nothing else of the ranges)
            k_hierarchy<<<(n - 1 + 255) / 256, 256, 0, stream>>>((int)n, keysSorted, childL, childR, rangeFirst, rangeLast, parentI, parentL); ctx->launches++;
        }
        k_refit<<<blocks, 256, 0, stream>>>((int)n, idsSorted, triLo, triHi, childL, childR, parentI, parentL, arrive, boxLo, boxHi); ctx->launches++;
    }
    else if (!(flags & GFX_BVH_BUILD_PLOC)) {
        // binned SAH, top-down: small-node lists ping-pong between keys / keysSorted (n/2 records of 16 B each), big-node
        // lists are tiny; counters = { next small, next big, internal nodes allocated }
        uint4* smallLists[2] = { reinterpret_cast<uint4*>(keys), reinterpret_cast<uint4*>(keysSorted) };
        uint4* bigLists[2] = { bigListStore[0], bigListStore[1] };
        uint4* hugeLists[2] = { hugeListStore[0], hugeListStore[1] };
        SahArgs sa;
        sa.n = n;
        sa.triLo = triLo; sa.triHi = triHi;
        sa.order = idsSorted; sa.scratch = ids;
        sa.childL = childL; sa.childR = childR; sa.count = rangeFirst;
        sa.boxLo = boxLo; sa.boxHi = boxHi;
        sa.counters = counters;
        // { small, big, huge } of the current level
        uint32_t sizes[3] = { n > kSahBigNode ? 0u : 1u, (n > kSahBigNode && n <= kSahHugeNode) ? 1u : 0u, n > kSahHugeNode ? 1u : 0u };
        const uint4 rootRec = make_uint4(0u, 0u, n, 0u);
        GFX_CUDA(ctx, cudaMemcpyAsync(sizes[2] ? hugeLists[0] : sizes[1] ? bigLists[0] : smallLists[0], &rootRec, 16, cudaMemcpyHostToDevice, stream));
        uint32_t hostSah[4] = { 0u, 0u, 1u, 0u }; // node 0 = root
        GFX_CUDA(ctx, cudaMemcpyAsync(counters, hostSah, 16, cudaMemcpyHostToDevice, stream));
        SahHugeArgs ha;
        ha.nodes = reinterpret_cast<SahHugeNode*>(hugeNodeStore);
        ha.blockLeft = hugeBlockStore;
        ha.blockRight = hugeBlockStore + hugeMaxBlocks;
        int cur = 0;
        uint32_t depth = 0;
        while (sizes[0] + sizes[1] + sizes[2] > 0) {
            sa.smallOut = smallLists[cur ^ 1];
            sa.bigOut = bigLists[cur ^ 1];
            sa.hugeOut = hugeLists[cur ^ 1];
            if (sizes[2]) { // multi-block split of the nodes above kSahHugeNode triangles
                sa.listIn = hugeLists[cur];
                sa.listSize = sizes[2];
                ha.a = sa;
                const uint32_t blocksUpper = n / kSahHugeChunk + sizes[2] + 1; // sum of ceil(num / chunk) over disjoint slices
                k_sahHugeInit<<<sizes[2], 128, 0, stream>>>(ha);
                k_sahHugeBounds<<<blocksUpper, 1024, 0, stream>>>(ha);
                k_sahHugeBin<<<blocksUpper, 1024, 0, stream>>>(ha);
                k_sahHugeEval<<<sizes[2], 32, 0, stream>>>(ha);
                k_sahHugeCount<<<blocksUpper, 1024, 0, stream>>>(ha);
                k_sahHugeOffsets<<<sizes[2], 32, 0, stream>>>(ha);
                k_sahHugeScatter<<<blocksUpper, 1024, 0, stream>>>(ha);
                k_sahHugeCopyBack<<<blocksUpper, 1024, 0, stream>>>(ha);
                ctx->launches += 8;
            }
            if (sizes[1]) {
                sa.listIn = bigLists[cur];
                sa.listSize = sizes[1];
                k_sahSplit<1024><<<sizes[1], 1024, 0, stream>>>(sa); ctx->launches++;
            }
            if (sizes[0]) {
                sa.listIn = smallLists[cur];
                sa.listSize = sizes[0];
                k_sahSplit<64><<<sizes[0], 64, 0, stream>>>(sa); ctx->launches++;
            }
            GFX_CUDA(ctx, cudaMemcpyAsync(hostSah, counters, 16, cudaMemcpyDeviceToHost, stream));
            GFX_CUDA(ctx, cudaStreamSynchronize(stream));
            sizes[0] = hostSah[0];
            sizes[1] = hostSah[1];
            sizes[2] = hostSah[3];
            const uint32_t zeros[2] = { 0u, 0u };
            GFX_CUDA(ctx, cudaMemcpyAsync(counters, zeros, 8, cudaMemcpyHostToDevice, stream));
            GFX_CUDA(ctx, cudaMemcpyAsync(counters + 3, zeros, 4, cudaMemcpyHostToDevice, stream));
            cur ^= 1;
            if (++depth > 4096 || sizes[1] > bigCapacity || sizes[2] > hugeCapacity) {
                ctx->setError("gfx_bvh_build: SAH split did not converge");
                return GFX_ERR_CUDA;
            }
        }
        k_sahLeafBoxes<<<blocks, 256, 0, stream>>>((int)n, idsSorted, triLo, triHi, boxLo, boxHi); ctx->launches++;
        rootRef = 0u;
    }
    else {
        // PLOC: clusters ping-pong between parentI / parentL, nearest neighbours in arrive, node counter in counters[3]
        uint32_t *clusters = parentI, *clustersOut = parentL, *nearest = arrive;
        uint32_t* numSelected = counters + 2;
        GFX_CUDA(ctx, cudaMemsetAsync(counters, 0, 16, stream));
        k_plocInit<<<blocks, 256, 0, stream>>>((int)n, idsSorted, triLo, triHi, clusters, boxLo, boxHi); ctx->launches++;
        int plocRadius = (int)((flags >> 16) & 0xFFu); // 0 = default
        if (plocRadius == 0) plocRadius = 16;
        if (plocRadius > kPlocMaxRadius) plocRadius = kPlocMaxRadius;
        uint32_t m = n;
        uint32_t passes = 0;
        while (m > 1) {
            const uint32_t mb = (m + kPlocBlock - 1) / kPlocBlock;
            k_plocNearest<<<mb, kPlocBlock, 0, stream>>>((int)m, (int)n, plocRadius, clusters, boxLo, boxHi, nearest);
            k_plocMerge<<<(m + 255) / 256, 256, 0, stream>>>((int)m, (int)n, clusters, nearest, childL, childR, rangeFirst, boxLo, boxHi,
                                                           counters + 3, clustersOut);
            cub::DeviceSelect::If(selTmp, selBytes, clustersOut, clusters, numSelected, (int)m, PlocValid(), stream);
            ctx->launches += 4;
            uint32_t newM = 0;
            GFX_CUDA(ctx, cudaMemcpyAsync(&newM, numSelected, 4, cudaMemcpyDeviceToHost, stream));
            GFX_CUDA(ctx, cudaStreamSynchronize(stream));
            if (newM >= m || ++passes > 4096) {
                ctx->setError("gfx_bvh_build: PLOC did not converge");
                return GFX_ERR_CUDA;
            }
            m = newM;
        }
        GFX_CUDA(ctx, cudaMemcpyAsync(&rootRef, clusters, 4, cudaMemcpyDeviceToHost, stream));
        GFX_CUDA(ctx, cudaStreamSynchronize(stream));
    }

    // collapse, level by level
    uint32_t hostCounters[4] = { 1u, 0u, 0u, 0u }; // node 0 = root is pre-allocated
    GFX_CUDA(ctx, cudaMemcpyAsync(counters, hostCounters, 16, cudaMemcpyHostToDevice, stream));
    const uint2 rootItem = make_uint2(0u, rootRef);
    GFX_CUDA(ctx, cudaMemcpyAsync(queueA, &rootItem, 8, cudaMemcpyHostToDevice, stream));
    CollapseArgs a;
    a.n = (int)n;
    a.maxLeaf = maxLeaf;
    a.childL = childL; a.childR = childR; a.count = rangeFirst;
    a.boxLo = boxLo; a.boxHi = boxHi; a.sortedIds = idsSorted;
    a.nodes = reinterpret_cast<uint4*>(B.nodes);
    a.primRefs = B.primRefs;
    a.counters = counters;
    uint32_t queueSize = 1;
    uint2 *qin = queueA, *qout = queueB;
    uint32_t levels = 0;
    while (queueSize > 0) {
        a.queueIn = qin;
        a.queueOut = qout;
        a.queueInSize = queueSize;
        k_collapse<<<(queueSize + 127) / 128, 128, 0, stream>>>(a); ctx->launches++;
        GFX_CUDA(ctx, cudaMemcpyAsync(hostCounters, counters, 16, cudaMemcpyDeviceToHost, stream));
        GFX_CUDA(ctx, cudaStreamSynchronize(stream));
        queueSize = hostCounters[2];
        const uint32_t zero = 0;
        GFX_CUDA(ctx, cudaMemcpyAsync(counters + 2, &zero, 4, cudaMemcpyHostToDevice, stream));
        std::swap(qin, qout);
        if (++levels > 4096) {
            ctx->setError("gfx_bvh_build: collapse did not converge");
            return GFX_ERR_CUDA;
        }
    }
    B.numNodes = hostCounters[0];
    B.numPrimRefs = hostCounters[1];
    B.levels = levels;
    uint32_t ob[6];
    GFX_CUDA(ctx, cudaMemcpy(ob, B.sceneBounds, 24, cudaMemcpyDeviceToHost));
    for (int i = 0; i < 6; ++i) {
        const uint32_t u = ob[i] ^ (ob[i] >= 0x80000000u ? 0x80000000u : 0xFFFFFFFFu);
        float f;
        memcpy(&f, &u, 4);
        (i < 3 ? B.sceneMin[i] : B.sceneMax[i - 3]) = f;
    }

    return GFX_OK;
}

// ---- 7. traversal tables ------------------------------------------------------------------------
// The reference layout keeps triangles in scene order behind a PrimitiveReference indirection (common_shared.h:1012-1025).
// The traverser reads a second copy in leaf order: leafTris[i] = tris[primRefs[i] & 0x7FFFFFFF] with the reference word
// (storage index + end-of-leaf bit) in the padding field, so a leaf costs one dependent fetch instead of two and the
// triangles of a leaf - and of the sibling leaves of a node - are adjacent in memory.
__global__ void k_leafTris(uint32_t numPrimRefs, const uint32_t* __restrict__ primRefs, const float4* __restrict__ tris,
                           float4* __restrict__ leafTris) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numPrimRefs)
        return;
    const uint32_t pr = primRefs[i];
    const float4* src = tris + 3 * (size_t)(pr & 0x7FFFFFFFu);
    float4* dst = leafTris + 3 * (size_t)i;
    dst[0] = src[0];
    dst[1] = src[1];
    float4 t2 = src[2];
    t2.w = __uint_as_float(pr);
    dst[2] = t2;
}

int finishBvh(gfx_ctx* ctx, cudaStream_t stream) {
    BvhState &B = ctx->bvh;
    if (B.numPrimRefs > B.leafTrisCapacity || !B.leafTris) {
        cudaFree(B.leafTris);
        B.leafTris = nullptr;
        B.leafTrisCapacity = 0;
        GFX_CUDA(ctx, cudaMalloc(&B.leafTris, (size_t)max(B.numPrimRefs, 1u) * 48));
        B.leafTrisCapacity = max(B.numPrimRefs, 1u);
    }
    if (B.numPrimRefs) {
        k_leafTris<<<(B.numPrimRefs + 255) / 256, 256, 0, stream>>>(B.numPrimRefs, B.primRefs, B.tris, B.leafTris);
        ctx->launches++;
        GFX_CUDA(ctx, cudaGetLastError());
    }
    return GFX_OK;
}

} // namespace gfx
