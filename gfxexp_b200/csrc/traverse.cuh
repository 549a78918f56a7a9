// traverse.cuh — per-thread stack traversal of the reference's 8-wide quantised BVH on sm_100a.
//
// Replaces optixTrace (utils/optix_util.h:575-584) for closest-hit and visibility rays, with the
// semantics of the only BVH traverser in the reference tree, bvh::traverse<8>
// (common/bvh_builder.cpp:1272-1649): children are visited leaf-groups-first, near to far, by the
// same key (entry distance, isInternal<<31); the ray/triangle test is bit-for-bit
// testRayVsTriangle (common/bvh_builder.cpp:1251-1270) on the explicit-FMA vector kernels of
// vec.cuh / oracle/vecmath.h.
//
// Differences by design (documented in DESIGN.md):
//  * ties in hit distance resolve to the smaller TriangleStorage index instead of "first found"
//    (makes the result independent of BVH topology, so a Morton LBVH and the reference SBVH give
//    identical hits);
//  * the slab test works on t = q * (scale/dir) + (origin-org)/dir with explicit FMAs and a 1e-5
//    relative slack, i.e. it is conservative w.r.t. AABB::intersect (common/basic_types.h:3450-3465);
//    it only decides which nodes are visited, never the hit itself.
//
// The traversal is exposed as a resumable state machine (TraversalState + traverseStep = one internal
// node incl. its leaf children) so that the wavefront kernel of trace.cu can refill finished lanes
// with new rays (persistent threads) while the fused kernels simply loop traverseStep to completion.
#pragma once
#include "scene.cuh"

namespace gfx {

struct Hit {
    float dist;
    uint32_t storageIndex; // 0xFFFFFFFF = miss
    uint32_t geomIndex;
    uint32_t primIndex;
    float bcB, bcC;
    uint32_t statNodes, statTris; // only maintained by the STATS instantiation
};

GFX_D bool testRayVsTriangle( // common/bvh_builder.cpp:1251-1270
    const f3 &rayOrg, const f3 &rayDir, const float distMin, const float distMax,
    const f3 &pA, const f3 &pB, const f3 &pC,
    float* hitDist, float* bcB, float* bcC) {
    const f3 eAB = pB - pA;
    const f3 eCA = pA - pC;
    const f3 hitNormal = cross(eCA, eAB);
    const f3 e = (1.0f / dot(hitNormal, rayDir)) * (pA - rayOrg);
    const f3 i = cross(rayDir, e);
    *bcB = dot(i, eCA);
    *bcC = dot(i, eAB);
    *hitDist = dot(hitNormal, e);
    return ((*hitDist < distMax) && (*hitDist > distMin) &&
            (*bcB >= 0.0f) && (*bcC >= 0.0f) && (*bcB + *bcC <= 1));
}

#define GFX_CSWAP(a, b) { const uint32_t lo_ = min(a, b); const uint32_t hi_ = max(a, b); a = lo_; b = hi_; }

constexpr int kStackSize = 64;
// The wavefront kernels keep the first kSmemStack entries of every lane's stack in shared memory, laid out [entry][thread] so
// that a warp's pushes and pops are conflict-free whatever the lanes' depths (a per-thread local-memory stack makes every push a
// divergent store: the push / pop section held 41 % of the trace kernel's stall samples in round 1); deeper entries - rare with
// an 8-wide tree - spill to the local array.
constexpr int kSmemStack = 16;
constexpr int kSmemStackThreads = 128; // block size of the wavefront kernels

struct TraversalState {
    f3 org, dir, idir;
    float tmin, tmax;
    Hit best;
    uint32_t nodeIdx;
    int sp;
    uint2* sstack;           // this thread's column of the shared-memory stack (wavefront kernels), else unused
    uint2 stack[kStackSize]; // (node index, truncated entry distance bits)
};
template <int SMEM_STRIDE> // threads per block of the shared-memory stack, 0 = local memory only
GFX_D void stackStore(TraversalState &st, int at, const uint2 &v) {
    if (SMEM_STRIDE > 0 && at < kSmemStack)
        st.sstack[at * SMEM_STRIDE] = v;
    else
        st.stack[SMEM_STRIDE > 0 ? at - kSmemStack : at] = v;
}
template <int SMEM_STRIDE>
GFX_D uint2 stackLoad(const TraversalState &st, int at) {
    if (SMEM_STRIDE > 0 && at < kSmemStack)
        return st.sstack[at * SMEM_STRIDE];
    return st.stack[SMEM_STRIDE > 0 ? at - kSmemStack : at];
}

GFX_D void traverseInit(TraversalState &st, const f3 &org, const f3 &dir, float tmin, float tmax) {
    st.org = org;
    st.dir = dir;
    st.tmin = tmin;
    st.tmax = tmax;
    st.best.dist = tmax;
    st.best.storageIndex = 0xFFFFFFFFu;
    st.best.geomIndex = 0xFFFFFFFFu;
    st.best.primIndex = 0xFFFFFFFFu;
    st.best.bcB = 0.0f;
    st.best.bcC = 0.0f;
    st.best.statNodes = 0;
    st.best.statTris = 0;
    // guarded reciprocal direction for the slab test only
    const float ooeps = 8.271806e-25f; // 2^-80
    const f3 sd(fabsf(dir.x) > ooeps ? dir.x : copysignf(ooeps, dir.x),
                fabsf(dir.y) > ooeps ? dir.y : copysignf(ooeps, dir.y),
                fabsf(dir.z) > ooeps ? dir.z : copysignf(ooeps, dir.z));
    st.idir = f3(1.0f / sd.x, 1.0f / sd.y, 1.0f / sd.z);
    st.nodeIdx = 0;
    st.sp = 0;
    st.sstack = nullptr;
}

// Leaf children whose triangle tests have been postponed (wavefront kernel): the start of the triangle chain and the
// entry distance of the leaf box.  A node step appends at most 8.
constexpr int kPendingLeaves = 12;
struct PendingLeaves {
    uint32_t idx[kPendingLeaves];
    float tn[kPendingLeaves];
    int n;
};

// One triangle of a leaf chain (leaf-ordered storage).  Returns true when an any-hit ray has found its occluder.
template <bool ANY_HIT, bool STATS>
GFX_D bool testLeafTriangle(const DevBvh &bvh, TraversalState &st, uint32_t idx, bool* endOfChain) {
    const float4* tp = bvh.leafTris + 3 * (size_t)idx;
    const float4 t0 = __ldg(tp + 0);
    const float4 t1 = __ldg(tp + 1);
    const float4 t2 = __ldg(tp + 2);
    const uint32_t pr = __float_as_uint(t2.w); // PrimitiveReference word: storage index | end-of-leaf << 31
    const uint32_t si = pr & 0x7FFFFFFFu;
    *endOfChain = (pr >> 31) != 0;
    float hitDist, bcB, bcC;
    if (STATS)
        ++st.best.statTris;
    const bool hit = testRayVsTriangle(st.org, st.dir, st.tmin, st.tmax,
                                       f3(t0.x, t0.y, t0.z), f3(t0.w, t1.x, t1.y), f3(t1.z, t1.w, t2.x),
                                       &hitDist, &bcB, &bcC);
    if (hit && (hitDist < st.best.dist || (hitDist == st.best.dist && si < st.best.storageIndex))) {
        st.best.dist = hitDist;
        st.best.storageIndex = si;
        st.best.geomIndex = __float_as_uint(t2.y);
        st.best.primIndex = __float_as_uint(t2.z);
        st.best.bcB = bcB;
        st.best.bcC = bcC;
        if (ANY_HIT)
            return true;
    }
    return false;
}

// Advances the newest postponed leaf of this lane by one triangle.  Returns true when an any-hit ray is occluded.
template <bool ANY_HIT, bool STATS>
GFX_D bool testPendingTriangle(const DevBvh &bvh, TraversalState &st, PendingLeaves &pend) {
    const int top = pend.n - 1;
    if (pend.tn[top] > st.best.dist) { // a closer hit has been found since the leaf was postponed
        pend.n = top;
        return false;
    }
    const uint32_t idx = pend.idx[top];
    bool end;
    if (testLeafTriangle<ANY_HIT, STATS>(bvh, st, idx, &end))
        return true;
    if (end)
        pend.n = top;
    else
        pend.idx[top] = idx + 1;
    return false;
}

// Processes node st.nodeIdx: slab-tests its children, intersects the triangle chains of the leaf
// children that are hit (or, with `pend`, postpones them), selects the next internal node.  Returns false when the
// traversal is finished.
template <bool ANY_HIT, bool STATS, bool DEFER = false, int SMEM_STRIDE = 0>
GFX_D bool traverseStep(const DevBvh &bvh, TraversalState &st, PendingLeaves* pend = nullptr) {
    const uint4* np = bvh.nodes + 5 * (size_t)st.nodeIdx;
    const uint4 n0 = __ldg(np + 0);
    const uint4 n1 = __ldg(np + 1);
    const uint4 n2 = __ldg(np + 2);
    const uint4 n3 = __ldg(np + 3);
    const uint4 n4 = __ldg(np + 4);
    if (STATS)
        ++st.best.statNodes;

    const uint32_t internalMask = n0.w >> 24;
    const float ax = __uint_as_float((n0.w & 0xFFu) << 23) * st.idir.x;
    const float ay = __uint_as_float(((n0.w >> 8) & 0xFFu) << 23) * st.idir.y;
    const float az = __uint_as_float(((n0.w >> 16) & 0xFFu) << 23) * st.idir.z;
    const float bx = (__uint_as_float(n0.x) - st.org.x) * st.idir.x;
    const float by = (__uint_as_float(n0.y) - st.org.y) * st.idir.y;
    const float bz = (__uint_as_float(n0.z) - st.org.z) * st.idir.z;

    // The sign of the ray direction decides which quantised plane of each axis is entered first, once per node and
    // axis instead of a min/max pair per child (same t values as min(tlo, thi) / max(tlo, thi)).
    const bool sx = st.idir.x < 0.0f, sy = st.idir.y < 0.0f, sz = st.idir.z < 0.0f;
    const uint32_t nearX[2] = { sx ? n3.z : n2.x, sx ? n3.w : n2.y }, farX[2] = { sx ? n2.x : n3.z, sx ? n2.y : n3.w };
    const uint32_t nearY[2] = { sy ? n4.x : n2.z, sy ? n4.y : n2.w }, farY[2] = { sy ? n2.z : n4.x, sy ? n2.w : n4.y };
    const uint32_t nearZ[2] = { sz ? n4.z : n3.x, sz ? n4.w : n3.y }, farZ[2] = { sz ? n3.x : n4.z, sz ? n3.y : n4.w };
    const uint32_t invalidNearX = sx ? 0u : 255u, invalidFarX = sx ? 255u : 0u; // (qminx, qmaxx) = (255, 0) marks an empty slot

    uint32_t keys[8];
#pragma unroll
    for (int slot = 0; slot < 8; ++slot) {
        const int sh = 8 * (slot & 3), w = slot >> 2;
        const uint32_t qnx = (nearX[w] >> sh) & 0xFFu, qfx = (farX[w] >> sh) & 0xFFu;
        const uint32_t qny = (nearY[w] >> sh) & 0xFFu, qfy = (farY[w] >> sh) & 0xFFu;
        const uint32_t qnz = (nearZ[w] >> sh) & 0xFFu, qfz = (farZ[w] >> sh) & 0xFFu;
        const bool valid = (qnx != invalidNearX) || (qfx != invalidFarX);
        const float tnx = __fmaf_rn((float)qnx, ax, bx), tfx = __fmaf_rn((float)qfx, ax, bx);
        const float tny = __fmaf_rn((float)qny, ay, by), tfy = __fmaf_rn((float)qfy, ay, by);
        const float tnz = __fmaf_rn((float)qnz, az, bz), tfz = __fmaf_rn((float)qfz, az, bz);
        const float tn = fmaxf(fmaxf(tnx, tny), fmaxf(tnz, st.tmin));
        const float tf = fminf(fminf(tfx, tfy), fminf(tfz, st.best.dist));
        const bool hit = valid && (tn <= tf * 1.00001f);
        const uint32_t isInternal = (internalMask >> slot) & 1u;
        keys[slot] = hit ? ((isInternal << 31) | ((__float_as_uint(tn) >> 1) & 0x7FFFFFF8u) | (uint32_t)slot)
                         : 0xFFFFFFFFu;
    }
    // 19-comparator network, ascending: leaf hits (near..far), internal hits (near..far), misses.
    GFX_CSWAP(keys[0], keys[2]); GFX_CSWAP(keys[1], keys[3]); GFX_CSWAP(keys[4], keys[6]); GFX_CSWAP(keys[5], keys[7]);
    GFX_CSWAP(keys[0], keys[4]); GFX_CSWAP(keys[1], keys[5]); GFX_CSWAP(keys[2], keys[6]); GFX_CSWAP(keys[3], keys[7]);
    GFX_CSWAP(keys[0], keys[1]); GFX_CSWAP(keys[2], keys[3]); GFX_CSWAP(keys[4], keys[5]); GFX_CSWAP(keys[6], keys[7]);
    GFX_CSWAP(keys[2], keys[4]); GFX_CSWAP(keys[3], keys[5]);
    GFX_CSWAP(keys[1], keys[4]); GFX_CSWAP(keys[3], keys[6]);
    GFX_CSWAP(keys[1], keys[2]); GFX_CSWAP(keys[3], keys[4]); GFX_CSWAP(keys[5], keys[6]);

    // ---- leaf children: intersect their triangle chains now (shrinks best.dist before descending)
    const uint32_t leafBase = n1.y;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t key = keys[k];
        if (key >= 0x80000000u)
            break;
        const uint32_t slot = key & 7u;
        const float tn = __uint_as_float((key & 0x7FFFFFF8u) << 1);
        if (tn > st.best.dist)
            continue;
        const uint32_t metas = slot < 4 ? n1.z : n1.w;
        uint32_t idx = leafBase + ((metas >> (8 * (slot & 3))) & 0xFFu);
        if (DEFER) {
            pend->idx[pend->n] = idx;
            pend->tn[pend->n] = tn;
            ++pend->n;
            continue;
        }
        while (true) {
            bool end;
            if (testLeafTriangle<ANY_HIT, STATS>(bvh, st, idx, &end))
                return false;
            if (end)
                break;
            ++idx;
        }
    }

    // ---- internal children: nearest becomes the next node, the others are pushed far -> near
    const uint32_t childBase = n1.x;
    // (A branch-free variant - stack positions from population counts, predicated stores - was measured in round 2 and is
    // gone: same hits, but G-buffer 0.67 -> 0.80 ms and visibility trace 0.90 -> 0.94 ms, profiles/r02_summary.md.)
    uint32_t next = 0xFFFFFFFFu, nextT = 0u;
#pragma unroll
    for (int k = 7; k >= 0; --k) {
        const uint32_t key = keys[k];
        if (key == 0xFFFFFFFFu || key < 0x80000000u)
            continue;
        const uint32_t slot = key & 7u;
        const uint32_t tnBits = (key & 0x7FFFFFF8u) << 1; // truncated entry distance (<= true tn)
        if (__uint_as_float(tnBits) > st.best.dist)
            continue;
        if (next != 0xFFFFFFFFu) {
            if (st.sp < kStackSize)
                stackStore<SMEM_STRIDE>(st, st.sp++, make_uint2(next, nextT));
            else if (bvh.overflowFlag)
                *bvh.overflowFlag = 1u;
        }
        next = childBase + __popc(internalMask & ((1u << slot) - 1u));
        nextT = tnBits;
    }
    if (next != 0xFFFFFFFFu) {
        st.nodeIdx = next;
        return true;
    }
    while (st.sp > 0) {
        const uint2 e = stackLoad<SMEM_STRIDE>(st, --st.sp);
        if (__uint_as_float(e.y) <= st.best.dist) {
            st.nodeIdx = e.x;
            return true;
        }
    }
    return false;
}

template <bool ANY_HIT, bool STATS = false>
GFX_D Hit traverseBvh(const DevBvh &bvh, const f3 &org, const f3 &dir, const float tmin, const float tmax) {
    TraversalState st;
    traverseInit(st, org, dir, tmin, tmax);
    if (bvh.numNodes == 0)
        return st.best;
    while (traverseStep<ANY_HIT, STATS>(bvh, st)) {
    }
    return st.best;
}
// the same with the first kSmemStack stack entries in shared memory: `sstack` = this thread's column of a
// [kSmemStack][STRIDE] uint2 array
template <bool ANY_HIT, int STRIDE>
GFX_D Hit traverseBvhSmemStack(const DevBvh &bvh, const f3 &org, const f3 &dir, const float tmin, const float tmax, uint2* sstack) {
    TraversalState st;
    traverseInit(st, org, dir, tmin, tmax);
    st.sstack = sstack;
    if (bvh.numNodes == 0)
        return st.best;
    while (traverseStep<ANY_HIT, false, false, STRIDE>(bvh, st)) {
    }
    return st.best;
}

} // namespace gfx
