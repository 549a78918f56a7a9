// wavefront.cuh — the persistent-thread ray tracing kernel shared by trace.cu (C-ABI ray batches, ReSTIR
// visibility queue) and pathtrace.cu (extension + shadow ray queues of the wavefront path tracer).
//
// Why persistent threads: incoherent rays of one warp visit very different numbers of nodes (the shadow
// rays of an 8x4 pixel tile go to 32 different lights), so a ray-per-thread launch idles most lanes while
// the longest traversal finishes.  Here a warp keeps 32 traversal state machines (traverse.cuh) and refills
// finished lanes from a global counter as soon as a quarter of them are idle; one atomic per refill.
//
// Writer concept: `template <bool ANY_HIT, bool STATS> void write(uint32_t ray, const TraversalState&) const`
// is called exactly once per ray, by the lane that traced it.
#pragma once
#include "traverse.cuh"

namespace gfx {

template <bool ANY_HIT, bool STATS, bool DEFER, typename Writer>
GFX_D void traceWavefrontBody(const DevBvh &bvh, const float4* __restrict__ rays, const uint32_t* __restrict__ numRaysPtr,
                              uint32_t numRaysImm, uint32_t* __restrict__ fetchCounter, const Writer &writer) {
    const uint32_t total = numRaysPtr ? *numRaysPtr : numRaysImm;
    if (total == 0 || bvh.numNodes == 0) {
        // nothing to traverse: every ray misses
        if (bvh.numNodes == 0) {
            TraversalState st;
            for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < total; r += gridDim.x * blockDim.x) {
                const float4 r1 = __ldg(rays + 2 * (size_t)r + 1);
                traverseInit(st, f3(0, 0, 0), f3(0, 0, 1), 0.0f, r1.w);
                writer.template write<ANY_HIT, STATS>(r, st);
            }
        }
        return;
    }
    const uint32_t lane = threadIdx.x & 31u;
    __shared__ uint2 sharedStack[kSmemStack][kSmemStackThreads];
    uint2* const myStack = &sharedStack[0][threadIdx.x];
    TraversalState st;
    bool active = false;
    uint32_t myRay = 0;
    if (DEFER) {
    // Postponed leaves: a node step only records the leaf children it hits; the triangle tests run when at least
    // kFlushLanes lanes have some to do (or a lane's list is full, or nobody can advance otherwise).  Measured by ncu on the
    // immediate version: the node step runs with 27.8 of 32 lanes, the triangle tests inside it with 6-12, and they
    // issue 60 % of the warp instructions.  A lane whose traversal has ended with leaves still postponed waits
    // (`draining`) for the next flush; an occluded any-hit ray learns it at the flush.
    constexpr int kFlushLanes = 16;
    PendingLeaves pend;
    pend.n = 0;
    bool draining = false;
    while (true) {
        // ---- refill idle lanes (one atomic per warp)
        const uint32_t idle = __ballot_sync(0xFFFFFFFFu, !active);
        if (idle) {
            const int leader = __ffs(idle) - 1;
            uint32_t base = 0;
            if ((int)lane == leader)
                base = atomicAdd(fetchCounter, (uint32_t)__popc(idle));
            base = __shfl_sync(0xFFFFFFFFu, base, leader);
            if (!active) {
                const uint32_t r = base + __popc(idle & ((1u << lane) - 1u));
                if (r < total) {
                    const float4 r0 = __ldg(rays + 2 * (size_t)r);
                    const float4 r1 = __ldg(rays + 2 * (size_t)r + 1);
                    traverseInit(st, f3(r0.x, r0.y, r0.z), f3(r1.x, r1.y, r1.z), r0.w, r1.w);
                    st.sstack = myStack;
                    myRay = r;
                    active = true;
                }
            }
        }
        if (!__any_sync(0xFFFFFFFFu, active))
            break;
#pragma unroll 1
        for (int it = 0; it < 8; ++it) {
            if (active && !draining && !traverseStep<ANY_HIT, STATS, true, kSmemStackThreads>(bvh, st, &pend))
                draining = true;
            const uint32_t have = __ballot_sync(0xFFFFFFFFu, active && pend.n > 0);
            const uint32_t running = __ballot_sync(0xFFFFFFFFu, active && !draining);
            const bool full = __any_sync(0xFFFFFFFFu, pend.n > kPendingLeaves - 8);
            if (have && (__popc(have) >= kFlushLanes || full || running == 0u)) {
                bool occluded = false;
                while (__any_sync(0xFFFFFFFFu, pend.n > 0)) {
                    if (pend.n > 0 && testPendingTriangle<ANY_HIT, STATS>(bvh, st, pend)) {
                        occluded = true;
                        pend.n = 0;
                    }
                }
                if (occluded)
                    draining = true; // the ray is finished whatever its stack still holds
            }
            if (active && draining && pend.n == 0) {
                writer.template write<ANY_HIT, STATS>(myRay, st);
                active = false;
                draining = false;
            }
            if (__popc(__ballot_sync(0xFFFFFFFFu, active && !draining)) <= 24)
                break;
        }
    }
    return;
    }
    while (true) {
        // ---- refill idle lanes (one atomic per warp)
        const uint32_t idle = __ballot_sync(0xFFFFFFFFu, !active);
        if (idle) {
            const int leader = __ffs(idle) - 1;
            uint32_t base = 0;
            if ((int)lane == leader)
                base = atomicAdd(fetchCounter, (uint32_t)__popc(idle));
            base = __shfl_sync(0xFFFFFFFFu, base, leader);
            if (!active) {
                const uint32_t r = base + __popc(idle & ((1u << lane) - 1u));
                if (r < total) {
                    const float4 r0 = __ldg(rays + 2 * (size_t)r);
                    const float4 r1 = __ldg(rays + 2 * (size_t)r + 1);
                    traverseInit(st, f3(r0.x, r0.y, r0.z), f3(r1.x, r1.y, r1.z), r0.w, r1.w);
                    st.sstack = myStack;
                    myRay = r;
                    active = true;
                }
            }
        }
        if (!__any_sync(0xFFFFFFFFu, active))
            break;
        // ---- advance every active lane by up to 8 nodes, leave early once a quarter of the warp is idle
#pragma unroll 1
        for (int it = 0; it < 8; ++it) {
            if (active && !traverseStep<ANY_HIT, STATS, false, kSmemStackThreads>(bvh, st)) {
                writer.template write<ANY_HIT, STATS>(myRay, st);
                active = false;
            }
            if (__popc(__ballot_sync(0xFFFFFFFFu, active)) <= 24)
                break;
        }
    }
}

// immediate leaf tests: closest-hit rays (a hit shrinks the search interval at once) and any-hit rays that are mostly
// occluded (path-tracer NEE: early termination matters more than lane utilisation)
template <bool ANY_HIT, bool STATS, typename Writer>
__global__ void __launch_bounds__(128) k_traceWavefront(DevBvh bvh, const float4* __restrict__ rays,
                                                        const uint32_t* __restrict__ numRaysPtr, uint32_t numRaysImm,
                                                        uint32_t* __restrict__ fetchCounter, Writer writer) {
    traceWavefrontBody<ANY_HIT, STATS, false>(bvh, rays, numRaysPtr, numRaysImm, fetchCounter, writer);
}
// postponed leaf tests: visibility rays towards resampled light samples (mostly unoccluded, so the whole path is walked)
template <bool ANY_HIT, bool STATS, typename Writer>
__global__ void __launch_bounds__(128) k_traceWavefrontDeferred(DevBvh bvh, const float4* __restrict__ rays,
                                                                const uint32_t* __restrict__ numRaysPtr, uint32_t numRaysImm,
                                                                uint32_t* __restrict__ fetchCounter, Writer writer) {
    traceWavefrontBody<ANY_HIT, STATS, true>(bvh, rays, numRaysPtr, numRaysImm, fetchCounter, writer);
}

static inline int wavefrontGrid() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // 9 x 128 threads per SM: what 56 registers admit (measured 8 / 9 / 12 / 16: 0.847 / 0.821 / 0.821 / 0.822 ms per
    // visibility trace)
    return sms * 9;
}

} // namespace gfx
