// nrc_pathtrace.cu — the Neural Radiance Caching path tracer and its bookkeeping kernels on sm_100a.
//
// Replaces pathTracing.setEntryPoint(NRC) + optixPipeline.launch (neural_radiance_caching_main.cpp:2281-2289) with the
// programs pathTrace_raygen_generic<true> / pathTrace_closestHit_generic<true> / createRadianceQuery
// (neural_radiance_caching/gpu_kernels/optix_pathtracing_kernels.cu:12-34, 95-361, 363-623) and the PURE_CUDA kernels
// preprocessNRC, accumulateInferredRadianceValues, propagateRadianceValues, shuffleTrainingData
// (neural_radiance_caching/gpu_kernels/nrc_setup_kernels.cu:6-49, 51-92, 94-138, 140-216).
//
// Same wavefront pipeline as pathtrace.cu (one path vertex per round, compacted ray queues, persistent trace
// kernel); what NRC adds per round is the training-vertex allocation.  The reference hands out records with
// a global atomicAdd (:216, :571), which makes the record order - and with it the training batches and the
// network weights - depend on GPU scheduling.  Here the training path of each tile stages its vertex in a
// per-tile slot and a scan in tile order numbers them (k_nrcCommitScan / k_nrcCommitScatter): frames are
// reproducible bit for bit, every rank of a multi-GPU run derives identical training data, and no host
// read-back is needed anywhere in the frame (the reference synchronises to read numTrainingData and tileSize,
// neural_radiance_caching_main.cpp:2291-2304; here the inference launch reads its size from device memory).
#include "pathtrace.cuh"

namespace gfx {

constexpr float kPathTerminationFactor = 0.01f;        // neural_radiance_caching_shared.h:7
constexpr uint32_t kNumTrainingDataPerFrame = 1u << 16; // :8
constexpr uint32_t kTrainBufferSize = 2 * kNumTrainingDataPerFrame;
constexpr uint32_t kInvalidVertexDataIndex = 0x007FFFFFu;
constexpr uint32_t kMaxNrcRounds = 62;                  // pathLength is a 6-bit payload field

enum { // words of the state block (GFX_BUF_NRC_STATE)
    NRC_NUM_TRAINING_DATA = 0, NRC_TILE_SIZE = 2, NRC_OFFSET_UNBIASED_TILE = 6, NRC_OFFSET_TRAINING_PATH = 7,
    NRC_TARGET_MIN = 8, NRC_TARGET_MAX = 11, NRC_TARGET_AVG = 20, NRC_NUM_INFERENCE_QUERIES = 26, NRC_NUM_SUFFIX_QUERIES = 27
};
enum { // per-path flags (pathA.z)
    NRC_F_RENDERING_ENDS_WITH_CACHE = 1u, NRC_F_TRAINING_PATH = 2u, NRC_F_UNBIASED_TILE = 4u, NRC_F_PRIMARY_HIT = 8u
};

struct DevNrc {
    uint32_t numSuffixes;
    float* inferenceQuery;
    uint4* terminalInfo;
    float* inferredRadiance;
    float* frameContribution;
    float* trainQuery[2];
    float* trainTarget[2];
    uint4* trainVertexInfo;
    uint32_t* suffixTerminal;
    uint32_t* shufflers;
    uint32_t* state;
    float4* pathA;
    float4* pathB;
    float4* shadowPending2;
    uint32_t* tilePrev;
    uint32_t* tileSuffixEnded;
    uint32_t* stagedFlags;
    uint32_t* stagedIndex;
    float* stagedQuery;
    float4* stagedThroughput;
    float4* stagedNEE;
    uint32_t* shardCounts; // [0 .. shardWorld) the ranks' vertex counts of this round, [64] this rank's own
    uint32_t shardRank, shardWorld;
};

static DevNrc makeDevNrc(const gfx_ctx* ctx) {
    const FrameState::Nrc &N = ctx->frame.nrc;
    DevNrc d;
    d.numSuffixes = N.numSuffixes;
    d.inferenceQuery = N.inferenceQuery;
    d.terminalInfo = N.terminalInfo;
    d.inferredRadiance = N.inferredRadiance;
    d.frameContribution = N.frameContribution;
    for (int i = 0; i < 2; ++i) {
        d.trainQuery[i] = N.trainQuery[i];
        d.trainTarget[i] = N.trainTarget[i];
    }
    d.trainVertexInfo = N.trainVertexInfo;
    d.suffixTerminal = N.suffixTerminal;
    d.shufflers = N.shufflers;
    d.state = N.state;
    d.pathA = N.pathA;
    d.pathB = N.pathB;
    d.shadowPending2 = N.shadowPending2;
    d.tilePrev = N.tilePrev;
    d.tileSuffixEnded = N.tileSuffixEnded;
    d.stagedFlags = N.stagedFlags;
    d.stagedIndex = N.stagedIndex;
    d.stagedQuery = N.stagedQuery;
    d.stagedThroughput = N.stagedThroughput;
    d.stagedNEE = N.stagedNEE;
    d.shardCounts = N.shardCounts;
    d.shardRank = (uint32_t)N.shardRank;
    d.shardWorld = N.shardComm ? (uint32_t)N.shardWorld : 1u;
    return d;
}

int ensureNrcFrame(gfx_ctx* ctx) {
    FrameState &F = ctx->frame;
    FrameState::Nrc &N = F.nrc;
    if (N.created)
        return GFX_OK;
    const size_t n = (size_t)F.W * F.H;
    // W*H/16 in the reference (neural_radiance_caching_main.cpp:1151), rounded up per axis so that 4x4 tiles of an
    // image whose size is not a multiple of 4 still own a slot
    N.numSuffixes = ((F.W + 3) / 4) * ((F.H + 3) / 4);
    N.queryCapacity = (uint32_t)((n + N.numSuffixes + 127) / 128 * 128);
    const size_t S = N.numSuffixes, Q = N.queryCapacity;
    auto alloc = [&](void** p, size_t bytes) {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess)
            e = cudaMemset(*p, 0, bytes);
        return e;
    };
    GFX_CUDA(ctx, alloc((void**)&N.inferenceQuery, Q * 56));
    GFX_CUDA(ctx, alloc((void**)&N.terminalInfo, n * 16));
    GFX_CUDA(ctx, alloc((void**)&N.inferredRadiance, Q * 12));
    GFX_CUDA(ctx, alloc((void**)&N.frameContribution, n * 12));
    for (int i = 0; i < 2; ++i) {
        GFX_CUDA(ctx, alloc((void**)&N.trainQuery[i], (size_t)kTrainBufferSize * 56));
        GFX_CUDA(ctx, alloc((void**)&N.trainTarget[i], (size_t)kTrainBufferSize * 12));
    }
    GFX_CUDA(ctx, alloc((void**)&N.trainVertexInfo, (size_t)kTrainBufferSize * 16));
    GFX_CUDA(ctx, alloc((void**)&N.suffixTerminal, S * 4));
    GFX_CUDA(ctx, alloc((void**)&N.shufflers, (size_t)kNumTrainingDataPerFrame * 4));
    GFX_CUDA(ctx, alloc((void**)&N.state, 32 * 4));
    GFX_CUDA(ctx, alloc((void**)&N.pathA, n * 16));
    GFX_CUDA(ctx, alloc((void**)&N.pathB, n * 16));
    GFX_CUDA(ctx, alloc((void**)&N.shadowPending2, n * 16));
    GFX_CUDA(ctx, alloc((void**)&N.tilePrev, S * 4));
    GFX_CUDA(ctx, alloc((void**)&N.tileSuffixEnded, S * 4));
    GFX_CUDA(ctx, alloc((void**)&N.stagedFlags, S * 4));
    GFX_CUDA(ctx, alloc((void**)&N.stagedIndex, S * 4));
    GFX_CUDA(ctx, alloc((void**)&N.stagedQuery, S * 56));
    GFX_CUDA(ctx, alloc((void**)&N.stagedThroughput, S * 16));
    GFX_CUDA(ctx, alloc((void**)&N.stagedNEE, S * 16));
    GFX_CUDA(ctx, alloc((void**)&N.shardCounts, 128 * 4));
    // host-side initial values (neural_radiance_caching_main.cpp:1155-1193)
    std::vector<uint32_t> suffix(S, kInvalidVertexDataIndex);
    GFX_CUDA(ctx, cudaMemcpy(N.suffixTerminal, suffix.data(), S * 4, cudaMemcpyHostToDevice));
    std::vector<uint32_t> shufflers(kNumTrainingDataPerFrame);
    uint32_t lcg = 471313181u;
    for (uint32_t i = 0; i < kNumTrainingDataPerFrame; ++i) {
        lcg = (lcg * 1103515245u + 12345u) % (1u << 31);
        shufflers[i] = lcg;
    }
    GFX_CUDA(ctx, cudaMemcpy(N.shufflers, shufflers.data(), shufflers.size() * 4, cudaMemcpyHostToDevice));
    uint32_t state[32] = {};
    state[NRC_TILE_SIZE + 0] = state[NRC_TILE_SIZE + 1] = state[NRC_TILE_SIZE + 2] = state[NRC_TILE_SIZE + 3] = 8;
    GFX_CUDA(ctx, cudaMemcpy(N.state, state, sizeof(state), cudaMemcpyHostToDevice));
    N.created = true;
    return GFX_OK;
}

GFX_D int32_t floatToOrderedInt(float v) { // basic_types.h:411-418
    const int32_t i = __float_as_int(v);
    return i >= 0 ? i : i ^ 0x7FFFFFFF;
}

// optix_pathtracing_kernels.cu:12-16
GFX_D void convertToPolar(const f3 &dir, float* phi, float* theta) {
    const float z = fminf(fmaxf(dir.z, -1.0f), 1.0f);
    *theta = dm_acos(z);
    *phi = dm_atan2(dir.y, dir.x);
}

// optix_pathtracing_kernels.cu:18-34; AABB::normalize (basic_types.h:3425-3427); BSDF::getSurfaceParameters
// (common_device.cuh:342-347, 525-531).  `dst` is 8-byte aligned (56-byte records).
GFX_D void createRadianceQuery(const DevFrameParams &p, const f3 &positionInWorld, const f3 &normalInWorld,
                               const f3 &scatteredDirInWorld, const BSDF &bsdf, float* dst) {
    const f3 a = positionInWorld - p.sceneAabbMin, d = p.sceneAabbMax - p.sceneAabbMin;
    float q[14];
    q[0] = d.x != 0 ? a.x / d.x : 0.0f;
    q[1] = d.y != 0 ? a.y / d.y : 0.0f;
    q[2] = d.z != 0 ? a.z / d.z : 0.0f;
    convertToPolar(normalInWorld, &q[3], &q[4]);
    convertToPolar(scatteredDirInWorld, &q[5], &q[6]);
    q[7] = 1 - dm_exp(-bsdf.roughness);
    q[8] = bsdf.diffuseColor.x; q[9] = bsdf.diffuseColor.y; q[10] = bsdf.diffuseColor.z;
    q[11] = bsdf.specularF0Color.x; q[12] = bsdf.specularF0Color.y; q[13] = bsdf.specularF0Color.z;
    float2* o = reinterpret_cast<float2*>(dst);
#pragma unroll
    for (int i = 0; i < 7; ++i)
        o[i] = make_float2(q[2 * i], q[2 * i + 1]);
}
GFX_D void copyQuery(float* dst, const float* src) {
    const float2* s = reinterpret_cast<const float2*>(src);
    float2* o = reinterpret_cast<float2*>(dst);
#pragma unroll
    for (int i = 0; i < 7; ++i)
        o[i] = s[i];
}

GFX_D uint4 packTerminalInfo(const f3 &alpha, uint32_t pathLength, bool hasQuery, bool isTrainingPixel, bool isUnbiasedTile) {
    return make_uint4(__float_as_uint(alpha.x), __float_as_uint(alpha.y), __float_as_uint(alpha.z),
                      (hasQuery ? 1u : 0u) | ((pathLength & 0xFFu) << 1) | ((isTrainingPixel ? 1u : 0u) << 9) |
                          ((isUnbiasedTile ? 1u : 0u) << 10));
}
GFX_D uint32_t packSuffixTerminal(uint32_t prev, bool hasQuery, uint32_t pathLength) {
    return (prev & 0x7FFFFFu) | ((hasQuery ? 1u : 0u) << 23) | ((pathLength & 0xFFu) << 24);
}

// ---------------------------------------------------------------------------------------------------------
// preprocessNRC (nrc_setup_kernels.cu:6-49) + reset of the per-tile staging state
__global__ void k_nrcPreprocess(DevNrc n, uint32_t W, uint32_t H, uint32_t bufIdx, uint32_t offsetToSelectUnbiasedTile,
                                uint32_t offsetToSelectTrainingPath, uint32_t isNewSequence) {
    const uint32_t linearIndex = blockDim.x * blockIdx.x + threadIdx.x;
    if (linearIndex >= n.numSuffixes)
        return;
    const uint32_t prevBufIdx = (bufIdx + 1) % 2;
    if (linearIndex == 0) {
        uint32_t newTileSize[2];
        if (isNewSequence) {
            newTileSize[0] = newTileSize[1] = 8;
        }
        else {
            const uint32_t prevNumTrainingData = n.state[NRC_NUM_TRAINING_DATA + prevBufIdx];
            const float r = sqrtf(static_cast<float>(prevNumTrainingData) / kNumTrainingDataPerFrame);
            for (int c = 0; c < 2; ++c) {
                const uint32_t cur = n.state[NRC_TILE_SIZE + 2 * prevBufIdx + c];
                newTileSize[c] = min(max(dm_f2uint(cur * r), 4u), 128u);
            }
        }
        n.state[NRC_TILE_SIZE + 2 * bufIdx + 0] = newTileSize[0];
        n.state[NRC_TILE_SIZE + 2 * bufIdx + 1] = newTileSize[1];
        n.state[NRC_NUM_TRAINING_DATA + bufIdx] = 0;
        n.state[NRC_OFFSET_UNBIASED_TILE] = offsetToSelectUnbiasedTile;
        n.state[NRC_OFFSET_TRAINING_PATH] = offsetToSelectTrainingPath;
        const float inf = __int_as_float(0x7F800000);
        for (int c = 0; c < 3; ++c) {
            n.state[NRC_TARGET_MIN + 6 * bufIdx + c] = (uint32_t)floatToOrderedInt(inf);
            n.state[NRC_TARGET_MAX + 6 * bufIdx + c] = (uint32_t)floatToOrderedInt(-inf);
            n.state[NRC_TARGET_AVG + 3 * bufIdx + c] = __float_as_uint(0.0f);
        }
        // the launch size of the inference pass, computed by the host in the reference (:2301-2304)
        const uint32_t numTilesX = (W + newTileSize[0] - 1) / newTileSize[0], numTilesY = (H + newTileSize[1] - 1) / newTileSize[1];
        n.state[NRC_NUM_INFERENCE_QUERIES] = (W * H + numTilesX * numTilesY + 127) / 128 * 128;
        n.state[NRC_NUM_SUFFIX_QUERIES] = (numTilesX * numTilesY + 127) / 128 * 128; // a strip's second launch (gfx_nrc_frame_infer_rows)
    }
    n.suffixTerminal[linearIndex] = packSuffixTerminal(kInvalidVertexDataIndex, false, 0);
    n.tilePrev[linearIndex] = kInvalidVertexDataIndex;
    n.tileSuffixEnded[linearIndex] = 0;
    n.stagedFlags[linearIndex] = 0;
    n.stagedIndex[linearIndex] = 0xFFFFFFFFu;
}

// ---------------------------------------------------------------------------------------------------------
struct NrcVertexRequest {
    bool wantVertex;
    uint32_t tile, pathLength;
    bool fromRayGen;
};

// queues the rays of a vertex like emitRays() and, for a training path, stages its training vertex
GFX_D void emitRaysNrc(const DevScene &s, const DevPathState &ps, const DevNrc &n, uint32_t* roundCounters, uint32_t nextQueue,
                       uint32_t lane, uint32_t pix, const f3 &positionInWorld, const VertexOutput &v, bool alive,
                       const NrcVertexRequest &req) {
    const bool wantShadow = alive && v.wantShadow;
    const bool wantExt = alive && v.wantExtension;
    const uint32_t shadowSlot = allocQueueSlot(roundCounters + 2, wantShadow, lane);
    const uint32_t extSlot = allocQueueSlot(roundCounters + 0, wantExt, lane);
    if (wantShadow) {
        ps.shadowRays[2 * (size_t)shadowSlot] = make_float4(positionInWorld.x, positionInWorld.y, positionInWorld.z, 0.0f);
        ps.shadowRays[2 * (size_t)shadowSlot + 1] = make_float4(v.shadowDir.x, v.shadowDir.y, v.shadowDir.z, v.shadowTmax);
        ps.shadowPixel[shadowSlot] = pix;
        ps.shadowPending[shadowSlot] = v.pending;
        n.shadowPending2[shadowSlot] = make_float4(v.neeUnoccluded.x, v.neeUnoccluded.y, v.neeUnoccluded.z,
                                                   __uint_as_float(alive && req.wantVertex ? req.tile : 0xFFFFFFFFu));
    }
    if (wantExt) {
        ps.extRays[nextQueue][2 * (size_t)extSlot] = make_float4(positionInWorld.x, positionInWorld.y, positionInWorld.z, 0.0f);
        ps.extRays[nextQueue][2 * (size_t)extSlot + 1] = make_float4(v.nextDir.x, v.nextDir.y, v.nextDir.z, 3.402823466e+38f);
        ps.extPixel[nextQueue][extSlot] = pix;
    }
    if (alive && req.wantVertex) {
        n.stagedFlags[req.tile] = 1u | (req.fromRayGen ? 2u : 0u) | (req.pathLength << 8);
        n.stagedThroughput[req.tile] = make_float4(v.localThroughput.x, v.localThroughput.y, v.localThroughput.z, 0.0f);
        n.stagedNEE[req.tile] = make_float4(v.directContNEE.x, v.directContNEE.y, v.directContNEE.z, 0.0f);
    }
    const uint32_t cnt = __popc(__ballot_sync(0xFFFFFFFFu, wantShadow)) + __popc(__ballot_sync(0xFFFFFFFFu, wantExt));
    if (lane == 0 && cnt)
        atomicAdd(s.rayCounter, (unsigned long long)cnt);
}

// pathTrace_raygen_generic<true> up to the path extension loop (optix_pathtracing_kernels.cu:95-283)
__global__ void __launch_bounds__(64, kBounceMinBlocks) k_nrcFirstHit(DevScene s, DevFrame f, DevFrameParams p, DevPathState ps, DevNrc n) {
    const uint32_t x = blockIdx.x * 8 + threadIdx.x;
    const uint32_t y = p.y0 + blockIdx.y * 8 + threadIdx.y;
    const uint32_t lane = (threadIdx.x + threadIdx.y * blockDim.x) & 31u;
    const bool inside = x < f.W && y < p.y1;
    const uint32_t pix = inside ? y * f.W + x : 0u;

    bool alive = false;
    f3 positionInWorld(0.0f);
    VertexOutput v;
    v.wantShadow = v.wantExtension = false;
    NrcVertexRequest req;
    req.wantVertex = false;
    req.tile = 0;
    req.pathLength = 1;
    req.fromRayGen = true;
    if (inside) {
        // dynamic tiles: one training path per tile, one tile in 16 unbiased (:107-136)
        const uint32_t tileSizeX = n.state[NRC_TILE_SIZE + 2 * p.bufferIndex], tileSizeY = n.state[NRC_TILE_SIZE + 2 * p.bufferIndex + 1];
        const uint32_t numPixelsInTile = tileSizeX * tileSizeY;
        const uint32_t localLinearIndex = (y % tileSizeY) * tileSizeX + (x % tileSizeX);
        const bool isTrainingPath = (localLinearIndex + n.state[NRC_OFFSET_TRAINING_PATH]) % numPixelsInTile == 0;
        const uint32_t numTilesX = (f.W + tileSizeX - 1) / tileSizeX;
        const uint32_t tileX = x / tileSizeX, tileY = y / tileSizeY;
        const uint32_t linearTileIndex = tileY * numTilesX + tileX;
        const uint32_t localLinearTileIndex = (tileY % 4) * 4 + (tileX % 4);
        const bool isUnbiasedTrainingTile = (localLinearTileIndex + n.state[NRC_OFFSET_UNBIASED_TILE]) % 16 == 0;
        uint32_t flags = (isTrainingPath ? NRC_F_TRAINING_PATH : 0u) | (isUnbiasedTrainingTile ? NRC_F_UNBIASED_TILE : 0u);
        float primaryPathSpread = 0.0f;

        const uint4 gb0 = f.gb0[p.bufferIndex][pix];
        f3 radiance(0.001f, 0.001f, 0.001f);
        if (gb0.x != 0xFFFFFFFFu) {
            flags |= NRC_F_PRIMARY_HIT;
            const DevInstance* inst = s.instances + gb0.x;
            const DevMesh mesh = s.meshes[gb0.y];
            const float bcB = decodeBarycentric((uint16_t)(gb0.w & 0xFFFFu));
            const float bcC = decodeBarycentric((uint16_t)(gb0.w >> 16));
            SurfacePoint sp;
            computeSurfacePointFromGBuffer(s, inst, mesh, gb0.z, bcB, bcC, &sp);

            const f3 alpha(1.0f);
            PCG32RNG rng{ f.rng[pix] };
            const GfxMaterialDesc* mat = s.materials + mesh.materialSlot;
            f3 vOut = p.camera.position - sp.positionInWorld;
            const float primaryDist2 = sqLength(vOut);
            vOut /= sqrtf(primaryDist2);
            const float primaryDotVN = dot(vOut, sp.geometricNormalInWorld);
            const float frontHit = primaryDotVN >= 0.0f ? 1.0f : -1.0f;
            positionInWorld = offsetRayOrigin(sp.positionInWorld, frontHit * sp.geometricNormalInWorld);
            primaryPathSpread = primaryDist2 / (4 * kPi * fabsf(primaryDotVN));
            const ReferenceFrame shadingFrame(sp.shadingNormalInWorld, sp.texCoord0DirInWorld);
            const f3 vOutLocal = shadingFrame.toLocal(vOut);

            radiance = f3(0.0f);
            if (vOutLocal.z > 0 && mat->hasEmittance)
                radiance += alpha * f3(mat->emittance[0], mat->emittance[1], mat->emittance[2]) / kPi;
            const BSDF bsdf = setupBsdfAtHit(s, mesh, gb0.z, bcB, bcC);
            shadeVertex(s, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, &radiance, &v);
            f.rng[pix] = rng.state;
            ps.alphaPdf[pix] = make_float4(v.alpha.x, v.alpha.y, v.alpha.z, v.dirPDensity);
            n.pathB[pix] = make_float4(v.localThroughput.x, v.localThroughput.y, v.localThroughput.z, 0.0f);
            alive = true;
            if (isTrainingPath) { // :213-248
                req.wantVertex = true;
                req.tile = linearTileIndex;
                createRadianceQuery(p, positionInWorld, shadingFrame.normal, vOut, bsdf, n.stagedQuery + 14 * (size_t)linearTileIndex);
            }
        }
        else if (s.env.enabled) { // :323-331: the environment seen directly; the miss program left (u, v) in the barycentrics
            radiance = s.env.powerCoeff * envFetch(s.env, decodeBarycentric((uint16_t)(gb0.w & 0xFFFFu)), decodeBarycentric((uint16_t)(gb0.w >> 16)));
        }
        ps.radiance[pix] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
        n.pathA[pix] = make_float4(primaryPathSpread, 0.0f, __uint_as_float(flags | (1u << 8)), __uint_as_float(linearTileIndex));
    }
    emitRaysNrc(s, ps, n, ps.counters, 0u, lane, pix, positionInWorld, v, alive, req);
}

// pathTrace_closestHit_generic<true> (:363-623) + the loop bookkeeping (:285-311) on the queue of live paths
__global__ void __launch_bounds__(64, kBounceMinBlocks) k_nrcBounce(DevScene s, DevFrame f, DevFrameParams p, DevPathState ps, DevNrc n, uint32_t round) {
    const uint32_t curQueue = round & 1u, nextQueue = curQueue ^ 1u;
    const uint32_t* roundCounters = ps.counters + 4 * round;
    uint32_t* nextCounters = ps.counters + 4 * (round + 1);
    const uint32_t count = roundCounters[0];
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warpsPerGrid = gridDim.x * (blockDim.x >> 5);
    const uint32_t warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const float initImportance = sRGB_calcLuminance(f3(1.0f));
    const uint32_t pathLength = round + 2;
    const bool maxLengthTerminate = (pathLength >= p.maxPathLength && p.maxPathLength > 0) || pathLength >= kMaxNrcRounds;
    const size_t suffixOffset = (size_t)f.W * f.H;

    for (uint32_t base = warp * 32u; base < count; base += warpsPerGrid * 32u) {
        const uint32_t slot = base + lane;
        bool alive = false;
        uint32_t pix = 0;
        f3 positionInWorld(0.0f);
        VertexOutput v;
        v.wantShadow = v.wantExtension = false;
        NrcVertexRequest req;
        req.wantVertex = false;
        req.tile = 0;
        req.pathLength = pathLength;
        req.fromRayGen = false;
        if (slot < count) {
            pix = ps.extPixel[curQueue][slot];
            const uint4 hit = ps.extHits[slot];
            float4 pa = n.pathA[pix];
            uint32_t flags = (__float_as_uint(pa.z) & 0xFFu) | (pathLength << 8);
            const uint32_t tile = __float_as_uint(pa.w);
            const bool isTrainingPath = flags & NRC_F_TRAINING_PATH, isUnbiasedTrainingTile = flags & NRC_F_UNBIASED_TILE;
            bool renderingPathEndsWithCache = flags & NRC_F_RENDERING_ENDS_WITH_CACHE;
            float curSqrtPathSpread = pa.y;
            const float primaryPathSpread = pa.x;

            // one pass through the closest-hit program; `break` = return
            do {
                if (hit.y == 0xFFFFFFFFu) { // pathTrace_miss_generic (:625-672): implicit environment light, MIS
                    if (s.env.enabled) {
                        const float4 r1 = ps.extRays[curQueue][2 * (size_t)slot + 1];
                        const float4 ap = ps.alphaPdf[pix];
                        const f3 directContImplicit = evaluateEnvLightOnMiss(s, f3(r1.x, r1.y, r1.z), ap.w, true);
                        float4 rad = ps.radiance[pix];
                        const f3 add = f3(ap.x, ap.y, ap.z) * directContImplicit;
                        rad.x += add.x; rad.y += add.y; rad.z += add.z;
                        ps.radiance[pix] = rad;
                        const uint32_t prevTrainDataIndex = isTrainingPath ? n.tilePrev[tile] : kInvalidVertexDataIndex;
                        if (isTrainingPath && prevTrainDataIndex != kInvalidVertexDataIndex) {
                            const float4 pb = n.pathB[pix];
                            const f3 addT = f3(pb.x, pb.y, pb.z) * directContImplicit;
                            float* tgt = n.trainTarget[0] + 3 * (size_t)prevTrainDataIndex;
                            tgt[0] += addT.x; tgt[1] += addT.y; tgt[2] += addT.z;
                        }
                    }
                    break;
                }
                const float4 r0 = ps.extRays[curQueue][2 * (size_t)slot];
                const float4 r1 = ps.extRays[curQueue][2 * (size_t)slot + 1];
                const f3 rayOrigin(r0.x, r0.y, r0.z), rayDir(r1.x, r1.y, r1.z);
                const float4 ap = ps.alphaPdf[pix];
                f3 alpha(ap.x, ap.y, ap.z);
                const float prevDirPDensity = ap.w;
                const float4 rad = ps.radiance[pix];
                f3 radiance(rad.x, rad.y, rad.z);
                PCG32RNG rng{ f.rng[pix] };
                const uint32_t prevTrainDataIndex = isTrainingPath ? n.tilePrev[tile] : kInvalidVertexDataIndex;
                bool trainingSuffixEndsWithCache = isTrainingPath ? n.tileSuffixEnded[tile] != 0 : false;

                const uint2 im = __ldg(s.geomToInstMesh + hit.x);
                const DevInstance* inst = s.instances + im.x;
                const DevMesh mesh = s.meshes[im.y];
                SurfacePoint sp;
                computeSurfacePointAtHit(s, inst, mesh, hit.y, __uint_as_float(hit.z), __uint_as_float(hit.w), &sp);
                const GfxMaterialDesc* mat = s.materials + mesh.materialSlot;

                const f3 vOut = normalize(-rayDir);
                const float frontHit = dot(vOut, sp.geometricNormalInWorld) >= 0.0f ? 1.0f : -1.0f;
                const ReferenceFrame shadingFrame(sp.shadingNormalInWorld, sp.texCoord0DirInWorld);
                positionInWorld = offsetRayOrigin(sp.positionInWorld, frontHit * sp.geometricNormalInWorld);
                const f3 vOutLocal = shadingFrame.toLocal(vOut);

                const float dist2 = sqLength(positionInWorld - rayOrigin);
                curSqrtPathSpread += sqrtf(dist2 / (prevDirPDensity * fabsf(vOutLocal.z)));

                // what happens to the path state whichever way the program returns
                auto commitState = [&]() {
                    f.rng[pix] = rng.state;
                    ps.radiance[pix] = make_float4(radiance.x, radiance.y, radiance.z, 0.0f);
                };

                // implicit light sampling (:417-445)
                if (vOutLocal.z > 0 && mat->hasEmittance) {
                    const f3 emittance(mat->emittance[0], mat->emittance[1], mat->emittance[2]);
                    const float lightPDensity = sp.hypAreaPDensity * dist2 / vOutLocal.z;
                    const float bsdfPDensity = prevDirPDensity;
                    const float misWeight = pow2f(bsdfPDensity) / (pow2f(bsdfPDensity) + pow2f(lightPDensity));
                    const f3 directContImplicit = emittance * (misWeight / kPi);
                    radiance += alpha * directContImplicit;
                    if (isTrainingPath && prevTrainDataIndex != kInvalidVertexDataIndex) {
                        const float4 pb = n.pathB[pix];
                        const f3 add = f3(pb.x, pb.y, pb.z) * directContImplicit;
                        float* tgt = n.trainTarget[0] + 3 * (size_t)prevTrainDataIndex;
                        tgt[0] += add.x; tgt[1] += add.y; tgt[2] += add.z;
                    }
                }

                // Russian roulette (:447-469)
                bool performRR = true;
                bool terminatedByRR = false;
                float recContinueProb = 1.0f;
                if (isTrainingPath)
                    performRR = pathLength > 2;
                if (performRR) {
                    const float continueProb = fminf(sRGB_calcLuminance(alpha) / initImportance, 1.0f);
                    if (rng.getFloat0cTo1o() >= continueProb || maxLengthTerminate) {
                        if (renderingPathEndsWithCache && isTrainingPath && isUnbiasedTrainingTile) {
                            commitState();
                            break;
                        }
                        terminatedByRR = true;
                    }
                    recContinueProb = 1.0f / continueProb;
                }

                const BSDF bsdf = setupBsdfAtHit(s, mesh, hit.y, __uint_as_float(hit.z), __uint_as_float(hit.w));

                // termination into the cache by the spread heuristic (:474-531)
                bool endsWithCache = pow2f(curSqrtPathSpread) > kPathTerminationFactor * primaryPathSpread;
                if (renderingPathEndsWithCache && isTrainingPath && isUnbiasedTrainingTile)
                    endsWithCache = false;
                if (endsWithCache) {
                    if (!renderingPathEndsWithCache) {
                        createRadianceQuery(p, positionInWorld, shadingFrame.normal, vOut, bsdf, n.inferenceQuery + 14 * (size_t)pix);
                        n.terminalInfo[pix] = packTerminalInfo(alpha, pathLength, true, isTrainingPath, isUnbiasedTrainingTile);
                        renderingPathEndsWithCache = true;
                        flags |= NRC_F_RENDERING_ENDS_WITH_CACHE;
                        if (isTrainingPath) {
                            curSqrtPathSpread = 0;
                        }
                        else {
                            commitState();
                            break;
                        }
                    }
                    else {
                        if (!trainingSuffixEndsWithCache) {
                            createRadianceQuery(p, positionInWorld, shadingFrame.normal, vOut, bsdf,
                                                n.inferenceQuery + 14 * (suffixOffset + tile));
                            n.suffixTerminal[tile] = packSuffixTerminal(prevTrainDataIndex, true, pathLength);
                            n.tileSuffixEnded[tile] = 1;
                        }
                        commitState();
                        break;
                    }
                }

                if (terminatedByRR) {
                    commitState();
                    break;
                }
                alpha *= recContinueProb;
                if (isTrainingPath && prevTrainDataIndex != kInvalidVertexDataIndex) {
                    uint4* vi = n.trainVertexInfo + prevTrainDataIndex;
                    uint4 t = *vi;
                    t.x = __float_as_uint(__uint_as_float(t.x) * recContinueProb);
                    t.y = __float_as_uint(__uint_as_float(t.y) * recContinueProb);
                    t.z = __float_as_uint(__uint_as_float(t.z) * recContinueProb);
                    *vi = t;
                }

                shadeVertex(s, positionInWorld, vOutLocal, shadingFrame, bsdf, rng, alpha, &radiance, &v);
                ps.alphaPdf[pix] = make_float4(v.alpha.x, v.alpha.y, v.alpha.z, v.dirPDensity);
                n.pathB[pix] = make_float4(v.localThroughput.x, v.localThroughput.y, v.localThroughput.z, 0.0f);
                alive = true;
                commitState();

                if (isTrainingPath && !trainingSuffixEndsWithCache) { // :568-617
                    req.wantVertex = true;
                    req.tile = tile;
                    createRadianceQuery(p, positionInWorld, shadingFrame.normal, vOut, bsdf, n.stagedQuery + 14 * (size_t)tile);
                }
            } while (false);

            pa.y = curSqrtPathSpread;
            pa.z = __uint_as_float(flags);
            n.pathA[pix] = pa;
        }
        emitRaysNrc(s, ps, n, nextCounters, nextQueue, lane, pix, positionInWorld, v, alive, req);
    }
}

// numbers the training vertices staged in this round in tile order: a single block scans the per-tile flags ...
__global__ void __launch_bounds__(1024) k_nrcCommitScan(DevNrc n, uint32_t bufIdx, uint32_t W, uint32_t H) {
    __shared__ uint32_t warpSums[32];
    __shared__ uint32_t blockTotal;
    const uint32_t tid = threadIdx.x;
    // only the tiles of this frame's tile size can hold a staged vertex
    const uint32_t tileSizeX = n.state[NRC_TILE_SIZE + 2 * bufIdx], tileSizeY = n.state[NRC_TILE_SIZE + 2 * bufIdx + 1];
    const uint32_t numTiles = min(((W + tileSizeX - 1) / tileSizeX) * ((H + tileSizeY - 1) / tileSizeY), n.numSuffixes);
    const uint32_t chunk = (numTiles + blockDim.x - 1) / blockDim.x;
    const uint32_t begin = min(tid * chunk, numTiles), end = min(begin + chunk, numTiles);
    uint32_t local = 0;
    for (uint32_t t = begin; t < end; ++t)
        local += n.stagedFlags[t] & 1u;
    // exclusive scan of `local` over the block
    uint32_t incl = local;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if ((tid & 31u) >= (uint32_t)d)
            incl += o;
    }
    if ((tid & 31u) == 31u)
        warpSums[tid >> 5] = incl;
    __syncthreads();
    if (tid < 32) {
        uint32_t w = warpSums[tid], wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, wi, d);
            if (tid >= (uint32_t)d)
                wi += o;
        }
        warpSums[tid] = wi - w;
        if (tid == 31)
            blockTotal = wi;
    }
    __syncthreads();
    // sharded over ranks: the numbers are local until the ranks' counts of this round have been gathered (k_nrcCommitScatter
    // adds the vertices of the earlier rounds and of the ranks above, k_nrcCommitAdvance moves the counter on)
    const bool sharded = n.shardWorld > 1;
    uint32_t rank = (sharded ? 0u : n.state[NRC_NUM_TRAINING_DATA + bufIdx]) + warpSums[tid >> 5] + (incl - local);
    for (uint32_t t = begin; t < end; ++t)
        if (n.stagedFlags[t] & 1u)
            n.stagedIndex[t] = rank++;
    __syncthreads();
    if (tid == 0) {
        if (sharded)
            n.shardCounts[64] = blockTotal;
        else
            n.state[NRC_NUM_TRAINING_DATA + bufIdx] += blockTotal; // the counter keeps counting past the buffer size (:216)
    }
}

__global__ void k_nrcCommitAdvance(DevNrc n, uint32_t bufIdx) {
    uint32_t total = 0;
    for (uint32_t r = 0; r < n.shardWorld; ++r)
        total += n.shardCounts[r];
    n.state[NRC_NUM_TRAINING_DATA + bufIdx] += total;
}

// ... and every staged vertex is moved to the record it was given (:213-248, :568-617)
__global__ void k_nrcCommitScatter(DevNrc n, uint32_t numPixels, uint32_t bufIdx) {
    const uint32_t tile = blockDim.x * blockIdx.x + threadIdx.x;
    if (tile >= n.numSuffixes)
        return;
    const uint32_t flags = n.stagedFlags[tile];
    if (!(flags & 1u))
        return;
    n.stagedFlags[tile] = 0;
    uint32_t trainDataIndex = n.stagedIndex[tile];
    if (n.shardWorld > 1) { // tile order across ranks = rank order: strips are runs of tile rows
        trainDataIndex += n.state[NRC_NUM_TRAINING_DATA + bufIdx];
        for (uint32_t r = 0; r < n.shardRank; ++r)
            trainDataIndex += n.shardCounts[r];
        n.stagedIndex[tile] = trainDataIndex;
    }
    const uint32_t prev = n.tilePrev[tile];
    const uint32_t pathLength = flags >> 8;
    const float* query = n.stagedQuery + 14 * (size_t)tile;
    if (trainDataIndex < kTrainBufferSize) {
        copyQuery(n.trainQuery[0] + 14 * (size_t)trainDataIndex, query);
        const float4 lt = n.stagedThroughput[tile];
        n.trainVertexInfo[trainDataIndex] = make_uint4(__float_as_uint(lt.x), __float_as_uint(lt.y), __float_as_uint(lt.z),
                                                       (prev & 0x7FFFFFu) | ((pathLength & 0xFFu) << 23));
        const float4 nee = n.stagedNEE[tile];
        float* tgt = n.trainTarget[0] + 3 * (size_t)trainDataIndex;
        tgt[0] = nee.x; tgt[1] = nee.y; tgt[2] = nee.z;
        n.tilePrev[tile] = trainDataIndex;
    }
    else if (flags & 2u) {
        n.tilePrev[tile] = kInvalidVertexDataIndex; // :244-246
        n.stagedIndex[tile] = 0xFFFFFFFFu;
    }
    else { // buffer full: the training suffix ends here with a query (:605-616)
        copyQuery(n.inferenceQuery + 14 * ((size_t)numPixels + tile), query);
        n.suffixTerminal[tile] = packSuffixTerminal(prev, true, pathLength);
        n.tileSuffixEnded[tile] = 1;
        n.stagedIndex[tile] = 0xFFFFFFFFu;
    }
}

// ray-gen epilogue (:312-346)
__global__ void __launch_bounds__(256) k_nrcFinish(DevFrame f, DevPathState ps, DevNrc n, uint32_t firstPixel, uint32_t endPixel) {
    const uint32_t pix = firstPixel + blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= endPixel)
        return;
    const float4 pa = n.pathA[pix];
    const uint32_t flags = __float_as_uint(pa.z);
    const uint32_t tile = __float_as_uint(pa.w);
    const uint32_t pathLength = flags >> 8;
    const bool isTrainingPath = flags & NRC_F_TRAINING_PATH;
    if ((flags & NRC_F_PRIMARY_HIT) && isTrainingPath && n.tileSuffixEnded[tile] == 0)
        n.suffixTerminal[tile] = packSuffixTerminal(n.tilePrev[tile], false, pathLength);
    if (!(flags & NRC_F_RENDERING_ENDS_WITH_CACHE))
        n.terminalInfo[pix] = packTerminalInfo(f3(0.0f), pathLength, false, isTrainingPath, flags & NRC_F_UNBIASED_TILE);
    const float4 rad = ps.radiance[pix];
    float* c = n.frameContribution + 3 * (size_t)pix;
    c[0] = rad.x; c[1] = rad.y; c[2] = rad.z;
}

struct NrcShadowWriter { // ShadowAccumulateWriter + the NEE target of the training vertex staged with the ray
    const uint32_t* shadowPixel;
    const float4* pending;
    const float4* pending2;
    float4* radiance;
    const uint32_t* stagedIndex;
    float* trainTarget;
    template <bool ANY_HIT, bool STATS>
    GFX_D void write(uint32_t ray, const TraversalState &st) const {
        const float4 c = pending[ray];
        const bool unoccluded = st.best.storageIndex == 0xFFFFFFFFu;
        if (!unoccluded && isfinite(c.w))
            return;
        float4* dst = radiance + shadowPixel[ray];
        float4 r = *dst;
        if (unoccluded) {
            r.x += c.x; r.y += c.y; r.z += c.z;
            const float4 c2 = pending2[ray];
            const uint32_t tile = __float_as_uint(c2.w);
            if (tile != 0xFFFFFFFFu) {
                const uint32_t idx = stagedIndex[tile];
                if (idx != 0xFFFFFFFFu) {
                    float* tgt = trainTarget + 3 * (size_t)idx;
                    tgt[0] = c2.x; tgt[1] = c2.y; tgt[2] = c2.z;
                }
            }
        }
        else {
            const float nan = __int_as_float(0x7FC00000);
            r.x += nan; r.y += nan; r.z += nan;
        }
        *dst = r;
    }
};

int launchPathTraceNrc(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params) {
    int rc = ensurePathTraceBuffers(ctx);
    if (rc != GFX_OK)
        return rc;
    rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    FrameState &F = ctx->frame;
    const DevFrameParams p = makeDevParams(ctx, params);
    // a strip of rows (tileOriginY / tileRows) is one rank's share of a frame sharded with gfx_nrc_shard: the training
    // vertices are numbered over the whole frame, so a strip without the other ranks would leave holes in the records
    const bool sharded = F.nrc.shardComm != nullptr && F.nrc.shardWorld > 1;
    if (!sharded && (p.y0 != 0 || p.y1 != F.H)) {
        ctx->setError("gfx_pathtrace_launch(GFX_PT_NRC): strips need gfx_nrc_shard (the training records span the frame)");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    if (p.y0 >= p.y1) {
        ctx->setError("gfx_pathtrace_launch(GFX_PT_NRC): empty strip");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    typedef int (*NcclAllGatherFn)(const void*, void*, size_t, int, void*, cudaStream_t);
    const NcclAllGatherFn allGather = sharded ? reinterpret_cast<NcclAllGatherFn>(ncclSymbol("ncclAllGather")) : nullptr;
    if (sharded && !allGather) {
        ctx->setError("gfx_pathtrace_launch(GFX_PT_NRC): ncclAllGather not found (load NCCL in the host process)");
        return GFX_ERR_UNSUPPORTED;
    }
    const DevScene s = ctx->devScene(params);
    const DevFrame f = ctx->devFrame();
    const DevPathState ps = makePathState(ctx);
    const DevNrc n = makeDevNrc(ctx);
    const uint32_t numPixels = F.W * F.H;

    const uint32_t maxPathLength = params->maxPathLength;
    // a training path is exempt from Russian roulette at pathLength 2 (:452-453), so even maxPathLength <= 2 needs
    // the round with pathLength 3
    const uint32_t numRounds = (maxPathLength > 0 ? min(max(maxPathLength, 3u), kMaxNrcRounds) : kMaxNrcRounds) - 1u;
    GFX_CUDA(ctx, cudaMemsetAsync(F.ptCounters, 0, (kMaxPathRounds + 1) * 16, stream));

    const dim3 block(8, 8);
    const dim3 grid((F.W + 7) / 8, (p.y1 - p.y0 + 7) / 8);
    const uint32_t scatterGrid = (n.numSuffixes + 127) / 128;
    int commitError = 0;
    auto commit = [&]() {
        GFX_TIMED(ctx, stream, "nrc_commit");
        k_nrcCommitScan<<<1, 1024, 0, stream>>>(n, p.bufferIndex, F.W, F.H);
        if (sharded) // one word per rank and round: the only exchange the path tracer needs
            commitError |= allGather(n.shardCounts + 64, n.shardCounts, 1, 3 /* ncclUint32 */, F.nrc.shardComm, stream);
        k_nrcCommitScatter<<<scatterGrid, 128, 0, stream>>>(n, numPixels, p.bufferIndex);
        ctx->launches += 2;
        if (sharded) {
            k_nrcCommitAdvance<<<1, 1, 0, stream>>>(n, p.bufferIndex);
            ctx->launches++;
        }
    };
    { GFX_TIMED(ctx, stream, "nrc_first_hit"); k_nrcFirstHit<<<grid, block, 0, stream>>>(s, f, p, ps, n); }
    commit();
    ctx->launches += 1;
    const int traceGrid = wavefrontGrid();
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    const NrcShadowWriter shadowWriter{ ps.shadowPixel, ps.shadowPending, n.shadowPending2, ps.radiance, n.stagedIndex, n.trainTarget[0] };
    const ExtensionHitWriter extWriter{ ps.extHits };
    for (uint32_t round = 0; round < numRounds; ++round) {
        uint32_t* c = F.ptCounters + 4 * round;
        { GFX_TIMED(ctx, stream, "nrc_trace_shadow"); k_traceWavefront<true, false><<<traceGrid, 128, 0, stream>>>(s.bvh, ps.shadowRays, c + 2, 0u, c + 3, shadowWriter); }
        { GFX_TIMED(ctx, stream, "nrc_trace_extension"); k_traceWavefront<false, false><<<traceGrid, 128, 0, stream>>>(s.bvh, ps.extRays[round & 1], c + 0, 0u, c + 1, extWriter); }
        { GFX_TIMED(ctx, stream, "nrc_bounce"); k_nrcBounce<<<sms * 16, 64, 0, stream>>>(s, f, p, ps, n, round); }
        commit();
        ctx->launches += 3;
    }
    // shadow rays requested by the last round (a training path may still have sampled a light there)
    {
        uint32_t* c = F.ptCounters + 4 * numRounds;
        k_traceWavefront<true, false><<<traceGrid, 128, 0, stream>>>(s.bvh, ps.shadowRays, c + 2, 0u, c + 3, shadowWriter);
        ctx->launches++;
    }
    const uint32_t firstPixel = p.y0 * F.W, endPixel = p.y1 * F.W;
    { GFX_TIMED(ctx, stream, "nrc_finish");
    k_nrcFinish<<<(endPixel - firstPixel + 255) / 256, 256, 0, stream>>>(f, ps, n, firstPixel, endPixel); }
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    if (commitError) {
        ctx->setError("gfx_pathtrace_launch(GFX_PT_NRC): ncclAllGather of the training-vertex counts failed");
        return GFX_ERR_CUDA;
    }
    return GFX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// nrc_setup_kernels.cu:51-92
__global__ void __launch_bounds__(256) k_nrcAccumulate(DevFrame f, DevFrameParams p, DevNrc n) {
    const uint32_t i = p.y0 * f.W + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.y1 * f.W)
        return;
    const uint4 t = n.terminalInfo[i];
    const f3 alpha(__uint_as_float(t.x), __uint_as_float(t.y), __uint_as_float(t.z));
    const float* dc = n.frameContribution + 3 * (size_t)i;
    const f3 directCont(dc[0], dc[1], dc[2]);
    f3 radiance(0.0f);
    if (t.w & 1u) {
        const float* r = n.inferredRadiance + 3 * (size_t)i;
        radiance = max3(f3(r[0], r[1], r[2]), f3(0.0f));
        if (p.radianceScale > 0)
            radiance /= p.radianceScale;
        const float* q = n.inferenceQuery + 14 * (size_t)i;
        radiance *= (f3(q[8], q[9], q[10]) + f3(q[11], q[12], q[13]));
    }
    const f3 indirectCont = alpha * radiance;
    const f3 contribution = directCont + indirectCont;
    f3 prevColorResult(0.0f);
    if (p.numAccumFrames > 0) {
        const float4 b = f.beauty[i];
        prevColorResult = f3(b.x, b.y, b.z);
    }
    const float curWeight = 1.0f / (1 + p.numAccumFrames);
    const f3 colorResult = (1 - curWeight) * prevColorResult + curWeight * contribution;
    f.beauty[i] = make_float4(colorResult.x, colorResult.y, colorResult.z, 1.0f);
}

// nrc_setup_kernels.cu:94-138
__global__ void __launch_bounds__(128) k_nrcPropagate(DevFrameParams p, DevNrc n, uint32_t numPixels) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n.numSuffixes)
        return;
    const uint32_t ti = n.suffixTerminal[i];
    const uint32_t prev = ti & 0x7FFFFFu;
    if (prev == kInvalidVertexDataIndex)
        return;
    f3 contribution(0.0f);
    if ((ti >> 23) & 1u) {
        const float* r = n.inferredRadiance + 3 * ((size_t)numPixels + i);
        contribution = max3(f3(r[0], r[1], r[2]), f3(0.0f));
        if (p.radianceScale > 0)
            contribution /= p.radianceScale;
        const float* q = n.inferenceQuery + 14 * ((size_t)numPixels + i);
        contribution *= (f3(q[8], q[9], q[10]) + f3(q[11], q[12], q[13]));
    }
    uint32_t last = prev;
    while (last != kInvalidVertexDataIndex) {
        const uint4 vi = n.trainVertexInfo[last];
        float* tgt = n.trainTarget[0] + 3 * (size_t)last;
        const f3 indirectCont = f3(__uint_as_float(vi.x), __uint_as_float(vi.y), __uint_as_float(vi.z)) * contribution;
        contribution = f3(tgt[0], tgt[1], tgt[2]) + indirectCont;
        const float* q = n.trainQuery[0] + 14 * (size_t)last;
        const f3 refFactor = f3(q[8], q[9], q[10]) + f3(q[11], q[12], q[13]);
        tgt[0] = refFactor.x != 0 ? contribution.x / refFactor.x : 0.0f;
        tgt[1] = refFactor.y != 0 ? contribution.y / refFactor.y : 0.0f;
        tgt[2] = refFactor.z != 0 ? contribution.z / refFactor.z : 0.0f;
        last = vi.w & 0x7FFFFFu;
    }
}

// nrc_setup_kernels.cu:140-216
__global__ void __launch_bounds__(256) k_nrcShuffle(DevFrameParams p, DevNrc n) {
    const uint32_t linearIndex = blockDim.x * blockIdx.x + threadIdx.x;
    const uint32_t bufIdx = p.bufferIndex;
    const uint32_t numTrainingData = n.state[NRC_NUM_TRAINING_DATA + bufIdx];
    __shared__ int32_t smMin[3], smMax[3];
    __shared__ float smAvg[3];
    if (numTrainingData > 0) {
        uint32_t lcg = n.shufflers[linearIndex];
        lcg = (lcg * 1103515245u + 12345u) % (1u << 31);
        n.shufflers[linearIndex] = lcg;
        const uint32_t dstIdx = lcg % kNumTrainingDataPerFrame;
        const uint32_t srcIdx = linearIndex % min(numTrainingData, kTrainBufferSize);
        float q[14];
        const float2* src = reinterpret_cast<const float2*>(n.trainQuery[0] + 14 * (size_t)srcIdx);
        bool valid = true;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const float2 v = src[i];
            q[2 * i] = v.x;
            q[2 * i + 1] = v.y;
            valid = valid && isfinite(v.x) && isfinite(v.y);
        }
        const float* ts = n.trainTarget[0] + 3 * (size_t)srcIdx;
        float tgt[3] = { ts[0], ts[1], ts[2] };
        if (!valid) {
#pragma unroll
            for (int i = 0; i < 14; ++i)
                q[i] = 0.0f;
        }
        if (!(isfinite(tgt[0]) && isfinite(tgt[1]) && isfinite(tgt[2])))
            tgt[0] = tgt[1] = tgt[2] = 0.0f;

        if (threadIdx.x == 0) {
            const float inf = __int_as_float(0x7F800000);
            for (int c = 0; c < 3; ++c) {
                smMin[c] = floatToOrderedInt(inf);
                smMax[c] = floatToOrderedInt(-inf);
                smAvg[c] = 0.0f;
            }
        }
        __syncthreads();
        for (int c = 0; c < 3; ++c) {
            atomicMin(&smMin[c], floatToOrderedInt(tgt[c]));
            atomicMax(&smMax[c], floatToOrderedInt(tgt[c]));
            atomicAdd(&smAvg[c], tgt[c] * (1.0f / kNumTrainingDataPerFrame));
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int c = 0; c < 3; ++c) {
                atomicMin(reinterpret_cast<int32_t*>(n.state + NRC_TARGET_MIN + 6 * bufIdx + c), smMin[c]);
                atomicMax(reinterpret_cast<int32_t*>(n.state + NRC_TARGET_MAX + 6 * bufIdx + c), smMax[c]);
                atomicAdd(reinterpret_cast<float*>(n.state + NRC_TARGET_AVG + 3 * bufIdx + c), smAvg[c]);
            }
        }
        for (int c = 0; c < 3; ++c) {
            if (p.radianceScale > 0)
                tgt[c] *= p.radianceScale;
            tgt[c] = fminf(tgt[c], 1e+6f);
        }
        float2* dst = reinterpret_cast<float2*>(n.trainQuery[1] + 14 * (size_t)dstIdx);
#pragma unroll
        for (int i = 0; i < 7; ++i)
            dst[i] = make_float2(q[2 * i], q[2 * i + 1]);
        float* td = n.trainTarget[1] + 3 * (size_t)dstIdx;
        td[0] = tgt[0]; td[1] = tgt[1]; td[2] = tgt[2];
    }
    else {
        float2* dst = reinterpret_cast<float2*>(n.trainQuery[1] + 14 * (size_t)linearIndex);
#pragma unroll
        for (int i = 0; i < 7; ++i)
            dst[i] = make_float2(0.0f, 0.0f);
        float* td = n.trainTarget[1] + 3 * (size_t)linearIndex;
        td[0] = td[1] = td[2] = 0.0f;
    }
}

int launchNrcPreprocess(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params, uint32_t offsetToSelectUnbiasedTile,
                        uint32_t offsetToSelectTrainingPath, int isNewSequence) {
    const int rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    const DevNrc n = makeDevNrc(ctx);
    GFX_TIMED(ctx, stream, "nrc_preprocess");
    if (n.shardWorld > 1) { // the ranks' records are merged by an integer sum (launchNrcPass, propagate): start from zero
        GFX_CUDA(ctx, cudaMemsetAsync(n.trainQuery[0], 0, (size_t)kTrainBufferSize * 56, stream));
        GFX_CUDA(ctx, cudaMemsetAsync(n.trainTarget[0], 0, (size_t)kTrainBufferSize * 12, stream));
    }
    k_nrcPreprocess<<<(n.numSuffixes + 255) / 256, 256, 0, stream>>>(n, ctx->frame.W, ctx->frame.H, params->bufferIndex & 1,
                                                                     offsetToSelectUnbiasedTile, offsetToSelectTrainingPath,
                                                                     isNewSequence ? 1u : 0u);
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

int launchNrcPass(gfx_ctx* ctx, cudaStream_t stream, const GfxFrameParams* params, int pass) {
    const int rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    const DevNrc n = makeDevNrc(ctx);
    const DevFrameParams p = makeDevParams(ctx, params);
    const uint32_t numPixels = ctx->frame.W * ctx->frame.H;
    static const char* const kPassLabel[3] = { "nrc_accumulate", "nrc_propagate_merge", "nrc_shuffle" };
    GFX_TIMED(ctx, stream, kPassLabel[pass < 0 || pass > 2 ? 0 : pass]);
    switch (pass) {
    case 0: k_nrcAccumulate<<<((p.y1 - p.y0) * ctx->frame.W + 255) / 256, 256, 0, stream>>>(ctx->devFrame(), p, n); break;
    case 1:
        k_nrcPropagate<<<(n.numSuffixes + 127) / 128, 128, 0, stream>>>(p, n, numPixels);
        if (n.shardWorld > 1) {
            // every rank trains on all records (the weights stay replicated): each record was written by exactly one rank
            // and is zero elsewhere, so an unsigned integer sum over the ranks reproduces its bits
            typedef int (*NcclAllReduceFn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
            const NcclAllReduceFn allReduce = reinterpret_cast<NcclAllReduceFn>(ncclSymbol("ncclAllReduce"));
            if (!allReduce) {
                ctx->setError("gfx_nrc_propagate: ncclAllReduce not found (load NCCL in the host process)");
                return GFX_ERR_UNSUPPORTED;
            }
            void* comm = ctx->frame.nrc.shardComm;
            int e = allReduce(n.trainQuery[0], n.trainQuery[0], (size_t)kTrainBufferSize * 14, 3 /* ncclUint32 */, 0 /* ncclSum */, comm, stream);
            e |= allReduce(n.trainTarget[0], n.trainTarget[0], (size_t)kTrainBufferSize * 3, 3, 0, comm, stream);
            if (e) {
                ctx->setError("gfx_nrc_propagate: ncclAllReduce of the training records failed");
                return GFX_ERR_CUDA;
            }
        }
        break;
    case 2: k_nrcShuffle<<<kNumTrainingDataPerFrame / 256, 256, 0, stream>>>(p, n); break;
    default: ctx->setError("unknown NRC pass"); return GFX_ERR_INVALID_ARGUMENT;
    }
    ctx->launches++;
    GFX_CUDA(ctx, cudaGetLastError());
    return GFX_OK;
}

} // namespace gfx
