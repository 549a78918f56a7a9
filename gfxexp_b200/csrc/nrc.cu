// nrc.cu — the Neural Radiance Cache network on sm_100a.
//
// Replaces NeuralRadianceCache::{initialize,infer,train} (neural_radiance_caching/network_interface.cu:
// 48-157) and the tiny-cuda-nn kernels behind it (ext/tiny-cuda-nn: kernel_grid<half,3,2>
// encodings/grid.h:132-304, kernel_one_blob encodings/oneblob.h:83-108, kernel_mlp_fused<64,...>
// src/fully_fused_mlp.cu:47-129 — nvcuda::wmma 16x16x16 half —, relative_l2_luminance_loss,
// adam_step, ema_step_half_precision).
//
// Inference (2.2 M queries per 1080p frame) is ONE fused kernel: each 128-thread CTA encodes 128
// queries (hash grid + one-blob + identity -> 64 fp16 features) straight into shared memory in the
// tcgen05 K-major core-matrix layout, then runs the 64->64->...->16 MLP on the 5th-generation tensor
// cores: tcgen05.mma (M=128, N=64|16, K=16, fp16 in, fp32 accumulate) issued by one thread with the
// accumulator in TMEM, tcgen05.ld back to registers for ReLU + fp16 rounding, activations written
// back to the same shared-memory tile for the next layer.  Weights (18 KB) stay resident in shared
// memory, pre-arranged in the UMMA layout by k_nrcPrepWeights.  No activation ever touches HBM: the
// compulsory traffic is 56 B in + 12 B out per query (SURVEY.md §8d).
//
// Training (4 x 16 384 samples per frame) is latency-bound and runs on CUDA cores: one block = 128
// samples, weights and activations in shared memory, dW reduced per block then atomically added.
#include "context.h"
#include <cuda_fp16.h>
#include <random>
#include <vector>
#include <cmath>

namespace gfx {

constexpr uint32_t kInputDims = 14, kOutputDims = 3, kWidth = 64, kPaddedOutput = 16;
constexpr uint32_t kLevels = 16, kLog2HashmapSize = 15, kBaseResolution = 16;
constexpr float kLossScale = 128.0f;

struct NrcLevel {
    uint32_t offset;      // grid entries
    uint32_t hashmapSize;
    float scale;
    uint32_t resolution;
};
struct NrcLevels { NrcLevel l[kLevels]; };

} // namespace gfx

struct gfx_nrc {
    gfx_ctx* ctx = nullptr;
    uint32_t numHiddenLayers = 2;
    float learningRate = 1e-2f;
    uint32_t numMatrixWeights = 0, numParams = 0;
    gfx::NrcLevels levels;
    __half* params = nullptr;     // current fp16 weights
    __half* paramsEma = nullptr;  // inference weights
    float* master = nullptr;
    float* m1 = nullptr;
    float* m2 = nullptr;
    uint32_t* steps = nullptr;
    unsigned long long* grads = nullptr; // loss-scaled gradients as 64-bit fixed point (2^-30 units): integer atomics
                                         // commute, so a training step is bit-reproducible whatever the block schedule
    float* loss = nullptr;        // device scalar
    uint4* ummaWeights = nullptr; // EMA MLP weights in the tcgen05 shared-memory layout
    uint4* trainBlobFwd = nullptr; // training weights, tcgen05 layouts: W_l [N x 64] and W_l^T [64 x K] K-major blobs
    uint4* trainBlobT = nullptr;
    float4* positions = nullptr;   // split inference scratch: packed query positions, grid features [tile][level][row] half2
    __half2* features = nullptr;
    uint32_t scratchQueries = 0;
    float* gradsFloat = nullptr;   // gfx_nrc_keep_gradients: the loss-scaled gradients of the last training step
    bool keepGradients = false;
    uint32_t globalStep = 0;
    bool ummaDirty = true;
};

namespace gfx {

GFX_D float quarticCdf(float x, float invRadius) { // tiny-cuda-nn common_device.h:478-483
    const float u = x * invRadius;
    const float u2 = u * u;
    const float u4 = u2 * u2;
    return fmaxf(0.0f, fminf(1.0f, (15.0f / 16.0f) * u * (1 - (2.0f / 3.0f) * u2 + (1.0f / 5.0f) * u4) + 0.5f));
}

// index % size without an integer division: hashed levels have power-of-two tables, dense levels only wrap for
// out-of-range positions
GFX_D uint32_t nrcWrap(uint32_t index, uint32_t size) {
    if ((size & (size - 1u)) == 0u)
        return index & (size - 1u);
    return index < size ? index : index % size;
}

// grid_index (grid.h:76-111) for the 8 corners of one cell: the per-axis terms of the dense stride sum or of the
// coherent prime hash are computed once, a corner is one 3-input add/xor plus the wrap. Everything that depends only
// on the level is warp-uniform.
struct NrcCellIndexer {
    uint32_t term[3][2];
    uint32_t size;
    bool hashed;
    GFX_D NrcCellIndexer(const NrcLevel &lv, const uint32_t posGrid[3]) {
        size = lv.hashmapSize;
        uint32_t stride = 1;
        uint32_t strides[3];
        bool used[3];
#pragma unroll
        for (uint32_t dim = 0; dim < 3; ++dim) {
            used[dim] = stride <= lv.hashmapSize;
            strides[dim] = stride;
            if (used[dim])
                stride *= lv.resolution;
        }
        hashed = lv.hashmapSize < stride;
        const uint32_t primes[3] = { 1u, 2654435761u, 805459861u };
#pragma unroll
        for (uint32_t dim = 0; dim < 3; ++dim) {
            const uint32_t m = hashed ? primes[dim] : (used[dim] ? strides[dim] : 0u);
            term[dim][0] = posGrid[dim] * m;
            term[dim][1] = term[dim][0] + m;
        }
    }
    // corner bit d of idx selects posGrid[d] + 1; returns the index of the first of the two features
    GFX_D uint32_t corner(uint32_t idx) const {
        const uint32_t a = term[0][idx & 1u], b = term[1][(idx >> 1) & 1u], c = term[2][(idx >> 2) & 1u];
        return nrcWrap(hashed ? (a ^ b ^ c) : (a + b + c), size) * 2u;
    }
};

GFX_D uint32_t nrcGridIndex(const NrcLevel &lv, const uint32_t pos[3]) { // grid.h:76-111
    uint32_t stride = 1;
    uint32_t index = 0;
#pragma unroll
    for (uint32_t dim = 0; dim < 3; ++dim) {
        if (stride <= lv.hashmapSize) {
            index += pos[dim] * stride;
            stride *= lv.resolution;
        }
    }
    if (lv.hashmapSize < stride)
        index = (pos[0] * 1u) ^ (pos[1] * 2654435761u) ^ (pos[2] * 805459861u);
    return (index % lv.hashmapSize) * 2u;
}

// OneBlob: 5 dims x 4 bins -> features 32..51, identity 52..57, ones 58..63 (q = the 14 query floats; q[0..2] unused)
GFX_D void nrcEncodeTail(const float* q, __half* tail) {
#pragma unroll
    for (uint32_t d = 0; d < 5; ++d) {
        const float x = q[3 + d];
        // kernel_one_blob_soa (tiny-cuda-nn oneblob.h:110-139; the composite encoding runs its nested encodings on SoA
        // slices): CDF at the five bin boundaries k / 4, each summed over the three periodic images
        float leftCdf = quarticCdf(-x, 4.0f) + quarticCdf(-x - 1.0f, 4.0f) + quarticCdf(-x + 1.0f, 4.0f);
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
            const float rightBoundary = 0.25f * (float)(k + 1); // scalbnf(k + 1, -2)
            const float rightCdf = quarticCdf(rightBoundary - x, 4.0f) + quarticCdf(rightBoundary - x - 1.0f, 4.0f) +
                                   quarticCdf(rightBoundary - x + 1.0f, 4.0f);
            tail[d * 4 + k] = __float2half(rightCdf - leftCdf);
            leftCdf = rightCdf;
        }
    }
#pragma unroll
    for (uint32_t d = 0; d < 6; ++d)
        tail[20 + d] = __float2half(q[8 + d]);
#pragma unroll
    for (uint32_t k = 26; k < 32; ++k)
        tail[k] = __float2half(1.0f);
}

// Encodes one query into 64 halves, delivered 8 at a time (chunk c = features 8c..8c+7) through `emit`.
// Arithmetic mirrors oracle/nrc.cpp::encode (half accumulation of the trilinear blend like kernel_grid).
template <typename Emit>
GFX_D void nrcEncode(const NrcLevels &levels, const __half* __restrict__ table, const float* __restrict__ in, Emit emit) {
    float q[kInputDims];
#pragma unroll
    for (uint32_t d = 0; d < kInputDims; ++d)
        q[d] = in[d];
    __half feat[8];
    // Measured on B200 (profiles/r01_summary.md, NRC inference A/B): this exact shape - one level at a time, the 8 gathers
    // interleaved with their index arithmetic - is 10 % faster than issuing the 8 gathers back to back, than 2x/4x
    // unrolling and than a division-free index; the encoder is bound by the L1's divergent-gather rate, not by issue.
#pragma unroll 1
    for (uint32_t l = 0; l < kLevels; ++l) {
        const NrcLevel lv = levels.l[l];
        const __half2* grid = reinterpret_cast<const __half2*>(table + (size_t)lv.offset * 2);
        float pos[3];
        uint32_t posGrid[3];
#pragma unroll
        for (uint32_t d = 0; d < 3; ++d) {
            pos[d] = q[d] * lv.scale + 0.5f;
            const int tmp = (int)floorf(pos[d]);
            posGrid[d] = (uint32_t)tmp;
            pos[d] -= (float)tmp;
        }
        __half r0 = __float2half(0.0f), r1 = __float2half(0.0f);
#pragma unroll
        for (uint32_t idx = 0; idx < 8; ++idx) {
            float weight = 1;
            uint32_t local[3];
#pragma unroll
            for (uint32_t d = 0; d < 3; ++d) {
                if ((idx & (1u << d)) == 0) {
                    weight *= 1 - pos[d];
                    local[d] = posGrid[d];
                }
                else {
                    weight *= pos[d];
                    local[d] = posGrid[d] + 1;
                }
            }
            const __half2 v = __ldg(grid + (nrcGridIndex(lv, local) >> 1));
            r0 = __float2half(__half2float(r0) + __half2float(__float2half(weight * __low2float(v))));
            r1 = __float2half(__half2float(r1) + __half2float(__float2half(weight * __high2float(v))));
        }
        feat[(l & 3) * 2 + 0] = r0;
        feat[(l & 3) * 2 + 1] = r1;
        if ((l & 3) == 3)
            emit(l >> 2, feat);
    }
    __half tail[32];
    nrcEncodeTail(q, tail);
#pragma unroll
    for (uint32_t c = 0; c < 4; ++c)
        emit(4 + c, tail + 8 * c);
}

// ---------------------------------------------------------------------------------------------
// tcgen05 helpers (PTX for sm_100a)
// ---------------------------------------------------------------------------------------------
GFX_D uint32_t smemU32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor): core matrices are
// 8 rows x 16 B stored contiguously; LBO = byte distance between the two K-halves of one MMA (K = 16),
// SBO = byte distance between consecutive 8-row groups.
GFX_D uint64_t makeSmemDesc(uint32_t addr, uint32_t lboBytes, uint32_t sboBytes) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lboBytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sboBytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46; // descriptor version for sm_100
    return d;               // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// instruction descriptor for kind::f16 (cute::UMMA::InstrDescriptor): D = F32, A = B = F16, K-major both
__host__ __device__ constexpr uint32_t makeInstrDesc(uint32_t M, uint32_t N) {
    return (1u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
GFX_D void umma(uint32_t tmemD, uint64_t aDesc, uint64_t bDesc, uint32_t iDesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n"
        :: "r"(tmemD), "l"(aDesc), "l"(bDesc), "r"(iDesc), "r"(accumulate) : "memory");
}
GFX_D void ummaCommit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smemU32(bar)) : "memory");
}
GFX_D void mbarInit(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smemU32(bar)), "r"(count) : "memory");
}
GFX_D void mbarWait(uint64_t* bar, uint32_t phase) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n"
        :: "r"(smemU32(bar)), "r"(phase) : "memory");
}
GFX_D void tmemLoad32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
GFX_D void tmemLoad4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
GFX_D void tmemWaitLd() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
GFX_D void tcFenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
GFX_D void tcFenceAfter() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
GFX_D void fenceProxyAsync() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// k_nrcPrepWeights: EMA MLP weights [out][in] -> per-layer K-major core-matrix blobs:
//   byte offset(layer, n, k) = layerBase + (k / 8) * (N * 16) + n * 16 + (k % 8) * 2
// ---------------------------------------------------------------------------------------------
__global__ void k_nrcPrepWeights(const __half* __restrict__ w, uint32_t numHiddenLayers, __half* __restrict__ blob) {
    const uint32_t total = numHiddenLayers * kWidth * kWidth + kPaddedOutput * kWidth;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        uint32_t layer = i / (kWidth * kWidth), rem = i % (kWidth * kWidth), N = kWidth;
        if (layer >= numHiddenLayers) {
            layer = numHiddenLayers;
            rem = i - numHiddenLayers * kWidth * kWidth;
            N = kPaddedOutput;
        }
        const uint32_t n = rem / kWidth, k = rem % kWidth;
        const uint32_t dst = layer * kWidth * kWidth + (k / 8) * (N * 8) + n * 8 + (k % 8);
        blob[dst] = w[i];
    }
}

// ---------------------------------------------------------------------------------------------
// k_nrcInfer: fused encode + MLP on tcgen05. 128 threads, persistent over 128-query tiles.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kTileRows = 128;
constexpr uint32_t kATileBytes = kTileRows * kWidth * 2; // 16 KB: 8 K-chunks x 128 rows x 16 B

__global__ void __launch_bounds__(128) k_nrcInfer(NrcLevels levels, const __half* __restrict__ table,
                                                  const uint4* __restrict__ ummaWeights, uint32_t numHiddenLayers,
                                                  const float* __restrict__ input, float* __restrict__ output,
                                                  uint32_t numDataImm, const uint32_t* __restrict__ numDataPtr) {
    // the batch size either comes with the launch or lives in device memory (NRC frame: W*H + #tiles, known
    // only on the device; the reference synchronises with the host for it)
    const uint32_t numData = numDataPtr ? *numDataPtr : numDataImm;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA = smem;                                    // activation tile (A operand)
    uint8_t* sW = smem + kATileBytes;                      // all weight blobs (B operands)
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmemBaseShared;

    const uint32_t tid = threadIdx.x;
    const uint32_t warp = tid >> 5;
    const uint32_t weightBytes = (numHiddenLayers * kWidth * kWidth + kPaddedOutput * kWidth) * 2;

    // resident weights (18 KB, once per persistent CTA): cooperative 16-byte copies.  One cp.async.bulk + mbarrier like the
    // training kernel measured neutral for the copy itself and 7 % slower overall because of the code ptxas then generates
    // for the encoder (profiles/r01_summary.md).
    if (tid == 0) {
        mbarInit(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t i = tid; i < weightBytes / 16; i += 128)
        reinterpret_cast<uint4*>(sW)[i] = __ldg(ummaWeights + i);
    if (warp == 0) { // TMEM: 64 fp32 accumulator columns x 128 lanes
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smemU32(&tmemBaseShared)), "r"(64u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fenceProxyAsync();
    tcFenceBefore();
    __syncthreads();
    tcFenceAfter();
    const uint32_t tmemBase = tmemBaseShared;
    const uint32_t tmemRow = tmemBase + ((warp * 32u) << 16); // this warp's 32 lanes

    const uint32_t aAddr = smemU32(sA);
    const uint32_t wAddr = smemU32(sW);
    const uint32_t idescHidden = makeInstrDesc(128, kWidth);
    const uint32_t idescOut = makeInstrDesc(128, kPaddedOutput);
    uint32_t phase = 0;

    const uint32_t numTiles = (numData + kTileRows - 1) / kTileRows;
    for (uint32_t tile = blockIdx.x; tile < numTiles; tile += gridDim.x) {
        const uint32_t row = tile * kTileRows + tid;
        // ---- encode this thread's query into the A tile: chunk c at c * 2048 + row * 16
        if (row < numData) {
            nrcEncode(levels, table, input + (size_t)row * kInputDims, [&](uint32_t c, const __half* f) {
                uint4 v;
                v.x = (uint32_t)__half_as_ushort(f[0]) | ((uint32_t)__half_as_ushort(f[1]) << 16);
                v.y = (uint32_t)__half_as_ushort(f[2]) | ((uint32_t)__half_as_ushort(f[3]) << 16);
                v.z = (uint32_t)__half_as_ushort(f[4]) | ((uint32_t)__half_as_ushort(f[5]) << 16);
                v.w = (uint32_t)__half_as_ushort(f[6]) | ((uint32_t)__half_as_ushort(f[7]) << 16);
                *reinterpret_cast<uint4*>(sA + c * (kTileRows * 16) + tid * 16) = v;
            });
        }
        else {
#pragma unroll
            for (uint32_t c = 0; c < 8; ++c)
                *reinterpret_cast<uint4*>(sA + c * (kTileRows * 16) + tid * 16) = make_uint4(0, 0, 0, 0);
        }

        for (uint32_t layer = 0; layer <= numHiddenLayers; ++layer) {
            const bool last = layer == numHiddenLayers;
            const uint32_t N = last ? kPaddedOutput : kWidth;
            // make the generic-proxy writes of sA visible to the tensor core, order against previous tcgen05.ld
            fenceProxyAsync();
            tcFenceBefore();
            __syncthreads();
            if (tid == 0) {
                tcFenceAfter();
                const uint32_t wLayer = wAddr + layer * kWidth * kWidth * 2;
#pragma unroll
                for (uint32_t k = 0; k < kWidth / 16; ++k) {
                    // K step k covers chunks 2k, 2k+1: A chunk stride 2048 B, B chunk stride N*16 B
                    const uint64_t aDesc = makeSmemDesc(aAddr + 2 * k * (kTileRows * 16), kTileRows * 16, 128);
                    const uint64_t bDesc = makeSmemDesc(wLayer + 2 * k * (N * 16), N * 16, 128);
                    umma(tmemBase, aDesc, bDesc, last ? idescOut : idescHidden, k > 0 ? 1u : 0u);
                }
                ummaCommit(&bar);
            }
            mbarWait(&bar, phase);
            phase ^= 1;
            tcFenceAfter();
            if (!last) {
                // epilogue: accumulator row -> ReLU -> fp16 -> back into the A tile
#pragma unroll
                for (uint32_t half_ = 0; half_ < 2; ++half_) {
                    uint32_t r[32];
                    tmemLoad32(tmemRow + half_ * 32, r);
                    tmemWaitLd();
#pragma unroll
                    for (uint32_t c = 0; c < 4; ++c) {
                        uint32_t packed[4];
#pragma unroll
                        for (uint32_t e = 0; e < 4; ++e) {
                            const float a = fmaxf(__uint_as_float(r[c * 8 + 2 * e]), 0.0f);
                            const float b = fmaxf(__uint_as_float(r[c * 8 + 2 * e + 1]), 0.0f);
                            packed[e] = (uint32_t)__half_as_ushort(__float2half(a)) | ((uint32_t)__half_as_ushort(__float2half(b)) << 16);
                        }
                        *reinterpret_cast<uint4*>(sA + (half_ * 4 + c) * (kTileRows * 16) + tid * 16) =
                            make_uint4(packed[0], packed[1], packed[2], packed[3]);
                    }
                }
            }
            else {
                uint32_t r[4];
                tmemLoad4(tmemRow, r);
                tmemWaitLd();
                if (row < numData) {
                    // trim_and_cast_from: half output -> float
                    output[(size_t)row * kOutputDims + 0] = __half2float(__float2half(__uint_as_float(r[0])));
                    output[(size_t)row * kOutputDims + 1] = __half2float(__float2half(__uint_as_float(r[1])));
                    output[(size_t)row * kOutputDims + 2] = __half2float(__float2half(__uint_as_float(r[2])));
                }
            }
        }
        // all warps are done reading TMEM / the A tile before the next tile overwrites them
        tcFenceBefore();
        __syncthreads();
        tcFenceAfter();
    }

    tcFenceBefore();
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmemBase), "r"(64u) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Inference, split form (default): the hash grid is the part of the network that is bound by divergent gathers - 128 dependent
// 4-byte reads per query out of a 2 MB table, i.e. 128 L1 wavefronts at ~2 clocks each (ncu, round 1: tensor pipe 0.9 % active;
// the fused kernel above and tiny-cuda-nn's kernel_grid both sit at 1.5-1.8 ms for 2.1 M queries on a B200).  One LEVEL of the
// table is only 128 KB, though (level 0: 16 KB), which fits in a B200 SM's shared memory, where a 32-lane gather costs ~3 clocks
// instead of ~66.  So:
//   k_nrcPackPositions   positions of the [N][14] queries -> float4 stream (read once per level below);
//   k_nrcGridEncode      grid = 16 levels x R replicas, one CTA per SM: the CTA pulls ITS level's table into shared memory with
//                        cp.async.bulk (TMA) + mbarrier once, then streams its share of the queries through it: coalesced
//                        position read, 8 shared-memory gathers, trilinear blend in half exactly like kernel_grid
//                        (grid.h:132-255), coalesced half2 store into features[tile][level][row] (8 KB per 128-query tile);
//   k_nrcInferMlp        per 128-query tile: two TMA bulk copies bring the tile's queries (7 KB) and grid features (8 KB) into
//                        shared memory (double-buffered: the next tile is in flight), the threads add one-blob + identity and
//                        lay the A tile out in UMMA core matrices, tcgen05.mma runs the 64->64->...->16 MLP as above, and the
//                        radiance leaves through a TMA bulk store.
// The features are the same halves, bit for bit, as nrcEncode's (tests/test_gpu_nrc.py::test_split_encoding_is_bit_exact).
// ---------------------------------------------------------------------------------------------
__global__ void k_nrcPackPositions(const float* __restrict__ input, float4* __restrict__ positions, uint32_t numDataImm,
                                   const uint32_t* __restrict__ numDataPtr) {
    const uint32_t numData = numDataPtr ? *numDataPtr : numDataImm;
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < numData; q += gridDim.x * blockDim.x) {
        const float* in = input + (size_t)q * kInputDims;
        positions[q] = make_float4(in[0], in[1], in[2], 0.0f);
    }
}

GFX_D void bulkLoad(void* smemDst, const void* globalSrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smemU32(smemDst)), "l"(globalSrc), "r"(bytes), "r"(smemU32(bar)) : "memory");
}
GFX_D void mbarExpectTx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smemU32(bar)), "r"(bytes) : "memory");
}

constexpr uint32_t kEncodeThreads = 1024;
constexpr uint32_t kTileFeatureBytes = kLevels * 128 * 4; // 8 KB per 128-query tile: [level][row] half2

__global__ void __launch_bounds__(kEncodeThreads, 1) k_nrcGridEncode(NrcLevels levels, const __half* __restrict__ table,
                                                                      const float4* __restrict__ positions,
                                                                      __half2* __restrict__ features, uint32_t replicas,
                                                                      uint32_t numDataImm, const uint32_t* __restrict__ numDataPtr) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar;
    const uint32_t numData = numDataPtr ? *numDataPtr : numDataImm;
    const uint32_t level = blockIdx.x / replicas, replica = blockIdx.x % replicas;
    const NrcLevel lv = levels.l[level];
    const uint32_t tableBytes = lv.hashmapSize * 4u;
    if (threadIdx.x == 0) {
        mbarInit(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbarExpectTx(&bar, tableBytes);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(table + (size_t)lv.offset * 2);
        for (uint32_t off = 0; off < tableBytes; off += 32768u)
            bulkLoad(smem + off, src + off, min(32768u, tableBytes - off), &bar);
    }
    __syncthreads();
    mbarWait(&bar, 0);
    __half2* grid = reinterpret_cast<__half2*>(smem);

    // level constants of grid_index (grid.h:76-111), hoisted: dense levels add strides, hashed levels xor prime products
    uint32_t stride = 1, strides[3];
    bool used[3];
#pragma unroll
    for (uint32_t dim = 0; dim < 3; ++dim) {
        used[dim] = stride <= lv.hashmapSize;
        strides[dim] = stride;
        if (used[dim])
            stride *= lv.resolution;
    }
    const bool hashed = lv.hashmapSize < stride;

    // Dense levels index x + y * res + z * res^2 with res a multiple of 16: the queries of a warp are consecutive pixels, whose
    // positions typically run along ONE grid axis, so along y or z all 32 lanes would hit the same shared-memory bank (measured:
    // the dense levels' CTAs took twice as long as the hashed ones' and set the kernel's duration).  Entries are therefore
    // permuted inside each aligned row of 32: entry i lives at i ^ swz(i >> 5), swz(r) = (r ^ (r >> 5)) & 31 - y and z
    // neighbours land in different banks.  Hashed levels are spread by the hash already.
    const bool swizzle = !hashed && (lv.hashmapSize & 31u) == 0u;
    const uint32_t swzMask = swizzle ? 31u : 0u;
    if (swizzle) {
        const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, numRows = lv.hashmapSize >> 5;
        for (uint32_t row = warp; row < numRows; row += kEncodeThreads / 32) {
            const __half2 v = grid[row * 32 + lane];
            __syncwarp();
            grid[row * 32 + (lane ^ ((row ^ (row >> 5)) & 31u))] = v;
        }
        __syncthreads();
    }

    // this replica's share of the 128-query tiles
    const uint32_t numTiles = (numData + 127u) / 128u;
    const uint32_t tilesPer = (numTiles + replicas - 1) / replicas;
    const uint32_t qBegin = min(replica * tilesPer, numTiles) * 128u;
    const uint32_t qEnd = min(min((replica + 1) * tilesPer, numTiles) * 128u, numData);

    const uint32_t primes[3] = { 1u, 2654435761u, 805459861u };
    uint32_t mul[3];
#pragma unroll
    for (uint32_t dim = 0; dim < 3; ++dim)
        mul[dim] = hashed ? primes[dim] : (used[dim] ? strides[dim] : 0u);
    const uint32_t size = lv.hashmapSize;
    const bool pow2 = (size & (size - 1u)) == 0u;

    for (uint32_t q = qBegin + threadIdx.x; q < qEnd; q += kEncodeThreads) {
        const float4 p = __ldg(positions + q);
        const float in[3] = { p.x, p.y, p.z };
        float pos[3];
        uint32_t term[3][2];
#pragma unroll
        for (uint32_t d = 0; d < 3; ++d) { // pos_fract, common_device.h:425-431
            pos[d] = in[d] * lv.scale + 0.5f;
            const int tmp = (int)floorf(pos[d]);
            pos[d] -= (float)tmp;
            term[d][0] = (uint32_t)tmp * mul[d];
            term[d][1] = term[d][0] + mul[d];
        }
        __half2 r = __floats2half2_rn(0.0f, 0.0f);
#pragma unroll
        for (uint32_t idx = 0; idx < 8; ++idx) {
            float weight = 1;
#pragma unroll
            for (uint32_t d = 0; d < 3; ++d)
                weight *= (idx & (1u << d)) == 0 ? 1 - pos[d] : pos[d];
            const uint32_t a = term[0][idx & 1u], b = term[1][(idx >> 1) & 1u], c = term[2][(idx >> 2) & 1u];
            uint32_t index = hashed ? (a ^ b ^ c) : (a + b + c);
            index = pow2 ? (index & (size - 1u)) : (index < size ? index : index % size);
            index ^= ((index >> 5) ^ (index >> 10)) & swzMask;
            const float2 v = __half22float2(grid[index]);
            // result += (half)(weight * (float)value) in half precision (grid.h:233-238); __hadd2 rounds the exact sum once,
            // which equals the float-add-then-round-to-half the oracle spells out (the fp32 sum of two halves only rounds when
            // the smaller one is below a quarter ulp of the larger)
            r = __hadd2(r, __floats2half2_rn(weight * v.x, weight * v.y));
        }
        features[((size_t)(q >> 7) * kLevels + level) * 128u + (q & 127u)] = r;
    }
}

// queries of one tile and its grid features, landed by TMA
struct NrcTileStage {
    float query[128 * kInputDims];    // 7168 B
    __half2 feat[kLevels * 128];      // 8192 B
};

__global__ void __launch_bounds__(128) k_nrcInferMlp(const uint4* __restrict__ ummaWeights, uint32_t numHiddenLayers,
                                                     const float* __restrict__ input, const __half2* __restrict__ features,
                                                     float* __restrict__ output, uint32_t numDataImm,
                                                     const uint32_t* __restrict__ numDataPtr) {
    const uint32_t numData = numDataPtr ? *numDataPtr : numDataImm;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA = smem;                                                        // activation tile (A operand), 16 KB
    NrcTileStage* stage = reinterpret_cast<NrcTileStage*>(smem + kATileBytes); // 2 x 15 KB
    float* sOut = reinterpret_cast<float*>(smem + kATileBytes + 2 * sizeof(NrcTileStage)); // 128 x 3 floats
    uint8_t* sW = smem + kATileBytes + 2 * sizeof(NrcTileStage) + 128 * kOutputDims * 4;   // weight blobs (B operands)
    __shared__ __align__(8) uint64_t bar, stageBar[2];
    __shared__ uint32_t tmemBaseShared;

    const uint32_t tid = threadIdx.x;
    const uint32_t warp = tid >> 5;
    const uint32_t weightBytes = (numHiddenLayers * kWidth * kWidth + kPaddedOutput * kWidth) * 2;
    const uint32_t numTiles = numData / kTileRows;

    auto requestTile = [&](uint32_t tile, uint32_t b) { // thread 0 only
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbarExpectTx(&stageBar[b], (uint32_t)sizeof(NrcTileStage));
        bulkLoad(stage[b].query, input + (size_t)tile * 128 * kInputDims, 128 * kInputDims * 4, &stageBar[b]);
        bulkLoad(stage[b].feat, features + (size_t)tile * kLevels * 128, kTileFeatureBytes, &stageBar[b]);
    };

    if (tid == 0) {
        mbarInit(&bar, 1);
        mbarInit(&stageBar[0], 1);
        mbarInit(&stageBar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (blockIdx.x < numTiles)
            requestTile(blockIdx.x, 0);
    }
    for (uint32_t i = tid; i < weightBytes / 16; i += 128)
        reinterpret_cast<uint4*>(sW)[i] = __ldg(ummaWeights + i);
    if (warp == 0) { // TMEM: 64 fp32 accumulator columns x 128 lanes
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smemU32(&tmemBaseShared)), "r"(64u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fenceProxyAsync();
    tcFenceBefore();
    __syncthreads();
    tcFenceAfter();
    const uint32_t tmemBase = tmemBaseShared;
    const uint32_t tmemRow = tmemBase + ((warp * 32u) << 16); // this warp's 32 lanes

    const uint32_t aAddr = smemU32(sA);
    const uint32_t wAddr = smemU32(sW);
    const uint32_t idescHidden = makeInstrDesc(128, kWidth);
    const uint32_t idescOut = makeInstrDesc(128, kPaddedOutput);
    uint32_t phase = 0, stagePhase0 = 0, stagePhase1 = 0, buf = 0;

    for (uint32_t tile = blockIdx.x; tile < numTiles; tile += gridDim.x, buf ^= 1u) {
        // prefetch the next tile into the other buffer (every thread finished reading it one tile ago: the end-of-tile barrier)
        if (tid == 0 && tile + gridDim.x < numTiles)
            requestTile(tile + gridDim.x, buf ^ 1u);
        if (buf == 0) {
            mbarWait(&stageBar[0], stagePhase0);
            stagePhase0 ^= 1u;
        }
        else {
            mbarWait(&stageBar[1], stagePhase1);
            stagePhase1 ^= 1u;
        }
        const NrcTileStage &st = stage[buf];

        // ---- this thread's row of the A tile: chunk c (8 features = 16 B) at c * 2048 + row * 16
#pragma unroll
        for (uint32_t c = 0; c < 4; ++c) { // hash grid: levels 4c .. 4c + 3
            uint4 v;
            v.x = *reinterpret_cast<const uint32_t*>(&st.feat[(4 * c + 0) * 128 + tid]);
            v.y = *reinterpret_cast<const uint32_t*>(&st.feat[(4 * c + 1) * 128 + tid]);
            v.z = *reinterpret_cast<const uint32_t*>(&st.feat[(4 * c + 2) * 128 + tid]);
            v.w = *reinterpret_cast<const uint32_t*>(&st.feat[(4 * c + 3) * 128 + tid]);
            *reinterpret_cast<uint4*>(sA + c * (kTileRows * 16) + tid * 16) = v;
        }
        {
            float q[kInputDims];
            q[0] = q[1] = q[2] = 0.0f;
#pragma unroll
            for (uint32_t d = 3; d < kInputDims; ++d)
                q[d] = st.query[tid * kInputDims + d];
            __half tail[32];
            nrcEncodeTail(q, tail);
#pragma unroll
            for (uint32_t c = 0; c < 4; ++c) {
                uint4 v;
                const __half* f = tail + 8 * c;
                v.x = (uint32_t)__half_as_ushort(f[0]) | ((uint32_t)__half_as_ushort(f[1]) << 16);
                v.y = (uint32_t)__half_as_ushort(f[2]) | ((uint32_t)__half_as_ushort(f[3]) << 16);
                v.z = (uint32_t)__half_as_ushort(f[4]) | ((uint32_t)__half_as_ushort(f[5]) << 16);
                v.w = (uint32_t)__half_as_ushort(f[6]) | ((uint32_t)__half_as_ushort(f[7]) << 16);
                *reinterpret_cast<uint4*>(sA + (4 + c) * (kTileRows * 16) + tid * 16) = v;
            }
        }

        for (uint32_t layer = 0; layer <= numHiddenLayers; ++layer) {
            const bool last = layer == numHiddenLayers;
            const uint32_t N = last ? kPaddedOutput : kWidth;
            // make the generic-proxy writes of sA visible to the tensor core, order against previous tcgen05.ld
            fenceProxyAsync();
            tcFenceBefore();
            __syncthreads();
            if (tid == 0) {
                tcFenceAfter();
                const uint32_t wLayer = wAddr + layer * kWidth * kWidth * 2;
#pragma unroll
                for (uint32_t k = 0; k < kWidth / 16; ++k) {
                    const uint64_t aDesc = makeSmemDesc(aAddr + 2 * k * (kTileRows * 16), kTileRows * 16, 128);
                    const uint64_t bDesc = makeSmemDesc(wLayer + 2 * k * (N * 16), N * 16, 128);
                    umma(tmemBase, aDesc, bDesc, last ? idescOut : idescHidden, k > 0 ? 1u : 0u);
                }
                ummaCommit(&bar);
            }
            mbarWait(&bar, phase);
            phase ^= 1;
            tcFenceAfter();
            if (!last) {
#pragma unroll
                for (uint32_t half_ = 0; half_ < 2; ++half_) {
                    uint32_t r[32];
                    tmemLoad32(tmemRow + half_ * 32, r);
                    tmemWaitLd();
#pragma unroll
                    for (uint32_t c = 0; c < 4; ++c) {
                        uint32_t packed[4];
#pragma unroll
                        for (uint32_t e = 0; e < 4; ++e) {
                            const float a = fmaxf(__uint_as_float(r[c * 8 + 2 * e]), 0.0f);
                            const float b = fmaxf(__uint_as_float(r[c * 8 + 2 * e + 1]), 0.0f);
                            packed[e] = (uint32_t)__half_as_ushort(__float2half(a)) | ((uint32_t)__half_as_ushort(__float2half(b)) << 16);
                        }
                        *reinterpret_cast<uint4*>(sA + (half_ * 4 + c) * (kTileRows * 16) + tid * 16) =
                            make_uint4(packed[0], packed[1], packed[2], packed[3]);
                    }
                }
            }
            else {
                uint32_t r[4];
                tmemLoad4(tmemRow, r);
                tmemWaitLd();
                // the previous tile's bulk store must have read sOut before it is overwritten
                if (tid == 0)
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                __syncthreads();
                // trim_and_cast_from: half output -> float
                sOut[tid * kOutputDims + 0] = __half2float(__float2half(__uint_as_float(r[0])));
                sOut[tid * kOutputDims + 1] = __half2float(__float2half(__uint_as_float(r[1])));
                sOut[tid * kOutputDims + 2] = __half2float(__float2half(__uint_as_float(r[2])));
            }
        }
        // all warps are done reading TMEM / the A tile / the stage before the next tile overwrites them
        fenceProxyAsync();
        tcFenceBefore();
        __syncthreads();
        tcFenceAfter();
        if (tid == 0) { // radiance of the tile: one TMA bulk store of 1536 contiguous bytes
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         :: "l"(output + (size_t)tile * 128 * kOutputDims), "r"(smemU32(sOut)), "r"(128u * kOutputDims * 4u) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (tid == 0)
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    tcFenceBefore();
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmemBase), "r"(64u) : "memory");
}

// test hook: the 64 encoded halves per query as the split pipeline produces them (pack -> grid encode -> tail)
__global__ void k_nrcAssembleEncoding(const float* __restrict__ input, const __half2* __restrict__ features, uint32_t numData,
                                      __half* __restrict__ out) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= numData)
        return;
    __half* o = out + (size_t)q * 64;
    for (uint32_t l = 0; l < kLevels; ++l) {
        const __half2 v = features[((size_t)(q >> 7) * kLevels + l) * 128u + (q & 127u)];
        o[2 * l] = __low2half(v);
        o[2 * l + 1] = __high2half(v);
    }
    float qv[kInputDims];
    for (uint32_t d = 0; d < kInputDims; ++d)
        qv[d] = input[(size_t)q * kInputDims + d];
    __half tail[32];
    nrcEncodeTail(qv, tail);
    for (uint32_t k = 0; k < 32; ++k)
        o[32 + k] = tail[k];
}

// ---------------------------------------------------------------------------------------------
// training step on CUDA cores: block = 128 samples
// ---------------------------------------------------------------------------------------------
// deterministic gradient accumulation: 2^-30 fixed point in 64 bits (range +-8.6e9, resolution 9.3e-10 on loss-scaled values)
constexpr float kGradFixedScale = 1073741824.0f;
GFX_D void atomicAddFixed(unsigned long long* p, float v) {
    atomicAdd(p, (unsigned long long)__float2ll_rn(v * kGradFixedScale));
}
GFX_D float fixedToFloat(unsigned long long v) {
    return (float)((double)(long long)v * (1.0 / 1073741824.0));
}

constexpr uint32_t kRowStride = 66; // halves per activation row in shared memory (conflict-free rows)

__global__ void __launch_bounds__(128) k_nrcTrain(NrcLevels levels, const __half* __restrict__ params, uint32_t numMatrixWeights,
                                                  uint32_t numHiddenLayers, const float* __restrict__ input,
                                                  const float* __restrict__ target, uint32_t numData,
                                                  unsigned long long* __restrict__ grads, float* __restrict__ lossOut) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t H = numHiddenLayers;
    __half* sW = reinterpret_cast<__half*>(smem);                              // numMatrixWeights
    __half* sAct = sW + numMatrixWeights;                                      // (H + 1) x 128 x kRowStride
    __half* sD = sAct + (size_t)(H + 1) * 128 * kRowStride;                    // 128 x kRowStride
    __shared__ float sLoss[4];

    const uint32_t tid = threadIdx.x;
    const uint32_t q = blockIdx.x * 128 + tid;
    const bool valid = q < numData;
    for (uint32_t i = tid; i < numMatrixWeights; i += 128)
        sW[i] = params[i];
    const __half* table = params + numMatrixWeights;

    __half* x = sAct + (size_t)tid * kRowStride;
    if (valid) {
        nrcEncode(levels, table, input + (size_t)q * kInputDims, [&](uint32_t c, const __half* f) {
#pragma unroll
            for (uint32_t e = 0; e < 8; ++e)
                x[c * 8 + e] = f[e];
        });
    }
    else {
        for (uint32_t e = 0; e < 64; ++e)
            x[e] = __float2half(0.0f);
    }
    __syncthreads();

    // forward
    for (uint32_t layer = 0; layer < H; ++layer) {
        const __half* W = sW + (size_t)layer * kWidth * kWidth;
        const __half* in = sAct + ((size_t)layer * 128 + tid) * kRowStride;
        __half* out = sAct + ((size_t)(layer + 1) * 128 + tid) * kRowStride;
        for (uint32_t j = 0; j < kWidth; ++j) {
            float acc = 0.0f;
#pragma unroll 8
            for (uint32_t i = 0; i < kWidth; ++i)
                acc += __half2float(W[j * kWidth + i]) * __half2float(in[i]);
            out[j] = __float2half(fmaxf(acc, 0.0f));
        }
    }
    __half o[kPaddedOutput];
    {
        const __half* W = sW + (size_t)H * kWidth * kWidth;
        const __half* in = sAct + ((size_t)H * 128 + tid) * kRowStride;
        for (uint32_t j = 0; j < kPaddedOutput; ++j) {
            float acc = 0.0f;
#pragma unroll 8
            for (uint32_t i = 0; i < kWidth; ++i)
                acc += __half2float(W[j * kWidth + i]) * __half2float(in[i]);
            o[j] = __float2half(acc);
        }
    }
    // loss + dL/dy (relative_l2_luminance.h:41-88)
    float localLoss = 0.0f;
    __half* d = sD + (size_t)tid * kRowStride;
    {
        const uint32_t nTotal = numData * kOutputDims;
        const float r = __half2float(o[0]), g = __half2float(o[1]), b = __half2float(o[2]);
        const float luminance = 0.299f * r + 0.587f * g + 0.114f * b;
        const float denom = luminance * luminance + 0.01f;
        for (uint32_t k = 0; k < kPaddedOutput; ++k) {
            float gr = 0.0f;
            if (k < kOutputDims && valid) {
                const float difference = __half2float(o[k]) - target[(size_t)q * kOutputDims + k];
                localLoss += difference * difference / denom / nTotal;
                gr = kLossScale * (2 * difference / denom) / nTotal;
            }
            d[k] = __float2half(gr);
        }
    }
    __syncthreads();

    // output layer: dW, then dL/d(hidden)
    {
        const uint32_t base = H * kWidth * kWidth;
        const __half* hin = sAct + (size_t)H * 128 * kRowStride;
        for (uint32_t p = tid; p < kPaddedOutput * kWidth; p += 128) {
            const uint32_t j = p / kWidth, i = p % kWidth;
            float acc = 0.0f;
            for (uint32_t s = 0; s < 128; ++s)
                acc += __half2float(sD[s * kRowStride + j]) * __half2float(hin[s * kRowStride + i]);
            if (acc != 0.0f)
                atomicAddFixed(grads + base + p, acc);
        }
        const __half* W = sW + (size_t)H * kWidth * kWidth;
        const __half* myIn = hin + (size_t)tid * kRowStride;
        __half dNext[64];
        for (uint32_t i = 0; i < kWidth; ++i) {
            float acc = 0.0f;
#pragma unroll
            for (uint32_t j = 0; j < kPaddedOutput; ++j)
                acc += __half2float(W[j * kWidth + i]) * __half2float(d[j]);
            dNext[i] = (H > 0 && !(__half2float(myIn[i]) > 0.0f)) ? __float2half(0.0f) : __float2half(acc);
        }
        __syncthreads();
        for (uint32_t i = 0; i < kWidth; ++i)
            d[i] = dNext[i];
        __syncthreads();
    }
    for (int layer = (int)H - 1; layer >= 0; --layer) {
        const uint32_t base = (uint32_t)layer * kWidth * kWidth;
        const __half* hin = sAct + (size_t)layer * 128 * kRowStride;
        for (uint32_t p = tid; p < kWidth * kWidth; p += 128) {
            const uint32_t j = p / kWidth, i = p % kWidth;
            float acc = 0.0f;
            for (uint32_t s = 0; s < 128; ++s)
                acc += __half2float(sD[s * kRowStride + j]) * __half2float(hin[s * kRowStride + i]);
            if (acc != 0.0f)
                atomicAddFixed(grads + base + p, acc);
        }
        const __half* W = sW + (size_t)layer * kWidth * kWidth;
        const __half* myIn = hin + (size_t)tid * kRowStride;
        __half dNext[64];
        for (uint32_t i = 0; i < kWidth; ++i) {
            float acc = 0.0f;
            for (uint32_t j = 0; j < kWidth; ++j)
                acc += __half2float(W[j * kWidth + i]) * __half2float(d[j]);
            dNext[i] = (layer > 0 && !(__half2float(myIn[i]) > 0.0f)) ? __float2half(0.0f) : __float2half(acc);
        }
        __syncthreads();
        for (uint32_t i = 0; i < kWidth; ++i)
            d[i] = dNext[i];
        __syncthreads();
    }

    // hash-grid backward (kernel_grid_backward, grid.h:306-429): scatter the first 32 input gradients
    if (valid) {
        unsigned long long* gGrid = grads + numMatrixWeights;
        const float* in = input + (size_t)q * kInputDims;
        for (uint32_t l = 0; l < kLevels; ++l) {
            const NrcLevel lv = levels.l[l];
            const float g0 = __half2float(d[l * 2 + 0]), g1 = __half2float(d[l * 2 + 1]);
            if (g0 == 0.0f && g1 == 0.0f)
                continue;
            float pos[3];
            uint32_t posGrid[3];
            for (uint32_t dd = 0; dd < 3; ++dd) {
                pos[dd] = in[dd] * lv.scale + 0.5f;
                const int tmp = (int)floorf(pos[dd]);
                posGrid[dd] = (uint32_t)tmp;
                pos[dd] -= (float)tmp;
            }
            const NrcCellIndexer indexer(lv, posGrid);
#pragma unroll
            for (uint32_t idx = 0; idx < 8; ++idx) {
                float weight = 1;
#pragma unroll
                for (uint32_t dd = 0; dd < 3; ++dd)
                    weight *= (idx & (1u << dd)) == 0 ? 1 - pos[dd] : pos[dd];
                const uint32_t gi = lv.offset * 2 + indexer.corner(idx);
                atomicAddFixed(gGrid + gi, weight * g0);
                atomicAddFixed(gGrid + gi + 1, weight * g1);
            }
        }
    }
    // block loss
    for (int off = 16; off > 0; off >>= 1)
        localLoss += __shfl_xor_sync(0xFFFFFFFFu, localLoss, off);
    if ((tid & 31) == 0)
        sLoss[tid >> 5] = localLoss;
    __syncthreads();
    if (tid == 0)
        atomicAdd(lossOut, sLoss[0] + sLoss[1] + sLoss[2] + sLoss[3]);
}

// ---------------------------------------------------------------------------------------------
// k_nrcTrainTc: the same training step with every matrix product on tcgen05 (forward, data gradients, weight gradients).
//
// Per CTA = 128 samples (kernel_mlp_fused + kernel_mlp_fused_backward of tiny-cuda-nn work on the same 128-row chunks,
// ext/tiny-cuda-nn/src/fully_fused_mlp.cu:47-129, 150-259; the weight gradients are its three split-K CUTLASS GEMMs,
// :822-873).  All operands are K-major core-matrix tiles in shared memory:
//   forward        Z_l     [128 x N]  = A_l [128 x 64]            x W_l^T   (B = W_l blob  [N x 64],  as in k_nrcInfer)
//   data gradient  dA_l    [128 x 64] = dZ_l [128 x K]            x W_l     (B = W_l^T blob [64 x K], K = 64 or 16)
//   weight grad    dW_l    [K x 64]   = dZ_l^T [K(<=64) x 128]    x A_l     (A = transposed dZ tile, B = transposed A_l tile,
//                                                                            K = 128 samples; issued with M = 128, rows >= 64
//                                                                            of the accumulator are ignored)
// The transposed tiles are written by the threads that own the rows (each thread holds its sample's dZ row in registers
// and re-reads its A_l row).  Accumulators live in three 64-column TMEM regions; one tcgen05.commit per phase.
// Rounding points match k_nrcTrain (activations and gradients are fp16 between layers, fp32 accumulation inside).
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kTTileBytes = 64 * 128 * 2; // transposed tile: 16 K-chunks x 64 rows x 16 B

__global__ void k_nrcPrepTrainWeights(const __half* __restrict__ w, uint32_t numHiddenLayers, __half* __restrict__ blobFwd,
                                      __half* __restrict__ blobT) {
    const uint32_t total = numHiddenLayers * kWidth * kWidth + kPaddedOutput * kWidth;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        uint32_t layer = i / (kWidth * kWidth), rem = i % (kWidth * kWidth), N = kWidth;
        if (layer >= numHiddenLayers) {
            layer = numHiddenLayers;
            rem = i - numHiddenLayers * kWidth * kWidth;
            N = kPaddedOutput;
        }
        const uint32_t j = rem / kWidth, in = rem % kWidth; // W_l[j][in]
        // forward blob: B[n = j][k = in]
        blobFwd[layer * kWidth * kWidth + (in / 8) * (N * 8) + j * 8 + (in % 8)] = w[i];
        // transposed blob: B[n = in][k = j], 64 rows per K-chunk
        blobT[layer * kWidth * kWidth + (j / 8) * (kWidth * 8) + in * 8 + (j % 8)] = w[i];
    }
}

__global__ void __launch_bounds__(128) k_nrcTrainTc(NrcLevels levels, const __half* __restrict__ params, uint32_t numMatrixWeights,
                                                    uint32_t numHiddenLayers, const uint4* __restrict__ blobFwd,
                                                    const uint4* __restrict__ blobT, const float* __restrict__ input,
                                                    const float* __restrict__ target, uint32_t numData,
                                                    unsigned long long* __restrict__ grads, float* __restrict__ lossOut) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t H = numHiddenLayers;
    const uint32_t weightBytes = numMatrixWeights * 2;
    uint8_t* sWf = smem;                                   // forward blobs
    uint8_t* sWt = sWf + weightBytes;                      // transposed blobs
    uint8_t* sAct = sWt + weightBytes;                     // (H + 1) activation tiles A_0..A_H, 16 KB each
    uint8_t* sDz = sAct + (H + 1) * kATileBytes;           // dZ tile [128 x 64] (K-major, rows = samples)
    uint8_t* sDzT = sDz + kATileBytes;                     // dZ^T tile [64 x 128] (rows = neurons, K = samples)
    uint8_t* sActT = sDzT + kTTileBytes;                   // A_l^T tile [64 x 128]; the M = 128 read of sDzT spills into it
    __shared__ __align__(8) uint64_t bar, weightBar;
    __shared__ uint32_t tmemBaseShared;
    __shared__ float sLoss[4];

    const uint32_t tid = threadIdx.x;
    const uint32_t warp = tid >> 5;
    const uint32_t q = blockIdx.x * 128 + tid;
    const bool valid = q < numData;
    const __half* table = params + numMatrixWeights;

    if (tid == 0) {
        mbarInit(&bar, 1);
        mbarInit(&weightBar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smemU32(&weightBar)), "r"(2 * weightBytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smemU32(sWf)), "l"(blobFwd), "r"(weightBytes), "r"(smemU32(&weightBar)) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smemU32(sWt)), "l"(blobT), "r"(weightBytes), "r"(smemU32(&weightBar)) : "memory");
    }
    if (warp == 0) { // TMEM: 3 accumulators of 64 fp32 columns (forward / data gradient / weight gradient) -> 256 columns
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smemU32(&tmemBaseShared)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }

    // encode this thread's sample into A_0
    if (valid) {
        nrcEncode(levels, table, input + (size_t)q * kInputDims, [&](uint32_t c, const __half* f) {
            uint4 v;
            v.x = (uint32_t)__half_as_ushort(f[0]) | ((uint32_t)__half_as_ushort(f[1]) << 16);
            v.y = (uint32_t)__half_as_ushort(f[2]) | ((uint32_t)__half_as_ushort(f[3]) << 16);
            v.z = (uint32_t)__half_as_ushort(f[4]) | ((uint32_t)__half_as_ushort(f[5]) << 16);
            v.w = (uint32_t)__half_as_ushort(f[6]) | ((uint32_t)__half_as_ushort(f[7]) << 16);
            *reinterpret_cast<uint4*>(sAct + c * (kTileRows * 16) + tid * 16) = v;
        });
    }
    else {
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c)
            *reinterpret_cast<uint4*>(sAct + c * (kTileRows * 16) + tid * 16) = make_uint4(0, 0, 0, 0);
    }
    fenceProxyAsync();
    tcFenceBefore();
    __syncthreads();
    tcFenceAfter();
    mbarWait(&weightBar, 0);
    const uint32_t tmemBase = tmemBaseShared;
    const uint32_t tmemRow = tmemBase + ((warp * 32u) << 16);
    const uint32_t tmemFwd = 0, tmemDa = 64, tmemDw = 128; // column offsets
    const uint32_t idesc64 = makeInstrDesc(128, kWidth), idesc16 = makeInstrDesc(128, kPaddedOutput);
    uint32_t phase = 0;

    // ---- forward
    for (uint32_t layer = 0; layer <= H; ++layer) {
        const bool last = layer == H;
        const uint32_t N = last ? kPaddedOutput : kWidth;
        if (tid == 0) {
            tcFenceAfter();
            const uint32_t aAddr = smemU32(sAct + layer * kATileBytes);
            const uint32_t wLayer = smemU32(sWf) + layer * kWidth * kWidth * 2;
#pragma unroll
            for (uint32_t k = 0; k < kWidth / 16; ++k)
                umma(tmemBase + tmemFwd, makeSmemDesc(aAddr + 2 * k * (kTileRows * 16), kTileRows * 16, 128),
                     makeSmemDesc(wLayer + 2 * k * (N * 16), N * 16, 128), last ? idesc16 : idesc64, k > 0 ? 1u : 0u);
            ummaCommit(&bar);
        }
        mbarWait(&bar, phase);
        phase ^= 1;
        tcFenceAfter();
        if (!last) {
            uint8_t* next = sAct + (layer + 1) * kATileBytes;
#pragma unroll
            for (uint32_t half_ = 0; half_ < 2; ++half_) {
                uint32_t r[32];
                tmemLoad32(tmemRow + tmemFwd + half_ * 32, r);
                tmemWaitLd();
#pragma unroll
                for (uint32_t c = 0; c < 4; ++c) {
                    uint32_t packed[4];
#pragma unroll
                    for (uint32_t e = 0; e < 4; ++e) {
                        const float a = fmaxf(__uint_as_float(r[c * 8 + 2 * e]), 0.0f);
                        const float b = fmaxf(__uint_as_float(r[c * 8 + 2 * e + 1]), 0.0f);
                        packed[e] = (uint32_t)__half_as_ushort(__float2half(a)) | ((uint32_t)__half_as_ushort(__float2half(b)) << 16);
                    }
                    *reinterpret_cast<uint4*>(next + (half_ * 4 + c) * (kTileRows * 16) + tid * 16) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                }
            }
            fenceProxyAsync();
            tcFenceBefore();
            __syncthreads();
        }
    }

    // ---- loss + dL/dy (relative_l2_luminance.h:41-88)
    __half d[64]; // this sample's gradient row of the current layer (dZ_l), fp16 like tiny-cuda-nn's backward buffers
    float localLoss = 0.0f;
    {
        uint32_t r[4];
        tmemLoad4(tmemRow + tmemFwd, r);
        tmemWaitLd();
        const __half o[3] = { __float2half(__uint_as_float(r[0])), __float2half(__uint_as_float(r[1])), __float2half(__uint_as_float(r[2])) };
        const uint32_t nTotal = numData * kOutputDims;
        const float rr = __half2float(o[0]), gg = __half2float(o[1]), bb = __half2float(o[2]);
        const float luminance = 0.299f * rr + 0.587f * gg + 0.114f * bb;
        const float denom = luminance * luminance + 0.01f;
#pragma unroll
        for (uint32_t k = 0; k < kPaddedOutput; ++k) {
            float gr = 0.0f;
            if (k < kOutputDims && valid) {
                const float difference = __half2float(o[k]) - target[(size_t)q * kOutputDims + k];
                localLoss += difference * difference / denom / nTotal;
                gr = kLossScale * (2 * difference / denom) / nTotal;
            }
            d[k] = __float2half(gr);
        }
    }

    // ---- backward, layer H (output, K = 16) down to 0
    for (int layer = (int)H; layer >= 0; --layer) {
        const uint32_t K = layer == (int)H ? kPaddedOutput : kWidth; // width of dZ_l
        const uint8_t* aTile = sAct + layer * kATileBytes;
        // dZ_l: row-major tile for the data gradient, transposed tile for the weight gradient; A_l transposed
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) {
            if (c >= K / 8)
                break;
            uint4 v;
            v.x = (uint32_t)__half_as_ushort(d[c * 8 + 0]) | ((uint32_t)__half_as_ushort(d[c * 8 + 1]) << 16);
            v.y = (uint32_t)__half_as_ushort(d[c * 8 + 2]) | ((uint32_t)__half_as_ushort(d[c * 8 + 3]) << 16);
            v.z = (uint32_t)__half_as_ushort(d[c * 8 + 4]) | ((uint32_t)__half_as_ushort(d[c * 8 + 5]) << 16);
            v.w = (uint32_t)__half_as_ushort(d[c * 8 + 6]) | ((uint32_t)__half_as_ushort(d[c * 8 + 7]) << 16);
            *reinterpret_cast<uint4*>(sDz + c * (kTileRows * 16) + tid * 16) = v;
        }
        {
            __half* dzT = reinterpret_cast<__half*>(sDzT + (tid / 8) * (64 * 16) + (tid % 8) * 2);
#pragma unroll
            for (uint32_t j = 0; j < 64; ++j)
                if (j < K)
                    dzT[j * 8] = d[j]; // element (row j, k = tid) of a [64 x 128] K-major tile
            __half* aT = reinterpret_cast<__half*>(sActT + (tid / 8) * (64 * 16) + (tid % 8) * 2);
#pragma unroll
            for (uint32_t c = 0; c < 8; ++c) {
                const uint4 v = *reinterpret_cast<const uint4*>(aTile + c * (kTileRows * 16) + tid * 16);
                const uint32_t w4[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
                for (uint32_t e = 0; e < 4; ++e) {
                    aT[(c * 8 + 2 * e) * 8] = __ushort_as_half((unsigned short)(w4[e] & 0xFFFFu));
                    aT[(c * 8 + 2 * e + 1) * 8] = __ushort_as_half((unsigned short)(w4[e] >> 16));
                }
            }
        }
        fenceProxyAsync();
        tcFenceBefore();
        __syncthreads();
        if (tid == 0) {
            tcFenceAfter();
            // data gradient dA_l = dZ_l x W_l  (K steps of 16 over dZ's width)
            const uint32_t dzAddr = smemU32(sDz);
            const uint32_t wtLayer = smemU32(sWt) + layer * kWidth * kWidth * 2;
            for (uint32_t k = 0; k < K / 16; ++k)
                umma(tmemBase + tmemDa, makeSmemDesc(dzAddr + 2 * k * (kTileRows * 16), kTileRows * 16, 128),
                     makeSmemDesc(wtLayer + 2 * k * (kWidth * 16), kWidth * 16, 128), idesc64, k > 0 ? 1u : 0u);
            // weight gradient dW_l = dZ_l^T x A_l  (K = 128 samples)
            const uint32_t dzTAddr = smemU32(sDzT), aTAddr = smemU32(sActT);
#pragma unroll
            for (uint32_t k = 0; k < kTileRows / 16; ++k)
                umma(tmemBase + tmemDw, makeSmemDesc(dzTAddr + 2 * k * (64 * 16), 64 * 16, 128),
                     makeSmemDesc(aTAddr + 2 * k * (64 * 16), 64 * 16, 128), idesc64, k > 0 ? 1u : 0u);
            ummaCommit(&bar);
        }
        mbarWait(&bar, phase);
        phase ^= 1;
        tcFenceAfter();

        // weight gradient rows 0..K-1 -> fixed-point global accumulation (thread j owns output neuron j); tcgen05.ld is
        // warp-collective, so whole warps take part and only the lanes that own a valid row accumulate
        if (warp < (K + 31) / 32) {
            const uint32_t base = (uint32_t)layer * kWidth * kWidth + tid * kWidth;
#pragma unroll
            for (uint32_t half_ = 0; half_ < 2; ++half_) {
                uint32_t r[32];
                tmemLoad32(tmemRow + tmemDw + half_ * 32, r);
                tmemWaitLd();
                if (tid < K) {
#pragma unroll
                    for (uint32_t i = 0; i < 32; ++i) {
                        const float g = __uint_as_float(r[i]);
                        if (g != 0.0f)
                            atomicAddFixed(grads + base + half_ * 32 + i, g);
                    }
                }
            }
        }
        // data gradient row -> dZ_{l-1} (ReLU mask of A_l = relu(Z_{l-1})), or the encoder gradient for layer 0
        {
            __half dNext[64];
#pragma unroll
            for (uint32_t half_ = 0; half_ < 2; ++half_) {
                uint32_t r[32];
                tmemLoad32(tmemRow + tmemDa + half_ * 32, r);
                tmemWaitLd();
#pragma unroll
                for (uint32_t c = 0; c < 4; ++c) {
                    const uint4 av = *reinterpret_cast<const uint4*>(aTile + (half_ * 4 + c) * (kTileRows * 16) + tid * 16);
                    const uint32_t w4[4] = { av.x, av.y, av.z, av.w };
#pragma unroll
                    for (uint32_t e = 0; e < 8; ++e) {
                        const __half act = __ushort_as_half((unsigned short)((w4[e >> 1] >> (16 * (e & 1))) & 0xFFFFu));
                        const float g = __uint_as_float(r[c * 8 + e]);
                        dNext[half_ * 32 + c * 8 + e] = (layer > 0 && !(__half2float(act) > 0.0f)) ? __float2half(0.0f) : __float2half(g);
                    }
                }
            }
#pragma unroll
            for (uint32_t i = 0; i < 64; ++i)
                d[i] = dNext[i];
        }
        tcFenceBefore();
        __syncthreads(); // everyone is done with the tiles and the accumulators of this layer
        tcFenceAfter();
    }

    // ---- hash-grid backward (kernel_grid_backward, grid.h:306-429): scatter the first 32 input gradients (parked in
    // this thread's row of the dZ tile so that the level loop can index them)
    __half* gradRow = reinterpret_cast<__half*>(sDz + (size_t)tid * 64);
#pragma unroll
    for (uint32_t i = 0; i < 32; ++i)
        gradRow[i] = d[i];
    if (valid) {
        unsigned long long* gGrid = grads + numMatrixWeights;
        const float* in = input + (size_t)q * kInputDims;
        for (uint32_t l = 0; l < kLevels; ++l) {
            const NrcLevel lv = levels.l[l];
            const float g0 = __half2float(gradRow[l * 2 + 0]), g1 = __half2float(gradRow[l * 2 + 1]);
            if (g0 == 0.0f && g1 == 0.0f)
                continue;
            float pos[3];
            uint32_t posGrid[3];
            for (uint32_t dd = 0; dd < 3; ++dd) {
                pos[dd] = in[dd] * lv.scale + 0.5f;
                const int tmp = (int)floorf(pos[dd]);
                posGrid[dd] = (uint32_t)tmp;
                pos[dd] -= (float)tmp;
            }
            const NrcCellIndexer indexer(lv, posGrid);
#pragma unroll
            for (uint32_t idx = 0; idx < 8; ++idx) {
                float weight = 1;
#pragma unroll
                for (uint32_t dd = 0; dd < 3; ++dd)
                    weight *= (idx & (1u << dd)) == 0 ? 1 - pos[dd] : pos[dd];
                const uint32_t gi = lv.offset * 2 + indexer.corner(idx);
                atomicAddFixed(gGrid + gi, weight * g0);
                atomicAddFixed(gGrid + gi + 1, weight * g1);
            }
        }
    }
    for (int off = 16; off > 0; off >>= 1)
        localLoss += __shfl_xor_sync(0xFFFFFFFFu, localLoss, off);
    if ((tid & 31) == 0)
        sLoss[warp] = localLoss;
    tcFenceBefore();
    __syncthreads();
    if (tid == 0)
        atomicAdd(lossOut, sLoss[0] + sLoss[1] + sLoss[2] + sLoss[3]);
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmemBase), "r"(256u) : "memory");
}

// adam_step (adam.h:49-115) + ema_step_half_precision (ema.h:61-77); clears the gradient for the next step
__global__ void k_nrcAdamEma(uint32_t numParams, uint32_t numMatrixWeights, float learningRate, float emaDebiasOld,
                             float emaDebiasNew, unsigned long long* __restrict__ grads, float* __restrict__ master,
                             __half* __restrict__ params, __half* __restrict__ paramsEma, float* __restrict__ m1,
                             float* __restrict__ m2, uint32_t* __restrict__ steps) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= numParams)
        return;
    const float beta1 = 0.9f, beta2 = 0.99f, epsilon = 1e-15f, l2Reg = 1e-6f, emaDecay = 0.99f;
    float gradient = __half2float(__float2half(fixedToFloat(grads[i]))) / kLossScale;
    grads[i] = 0ull;
    const bool matrix = i < numMatrixWeights;
    if (matrix || gradient != 0) {
        const float weightFp = master[i];
        if (matrix)
            gradient += l2Reg * weightFp;
        const float gradientSq = gradient * gradient;
        const float firstMoment = m1[i] = beta1 * m1[i] + (1 - beta1) * gradient;
        const float secondMoment = m2[i] = beta2 * m2[i] + (1 - beta2) * gradientSq;
        float lr = learningRate;
        const uint32_t currentStep = ++steps[i];
        lr *= sqrtf(1 - powf(beta2, (float)currentStep)) / (1 - powf(beta1, (float)currentStep));
        const float effectiveLr = fminf(fmaxf(lr / (sqrtf(secondMoment) + epsilon), 0.0f), 3.402823466e+38f);
        const float newWeight = weightFp - effectiveLr * firstMoment;
        master[i] = newWeight;
        params[i] = __float2half(newWeight);
    }
    const float filtered = (__half2float(paramsEma[i]) * emaDecay * emaDebiasOld + __half2float(params[i]) * (1 - emaDecay)) * emaDebiasNew;
    paramsEma[i] = __float2half(filtered);
}

// gfx_nrc_keep_gradients: the gradients k_nrcAdamEma is about to consume, as the half values tiny-cuda-nn would hold
// (loss-scaled by 128), widened to float
__global__ void k_nrcKeepGradients(uint32_t n, const unsigned long long* __restrict__ grads, float* __restrict__ dst) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        dst[i] = __half2float(__float2half(fixedToFloat(grads[i])));
}

__global__ void k_nrcFloatToHalf(uint32_t n, const float* __restrict__ src, __half* __restrict__ dst) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        dst[i] = __float2half(src[i]);
}

__global__ void k_nrcHalfToFloat(uint32_t n, const __half* __restrict__ src, float* __restrict__ dst) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        dst[i] = __half2float(src[i]);
}

static void setupLevels(gfx_nrc* n) { // grid.h:885-922
    uint32_t offset = 0;
    for (uint32_t l = 0; l < kLevels; ++l) {
        const float scale = exp2f(l * log2f(2.0f)) * kBaseResolution - 1.0f;
        const uint32_t resolution = (uint32_t)ceilf(scale) + 1;
        const double dense = pow((double)resolution, 3.0);
        uint32_t paramsInLevel = dense > (double)(0xFFFFFFFFu / 2) ? 0xFFFFFFFFu / 2 : resolution * resolution * resolution;
        paramsInLevel = (paramsInLevel + 7u) / 8u * 8u;
        paramsInLevel = paramsInLevel < (1u << kLog2HashmapSize) ? paramsInLevel : (1u << kLog2HashmapSize);
        n->levels.l[l] = NrcLevel{ offset, paramsInLevel, scale, resolution };
        offset += paramsInLevel;
    }
    n->numMatrixWeights = kWidth * kWidth * n->numHiddenLayers + kPaddedOutput * kWidth;
    n->numParams = n->numMatrixWeights + offset * 2;
}

// tiny-cuda-nn's pcg32 (dependencies/pcg32/pcg32.h:46-116): 64-bit LCG, XSH-RR output
struct Pcg32 {
    uint64_t state, inc;
    explicit Pcg32(uint64_t initstate, uint64_t initseq = 1u) {
        state = 0u;
        inc = (initseq << 1u) | 1u;
        nextUint();
        state += initstate;
        nextUint();
    }
    uint32_t nextUint() {
        const uint64_t oldstate = state;
        state = oldstate * 0x5851f42d4c957f2dULL + inc;
        const uint32_t xorshifted = (uint32_t)(((oldstate >> 18u) ^ oldstate) >> 27u);
        const uint32_t rot = (uint32_t)(oldstate >> 59u);
        return (xorshifted >> rot) | (xorshifted << ((~rot + 1u) & 31));
    }
    float nextFloat() {
        union { uint32_t u; float f; } x;
        x.u = (nextUint() >> 9) | 0x3f800000u;
        return x.f - 1.0f;
    }
};

// The parameters a freshly constructed tcnn::Trainer holds (trainer.h:54-60, 72-109): rng = pcg32{seed_seq{seed}[0]};
// NetworkWithInputEncoding::initialize_params (network_with_input_encoding.h:133-156) initialises the network first -
// FullyFusedMLP: every weight matrix Xavier-uniform on the host, next_float() * 2 * scale - scale with
// scale = sqrt(6 / (fan_in + fan_out)) (fully_fused_mlp.cu:922-949, gpu_matrix.h:292-307) - then the encoding: the hash grid
// U(-1e-4, 1e-4) by generate_random_uniform (grid.h:1267-1272, random.h:65-100), a kernel in which thread i jumps the stream
// ahead by 4 i and writes elements i, i + T, i + 2T, i + 3T (T = total threads) with val * (upper - lower) + lower, one FMA
// under nvcc's default contraction.  One-blob and identity have no parameters.
static void tcnnInitialParams(uint32_t seed, uint32_t numHiddenLayers, uint32_t numMatrixWeights, uint32_t numParams,
                              std::vector<float>* master) {
    std::seed_seq seq{ seed };
    std::vector<uint32_t> seeds(2);
    seq.generate(seeds.begin(), seeds.end());
    Pcg32 rng(seeds.front());
    master->assign(numParams, 0.0f);
    size_t pos = 0;
    for (uint32_t m = 0; m <= numHiddenLayers; ++m) {
        const uint32_t rows = m == numHiddenLayers ? kPaddedOutput : kWidth, cols = kWidth; // fan_out = rows, fan_in = cols
        const float scale = 1.0f * std::sqrt(6.0f / (float)(cols + rows));
        for (uint32_t i = 0; i < rows * cols; ++i)
            (*master)[pos++] = rng.nextFloat() * 2.0f * scale - scale;
    }
    const size_t n = numParams - numMatrixWeights;
    const size_t threadsNeeded = (n + 3) / 4;
    const size_t totalThreads = (threadsNeeded + 127) / 128 * 128; // n_blocks_linear(n_threads) * n_threads_linear
    std::vector<float> stream(totalThreads * 4);
    for (float &f : stream)
        f = rng.nextFloat();
    const float upper = 1e-4f, lower = -1e-4f;
    for (size_t i = 0; i < totalThreads; ++i)
        for (size_t j = 0; j < 4; ++j) {
            const size_t idx = i + totalThreads * j;
            if (idx >= n)
                break;
            (*master)[numMatrixWeights + idx] = fmaf(stream[i * 4 + j], upper - lower, lower);
        }
}

} // namespace gfx

using namespace gfx;

#define NRC_CUDA(nrc, call) GFX_CUDA((nrc)->ctx, call)

extern "C" {

int gfx_nrc_train(gfx_nrc* n, void* stream, const float* inputData, const float* targetData, uint32_t numData, float* lossOnHost);
int gfx_nrc_reset(gfx_nrc* n, uint32_t seed);
void gfx_nrc_destroy(gfx_nrc* n);

int gfx_nrc_create(gfx_ctx* ctx, uint32_t numHiddenLayers, float learningRate, gfx_nrc** out) {
    if (!ctx || !out)
        return GFX_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (numHiddenLayers < 1 || numHiddenLayers > 8) {
        ctx->setError("gfx_nrc_create: numHiddenLayers must be in 1..8");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    GFX_CUDA(ctx, cudaSetDevice(ctx->device));
    gfx_nrc* n = new gfx_nrc();
    n->ctx = ctx;
    n->numHiddenLayers = numHiddenLayers;
    n->learningRate = learningRate;
    setupLevels(n);
    const size_t P = n->numParams;
    GFX_CUDA(ctx, cudaMalloc(&n->params, P * 2));
    GFX_CUDA(ctx, cudaMalloc(&n->paramsEma, P * 2));
    GFX_CUDA(ctx, cudaMalloc(&n->master, P * 4));
    GFX_CUDA(ctx, cudaMalloc(&n->m1, P * 4));
    GFX_CUDA(ctx, cudaMalloc(&n->m2, P * 4));
    GFX_CUDA(ctx, cudaMalloc(&n->steps, P * 4));
    GFX_CUDA(ctx, cudaMalloc(&n->grads, P * 8));
    GFX_CUDA(ctx, cudaMalloc(&n->loss, 16));
    GFX_CUDA(ctx, cudaMalloc(&n->ummaWeights, (size_t)n->numMatrixWeights * 2));
    GFX_CUDA(ctx, cudaMalloc(&n->trainBlobFwd, (size_t)n->numMatrixWeights * 2));
    GFX_CUDA(ctx, cudaMalloc(&n->trainBlobT, (size_t)n->numMatrixWeights * 2));
    GFX_CUDA(ctx, cudaMemset(n->params, 0, P * 2));
    GFX_CUDA(ctx, cudaMemset(n->paramsEma, 0, P * 2));
    GFX_CUDA(ctx, cudaMemset(n->master, 0, P * 4));
    GFX_CUDA(ctx, cudaMemset(n->m1, 0, P * 4));
    GFX_CUDA(ctx, cudaMemset(n->m2, 0, P * 4));
    GFX_CUDA(ctx, cudaMemset(n->steps, 0, P * 4));
    GFX_CUDA(ctx, cudaMemset(n->grads, 0, P * 8));
    const int rc = gfx_nrc_reset(n, 1337u); // tcnn::Trainer's default seed: a fresh cache equals the reference's fresh cache
    if (rc != GFX_OK) {
        gfx_nrc_destroy(n);
        return rc;
    }
    *out = n;
    return GFX_OK;
}

int gfx_nrc_reset(gfx_nrc* n, uint32_t seed) {
    if (!n)
        return GFX_ERR_INVALID_ARGUMENT;
    const size_t P = n->numParams;
    std::vector<float> master;
    tcnnInitialParams(seed, n->numHiddenLayers, n->numMatrixWeights, n->numParams, &master);
    NRC_CUDA(n, cudaMemcpy(n->master, master.data(), P * 4, cudaMemcpyHostToDevice));
    k_nrcFloatToHalf<<<(n->numParams + 255) / 256, 256>>>(n->numParams, n->master, n->params); // trainer.h:104-107
    n->ctx->launches++;
    NRC_CUDA(n, cudaMemset(n->paramsEma, 0, P * 2)); // EmaOptimizer::allocate zeroes the inference weights (ema.h:88-100)
    NRC_CUDA(n, cudaMemset(n->m1, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->m2, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->steps, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->grads, 0, P * 8));
    n->globalStep = 0;
    n->ummaDirty = true;
    NRC_CUDA(n, cudaDeviceSynchronize());
    return GFX_OK;
}

int gfx_nrc_keep_gradients(gfx_nrc* n, int on) {
    if (!n)
        return GFX_ERR_INVALID_ARGUMENT;
    if (on && !n->gradsFloat)
        NRC_CUDA(n, cudaMalloc(&n->gradsFloat, (size_t)n->numParams * 4));
    n->keepGradients = on != 0;
    return GFX_OK;
}

int gfx_nrc_read(gfx_nrc* n, int which, void* hostOut, size_t bytes) {
    if (!n || !hostOut)
        return GFX_ERR_INVALID_ARGUMENT;
    const size_t P = n->numParams;
    const void* src = nullptr;
    size_t need = P * 2;
    switch (which) {
    case GFX_NRC_READ_MASTER: src = n->master; need = P * 4; break;
    case GFX_NRC_READ_TRAINING: src = n->params; break;
    case GFX_NRC_READ_INFERENCE: src = n->paramsEma; break;
    case GFX_NRC_READ_GRADIENTS: src = n->gradsFloat; need = P * 4; break;
    default: return GFX_ERR_INVALID_ARGUMENT;
    }
    if (!src)
        return GFX_ERR_NOT_READY;
    if (bytes != need)
        return GFX_ERR_INVALID_ARGUMENT;
    NRC_CUDA(n, cudaDeviceSynchronize());
    NRC_CUDA(n, cudaMemcpy(hostOut, src, need, cudaMemcpyDeviceToHost));
    return GFX_OK;
}

void gfx_nrc_destroy(gfx_nrc* n) {
    if (!n)
        return;
    cudaFree(n->params); cudaFree(n->paramsEma); cudaFree(n->master); cudaFree(n->m1); cudaFree(n->m2);
    cudaFree(n->steps); cudaFree(n->grads); cudaFree(n->loss); cudaFree(n->ummaWeights); cudaFree(n->trainBlobFwd); cudaFree(n->trainBlobT); cudaFree(n->gradsFloat); cudaFree(n->positions); cudaFree(n->features);
    delete n;
}

uint32_t gfx_nrc_num_params(gfx_nrc* n) { return n ? n->numParams : 0; }

int gfx_nrc_set_params(gfx_nrc* n, const void* hostHalfParams, size_t bytes) {
    if (!n || !hostHalfParams || bytes != (size_t)n->numParams * 2)
        return GFX_ERR_INVALID_ARGUMENT;
    const size_t P = n->numParams;
    NRC_CUDA(n, cudaMemcpy(n->params, hostHalfParams, bytes, cudaMemcpyHostToDevice));
    NRC_CUDA(n, cudaMemcpy(n->paramsEma, n->params, bytes, cudaMemcpyDeviceToDevice));
    k_nrcHalfToFloat<<<(n->numParams + 255) / 256, 256>>>(n->numParams, n->params, n->master);
    n->ctx->launches++;
    NRC_CUDA(n, cudaMemset(n->m1, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->m2, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->steps, 0, P * 4));
    NRC_CUDA(n, cudaMemset(n->grads, 0, P * 8));
    n->globalStep = 0;
    n->ummaDirty = true;
    NRC_CUDA(n, cudaDeviceSynchronize());
    return GFX_OK;
}

int gfx_nrc_get_params(gfx_nrc* n, void* hostHalfParams, size_t bytes) {
    if (!n || !hostHalfParams || bytes != (size_t)n->numParams * 2)
        return GFX_ERR_INVALID_ARGUMENT;
    NRC_CUDA(n, cudaMemcpy(hostHalfParams, n->paramsEma, bytes, cudaMemcpyDeviceToHost));
    return GFX_OK;
}

static int nrcEnsureScratch(gfx_nrc* n, uint32_t numQueries) {
    if (numQueries <= n->scratchQueries)
        return GFX_OK;
    cudaFree(n->positions);
    cudaFree(n->features);
    n->positions = nullptr;
    n->features = nullptr;
    n->scratchQueries = 0;
    NRC_CUDA(n, cudaMalloc(&n->positions, (size_t)numQueries * 16));
    NRC_CUDA(n, cudaMalloc(&n->features, (size_t)numQueries * kLevels * 4));
    n->scratchQueries = numQueries;
    return GFX_OK;
}

// pack + grid encode (the two kernels in front of k_nrcInferMlp); numData (or *numDataPtr) is a multiple of 128
static int nrcGridEncodeLaunch(gfx_nrc* n, cudaStream_t s, const float* inputData, uint32_t numData, const uint32_t* numDataPtr,
                               bool emaTable) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    { GFX_TIMED(n->ctx, s, "nrc_pack_positions");
    k_nrcPackPositions<<<sms * 4, 256, 0, s>>>(inputData, n->positions, numData, numDataPtr); }
    n->ctx->launches++;
    const uint32_t replicas = (uint32_t)sms / kLevels > 0 ? (uint32_t)sms / kLevels : 1u;
    const size_t smem = (size_t)(1u << kLog2HashmapSize) * 4;
    NRC_CUDA(n, cudaFuncSetAttribute(k_nrcGridEncode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    { GFX_TIMED(n->ctx, s, "nrc_grid_encode");
    k_nrcGridEncode<<<kLevels * replicas, kEncodeThreads, smem, s>>>(n->levels, (emaTable ? n->paramsEma : n->params) + n->numMatrixWeights,
                                                                     n->positions, n->features, replicas, numData, numDataPtr); }
    n->ctx->launches++;
    NRC_CUDA(n, cudaGetLastError());
    return GFX_OK;
}

static int nrcInferLaunch(gfx_nrc* n, cudaStream_t s, const float* inputData, float* predictionData, uint32_t numData,
                          const uint32_t* numDataPtr) {
    if (n->ummaDirty) {
        k_nrcPrepWeights<<<32, 256, 0, s>>>(n->paramsEma, n->numHiddenLayers, reinterpret_cast<__half*>(n->ummaWeights));
        n->ctx->launches++;
        n->ummaDirty = false;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const uint32_t numTiles = numData / kTileRows; // upper bound when numDataPtr is given
    // buffers the TMA bulk copies cannot take (not 16-byte aligned) go through the one-kernel form: encode by L2 gathers
    // inside the MLP kernel
    const bool aligned = (reinterpret_cast<uintptr_t>(inputData) & 15u) == 0 && (reinterpret_cast<uintptr_t>(predictionData) & 15u) == 0;
    if (!aligned) {
        const size_t smem = kATileBytes + (size_t)n->numMatrixWeights * 2;
        NRC_CUDA(n, cudaFuncSetAttribute(k_nrcInfer, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const uint32_t grid = numTiles < (uint32_t)sms * 6 ? numTiles : (uint32_t)sms * 6;
        GFX_TIMED(n->ctx, s, "nrc_infer");
        k_nrcInfer<<<grid, 128, smem, s>>>(n->levels, n->paramsEma + n->numMatrixWeights, n->ummaWeights, n->numHiddenLayers,
                                           inputData, predictionData, numData, numDataPtr);
        n->ctx->launches++;
        NRC_CUDA(n, cudaGetLastError());
        return GFX_OK;
    }
    int rc = nrcEnsureScratch(n, numData);
    if (rc != GFX_OK)
        return rc;
    rc = nrcGridEncodeLaunch(n, s, inputData, numData, numDataPtr, true);
    if (rc != GFX_OK)
        return rc;
    const size_t smem = kATileBytes + 2 * sizeof(NrcTileStage) + 128 * kOutputDims * 4 + (size_t)n->numMatrixWeights * 2;
    NRC_CUDA(n, cudaFuncSetAttribute(k_nrcInferMlp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t ctasPerSm = (uint32_t)(220 * 1024 / (smem + 1024));
    const uint32_t maxGrid = (uint32_t)sms * (ctasPerSm ? ctasPerSm : 1u);
    const uint32_t grid = numTiles < maxGrid ? numTiles : maxGrid;
    GFX_TIMED(n->ctx, s, "nrc_infer");
    k_nrcInferMlp<<<grid, 128, smem, s>>>(n->ummaWeights, n->numHiddenLayers, inputData, n->features, predictionData, numData, numDataPtr);
    n->ctx->launches++;
    NRC_CUDA(n, cudaGetLastError());
    return GFX_OK;
}

// test hook (gfx_nrc_encode_debug): the encoded network input of numData queries, [numData][64] halves, through the split path
static int nrcEncodeDebug(gfx_nrc* n, cudaStream_t s, const float* inputData, uint32_t numData, void* outHalf) {
    int rc = nrcEnsureScratch(n, numData);
    if (rc != GFX_OK)
        return rc;
    rc = nrcGridEncodeLaunch(n, s, inputData, numData, nullptr, true);
    if (rc != GFX_OK)
        return rc;
    k_nrcAssembleEncoding<<<(numData + 127) / 128, 128, 0, s>>>(inputData, n->features, numData, reinterpret_cast<__half*>(outHalf));
    n->ctx->launches++;
    NRC_CUDA(n, cudaGetLastError());
    return GFX_OK;
}

int gfx_nrc_infer(gfx_nrc* n, void* stream, const float* inputData, float* predictionData, uint32_t numData) {
    if (!n || (!inputData && numData) || (!predictionData && numData))
        return GFX_ERR_INVALID_ARGUMENT;
    if (numData & 0x7F) { // network_interface.cu:143 Assert((numData & 0x7F) == 0)
        n->ctx->setError("gfx_nrc_infer: numData must be a multiple of 128");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    if (numData == 0)
        return GFX_OK;
    return nrcInferLaunch(n, (cudaStream_t)stream, inputData, predictionData, numData, nullptr);
}

int gfx_nrc_encode_debug(gfx_nrc* n, void* stream, const float* inputData, uint32_t numData, void* outHalf) {
    if (!n || !inputData || !outHalf || (numData & 0x7F))
        return GFX_ERR_INVALID_ARGUMENT;
    if (numData == 0)
        return GFX_OK;
    return nrcEncodeDebug(n, (cudaStream_t)stream, inputData, numData, outHalf);
}

int gfx_nrc_frame_infer(gfx_ctx* ctx, gfx_nrc* n, void* stream) {
    if (!ctx || !n || n->ctx != ctx)
        return GFX_ERR_INVALID_ARGUMENT;
    if (!ctx->frame.created)
        return GFX_ERR_NOT_READY;
    const int rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    const FrameState::Nrc &N = ctx->frame.nrc;
    // numInferenceQueries = pad128(W*H + #tiles) was left in the state block by gfx_nrc_preprocess
    return nrcInferLaunch(n, (cudaStream_t)stream, N.inferenceQuery, N.inferredRadiance, N.queryCapacity, N.state + 26);
}

int gfx_nrc_frame_infer_rows(gfx_ctx* ctx, gfx_nrc* n, void* stream, uint32_t rowLo, uint32_t rowHi) {
    if (!ctx || !n || n->ctx != ctx)
        return GFX_ERR_INVALID_ARGUMENT;
    if (!ctx->frame.created)
        return GFX_ERR_NOT_READY;
    int rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    const FrameState::Nrc &N = ctx->frame.nrc;
    const uint32_t W = ctx->frame.W, H = ctx->frame.H;
    if (rowLo >= rowHi || rowHi > H)
        return GFX_ERR_INVALID_ARGUMENT;
    const size_t numPixels = (size_t)W * H, first = (size_t)rowLo * W;
    if ((first & 127u) || (numPixels & 127u)) {
        ctx->setError("gfx_nrc_frame_infer_rows: rowLo * width and width * height must be multiples of the 128-query tile");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    // the strip's terminal queries (one per pixel; the tail of the last 128-query tile reads into the next rows, whose
    // predictions this rank does not use) ...
    const uint32_t numRowQueries = (uint32_t)((((size_t)(rowHi - rowLo) * W + 127) / 128) * 128);
    const uint32_t rowQueries = (uint32_t)(first + numRowQueries <= N.queryCapacity ? numRowQueries : N.queryCapacity - first);
    rc = nrcInferLaunch(n, (cudaStream_t)stream, N.inferenceQuery + 14 * first, N.inferredRadiance + 3 * first, rowQueries, nullptr);
    if (rc != GFX_OK)
        return rc;
    // ... and the training-suffix queries of all tiles (slots of the other ranks' tiles hold stale queries: their
    // predictions are never read here, propagation only walks the suffixes this rank traced)
    const uint32_t suffixCapacity = (uint32_t)(N.queryCapacity - numPixels);
    return nrcInferLaunch(n, (cudaStream_t)stream, N.inferenceQuery + 14 * numPixels, N.inferredRadiance + 3 * numPixels, suffixCapacity,
                          N.state + 27);
}

int gfx_nrc_frame_train(gfx_ctx* ctx, gfx_nrc* n, void* stream, float* lossOnHost) {
    if (!ctx || !n || n->ctx != ctx)
        return GFX_ERR_INVALID_ARGUMENT;
    if (!ctx->frame.created)
        return GFX_ERR_NOT_READY;
    int rc = ensureNrcFrame(ctx);
    if (rc != GFX_OK)
        return rc;
    const FrameState::Nrc &N = ctx->frame.nrc;
    // neural_radiance_caching_main.cpp:2350-2365: four steps over quarters of the shuffled 65 536 records
    const uint32_t batchSize = 65536 / 4;
    for (uint32_t step = 0; step < 4 && rc == GFX_OK; ++step)
        rc = gfx_nrc_train(n, stream, N.trainQuery[1] + (size_t)step * batchSize * 14, N.trainTarget[1] + (size_t)step * batchSize * 3,
                           batchSize, step == 3 ? lossOnHost : nullptr);
    return rc;
}

int gfx_nrc_train(gfx_nrc* n, void* stream, const float* inputData, const float* targetData, uint32_t numData, float* lossOnHost) {
    if (!n || !inputData || !targetData)
        return GFX_ERR_INVALID_ARGUMENT;
    if (numData & 0x7F) {
        n->ctx->setError("gfx_nrc_train: numData must be a multiple of 128");
        return GFX_ERR_INVALID_ARGUMENT;
    }
    if (numData == 0)
        return GFX_OK;
    cudaStream_t s = (cudaStream_t)stream;
    NRC_CUDA(n, cudaMemsetAsync(n->loss, 0, 4, s));
    // Fully-connected layers on tcgen05 (forward, data gradient and weight gradient); the CUDA-core kernel stays for deep
    // networks (more than 3 hidden layers) whose activation tiles do not fit in shared memory.
    if (n->numHiddenLayers <= 3) {
        const size_t smem = (size_t)n->numMatrixWeights * 4 + (size_t)(n->numHiddenLayers + 1) * kATileBytes + 3 * (size_t)kATileBytes;
        NRC_CUDA(n, cudaFuncSetAttribute(k_nrcTrainTc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        { GFX_TIMED(n->ctx, s, "nrc_train_prep_weights");
        k_nrcPrepTrainWeights<<<32, 256, 0, s>>>(n->params, n->numHiddenLayers, reinterpret_cast<__half*>(n->trainBlobFwd),
                                                 reinterpret_cast<__half*>(n->trainBlobT)); }
        n->ctx->launches++;
        { GFX_TIMED(n->ctx, s, "nrc_train_fwd_bwd");
        k_nrcTrainTc<<<numData / 128, 128, smem, s>>>(n->levels, n->params, n->numMatrixWeights, n->numHiddenLayers,
                                                      n->trainBlobFwd, n->trainBlobT, inputData, targetData, numData, n->grads,
                                                      n->loss); }
    }
    else {
        const size_t smem = ((size_t)n->numMatrixWeights + (size_t)(n->numHiddenLayers + 2) * 128 * kRowStride) * 2;
        NRC_CUDA(n, cudaFuncSetAttribute(k_nrcTrain, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        { GFX_TIMED(n->ctx, s, "nrc_train_fwd_bwd");
        k_nrcTrain<<<numData / 128, 128, smem, s>>>(n->levels, n->params, n->numMatrixWeights, n->numHiddenLayers, inputData,
                                                    targetData, numData, n->grads, n->loss); }
    }
    n->ctx->launches++;
    if (n->keepGradients) {
        k_nrcKeepGradients<<<(n->numParams + 255) / 256, 256, 0, s>>>(n->numParams, n->grads, n->gradsFloat);
        n->ctx->launches++;
    }
    ++n->globalStep;
    const float emaDecay = 0.99f;
    const float emaDebiasOld = 1 - (float)pow((double)emaDecay, (double)(n->globalStep - 1));
    const float emaDebiasNew = 1.0f / (1 - (float)pow((double)emaDecay, (double)n->globalStep));
    { GFX_TIMED(n->ctx, s, "nrc_adam_ema");
    k_nrcAdamEma<<<(n->numParams + 255) / 256, 256, 0, s>>>(n->numParams, n->numMatrixWeights, n->learningRate, emaDebiasOld,
                                                            emaDebiasNew, n->grads, n->master, n->params, n->paramsEma,
                                                            n->m1, n->m2, n->steps); }
    n->ctx->launches++;
    n->ummaDirty = true;
    NRC_CUDA(n, cudaGetLastError());
    if (lossOnHost) { // network_interface.cu:155-156: optional blocking read-back
        NRC_CUDA(n, cudaMemcpyAsync(lossOnHost, n->loss, 4, cudaMemcpyDeviceToHost, s));
        NRC_CUDA(n, cudaStreamSynchronize(s));
    }
    return GFX_OK;
}

} // extern "C"
