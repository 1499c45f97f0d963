// plen_actor_tc.cu -- Actor.forward (plen_ros/src/plen_ros_helpers/td3.py:45-57) for N observations on the 5th-generation
// tensor cores: tcgen05.mma (kind::f16, FP16 operands, FP32 accumulators in TMEM), part of libplen_b200.so.  sm_100a only.
//
// This is the one place on the path where the work is a dense contraction with a large M (N observations x 26-256-256-18,
// N = 16k .. 1M robots), so it goes to the tensor cores; the fp32 CUDA-core kernel (plen_actor_forward) stays the
// parity path (1e-5 against the reference's fp32 checkpoints), this one is the throughput path for rollouts
// (FP16 operands, 11-bit significands: on the shipped checkpoint mean action error 4.5e-4, max 0.12 against fp32, bound
// stated and tested in tests/test_td3_gpu.py; BF16 operands measured mean 4.2e-3 / max 0.59 there and were dropped).
// Against a float64 model that rounds where this kernel rounds, the residual is the accumulation order alone: median 6e-14,
// 99.9th percentile 4.8e-4 on the shipped checkpoint (tests/test_td3_kernels_gpu.py).
//
// One persistent CTA per SM, 128 threads, M = 128 observations per tile:
//   * all three weight matrices live in shared memory as FP16 for the whole kernel (W2 128 KB, W1 / W3 16 KB each, K
//     padded 26 -> 32, N padded 18 -> 32), in the canonical K-major no-swizzle UMMA layout (8 x 16 B core matrices);
//   * the activations of the tile (128 x 256 FP16, 64 KB) are the A operand, rewritten in place by every epilogue;
//   * per layer ONE thread issues K / 16 tcgen05.mma (128 x N x 16) into TMEM and commits to an mbarrier; the four warps
//     then read their 32 TMEM lanes with tcgen05.ld (32x32b.x32), add the bias, apply ReLU, convert to FP16 and store
//     the next A operand (layer 3: tanh, exploration noise, clip, store the actions).
// No TMA: the operands are produced by the threads themselves (fp32 -> fp16 conversion), so they are written with
// ordinary stores followed by fence.proxy.async.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/plen_b200.h"
#include "plen_tc_common.cuh"

extern "C" int plen_td3_set_error(int code, const char *msg, const char *detail);      // plen_td3.cu

namespace {

using namespace plen_tc;

constexpr int TM = 128, HID = 256, K1 = 32, N3 = 32;
constexpr uint32_t OFF_W2 = 0, OFF_W1 = OFF_W2 + HID * HID * 2, OFF_W3 = OFF_W1 + HID * K1 * 2, OFF_A = OFF_W3 + N3 * HID * 2,
                   OFF_BIAS = OFF_A + TM * HID * 2, OFF_BAR = OFF_BIAS + (2 * HID + N3) * 4, OFF_TPTR = OFF_BAR + 8,
                   TC_SMEM = OFF_TPTR + 8;
static_assert(TC_SMEM <= 232448, "shared memory budget of one CTA");

// byte offset of element (row, k) of an R-row K-major operand in the canonical no-swizzle layout:
// core matrix = 8 rows x 16 bytes (8 fp16 of K), contiguous; core matrices of consecutive row groups are adjacent
// (SBO = 128 B), core matrices of consecutive K groups are R * 16 B apart (LBO)
__device__ __forceinline__ uint32_t canon(int row, int k, int R) {
    return (uint32_t)((k >> 3) * (R * 16) + (row >> 3) * 128 + (row & 7) * 16 + (k & 7) * 2);
}

// two fp32 -> packed FP16 (saturating: a hidden activation beyond +-65504 would otherwise become inf)
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    __half2 v = __floats2half2_rn(fminf(fmaxf(lo, -65504.0f), 65504.0f), fminf(fmaxf(hi, -65504.0f), 65504.0f));
    return *reinterpret_cast<uint32_t *>(&v);
}
__device__ __forceinline__ uint32_t mixh(uint64_t x) {     // splitmix64 finaliser (same generator as plen_actor_forward)
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return (uint32_t)((x ^ (x >> 31)) >> 32);
}

// 8 consecutive K entries of row `row` (fp32 in global memory, zero beyond kmax) -> one 16-byte chunk of the operand
__device__ __forceinline__ void stage_chunk(unsigned char *dst, const float *src_row, int k0, int kmax, bool row_ok) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = (row_ok && k0 + i < kmax) ? src_row[k0 + i] : 0.0f;
    uint4 q = {pack_f16(v[0], v[1]), pack_f16(v[2], v[3]), pack_f16(v[4], v[5]), pack_f16(v[6], v[7])};
    *reinterpret_cast<uint4 *>(dst) = q;
}

__global__ void __launch_bounds__(128, 1)
k_actor_forward_tc(const float *__restrict__ w1, const float *__restrict__ b1, const float *__restrict__ w2,
                   const float *__restrict__ b2, const float *__restrict__ w3, const float *__restrict__ b3,
                   const float *__restrict__ obs, int n, float max_action, float noise_std, uint64_t seed,
                   float *__restrict__ act) {
    extern __shared__ __align__(128) unsigned char sm[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(sm);
    const uint32_t bar = sbase + OFF_BAR;
    float *bias = reinterpret_cast<float *>(sm + OFF_BIAS);
    volatile uint32_t *tptr = reinterpret_cast<volatile uint32_t *>(sm + OFF_TPTR);

    // ---- one-time set-up: weights -> FP16 canonical operands, biases, mbarrier, TMEM (512 columns: two 256-wide accumulators)
    for (int e = tid; e < HID * (HID / 8); e += 128) {          // W2 [256][256]
        const int nrow = e & (HID - 1), kg = e >> 8;
        stage_chunk(sm + OFF_W2 + canon(nrow, kg * 8, HID), w2 + (size_t)nrow * HID, kg * 8, HID, true);
    }
    for (int e = tid; e < HID * (K1 / 8); e += 128) {           // W1 [256][26 -> 32]
        const int nrow = e & (HID - 1), kg = e >> 8;
        stage_chunk(sm + OFF_W1 + canon(nrow, kg * 8, HID), w1 + (size_t)nrow * PLEN_OBS, kg * 8, PLEN_OBS, true);
    }
    for (int e = tid; e < N3 * (HID / 8); e += 128) {           // W3 [18 -> 32][256]
        const int nrow = e & (N3 - 1), kg = e >> 5;
        stage_chunk(sm + OFF_W3 + canon(nrow, kg * 8, N3), w3 + (size_t)nrow * HID, kg * 8, HID, nrow < PLEN_NJ);
    }
    for (int e = tid; e < HID; e += 128) { bias[e] = b1[e]; bias[HID + e] = b2[e]; }
    if (tid < N3) bias[2 * HID + tid] = (tid < PLEN_NJ) ? b3[tid] : 0.0f;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(sbase + OFF_TPTR), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tptr;
    const uint32_t lane_base = tmem + ((uint32_t)(32 * warp) << 16);       // this warp's 32 TMEM lanes (rows 32 warp ..)
    const uint32_t idesc256 = instr_desc(TM, HID), idesc32 = instr_desc(TM, N3);
    uint32_t parity = 0;
    bool poisoned = false;                                                  // an mbarrier wait was abandoned: write NaN actions
    const int row = tid;                                                    // row of the tile owned in every epilogue

    const int n_tiles = (n + TM - 1) / TM;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int grow = tile * TM + row;
        // ---- A <- observations (K padded to 32)
#pragma unroll
        for (int kg = 0; kg < K1 / 8; kg++)
            stage_chunk(sm + OFF_A + canon(row, kg * 8, TM), obs + (size_t)grow * PLEN_OBS, kg * 8, PLEN_OBS, grow < n);
        fence_async_smem();
        fence_before();
        __syncthreads();
        // ---- layer 1: D1[128 x 256] (TMEM columns 0..255) = A[128 x 32] W1^T
        if (tid == 0) {
            fence_after();
#pragma unroll
            for (int ks = 0; ks < K1 / 16; ks++)
                mma_f16(tmem, smem_desc(sbase + OFF_A + ks * 2 * (TM * 16), TM * 16, 128),
                         smem_desc(sbase + OFF_W1 + ks * 2 * (HID * 16), HID * 16, 128), idesc256, ks > 0);
            mma_commit(bar);
        }
        poisoned |= !mbar_wait(bar, parity); parity ^= 1;
        fence_after();
        // ---- epilogue 1: A <- fp16(relu(D1 + b1))
#pragma unroll 1
        for (int c = 0; c < HID / 32; c++) {
            uint32_t r[32];
            tmem_ld32(lane_base + 32 * c, r);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; i++) v[i] = fmaxf(__uint_as_float(r[8 * q + i]) + bias[32 * c + 8 * q + i], 0.0f);
                uint4 o = {pack_f16(v[0], v[1]), pack_f16(v[2], v[3]), pack_f16(v[4], v[5]), pack_f16(v[6], v[7])};
                *reinterpret_cast<uint4 *>(sm + OFF_A + canon(row, 32 * c + 8 * q, TM)) = o;
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        // ---- layer 2: D2 (TMEM columns 256..511) = A[128 x 256] W2^T
        if (tid == 0) {
            fence_after();
#pragma unroll
            for (int ks = 0; ks < HID / 16; ks++)
                mma_f16(tmem + 256, smem_desc(sbase + OFF_A + ks * 2 * (TM * 16), TM * 16, 128),
                         smem_desc(sbase + OFF_W2 + ks * 2 * (HID * 16), HID * 16, 128), idesc256, ks > 0);
            mma_commit(bar);
        }
        poisoned |= !mbar_wait(bar, parity); parity ^= 1;
        fence_after();
#pragma unroll 1
        for (int c = 0; c < HID / 32; c++) {
            uint32_t r[32];
            tmem_ld32(lane_base + 256 + 32 * c, r);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; i++) v[i] = fmaxf(__uint_as_float(r[8 * q + i]) + bias[HID + 32 * c + 8 * q + i], 0.0f);
                uint4 o = {pack_f16(v[0], v[1]), pack_f16(v[2], v[3]), pack_f16(v[4], v[5]), pack_f16(v[6], v[7])};
                *reinterpret_cast<uint4 *>(sm + OFF_A + canon(row, 32 * c + 8 * q, TM)) = o;
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        // ---- layer 3: D3[128 x 32] (TMEM columns 0..31) = A[128 x 256] W3^T
        if (tid == 0) {
            fence_after();
#pragma unroll
            for (int ks = 0; ks < HID / 16; ks++)
                mma_f16(tmem, smem_desc(sbase + OFF_A + ks * 2 * (TM * 16), TM * 16, 128),
                         smem_desc(sbase + OFF_W3 + ks * 2 * (N3 * 16), N3 * 16, 128), idesc32, ks > 0);
            mma_commit(bar);
        }
        poisoned |= !mbar_wait(bar, parity); parity ^= 1;
        fence_after();
        {
            uint32_t r[32];
            tmem_ld32(lane_base, r);
            if (grow < n) {
#pragma unroll
                for (int j = 0; j < PLEN_NJ; j++) {
                    float v = max_action * tanhf(__uint_as_float(r[j]) + bias[2 * HID + j]);         // td3.py:56
                    if (noise_std > 0.0f) {       // plen_td3.py:101-104, same counter-based draw as plen_actor_forward
                        const uint64_t ctr = seed * 0x100000001B3ull + (uint64_t)grow * 32u + (uint64_t)j;
                        const float u1 = (mixh(ctr) + 1.0f) * 2.3283064e-10f, u2 = mixh(ctr ^ 0xA5A5A5A5DEADBEEFull) * 2.3283064e-10f;
                        v += noise_std * sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
                        v = fminf(fmaxf(v, -max_action), max_action);
                    }
                    act[(size_t)grow * PLEN_NJ + j] = poisoned ? __int_as_float(0x7fc00000) : v;
                }
            }
        }
        fence_before();
        __syncthreads();      // the next tile's MMAs overwrite TMEM columns 0.. and the A operand
        fence_after();
    }
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512u) : "memory");
}

}  // namespace

extern "C" int plen_actor_forward_tc(int device, const float *w1, const float *b1, const float *w2, const float *b2,
                                       const float *w3, const float *b3, const float *obs_dev, int n, float max_action,
                                       float noise_std, unsigned long long seed, float *action_dev, void *stream) {
    if (!w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !obs_dev || !action_dev || n <= 0)
        return plen_td3_set_error(PLEN_E_ARG, "plen_actor_forward_tc: bad arguments", "");
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return plen_td3_set_error(PLEN_E_CUDA, "plen_actor_forward_tc: ", cudaGetErrorString(e));
    static int sm_count[64] = {0};
    const int di = device < 64 ? device : 63;
    if (sm_count[di] == 0) {
        e = cudaFuncSetAttribute(k_actor_forward_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM);
        if (e != cudaSuccess) return plen_td3_set_error(PLEN_E_CUDA, "plen_actor_forward_tc: ", cudaGetErrorString(e));
        int c = 0;
        cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, device);
        sm_count[di] = c > 0 ? c : 148;
    }
    const int tiles = (n + TM - 1) / TM;
    const int grid = tiles < sm_count[di] ? tiles : sm_count[di];
    k_actor_forward_tc<<<grid, 128, TC_SMEM, (cudaStream_t)stream>>>(w1, b1, w2, b2, w3, b3, obs_dev, n, max_action, noise_std, seed,
                                                                   action_dev);
    e = cudaGetLastError();
    if (e != cudaSuccess) return plen_td3_set_error(PLEN_E_CUDA, "plen_actor_forward_tc: ", cudaGetErrorString(e));
    return PLEN_OK;
}

/* 1 if any tensor-core actor launch on the current device ever abandoned an mbarrier wait (diagnostic, synchronises) */
extern "C" int plen_actor_tc_timed_out(void) {
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, plen_tc::g_tc_timeout, sizeof v) != cudaSuccess) return -1;
    return v;
}
