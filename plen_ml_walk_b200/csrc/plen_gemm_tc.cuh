// plen_gemm_tc.cuh -- the learner's strided GEMM on the 5th-generation tensor cores (tcgen05.mma kind::tf32, FP32
// accumulators in TMEM).  Included by plen_td3_learn.cu only; same Gemm descriptor and the same fused epilogues as the FP32
// kernel k_gemm, so every product of TD3Agent.train (td3.py:259-356) -- X W^T forward, dY W backward-data, dY^T X
// backward-weight with its bias-gradient row sum -- is routed here once the minibatch is large (>= 512 rows).
//
// Precision: 3xTF32.  TF32 keeps the fp32 exponent (loss gradients of order 1e-7 .. 1e2 need no loss scaling) but only a
// 10-bit mantissa, and a plain TF32 forward pass moves pre-activations by ~3e-4: enough to flip the ReLU mask of a few
// entries per column, each flip a full-size term of a weight gradient (measured: 2-5 % of the largest entry of the hidden
// layers' gradients at a minibatch of 1024, r2_tc2).  Every operand is therefore split when it is staged,
//     x = hi + lo,   hi = rna_tf32(x),   lo = rna_tf32(x - hi),
// and each product is accumulated as  A_lo B_hi + A_hi B_lo + A_hi B_hi  (the dropped A_lo B_lo term is 2^-22 relative):
// fp32-level accuracy from three tensor-core passes, which cost nothing here -- the update is latency bound, not MMA bound.
// Measured against float64 on a B200 (tests/test_td3_kernels_gpu.py): per entry, relative to (|A| |B|)_mn, 1.6-3.0x the
// FP32 kernel's error on the forward / backward-data products and 5-6x on the split-K backward-weight products (the
// tensor cores' FP32 accumulation is coarser than round-to-nearest FMA chains), at most 9.6e-7, 2000x below one TF32 pass.
//
// One CTA = one 128 x 128 output tile, 512 threads.  K advances in steps of 32 through a two-stage shared-memory ring:
//   * all threads fetch A (128 x 32) and B (128 x 32) tiles from global memory into registers TWO steps ahead -- arbitrary
//     (row, k) strides, coalesced along whichever is 1 -- split them into hi / lo and store both in the canonical no-swizzle
//     K-major UMMA layout (core matrix = 8 rows x 16 B; core matrices of consecutive row groups 128 B apart, of consecutive
//     k groups LBO = 128 * 16 + 16 B apart: the 16 B of padding make the k-fast staging stores bank-conflict free).  The
//     staging therefore transposes MN-major sources (the weights of a backward-data product, both operands of a
//     backward-weight product) for free and no second operand layout is needed.
//   * one thread issues twelve tcgen05.mma (128 x N x 8, three per 8-wide k slice) per stage and commits them to the stage's
//     mbarrier; the commit of stage s is what frees its buffer two steps later.
//   * epilogue: the sixteen warps read 32 TMEM lanes x 32 columns each (tcgen05.ld 32x32b.x32; warp w: lanes 32 (w & 3),
//     columns 32 (w >> 2)), apply the
//     epilogue of the product (bias / ReLU / tanh / noise / ReLU mask / tanh gradient) and store (split-K products: atomicAdd
//     into a zeroed output).
// No TMA: the operands are split and re-laid out by the threads, not copied.
#pragma once

#include "plen_tc_common.cuh"

namespace tcg {

using namespace plen_tc;

constexpr int BM = 128, BN = 128, BK = 32, KG = BK / 4;       // KG k-groups of 4 TF32 words (16 B) per stage
constexpr int NT = 512;                                        // threads per CTA (16 warps: the staging is instruction-latency bound)
constexpr int CH = KG * BM / NT;                               // 16-byte chunks of one operand tile per thread (2)
constexpr uint32_t LBO = BM * 16 + 16;                         // bytes between the core matrices of consecutive k groups
constexpr uint32_t PART = KG * LBO;                            // one operand tile, hi or lo part
constexpr uint32_t STAGE = 4 * PART;                           // A hi | A lo | B hi | B lo
constexpr uint32_t OFF_BAR = 2 * STAGE, OFF_TPTR = OFF_BAR + 16, SMEM = OFF_TPTR + 16;
static_assert(BM == BN && PART % 16 == 0 && SMEM <= 200 * 1024 && CH * NT == KG * BM, "tile shape");

__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// chunk i of thread tid: k group kg of row r of a 128 x 32 operand tile
//   k-fast (k stride 1): e = tid + 512 i -> kg = e & 7, r = e >> 3 (8 lanes read 128 contiguous bytes of a row)
//   otherwise          : r = tid & 127, kg = (tid >> 7) + 4 i     (32 lanes read 32 consecutive rows of one k)
template <bool kfast>
__device__ __forceinline__ void chunk_of(int tid, int i, int &r, int &kg) {
    const int e = tid + NT * i;
    r = kfast ? (e >> 3) : (tid & 127);
    kg = kfast ? (e & 7) : ((tid >> 7) + (NT / 128) * i);
}

// 128 rows x 32 k of an operand -> 8 registers of this thread.  element (row, k) = base[row * rs + k * ks];
// rows >= n_rows and k >= k_hi read as zero.
template <bool kfast>
__device__ __forceinline__ void fetch_tile(const float *base, long long rs, long long ks, int row0, int n_rows, int k0, int k_hi,
                                           int tid, float (&v)[4 * CH]) {
#pragma unroll
    for (int i = 0; i < CH; i++) {
        int r, kg;
        chunk_of<kfast>(tid, i, r, kg);
        const int row = row0 + r, k = k0 + 4 * kg;
        const float *p = base + (long long)row * rs + (long long)k * ks;
        const bool row_ok = row < n_rows;
        if (kfast && row_ok && k + 3 < k_hi && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
            const float4 q = *reinterpret_cast<const float4 *>(p);
            v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) v[4 * i + j] = (row_ok && k + j < k_hi) ? p[j * ks] : 0.0f;
        }
    }
}

// split into hi / lo TF32 parts and store both (hi at `dst`, lo at `dst + PART`) in the canonical layout
template <bool kfast>
__device__ __forceinline__ void store_tile(unsigned char *dst, int tid, const float (&v)[4 * CH]) {
#pragma unroll
    for (int i = 0; i < CH; i++) {
        int r, kg;
        chunk_of<kfast>(tid, i, r, kg);
        float4 h, l;
        h.x = to_tf32(v[4 * i]); h.y = to_tf32(v[4 * i + 1]); h.z = to_tf32(v[4 * i + 2]); h.w = to_tf32(v[4 * i + 3]);
        l.x = to_tf32(v[4 * i] - h.x); l.y = to_tf32(v[4 * i + 1] - h.y); l.z = to_tf32(v[4 * i + 2] - h.z); l.w = to_tf32(v[4 * i + 3] - h.w);
        unsigned char *q = dst + kg * LBO + (r >> 3) * 128 + (r & 7) * 16;
        *reinterpret_cast<float4 *>(q) = h;
        *reinterpret_cast<float4 *>(q + PART) = l;
    }
}

// Gemm / EPI_* / CallParams / mix32 come from plen_td3_learn.cu (this header is included after their definitions).
// Launched only for minibatches whose gradient buffers are zeroed first (plen_td3_learn.cu: SPLIT_K_MIN_BATCH): the
// bias-gradient row sums are always accumulated atomically (four threads share a row).
// Three instances cover the learner: <true, true, EPI_BIAS_RELU> forward of a hidden layer, <true, false, EPI_RELUMASK>
// backward-data, <false, false, EPI_NONE> backward-weight (+ bias-gradient row sums).  The operand majors and the epilogue
// are template parameters to keep each instance's code small: the kernel runs ONCE per CTA, so its instruction stream is
// fetched cold (the first build, one 157 KB instance, spent half of its warp latency in no_instruction stalls: r2_tc4).
template <bool AKF, bool BKF, int EPI>
__global__ void __launch_bounds__(NT, 1) k_gemm_tc(const Gemm g) {
    extern __shared__ __align__(128) unsigned char sm[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int z = blockIdx.z % g.nz, split = blockIdx.z / g.nz, m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int k_lo = split * g.k_chunk, k_hi = min(g.K, k_lo + g.k_chunk);
    const int nk = (k_hi - k_lo + BK - 1) / BK;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(sm);
    const uint32_t bar0 = sbase + OFF_BAR;
    volatile uint32_t *tptr = reinterpret_cast<volatile uint32_t *>(sm + OFF_TPTR);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0 + 8) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(sbase + OFF_TPTR), "r"((uint32_t)BN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tptr;

    const float *a = g.a + z * g.az, *b = g.b + z * g.bz;
    // MMA N: the valid columns of this tile rounded up to 16 (B rows beyond N are staged as zeros)
    const int n_valid = min(BN, g.N - n0);
    const uint32_t idesc = instr_desc_tf32(BM, (n_valid + 15) & ~15);
    const uint64_t desc0 = smem_desc(sbase, LBO, 128);              // descriptor of the A hi part of stage 0
    const bool do_rs = EPI == EPI_NONE && g.rowsum != nullptr && blockIdx.x == 0;      // bias gradient: row sums of A (m-fast there: row = tid & 127)
    float rs = 0.0f;
    bool poisoned = false;

    // register sets 0 / 1 hold the operands of the even / odd steps, fetched two steps ahead of their use
    float va0[4 * CH], vb0[4 * CH], va1[4 * CH], vb1[4 * CH];
    fetch_tile<AKF>(a, g.am, g.ak, m0, g.M, k_lo, k_hi, tid, va0);
    fetch_tile<BKF>(b, g.bn, g.bk, n0, g.N, k_lo, k_hi, tid, vb0);
    fetch_tile<AKF>(a, g.am, g.ak, m0, g.M, k_lo + BK, k_hi, tid, va1);      // (reads zeros when nk == 1)
    fetch_tile<BKF>(b, g.bn, g.bk, n0, g.N, k_lo + BK, k_hi, tid, vb1);
#define TC_STEP(kt_, va_, vb_)                                                                                         \
    {                                                                                                                  \
        const int kt = (kt_), s = kt & 1;                                                                              \
        if (kt >= 2) poisoned |= !mbar_wait(bar0 + 8 * s, ((kt >> 1) - 1) & 1); /* MMAs of step kt - 2 have read buffer s */ \
        unsigned char *stg = sm + s * STAGE;                                                                           \
        store_tile<AKF>(stg, tid, va_);                                                                                \
        store_tile<BKF>(stg + 2 * PART, tid, vb_);                                                                     \
        if (do_rs) {                                                                                                   \
            _Pragma("unroll") for (int i = 0; i < 4 * CH; i++) rs += va_[i];                                           \
        }                                                                                                              \
        if (kt + 2 < nk) {                                                                                             \
            fetch_tile<AKF>(a, g.am, g.ak, m0, g.M, k_lo + (kt + 2) * BK, k_hi, tid, va_);                              \
            fetch_tile<BKF>(b, g.bn, g.bk, n0, g.N, k_lo + (kt + 2) * BK, k_hi, tid, vb_);                              \
        }                                                                                                              \
        fence_async_smem();                                                                                            \
        fence_before();                                                                                                \
        __syncthreads();                                                                                               \
        if (tid == 0) {                                                                                                \
            fence_after();                                                                                             \
            /* the start-address field (bytes >> 4) is the low end of a descriptor: part / slice offsets are plain adds */ \
            const uint64_t ah = desc0 + ((uint64_t)(s * STAGE) >> 4), al = ah + (PART >> 4), bh = ah + (2 * PART >> 4),   \
                           bl = ah + (3 * PART >> 4);                                                                   \
            _Pragma("unroll") for (int ks = 0; ks < BK / 8; ks++) {                                                    \
                const uint64_t o = (uint64_t)(ks * 2 * LBO) >> 4;                                                      \
                mma_tf32(tmem, al + o, bh + o, idesc, (kt > 0 || ks > 0) ? 1u : 0u);                                   \
                mma_tf32(tmem, ah + o, bl + o, idesc, 1u);                                                             \
                mma_tf32(tmem, ah + o, bh + o, idesc, 1u);                                                             \
            }                                                                                                          \
            mma_commit(bar0 + 8 * s);                                                                                  \
        }                                                                                                              \
    }
    for (int kt2 = 0; kt2 < nk; kt2 += 2) {
        TC_STEP(kt2, va0, vb0);
        if (kt2 + 1 < nk) TC_STEP(kt2 + 1, va1, vb1);
    }
#undef TC_STEP
    // commits complete in order: the last one covers every MMA of the tile
    if (nk > 0) poisoned |= !mbar_wait(bar0 + 8 * ((nk - 1) & 1), ((nk - 1) >> 1) & 1);
    fence_after();

    if (do_rs && m0 + (tid & 127) < g.M) atomicAdd(&g.rowsum[z * g.rowsum_z + m0 + (tid & 127)], rs);
    const int m = m0 + (tid & 127);                                  // TMEM lane = row of the tile
    const uint32_t lane_base = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    float *crow = g.c + z * g.cz + (long long)m * g.ldc;
    const float nanv = __int_as_float(0x7fc00000);
    const int c0 = (warp >> 2) * 32;                                 // this warp's 32 columns of the tile
    if (c0 < n_valid) {
        uint32_t r[32];
        tmem_ld32(lane_base + c0, r);
        if (m < g.M) {
            const float *auxrow = g.aux ? g.aux + z * g.aux_z + (long long)m * g.ld_aux : nullptr;
            const float *brow = g.bias ? g.bias + z * g.bias_z : nullptr;
            const int nn = min(32, g.N - (n0 + c0));                 // valid columns of this slice
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j++) {
                const int n = n0 + c0 + j;
                float x = (nk > 0) ? __uint_as_float(r[j]) : 0.0f;
                if (j < nn) {
                    if (EPI == EPI_BIAS_RELU) x = fmaxf(x + brow[n], 0.0f);
                    else if (EPI == EPI_RELUMASK) x = (auxrow[n] > 0.0f) ? x : 0.0f;
                }
                v[j] = poisoned ? nanv : x;
            }
            float *dst = crow + n0 + c0;
            if (g.splits > 1) {
#pragma unroll
                for (int j = 0; j < 32; j++)
                    if (j < nn) atomicAdd(dst + j, v[j]);
            } else if (nn == 32 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
                for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4 *>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 32; j++)
                    if (j < nn) dst[j] = v[j];
            }
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"((uint32_t)BN) : "memory");
}

}  // namespace tcg
