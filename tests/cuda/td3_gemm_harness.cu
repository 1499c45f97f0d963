// td3_gemm_harness.cu -- TEST-ONLY: the TD3 learner's GEMM dispatch (launch() of plen_td3_learn.cu) callable on its own.
//
// Both library sources are included, not copied, so the anonymous-namespace Gemm descriptor, launch(), its split-K and
// tensor-core rules and the thread-local precision switch s_tc are exactly the library's.  (plen_td3.cu comes along for the
// replay-ring symbols plen_td3_learn.cu calls.)  Built by tests/td3_gemm_util.py with the library's nvcc flags.
#include "../../plen_ml_walk_b200/csrc/plen_td3.cu"
#include "../../plen_ml_walk_b200/csrc/plen_td3_learn.cu"

extern "C" {

// One product C[z] = epi(A[z] B[z]) through launch().
//   ptr[6]  : a, b, c, bias, aux, rowsum (the last three nullable)
//   st[12]  : az, am, ak, bz, bk, bn, cz, ldc, bias_z, aux_z, ld_aux, rowsum_z
//   dim[6]  : M, N, K, nz, epi, tc (tc = the learner's s_tc: 1 routes 128-row products to the 3xTF32 kernels)
//   p[3]    : p0, p1, p2 (max_action, policy_noise, noise_clip)
// A split-K or tensor-core product accumulates into C / rowsum: the caller zeroes them first, as the learner does.
// Returns the cudaError_t of the launch.
int harness_gemm(void *const *ptr, const long long *st, const int *dim, const float *p, unsigned long long seed, void *stream) {
    Gemm g;
    memset(&g, 0, sizeof g);
    g.a = (const float *)ptr[0]; g.b = (const float *)ptr[1]; g.c = (float *)ptr[2];
    g.bias = (const float *)ptr[3]; g.aux = (const float *)ptr[4]; g.rowsum = (float *)ptr[5];
    g.az = st[0]; g.am = st[1]; g.ak = st[2]; g.bz = st[3]; g.bk = st[4]; g.bn = st[5]; g.cz = st[6]; g.ldc = st[7];
    g.bias_z = st[8]; g.aux_z = st[9]; g.ld_aux = st[10]; g.rowsum_z = st[11];
    g.M = dim[0]; g.N = dim[1]; g.K = dim[2]; g.nz = dim[3]; g.epi = dim[4];
    g.p0 = p[0]; g.p1 = p[1]; g.p2 = p[2];
    g.seed = seed;
    g.cp = nullptr;
    if (dim[5]) {      // plen_td3_set_precision(t, 1) does the same for the library's kernels
        cudaError_t e = cudaFuncSetAttribute(tcg::k_gemm_tc<true, true, EPI_BIAS_RELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcg::SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tcg::k_gemm_tc<true, false, EPI_RELUMASK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcg::SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tcg::k_gemm_tc<false, false, EPI_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tcg::SMEM);
        if (e != cudaSuccess) return (int)e;
    }
    s_tc = dim[5] ? 1 : 0;
    launch(g, (cudaStream_t)stream);
    s_tc = 0;
    return (int)cudaGetLastError();
}

// this translation unit's copy of the tensor-core timeout flag (set when a k_gemm_tc launch abandoned an mbarrier wait)
int harness_tc_timed_out(void) {
    int v = 0;
    if (cudaMemcpyFromSymbol(&v, plen_tc::g_tc_timeout, sizeof v) != cudaSuccess) return -1;
    return v;
}

}  // extern "C"
