// tick_harness.cu -- TEST-ONLY: the two halves of a physics tick (k_dyn, then k_rank + k_solve / k_solve_x) launched one by one
// on a context of the library, so tests can read and write the buffer they meet at (solve records, extension records, sort
// keys, permutation) between them.
//
// plen_b200.cu is included, not copied: the kernels, their launch shapes, the dynamic shared-memory attributes plen_create
// sets and every plen_* entry point are exactly the library's.  Create the context with this library's own plen_create.
// Built by tests/tick_harness_util.py with the library's nvcc flags.
#include "../../plen_ml_walk_b200/csrc/plen_b200.cu"

extern "C" {

// device pointers of the per-robot buffers: d_state, d_srec, d_srx, d_key, d_perm, d_xgroups, d_man, d_scale, d_mass
// (d_srx / d_xgroups are NULL without link contacts, d_man without sole_manifold, d_mass before plen_set_env_mass).
// Returns the number of robots.
int th_buffers(plen_ctx *ctx, void **out) {
    out[0] = ctx->d_state; out[1] = ctx->d_srec; out[2] = ctx->d_srx; out[3] = ctx->d_key; out[4] = ctx->d_perm;
    out[5] = ctx->d_xgroups; out[6] = ctx->d_man; out[7] = ctx->d_scale; out[8] = ctx->d_mass;
    return ctx->n;
}

// sizes the tests check their layouts against
int th_sizes(int *out) {
    out[0] = SR_WORDS; out[1] = XR_WORDS; out[2] = PLEN_KEY_EXT; out[3] = RANK_KEY_MAX; out[4] = RANK_CLASSES; out[5] = RANK_TILE;
    out[6] = PLEN_SOLVE_ROBOTS; out[7] = MR_WORDS;
    return 8;
}

// k_dyn over the whole batch as tick 0 of launch_ticks runs it for plen_tick: targets_dev ([n][18], nullable = zero targets)
// are copied into d_tgt first, as plen_tick does; the context's scales, mass rows and manifolds apply, no command latency.
int th_dyn(plen_ctx *ctx, const float *targets_dev, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (targets_dev) {
        const cudaError_t e = cudaMemcpyAsync(ctx->d_tgt, targets_dev, sizeof(float) * PLEN_NJ * (size_t)ctx->n, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) return (int)e;
    }
    const bool boxes = ctx->dc.link_contacts != 0;
    launch_dyn(ctx, ctx->d_state, ctx->n, nullptr, targets_dev ? ctx->d_tgt : nullptr, ctx->d_srec, ctx->d_key, nullptr, nullptr, nullptr,
               ctx->d_scale, boxes ? ctx->d_srx : nullptr, ctx->d_man, ctx->d_mass, nullptr, 0, st);
    return (int)cudaGetLastError();
}

// k_rank over the whole batch: d_key -> d_perm (and d_xgroups with link contacts)
int th_rank(plen_ctx *ctx, void *stream) {
    const bool boxes = ctx->dc.link_contacts != 0;
    k_rank<<<rank_tiles(ctx->n), RANK_TILE, 0, (cudaStream_t)stream>>>(ctx->d_key, ctx->n, ctx->d_perm, boxes ? ctx->d_xgroups : nullptr);
    return (int)cudaGetLastError();
}

// the solve on whatever d_perm / d_xgroups hold: merged = 1 the merged k_solve<true>, 0 the split k_solve<false> + k_solve_x
// (with link contacts; without them k_solve<false> alone, as launch_ticks runs it)
int th_solve(plen_ctx *ctx, int merged, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const int n = ctx->n, nt = rank_tiles(n), ng = nt * (RANK_TILE / PLEN_SOLVE_ROBOTS);
    const bool boxes = ctx->dc.link_contacts != 0;
    if (!boxes) {
        k_solve<false><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, ctx->d_srec, ctx->d_perm, ctx->d_state, n, nt, nullptr, nullptr, ctx->d_key);
    } else if (merged) {
        k_solve<true><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, ctx->d_srec, ctx->d_perm, ctx->d_state, n, nt, ctx->d_xgroups, ctx->d_srx, ctx->d_key);
    } else {
        k_solve<false><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, ctx->d_srec, ctx->d_perm, ctx->d_state, n, nt, ctx->d_xgroups, ctx->d_srx, ctx->d_key);
        k_solve_x<<<nt * XS_SPLIT, 32, SOLVE_X_SMEM, st>>>(ctx->dc, ctx->d_srec, ctx->d_srx, ctx->d_key, ctx->d_perm, ctx->d_state, n, nt,
                                                          ctx->d_xgroups);
    }
    return (int)cudaGetLastError();
}

// PGS iteration cap and early-exit threshold of the context's later solves (residual_threshold < 0: no early exit), and the
// range size up to which plen_tick merges the box-contact groups into k_solve (launch_ticks: n <= merge_max)
void th_set_solver(plen_ctx *ctx, int iterations, float residual_threshold, int merge_max) {
    ctx->dc.iterations = iterations;
    ctx->dc.residual_threshold = residual_threshold;
    ctx->merge_max = merge_max;
}

}  // extern "C"
