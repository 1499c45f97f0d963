// plen_b200.cu -- kernels + C ABI of libplen_b200.so (see include/plen_b200.h).  sm_100a only, no CPU path.
//
// One env step = (k_dyn, k_solve) x substeps + k_post on the caller's stream:
//   k_dyn   one warp per robot: FK, CRBA, M^-1, v*, contacts, row set-up -> 6.4 KB solve record per robot (HBM)
//   k_rank  counting sort of the robots by contact load inside 1024-robot tiles -> permutation
//   k_solve four lanes per robot, eight robots per warp: projected Gauss-Seidel in the 30-dim operational space,
//           delta-v, integration
//   k_post  one warp per robot: observation, done, reward, counters, auto-reset
// The per-env state record is 96 words = 3 x 128 B lines, word w = 32 k + lane, so the warp-per-robot kernels touch it
// with fully coalesced lines.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "plen_host_tables.h"
#include "plen_solve.cuh"

using namespace plen;

// warps per CTA of the warp-per-robot kernels (k_dyn, k_post)
#ifndef DYN_WPC
#define DYN_WPC 10
#endif
#ifndef DYN_CTAS
#define DYN_CTAS 2     // resident k_dyn CTAs per SM the register cap is chosen for (2 x 10 warps; r2_ab4/5: 5 x 4 is 2.6 % slower with box contacts)
#endif
#ifndef PLEN_FAN_MAX_N
#define PLEN_FAN_MAX_N (1 << 30)     // plen_step of at most this many (and at least two sort tiles of) robots runs as concurrent ranges (0: never)
#endif
#ifndef PLEN_FAN_RANGES
#define PLEN_FAN_RANGES 2   // ... this many (<= PLEN_HOST_PIPE); measured: 2 beats 3 / 4 at every batch size (profiles/r1_v9_summary.md)
#endif
#ifndef PLEN_MERGE_MAX
#define PLEN_MERGE_MAX 32768  // ranges of at most this many robots solve box-contact groups inside k_solve, larger ones in k_solve_x (env PLEN_MERGE_MAX overrides: a dev knob)
#endif
#ifndef PLEN_HOST_PIPE
#define PLEN_HOST_PIPE 4      // ranges plen_step_host pipelines (copy of one range under the kernels of the others)
#endif

struct plen_ctx {
    int n, device, sm_count, merge_max, host_ranges, host_nw, host_w[2 * 4];
    plen_config cfg;
    plen_model model;
    DevConfig dc;
    EnvRanges er;
    float *d_tab, *d_state, *d_snapshot;
    float *d_srec;   // [n][SR_WORDS] solve records (k_dyn -> k_solve)
    float *d_srx;    // [n][XR_WORDS] extension records: box-contact rows of the robots whose link boxes touch the ground (rare)
    int *d_xgroups;  // [n_tiles] leading solver groups of every tile that hold such a robot (k_rank -> k_solve / k_solve_x)
    float *d_tgt;    // [n][18] servo targets of the current env step
    float *d_man;    // [n][PLEN_MAN_WORDS] persistent sole manifolds (cfg.sole_manifold = 1; NULL otherwise)
    float *d_hull;   // [2][PLEN_MAX_HULL][3] hull vertices of the feet (ditto)
    float *d_scale;  // [n][4] per-robot scales: friction, servo force limit, servo gain (plen_set_env_scales; all 1), and the
                     // command delay in ticks (word SC_LATENCY, plen_set_env_latency; read only while d_lat exists)
    float *d_mass;   // [n][MR_WORDS] per-robot body mass scales and torso payload (plen_set_env_mass; NULL until its first call)
    float *d_lat;    // [n][LAT_WORDS] per-robot command history ring (plen_set_env_latency; NULL until its first call)
    uint8_t *d_key;  // [n] contact-load sort key of the current tick (k_dyn -> k_rank)
    int *d_perm;     // [n_tiles * RANK_TILE] robots ordered by contact load inside each tile (k_rank -> k_solve)
    float *d_act, *d_obs, *d_rew;
    uint8_t *d_done, *d_tmo;
    unsigned long long *d_faults;   // robots retired by the numeric guard of k_post (plen_fault_count)
    cudaStream_t stream;
    cudaStream_t pipe[PLEN_HOST_PIPE];      // pipe[0] == stream; ranges of plen_step_host / of a fanned-out small plen_step
    cudaEvent_t fan_fork, fan_join[PLEN_HOST_PIPE];
    cudaEvent_t last_work;                  // recorded by every entry point that queues work on a caller stream; plen_step_host waits for it
    unsigned long long launches;            // kernels launched by plen_reset / plen_step / plen_step_host / plen_tick (plen_kernel_launches)
    // optional per-kernel timing of plen_step (plen_profile_enable): 2*substeps+2 events per recorded step
    cudaEvent_t *prof_ev;
    int prof_cap, prof_steps;
    char err[512];
};

static char g_err[512] = "";

static int fail(plen_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    snprintf(ctx ? ctx->err : g_err, 512, "%s", buf);
    return code;
}
#define CK(ctx, call)                                                                                       \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess) return fail(ctx, PLEN_E_CUDA, "%s: %s", #call, cudaGetErrorString(e_));      \
    } while (0)

// ------------------------------------------------------------------------------------------------ kernels
struct DynSmem {
    float tab[T_ROWS * 32];
    WarpScratch ws[DYN_WPC];
};

__device__ __forceinline__ DynSmem &stage_table(const float *tab_g) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DynSmem &sm = *reinterpret_cast<DynSmem *>(smem_raw);
    for (int i = threadIdx.x; i < T_ROWS * 32; i += blockDim.x) sm.tab[i] = tab_g[i];
    __syncthreads();
    return sm;
}

// First half of a tick, one warp per robot: FK, CRBA, M^-1, v*, contacts, row set-up -> solve record.
//   actions != NULL : agent-space actions of a new env step; the servo targets are derived (agent_to_env) and kept in tgt
//   actions == NULL : tgt holds the targets already (NULL = zero targets, the reset pose)
// 5 CTAs (20 warps) per SM: the register cap (<= 102) costs 16 B of spills outside the hot loops and measured +2.4 %
// MASS = true: the robots' mass rows (mrow, [n][MR_WORDS]) scale their bodies and add the torso payload; the false instance is
// the stock path, untouched by the option (launched whenever no mass row applies).
// lat != NULL (env steps once plen_set_env_latency was called; then scale != NULL too): tick `tick` of the step applies the
// robot's delayed command (latency_source) from its history ring, and tick 0 records the step's own targets in the ring.
template <bool MASS>
__global__ void __launch_bounds__(DYN_WPC * 32, DYN_CTAS)
k_dyn(const __grid_constant__ DevConfig dc, const __grid_constant__ EnvRanges er, const float *__restrict__ tab_g,
      const float *__restrict__ state, int n, const float *__restrict__ actions, float *__restrict__ tgt,
      float *__restrict__ srec, uint8_t *__restrict__ keys, float *dbg_minv, float *dbg_pos, float *dbg_rot,
      const float *__restrict__ scale, float *__restrict__ srx, float *__restrict__ man, const float *__restrict__ mrow,
      float *__restrict__ lat, int tick) {
    // The 4 KB model table is staged with cp.async while every warp already fetches its robot's state record and targets:
    // the two latencies overlap instead of adding up (the table wait used to sit in front of everything).
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DynSmem &sm = *reinterpret_cast<DynSmem *>(smem_raw);
    for (int i = threadIdx.x; i < T_ROWS * 32 / 4; i += blockDim.x)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((unsigned)__cvta_generic_to_shared(sm.tab + 4 * i)),
                     "l"(tab_g + 4 * i) : "memory");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    WarpScratch &ws = sm.ws[warp];
    const int env = blockIdx.x * DYN_WPC + warp;
    const bool has = env < n;
    float r0 = 0.0f, r1 = 0.0f, r2 = 0.0f, a_in = 0.0f;
    const bool jl = lane >= 6 && lane < 24;
    const size_t o = (size_t)(has ? env : 0) * PLEN_NJ + (jl ? lane - 6 : 0);
    if (has) {
        const float *rec = state + (size_t)env * PLEN_STATE_WORDS;
        r0 = gld(rec + lane); r1 = gld(rec + 32 + lane); r2 = gld(rec + 64 + lane);
        if (jl) a_in = actions ? gld(actions + o) : (tgt ? gld(tgt + o) : 0.0f);
    }
    vec4 sc; sc.x = sc.y = sc.z = sc.w = 1.0f;
    if (has && scale) sc = gld4(scale + 4 * (size_t)env);
    float mw = 1.0f;
    if (MASS && has) mw = gld(mrow + (size_t)env * MR_WORDS + lane);     // one 128-byte line per robot
    int lsrc = 0, ept = 0;
    float lv = 0.0f;       // the delayed targets (0: the reset-pose hold target of a command from before the last reset)
    if (lat && has) {
        ept = max((int)shfl(r1, W_EPT - 32), 0);
        lsrc = latency_source((int)sc.w, tick, dc.substeps, ept);
        if (lsrc > 0 && jl) lv = gld(lat + (size_t)env * LAT_WORDS + 32 * latency_slot(ept, lsrc) + lane);   // one ring row
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    if (!has) return;
    LaneState L;
    unpack_record(r0, r1, r2, ws, L, lane);
    L.fric_s = sc.x; L.motor_s = sc.y; L.kp_s = sc.z;
    L.mass_w = mw;
    if (jl) {
        if (actions) { L.tgt = agent_target(dc, er, lane - 6, a_in); tgt[o] = L.tgt; }
        else L.tgt = a_in;
        if (lat) {
            if (actions) lat[(size_t)env * LAT_WORDS + 32 * latency_slot(ept, 0) + lane] = L.tgt;   // this step joins the history
            if (lsrc != 0) L.tgt = lv;
        }
    }
    DebugOut dbg{dbg_minv ? dbg_minv + (size_t)env * 576 : nullptr, dbg_pos ? dbg_pos + (size_t)env * 72 : nullptr,
                 dbg_rot ? dbg_rot + (size_t)env * 216 : nullptr};
    tick_dynamics<MASS>(dc, sm.tab, ws, L, lane, srec + (size_t)env * SR_WORDS, keys + env, (dbg_minv || dbg_pos || dbg_rot) ? &dbg : nullptr,
                        srx ? srx + (size_t)env * XR_WORDS : nullptr, man ? man + (size_t)env * PLEN_MAN_WORDS : nullptr);
}

// Robots are grouped by contact load before the solve: k_rank counting-sorts the keys k_dyn wrote inside tiles of
// RANK_TILE robots (heaviest first) and writes the permutation k_solve reads, so that the eight robots of a solver warp
// have similar active-point counts (mean per-foot loop length 2.6 -> 1.9 slots on the bench workload) and the heavy
// warps of every tile are dispatched first.  The sort is stable, so the grouping is reproducible.
#define RANK_TILE 1024
#define RANK_KEY_MAX (PLEN_KEY_EXT + PLEN_MAX_BOX_POINTS - 1)
#define RANK_CLASSES 160      // RANK_KEY_MAX + 1 keys and one class for the slots beyond n, rounded up to a multiple of 32
static_assert(RANK_KEY_MAX + 2 <= RANK_CLASSES && RANK_CLASSES % 32 == 0 && RANK_KEY_MAX <= 255, "k_rank class table");
__global__ void __launch_bounds__(RANK_TILE)
k_rank(const uint8_t *__restrict__ keys, int n, int *__restrict__ perm, int *__restrict__ xgroups) {
    // STABLE counting sort (robots of a class keep their index order), so the grouping of robots into solver warps -- and
    // with it every bit of the step -- is reproducible run to run: rank inside the warp from match_any, warps of a class
    // in warp order through a [warp][class] count table.
    __shared__ unsigned short s_wcnt[RANK_TILE / 32][RANK_CLASSES];
    __shared__ int s_base[RANK_CLASSES];
    const int t = threadIdx.x, r = blockIdx.x * RANK_TILE + t, w = t >> 5, lane = t & 31;
    for (int i = t; i < (RANK_TILE / 32) * RANK_CLASSES; i += RANK_TILE) (&s_wcnt[0][0])[i] = 0;
    __syncthreads();
    // class 0 = heaviest (key RANK_KEY_MAX: box contacts, most points); robots beyond n sort last
    const int cls = (r < n) ? RANK_KEY_MAX - min(gld_u8(keys + r), RANK_KEY_MAX) : RANK_CLASSES - 1;
    const unsigned peers = __match_any_sync(0xffffffffu, cls);
    const int rank_in_warp = __popc(peers & ((1u << lane) - 1u));
    if (rank_in_warp == 0) s_wcnt[w][cls] = (unsigned short)__popc(peers);
    __syncthreads();
    if (t < RANK_CLASSES) {  // class totals, then (below) their exclusive scan
        int tot = 0;
        for (int k = 0; k < RANK_TILE / 32; k++) tot += s_wcnt[k][t];
        s_base[t] = tot;
    }
    __syncthreads();
    if (t < 32) {            // exclusive scan of the class counts: RANK_CLASSES / 32 per lane
        constexpr int PER = RANK_CLASSES / 32;
        int c[PER], sum = 0;
#pragma unroll
        for (int k = 0; k < PER; k++) { c[k] = s_base[PER * t + k]; sum += c[k]; }
        int incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, incl, d); if (t >= d) incl += o; }
        int run = incl - sum;
#pragma unroll
        for (int k = 0; k < PER; k++) { s_base[PER * t + k] = run; run += c[k]; }
    }
    __syncthreads();
    int pos = rank_in_warp;
    for (int k = 0; k < w; k++) pos += s_wcnt[k][cls];
    perm[blockIdx.x * RANK_TILE + s_base[cls] + pos] = r;
    // classes 0 .. PLEN_MAX_BOX_POINTS - 1 = robots with box contacts: they lead the tile; so many solver groups hold one
    if (t == 0 && xgroups) xgroups[blockIdx.x] = (s_base[PLEN_MAX_BOX_POINTS] + PLEN_SOLVE_ROBOTS - 1) / PLEN_SOLVE_ROBOTS;
}

// Second half of a tick, 4 lanes per robot: PGS + delta-v + integration, state record updated in place.
// A CTA is ONE warp = 8 robots (30.1 KB of G in shared memory, 7 CTAs per SM).  CTA b takes group b / n_tiles of tile
// b % n_tiles, so the heavy groups of all tiles run first and the tail of the grid is made of light ones.
#ifndef PLEN_SOLVE_MAXREG
#define PLEN_SOLVE_MAXREG 255
#endif
// MERGED = false: the plain instance only; groups that hold a box-contact robot return at once and k_solve_x takes them.
// MERGED = true : those groups run the EXT instance inside this launch (same footprint: the EXT rows are read from global
//                 memory).  Measured (r2_ab1): at 4,096 robots the merged launch saves the serial tail of a second, nearly
//                 empty launch per tick (0.751 vs 1.062 ms per env step); at 131,072 robots the plain kernel compiled alone
//                 is 1-2 % faster (251 registers, smaller code), so launch_ticks picks by range size (PLEN_MERGE_MAX).
template <bool MERGED>
__global__ void __maxnreg__(PLEN_SOLVE_MAXREG)
k_solve(const __grid_constant__ DevConfig dc, const float *__restrict__ srec, const int *__restrict__ perm,
        float *__restrict__ state, int n, int n_tiles, const int *__restrict__ xgroups, const float *__restrict__ srx,
        const uint8_t *__restrict__ keys) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *Gs = reinterpret_cast<float *>(smem_raw);
    const int lane = threadIdx.x;
    const int tile = blockIdx.x % n_tiles, grp = blockIdx.x / n_tiles;
    // the first xgroups[tile] groups of a tile hold the robots whose link boxes touch the ground (k_rank sorts them to the front)
    const bool xgrp = xgroups && grp < gld_i(xgroups + tile);
    if (!MERGED && xgrp) return;
    const int robot = gld_i(perm + tile * RANK_TILE + grp * PLEN_SOLVE_ROBOTS + (lane >> 2));
    const bool valid = robot < n;
    const size_t r = valid ? (size_t)robot : 0;
    if (MERGED && xgrp) {
        const bool isx = valid && gld_u8(keys + r) >= PLEN_KEY_EXT;
        const int nx = isx ? (int)gld(srx + r * XR_WORDS + XR_NX) : 0;
        solve_tick<1>(dc, srec + r * SR_WORDS, Gs + (size_t)(lane >> 2) * PLEN_GS_WORDS, state + r * PLEN_STATE_WORDS, lane, valid,
                         srx + r * XR_WORDS, nx);
    } else {
        solve_tick<0>(dc, srec + r * SR_WORDS, Gs + (size_t)(lane >> 2) * PLEN_GS_WORDS, state + r * PLEN_STATE_WORDS, lane, valid);
    }
}

// The EXT instance as its own launch (large ranges): XS_SPLIT CTAs per tile walk the tile's box-contact groups, so the grid
// does not grow with the (unknown to the host) number of such groups; most CTAs find none.
#ifndef XS_SPLIT
#define XS_SPLIT 16
#endif
__global__ void __maxnreg__(255)
k_solve_x(const __grid_constant__ DevConfig dc, const float *__restrict__ srec, const float *__restrict__ srx,
          const uint8_t *__restrict__ keys, const int *__restrict__ perm, float *__restrict__ state, int n, int n_tiles,
          const int *__restrict__ xgroups) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *Gs = reinterpret_cast<float *>(smem_raw);
    float *Xs = Gs + PLEN_SOLVE_ROBOTS * PLEN_GS_WORDS;
    const int lane = threadIdx.x;
    const int tile = blockIdx.x % n_tiles;
    const int ng = gld_i(xgroups + tile);
    for (int grp = blockIdx.x / n_tiles; grp < ng; grp += XS_SPLIT) {
        const int robot = gld_i(perm + tile * RANK_TILE + grp * PLEN_SOLVE_ROBOTS + (lane >> 2));
        const bool valid = robot < n;
        const size_t r = valid ? (size_t)robot : 0;
        const bool isx = valid && gld_u8(keys + r) >= PLEN_KEY_EXT;
        const int nx = isx ? (int)gld(srx + r * XR_WORDS + XR_NX) : 0;
        solve_tick<2>(dc, srec + r * SR_WORDS, Gs + (size_t)(lane >> 2) * PLEN_GS_WORDS, state + r * PLEN_STATE_WORDS, lane, valid,
                         srx + r * XR_WORDS, nx, Xs + (size_t)(lane >> 2) * PLEN_XS_WORDS);
        __syncwarp();
    }
}

// per-robot scales (domain randomisation): column c of d_scale <- the given array, or 1 when `init`
__global__ void k_set_scales(float *__restrict__ scale, int n, const float *fric, const float *motor, const float *kp, int init) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float *s = scale + 4 * (size_t)e;
    if (init) { s[0] = s[1] = s[2] = s[3] = 1.0f; }
    if (fric) s[0] = fric[e];
    if (motor) s[1] = motor[e];
    if (kp) s[2] = kp[e];
}

// per-robot mass rows: body scales [n][PLEN_BODIES] into words 0 and 6..23, payload [n][4] into words 24..27; NULL leaves a part
// as it is, `init` first writes unit rows (scale 1, payload 0, padding 1).  One thread per word.
__global__ void k_set_mass(float *__restrict__ mrow, int n, const float *scale, const float *payload, int init) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * MR_WORDS) return;
    const size_t e = i / MR_WORDS;
    const int w = (int)(i % MR_WORDS);
    const bool pay = w >= MR_PAYLOAD && w < MR_PAYLOAD + 4, body = w == 0 || (w >= 6 && w < MR_PAYLOAD);
    if (init) mrow[i] = pay ? 0.0f : 1.0f;
    if (scale && body) mrow[i] = scale[e * PLEN_BODIES + (w == 0 ? 0 : w - 5)];
    if (payload && pay) mrow[i] = payload[e * 4 + (w - MR_PAYLOAD)];
}

// ... and back; unit values when the context has no mass rows
__global__ void k_get_mass(const float *__restrict__ mrow, int n, float *scale, float *payload) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)n * MR_WORDS) return;
    const size_t e = i / MR_WORDS;
    const int w = (int)(i % MR_WORDS);
    const bool pay = w >= MR_PAYLOAD && w < MR_PAYLOAD + 4, body = w == 0 || (w >= 6 && w < MR_PAYLOAD);
    if (scale && body) scale[e * PLEN_BODIES + (w == 0 ? 0 : w - 5)] = mrow ? mrow[i] : 1.0f;
    if (payload && pay) payload[e * 4 + (w - MR_PAYLOAD)] = mrow ? mrow[i] : 0.0f;
}

// per-robot command latency, one thread per robot: the delay (clamped to 0 .. 2 substeps, so that no value can index out of
// the ring) into word SC_LATENCY of the scale row, the logical history [n][2][18] (last step, the step before) into the ring
// rows of the robot's episode counter.  NULL leaves a part as it is; `init` first sets delay 0 and fills every ring row with
// the robot's last targets (tgt), as if that command had been held.
__global__ void k_set_latency(float *__restrict__ scale, float *__restrict__ ring, const float *__restrict__ state,
                              const float *__restrict__ tgt, int n, int max_ticks, const int *ticks, const float *hist, int init) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float *row = ring + (size_t)e * LAT_WORDS;
    if (init) {
        scale[4 * (size_t)e + SC_LATENCY] = 0.0f;
        for (int s = 0; s < LAT_SLOTS; s++)
            for (int j = 0; j < PLEN_NJ; j++) row[32 * s + 6 + j] = tgt[(size_t)e * PLEN_NJ + j];
    }
    if (ticks) scale[4 * (size_t)e + SC_LATENCY] = (float)min(max(ticks[e], 0), max_ticks);
    if (hist) {
        const int ept = max((int)state[(size_t)e * PLEN_STATE_WORDS + W_EPT], 0);
        for (int s = 1; s <= 2; s++)
            for (int j = 0; j < PLEN_NJ; j++) row[32 * latency_slot(ept, s) + 6 + j] = hist[((size_t)e * 2 + s - 1) * PLEN_NJ + j];
    }
}

// ... and back; delay 0 and the last targets as history when the context has no ring
__global__ void k_get_latency(const float *__restrict__ scale, const float *__restrict__ ring, const float *__restrict__ state,
                              const float *__restrict__ tgt, int n, int *ticks, float *hist) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (ticks) ticks[e] = ring ? (int)scale[4 * (size_t)e + SC_LATENCY] : 0;
    if (hist) {
        const int ept = max((int)state[(size_t)e * PLEN_STATE_WORDS + W_EPT], 0);
        for (int s = 1; s <= 2; s++)
            for (int j = 0; j < PLEN_NJ; j++)
                hist[((size_t)e * 2 + s - 1) * PLEN_NJ + j] =
                    ring ? ring[(size_t)e * LAT_WORDS + 32 * latency_slot(ept, s) + 6 + j] : tgt[(size_t)e * PLEN_NJ + j];
    }
}

// After the last tick of an env step, one warp per robot: observation, done, reward, counters, auto-reset.
__global__ void __launch_bounds__(DYN_WPC * 32)
k_post(const __grid_constant__ DevConfig dc, const float *__restrict__ tab_g, float *__restrict__ state, int n,
       float *__restrict__ obs, float *__restrict__ reward, uint8_t *__restrict__ done, uint8_t *__restrict__ timeout,
       float *__restrict__ terminal_obs, const float *__restrict__ snapshot, unsigned long long *__restrict__ faults,
       float *__restrict__ man) {
    DynSmem &sm = stage_table(tab_g);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env = blockIdx.x * DYN_WPC + warp;
    if (env >= n) return;
    WarpScratch &ws = sm.ws[warp];
    LaneState L;
    load_record(state + (size_t)env * PLEN_STATE_WORDS, ws, L, lane);
    StepIO io{nullptr, obs + (size_t)env * PLEN_OBS, reward + env, done + env, timeout ? timeout + env : nullptr,
              terminal_obs ? terminal_obs + (size_t)env * PLEN_OBS : nullptr, snapshot, faults,
              man ? man + (size_t)env * PLEN_MAN_WORDS : nullptr};
    env_post(dc, sm.tab, ws, L, lane, io);
    store_record(state + (size_t)env * PLEN_STATE_WORDS, ws, L, lane);
}

__global__ void __launch_bounds__(DYN_WPC * 32)
k_observe(const float *__restrict__ state, int n, float *__restrict__ obs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DynSmem &sm = *reinterpret_cast<DynSmem *>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env = blockIdx.x * (blockDim.x >> 5) + warp;
    if (env >= n) return;
    WarpScratch &ws = sm.ws[warp];
    LaneState L;
    load_record(state + (size_t)env * PLEN_STATE_WORDS, ws, L, lane);
    observe(ws, L, lane);
    if (lane < PLEN_OBS) obs[(size_t)env * PLEN_OBS + lane] = ws.obs[lane];
}

// PlenWalkEnv.reset (plen_env.py:558-614): copy the post-reset snapshot into the selected envs
__global__ void k_reset(float *__restrict__ state, int n, const uint8_t *__restrict__ mask,
                        const float *__restrict__ snapshot, float *__restrict__ obs, float *__restrict__ man) {
    const int env = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (env >= n) return;
    if (mask && !mask[env]) return;
    float *rec = state + (size_t)env * PLEN_STATE_WORDS;
    rec[lane] = snapshot[lane];
    rec[32 + lane] = snapshot[32 + lane];
    rec[64 + lane] = snapshot[64 + lane];
    if (obs && lane < PLEN_OBS) obs[(size_t)env * PLEN_OBS + lane] = snapshot[PLEN_STATE_WORDS + lane];
    if (man) {
        for (int w = lane; w < PLEN_MAN_WORDS; w += 32) man[(size_t)env * PLEN_MAN_WORDS + w] = snapshot[PLEN_SNAP_MAN + w];
    }
}

__global__ void k_fill(float *__restrict__ state, int n, const float *__restrict__ rec96) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < (size_t)n * PLEN_STATE_WORDS) state[i] = rec96[i % PLEN_STATE_WORDS];
}

// aux = [lam_n[8], manifold bits, cnt, ds, hist_len, ep_t, last[6], sums[9], ep_ret]
__global__ void k_get_state(const float *__restrict__ state, int n, float *qpos, float *qvel, float *aux) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const float *r = state + (size_t)e * PLEN_STATE_WORDS;
    if (qpos) {
        float *o = qpos + (size_t)e * PLEN_QPOS;
        for (int k = 0; k < 3; k++) o[k] = r[W_POS + k];
        for (int k = 0; k < 4; k++) o[3 + k] = r[W_QUAT + k];
        for (int k = 0; k < 18; k++) o[7 + k] = r[W_Q + 6 + k];
    }
    if (qvel) {
        float *o = qvel + (size_t)e * PLEN_QVEL;
        for (int k = 0; k < 3; k++) { o[k] = r[W_U + 3 + k]; o[3 + k] = r[W_U + k]; }
        for (int k = 0; k < 18; k++) o[6 + k] = r[W_U + 6 + k];
    }
    if (aux) {
        float *o = aux + (size_t)e * PLEN_AUX_WORDS;
        for (int k = 0; k < 8; k++) o[k] = r[W_U + 24 + k];
        o[8] = r[W_MAN]; o[9] = r[W_CNT]; o[10] = r[W_DS]; o[11] = r[W_HIST]; o[12] = r[W_EPT];
        for (int k = 0; k < 6; k++) o[13 + k] = r[W_LAST + k];
        for (int k = 0; k < 9; k++) o[19 + k] = r[W_SUMS + k];
        o[28] = r[W_EPRET];
    }
}

__global__ void k_set_state(float *__restrict__ state, int n, const float *qpos, const float *qvel, const float *aux) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float *r = state + (size_t)e * PLEN_STATE_WORDS;
    if (qpos) {
        const float *o = qpos + (size_t)e * PLEN_QPOS;
        for (int k = 0; k < 3; k++) r[W_POS + k] = o[k];
        for (int k = 0; k < 4; k++) r[W_QUAT + k] = o[3 + k];
        for (int k = 0; k < 18; k++) r[W_Q + 6 + k] = o[7 + k];
    }
    if (qvel) {
        const float *o = qvel + (size_t)e * PLEN_QVEL;
        for (int k = 0; k < 3; k++) { r[W_U + 3 + k] = o[k]; r[W_U + k] = o[3 + k]; }
        for (int k = 0; k < 18; k++) r[W_U + 6 + k] = o[6 + k];
    }
    if (aux) {
        const float *o = aux + (size_t)e * PLEN_AUX_WORDS;
        for (int k = 0; k < 8; k++) r[W_U + 24 + k] = o[k];
        r[W_MAN] = o[8]; r[W_CNT] = o[9]; r[W_DS] = o[10]; r[W_HIST] = o[11]; r[W_EPT] = o[12];
        for (int k = 0; k < 6; k++) r[W_LAST + k] = o[13 + k];
        for (int k = 0; k < 9; k++) r[W_SUMS + k] = o[19 + k];
        r[W_EPRET] = o[28];
    }
}

// ---- sinewave gait + closed-form leg IK, float64, one thread per parameter set
// (trajectory_generator.py:54-152 foot_path, :154-167 assemble, :169-233 IK, :235-270; trajectory_eval.py:180-261)
namespace gait {
constexpr int NDS = 5, NSS = 10, NROW = 20;   // trajectory_generator.py:10-11
__device__ bool leg_ik(double x, double y, double z, bool right, double *out6) {
    const double l1 = 25.0, l2 = 40.0;                                 // :35-37
    const double Zx = x, Zy = y, Zz = l1 + l2 - z;                     // :181-183
    const double th1 = right ? atan2(-Zy, Zz) : atan2(Zy, Zz);         // :185-188
    const double arg = (Zx * Zx + Zy * Zy + Zz * Zz - l1 * l1 - l2 * l2) / (2.0 * l1 * l2);   // :190-192
    if (!(arg >= -1.0 && arg <= 1.0)) return false;                    // math.acos raises ValueError
    double th3 = acos(arg);
    const double sqrtyz = sqrt(Zy * Zy + Zz * Zz), hok = l1 / l2;      // :194-195
    double th2 = -atan2(sqrtyz * sin(th3) + Zx * cos(th3) + Zx * hok,
                        sqrtyz * cos(th3) + sqrtyz * hok - Zx * sin(th3));   // :197-199
    // real_ranges (plen_env.py:170-189): R knee [3] / L knee [9] = [-1.0, 1.57]; R thigh [2] = [-0.95, 1.2]; L [8] = [-1.2, 0.95]
    th3 = fmin(fmax(th3, -1.0), 1.57);                                 // :203-207 / :215-218
    if (right) th2 = fmin(fmax(th2, -0.95), 1.2); else th2 = fmin(fmax(th2, -1.2), 0.95);   // :209-212 / :220-223
    const double th4 = -(th2 + th3), th5 = right ? -th1 : th1;         // :225-230
    out6[0] = 0.0; out6[1] = th1; out6[2] = th2; out6[3] = th3; out6[4] = th4; out6[5] = th5;
    return true;
}
__device__ void foot_point(int seg, int i, double height, double stride, double bend, double sway, double bias, double *p) {
    // seg: 0 SS dominant, 1 DS dominant, 2 SS support, 3 DS support (trajectory_generator.py:66-125)
    const double PI = 3.141592653589793;
    double t;
    switch (seg) {
        case 0: t = i / (NSS - 1.0);
            p[0] = t * stride; p[1] = sin(-PI * ((1 / 3.0) * (1 + t))) * sway; p[2] = sin(t * PI) * height + bend; break;
        case 1: t = i / (2 * NDS - 1.0);
            p[0] = -stride * (t / 2.0); p[1] = sin(-PI * ((-1.0 / 3.0) + (2 / 3.0) * t)) * sway; p[2] = bend; break;
        case 2: t = i / (NSS - 1.0);
            p[0] = stride * ((1.0 / 2.0) - t) / 2.0; p[1] = sin(PI * ((1 / 3.0) * (1 + t))) * sway; p[2] = bend; break;
        default: t = i / (2.0 * NDS - 1.0);
            p[0] = stride * (1.0 - t) / 2.0; p[1] = sin(-PI * ((2.0 / 3.0) + (2 / 3.0) * t)) * sway; p[2] = bend; break;
    }
    if (bias != 0) p[0] = p[0] - bias;                                  // :128-132
}
// column c (0..19) of foot_walk_rfwd_r (dominant: DS 2nd half, SS, support-DS 1st half) or foot_walk_lfwd_r (:135-145)
__device__ void walk_point(bool dominant, int c, double h, double s, double b, double sw, double bias, double *p) {
    if (dominant) {
        if (c < NDS) foot_point(1, NDS + c, h, s, b, sw, bias, p);
        else if (c < NDS + NSS) foot_point(0, c - NDS, h, s, b, sw, bias, p);
        else foot_point(3, c - NDS - NSS, h, s, b, sw, bias, p);
    } else {
        if (c < NDS) foot_point(3, NDS + c, h, s, b, sw, bias, p);
        else if (c < NDS + NSS) foot_point(2, c - NDS, h, s, b, sw, bias, p);
        else foot_point(1, c - NDS - NSS, h, s, b, sw, bias, p);
    }
}
__device__ void assemble_row(const double *row12, double *out18) {     // trajectory_eval.py:180-205
    const double PI = 3.141592653589793;
    out18[0] = -row12[0]; out18[1] = -row12[1]; out18[2] = -row12[2]; out18[3] = -row12[3];
    out18[4] = row12[4]; out18[5] = row12[5];
    out18[6] = row12[6]; out18[7] = row12[7]; out18[8] = row12[8]; out18[9] = row12[9];
    out18[10] = -row12[10]; out18[11] = row12[11];
    out18[12] = PI / 5; out18[13] = PI / 8; out18[14] = 0; out18[15] = -PI / 5; out18[16] = PI / 8; out18[17] = 0;
}
}  // namespace gait

__global__ void k_gait_ik(const double *__restrict__ params, int n, double *__restrict__ traj, double *__restrict__ bend,
                          uint8_t *__restrict__ status) {
    using namespace gait;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    const double h = params[5 * g], s = params[5 * g + 1], b = params[5 * g + 2], sw = params[5 * g + 3],
                 bias = params[5 * g + 4];
    bool ok = true;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int half = 0; half < 2; half++) {          // 0: foot_walk_rfwd, 1: foot_walk_lfwd
        for (int c = 0; c < NROW; c++) {
            double pr[3], pl[3], row[12], out[18];
            // right leg follows *_r; left leg follows the complementary path with y negated (:154-167)
            walk_point(half == 0, c, h, s, b, sw, bias, pr);
            walk_point(half != 0, c, h, s, b, sw, bias, pl);
            pl[1] = -pl[1];
            bool good = leg_ik(pr[0], pr[1], pr[2], true, row) & leg_ik(pl[0], pl[1], pl[2], false, row + 6);
            if (good) assemble_row(row, out);
            else { ok = false; for (int k = 0; k < 18; k++) out[k] = nan; }
            for (int k = 0; k < 18; k++) traj[((size_t)g * 40 + half * NROW + c) * 18 + k] = out[k];
        }
    }
    {   // bend_legs (trajectory_generator.py:240-252, trajectory_eval.py:251-261)
        double row[12], out[18];
        bool good = leg_ik(0.0, 0.0, b, true, row) & leg_ik(0.0, 0.0, b, false, row + 6);
        if (good) {
            for (int k = 0; k < 12; k++) out[k] = row[k];
            for (int k = 12; k < 18; k++) out[k] = 0.0;
            out[13] = 0.5; out[16] = 0.5;
            for (int k = 0; k < 4; k++) out[k] = -out[k];
            out[10] = -out[10];
        } else { ok = false; for (int k = 0; k < 18; k++) out[k] = nan; }
        if (bend) for (int k = 0; k < 18; k++) bend[(size_t)g * 18 + k] = out[k];
    }
    if (!ok) {   // the reference generator raises for the whole parameter set: no partial trajectory survives
        for (int k = 0; k < 40 * 18; k++) traj[(size_t)g * 40 * 18 + k] = nan;
        if (bend) for (int k = 0; k < 18; k++) bend[(size_t)g * 18 + k] = nan;
    }
    if (status) status[g] = ok ? 0 : 1;
}


// ---- FP32 FMA-pipe peak (measurement aid; SURVEY.md 8d asks for it: MEASURED_PEAKS.json has no FP32 figure).
// Every thread runs 8 independent FFMA (mode 0) or 4 packed FFMA2 (mode 1, fma.rn.f32x2) chains; 2 flop per lane-FMA.
__global__ void __launch_bounds__(256)
k_fp32_peak(float *out, int iters, int mode, float seed) {
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = seed + (float)(threadIdx.x + k);
    const float x = 0.999f + seed, y = 1e-3f;
    if (mode == 0) {
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int r = 0; r < 16; r++)
#pragma unroll
                for (int k = 0; k < 8; k++) a[k] = fmaf(a[k], x, y);
        }
    } else {
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int r = 0; r < 16; r++)
#pragma unroll
                for (int k = 0; k < 8; k += 2)
                    asm volatile("{ .reg .b64 ra, rb, rc; mov.b64 ra, {%0, %1}; mov.b64 rb, {%2, %2}; mov.b64 rc, {%3, %3};\n\t"
                                 "fma.rn.f32x2 ra, ra, rb, rc; mov.b64 {%0, %1}, ra; }"
                                 : "+f"(a[k]), "+f"(a[k + 1]) : "f"(x), "f"(y));
        }
    }
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; k++) s += a[k];
    if (s == 12345.678f) out[0] = s;      // never true in practice: keeps the chains alive
}

// ------------------------------------------------------------------------------------------------ C ABI
static const size_t DYN_SMEM = sizeof(DynSmem);
static const size_t SOLVE_SMEM = sizeof(float) * PLEN_GS_WORDS * PLEN_SOLVE_ROBOTS;
static const size_t SOLVE_X_SMEM = sizeof(float) * (PLEN_GS_WORDS + PLEN_XS_WORDS) * PLEN_SOLVE_ROBOTS;
// k_dyn: one CTA per four robots.  (Measured slower: a persistent grid-stride walk, grid = resident CTAs, 3 %; CTAs that walk
// 2 / 4 / 8 consecutive groups, 1.7 / 3.6 / 4.4 % -- many short CTAs overlap their load phases best.)
static int dyn_grid(int n) { return (n + DYN_WPC - 1) / DYN_WPC; }
static int rank_tiles(int n) { return (n + RANK_TILE - 1) / RANK_TILE; }

// k_dyn over n robots; the MASS instance only when mass rows apply (mrow != NULL), the stock instance otherwise.  lat: the
// robots' command history rings (nullable), tick: index of the tick inside the env step
static void launch_dyn(plen_ctx *ctx, const float *state, int n, const float *actions, float *tgt, float *srec, uint8_t *key,
                       float *dbg_minv, float *dbg_pos, float *dbg_rot, const float *scale, float *srx, float *man,
                       const float *mrow, float *lat, int tick, cudaStream_t st) {
    if (mrow)
        k_dyn<true><<<dyn_grid(n), DYN_WPC * 32, DYN_SMEM, st>>>(ctx->dc, ctx->er, ctx->d_tab, state, n, actions, tgt, srec, key,
                                                                dbg_minv, dbg_pos, dbg_rot, scale, srx, man, mrow, lat, tick);
    else
        k_dyn<false><<<dyn_grid(n), DYN_WPC * 32, DYN_SMEM, st>>>(ctx->dc, ctx->er, ctx->d_tab, state, n, actions, tgt, srec, key,
                                                                 dbg_minv, dbg_pos, dbg_rot, scale, srx, man, nullptr, lat, tick);
}

// n_ticks physics ticks of 1/240 s: (k_dyn, k_solve) per tick.  `actions` (agent space) only on the first tick.
// ev (nullable): 2*n_ticks events recorded before each kernel.
static void launch_ticks(plen_ctx *ctx, float *state, int n, const float *actions, float *tgt, int n_ticks, cudaStream_t st,
                         cudaEvent_t *ev = nullptr, size_t off = 0) {
    // off: first robot of the range inside the context's per-robot scratch (solve records, sort keys, permutation);
    // state / actions / tgt are already offset by the caller.  Ranges start on RANK_TILE boundaries.
    float *srec = ctx->d_srec + off * SR_WORDS;
    uint8_t *key = ctx->d_key + off;
    int *perm = ctx->d_perm + off;
    const bool boxes = ctx->dc.link_contacts != 0;
    float *srx = boxes ? ctx->d_srx + off * XR_WORDS : nullptr;
    int *xg = boxes ? ctx->d_xgroups + off / RANK_TILE : nullptr;
    // persistent sole manifolds: the snapshot robot keeps its own behind its record
    float *man = !ctx->d_man ? nullptr : (state == ctx->d_snapshot ? ctx->d_snapshot + PLEN_SNAP_MAN : ctx->d_man + off * PLEN_MAN_WORDS);
    // per-robot scales and mass rows: never for the snapshot robot, which is settled under the nominal parameters
    const bool snap = state == ctx->d_snapshot;
    const float *scale = (snap || !ctx->d_scale) ? nullptr : ctx->d_scale + 4 * off;
    const float *mrow = (snap || !ctx->d_mass) ? nullptr : ctx->d_mass + MR_WORDS * off;
    // command latency: env steps only (agent actions); plen_tick and the snapshot settle run raw physics without it
    float *lat = (snap || !actions || !ctx->d_lat) ? nullptr : ctx->d_lat + LAT_WORDS * off;
    for (int t = 0; t < n_ticks; t++) {
        if (ev) cudaEventRecord(ev[2 * t], st);
        launch_dyn(ctx, state, n, t == 0 ? actions : nullptr, tgt, srec, key, nullptr, nullptr, nullptr, scale, srx, man, mrow, lat, t, st);
        if (ev) cudaEventRecord(ev[2 * t + 1], st);
        const int nt = rank_tiles(n);
        k_rank<<<nt, RANK_TILE, 0, st>>>(key, n, perm, xg);
        const int ng = nt * (RANK_TILE / PLEN_SOLVE_ROBOTS);
        if (!boxes) {
            k_solve<false><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, srec, perm, state, n, nt, nullptr, nullptr, key);
        } else if (n > ctx->merge_max) {
            // (k_solve_x on a side stream next to k_solve, fork / join per tick, was measured 1.4 % SLOWER at 131,072 robots
            // than running it behind k_solve -- r2_ab2: its few long warps take SM slots from the main launch early)
            k_solve<false><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, srec, perm, state, n, nt, xg, srx, key);
            k_solve_x<<<nt * XS_SPLIT, 32, SOLVE_X_SMEM, st>>>(ctx->dc, srec, srx, key, perm, state, n, nt, xg);
            ctx->launches += 1;
        } else {
            k_solve<true><<<ng, 32, SOLVE_SMEM, st>>>(ctx->dc, srec, perm, state, n, nt, xg, srx, key);
        }
        ctx->launches += 3;
    }
}

// One env step of robots [off, off + cnt) on stream st (all pointers are whole-batch base pointers)
static void launch_step_range(plen_ctx *ctx, size_t off, int cnt, const float *actions_dev, float *obs_dev, float *reward_dev,
                              uint8_t *done_dev, uint8_t *timeout_dev, float *terminal_obs_dev, cudaStream_t st, cudaEvent_t *ev, int nev) {
    float *state = ctx->d_state + off * PLEN_STATE_WORDS;
    launch_ticks(ctx, state, cnt, actions_dev + off * PLEN_NJ, ctx->d_tgt + off * PLEN_NJ, ctx->cfg.substeps, st, ev, off);
    if (ev) cudaEventRecord(ev[nev - 2], st);
    k_post<<<dyn_grid(cnt), DYN_WPC * 32, DYN_SMEM, st>>>(ctx->dc, ctx->d_tab, state, cnt, obs_dev + off * PLEN_OBS, reward_dev + off,
                                                         done_dev + off, timeout_dev ? timeout_dev + off : nullptr,
                                                         terminal_obs_dev ? terminal_obs_dev + off * PLEN_OBS : nullptr, ctx->d_snapshot,
                                                         ctx->d_faults, ctx->d_man ? ctx->d_man + off * PLEN_MAN_WORDS : nullptr);
    ctx->launches += 1;
    if (ev) cudaEventRecord(ev[nev - 1], st);
}

// Remember the last work queued on a caller stream so that plen_step_host (private streams) can order itself after it.
// A capturing stream is left alone: an event recorded into a graph cannot be waited for from outside the capture.
static cudaError_t mark_work(plen_ctx *ctx, cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaError_t e = cudaStreamIsCapturing(st, &cs);
    if (e != cudaSuccess) return e;
    if (cs != cudaStreamCaptureStatusNone) return cudaSuccess;
    return cudaEventRecord(ctx->last_work, st);
}

extern "C" {

const char *plen_version(void) { return "plen_b200 0.3 (sm_100a)"; }

int plen_default_config(plen_config *cfg, int joint_act) {
    if (!cfg) return fail(nullptr, PLEN_E_ARG, "cfg is NULL");
    return default_config(cfg, joint_act);
}

const char *plen_last_error(const plen_ctx *ctx) { return ctx ? ctx->err : g_err; }
int plen_num_envs(const plen_ctx *ctx) { return ctx ? ctx->n : 0; }
unsigned long long plen_kernel_launches(const plen_ctx *ctx) { return ctx ? ctx->launches : 0; }

void plen_destroy(plen_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaFree(ctx->d_tab); cudaFree(ctx->d_state); cudaFree(ctx->d_snapshot); cudaFree(ctx->d_srec); cudaFree(ctx->d_srx); cudaFree(ctx->d_xgroups); cudaFree(ctx->d_tgt); cudaFree(ctx->d_key); cudaFree(ctx->d_perm); cudaFree(ctx->d_scale); cudaFree(ctx->d_mass); cudaFree(ctx->d_lat); cudaFree(ctx->d_man); cudaFree(ctx->d_hull);
    cudaFree(ctx->d_act); cudaFree(ctx->d_obs); cudaFree(ctx->d_rew); cudaFree(ctx->d_done); cudaFree(ctx->d_tmo); cudaFree(ctx->d_faults);
    for (int k = 1; k < PLEN_HOST_PIPE; k++)
        if (ctx->pipe[k]) cudaStreamDestroy(ctx->pipe[k]);
    if (ctx->fan_fork) cudaEventDestroy(ctx->fan_fork);
    if (ctx->last_work) cudaEventDestroy(ctx->last_work);
    for (int k = 0; k < PLEN_HOST_PIPE; k++)
        if (ctx->fan_join[k]) cudaEventDestroy(ctx->fan_join[k]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->prof_ev) {
        for (int i = 0; i < ctx->prof_cap * (2 * ctx->cfg.substeps + 2); i++) cudaEventDestroy(ctx->prof_ev[i]);
        free(ctx->prof_ev);
    }
    delete ctx;
}

static int create_impl(plen_ctx *ctx) {
    const int n = ctx->n;
    ctx->merge_max = getenv("PLEN_MERGE_MAX") ? atoi(getenv("PLEN_MERGE_MAX")) : PLEN_MERGE_MAX;
    ctx->host_ranges = getenv("PLEN_HOST_RANGES") ? atoi(getenv("PLEN_HOST_RANGES")) : 0;      // dev knob: ranges of plen_step_host (0 = by size)
    ctx->host_nw = 0;
    if (const char *sp = getenv("PLEN_HOST_SPLIT")) {       // dev knob: relative sizes of the ranges of plen_step_host
        while (*sp && ctx->host_nw < 2 * PLEN_HOST_PIPE) {
            const int w = atoi(sp);
            if (w > 0) ctx->host_w[ctx->host_nw++] = w;
            while (*sp && *sp != ',') sp++;
            if (*sp == ',') sp++;
        }
    }
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaFuncSetAttribute(k_dyn<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DYN_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_dyn<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DYN_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_post, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DYN_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_observe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DYN_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_solve<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SOLVE_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_solve<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SOLVE_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_solve_x, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SOLVE_X_SMEM));
    CK(ctx, cudaFuncSetAttribute(k_solve<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(ctx, cudaFuncSetAttribute(k_solve_x, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    // both hot kernels are occupancy-limited by shared memory: ask for the largest carve-out (7 k_solve CTAs per SM)
    CK(ctx, cudaFuncSetAttribute(k_solve<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(ctx, cudaFuncSetAttribute(k_dyn<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(ctx, cudaFuncSetAttribute(k_dyn<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->pipe[0] = ctx->stream;
    for (int k = 1; k < PLEN_HOST_PIPE; k++) CK(ctx, cudaStreamCreateWithFlags(&ctx->pipe[k], cudaStreamNonBlocking));
    CK(ctx, cudaEventCreateWithFlags(&ctx->fan_fork, cudaEventDisableTiming));
    CK(ctx, cudaEventCreateWithFlags(&ctx->last_work, cudaEventDisableTiming));
    for (int k = 0; k < PLEN_HOST_PIPE; k++) CK(ctx, cudaEventCreateWithFlags(&ctx->fan_join[k], cudaEventDisableTiming));
    float tab[T_ROWS * 32], rec[PLEN_STATE_WORDS];
    build_table(&ctx->model, &ctx->cfg, tab);
    build_devconfig(&ctx->model, &ctx->cfg, &ctx->dc, &ctx->er);
    CK(ctx, cudaMalloc(&ctx->d_tab, sizeof tab));
    CK(ctx, cudaMalloc(&ctx->d_state, sizeof(float) * PLEN_STATE_WORDS * (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_snapshot, sizeof(float) * PLEN_SNAP_WORDS));
    CK(ctx, cudaMemset(ctx->d_snapshot, 0, sizeof(float) * PLEN_SNAP_WORDS));
    if (ctx->dc.sole_manifold) {
        CK(ctx, cudaMalloc(&ctx->d_man, sizeof(float) * PLEN_MAN_WORDS * (size_t)n));
        CK(ctx, cudaMalloc(&ctx->d_hull, sizeof(float) * 2 * PLEN_MAX_HULL * 3));
        CK(ctx, cudaMemcpy(ctx->d_hull, ctx->model.foot_hull, sizeof(float) * 2 * PLEN_MAX_HULL * 3, cudaMemcpyHostToDevice));
        ctx->dc.hull = ctx->d_hull;
    }
    CK(ctx, cudaMalloc(&ctx->d_srec, sizeof(float) * SR_WORDS * (size_t)n));
    if (ctx->dc.link_contacts) {
        CK(ctx, cudaMalloc(&ctx->d_srx, sizeof(float) * XR_WORDS * ((size_t)n + 1)));      // + 1: the snapshot robot's record
        CK(ctx, cudaMalloc(&ctx->d_xgroups, sizeof(int) * ((size_t)rank_tiles(n) + 1)));
    }
    CK(ctx, cudaMalloc(&ctx->d_tgt, sizeof(float) * PLEN_NJ * (size_t)n));
    // the reset-pose hold target until the first step: plen_set_env_latency seeds the command history from these
    CK(ctx, cudaMemset(ctx->d_tgt, 0, sizeof(float) * PLEN_NJ * (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_key, (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_perm, sizeof(int) * (size_t)rank_tiles(n) * RANK_TILE));
    CK(ctx, cudaMalloc(&ctx->d_scale, sizeof(float) * 4 * (size_t)n));
    k_set_scales<<<(n + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_scale, n, nullptr, nullptr, nullptr, 1);
    CK(ctx, cudaMalloc(&ctx->d_act, sizeof(float) * PLEN_NJ * (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_obs, sizeof(float) * PLEN_OBS * (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_rew, sizeof(float) * (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_done, (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_tmo, (size_t)n));
    CK(ctx, cudaMalloc(&ctx->d_faults, sizeof(unsigned long long)));
    CK(ctx, cudaMemset(ctx->d_faults, 0, sizeof(unsigned long long)));
    CK(ctx, cudaMemcpy(ctx->d_tab, tab, sizeof tab, cudaMemcpyHostToDevice));
    // post-reset snapshot: teleport to the start pose, zero joints and targets, settle for reset_ticks (plen_env.py:561-574)
    init_record(&ctx->cfg, rec);
    CK(ctx, cudaMemcpy(ctx->d_snapshot, rec, sizeof rec, cudaMemcpyHostToDevice));
    launch_ticks(ctx, ctx->d_snapshot, 1, nullptr, nullptr, ctx->cfg.reset_ticks, ctx->stream);
    k_observe<<<1, 32, DYN_SMEM, ctx->stream>>>(ctx->d_snapshot, 1, ctx->d_snapshot + PLEN_STATE_WORDS);
    k_reset<<<(n * 32 + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_state, n, nullptr, ctx->d_snapshot, nullptr, ctx->d_man);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return PLEN_OK;
}

plen_ctx *plen_create(const plen_config *cfg, const plen_model *model, int n_envs, int device) {
    if (!cfg || !model || n_envs <= 0) { fail(nullptr, PLEN_E_ARG, "plen_create: bad arguments"); return nullptr; }
    if (cfg->sole_manifold && (model->n_hull[0] <= 0 || model->n_hull[1] <= 0 || model->n_hull[0] > PLEN_MAX_HULL ||
                               model->n_hull[1] > PLEN_MAX_HULL || !(cfg->support_tie >= 0.0f))) {
        fail(nullptr, PLEN_E_ARG, "plen_create: sole_manifold = 1 needs 1..%d hull vertices per foot in the model (got %d, %d) and "
                                  "support_tie >= 0", PLEN_MAX_HULL, model->n_hull[0], model->n_hull[1]);
        return nullptr;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        fail(nullptr, PLEN_E_CUDA, "plen_create: no usable CUDA device %d (%s); this library has no CPU fallback", device,
             e == cudaSuccess ? "device count 0 or index out of range" : cudaGetErrorString(e));
        return nullptr;
    }
    plen_ctx *ctx = new (std::nothrow) plen_ctx();
    if (!ctx) { fail(nullptr, PLEN_E_ARG, "out of host memory"); return nullptr; }
    memset(ctx, 0, sizeof *ctx);
    ctx->n = n_envs; ctx->device = device; ctx->cfg = *cfg; ctx->model = *model;
    ctx->sm_count = 148;
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (ctx->sm_count <= 0) ctx->sm_count = 148;
    if (create_impl(ctx) != PLEN_OK) {
        snprintf(g_err, sizeof g_err, "%s", ctx->err);
        plen_destroy(ctx);
        return nullptr;
    }
    return ctx;
}

int plen_reset(plen_ctx *ctx, const uint8_t *mask_dev, float *obs_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    k_reset<<<(ctx->n * 32 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d_state, ctx->n, mask_dev, ctx->d_snapshot, obs_dev, ctx->d_man);
    ctx->launches += 1;
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_step(plen_ctx *ctx, const float *actions_dev, float *obs_dev, float *reward_dev, uint8_t *done_dev,
              uint8_t *timeout_dev, float *terminal_obs_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    if (!actions_dev || !obs_dev || !reward_dev || !done_dev) return fail(ctx, PLEN_E_ARG, "plen_step: NULL buffer");
    CK(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int nev = 2 * ctx->cfg.substeps + 2;
    cudaEvent_t *ev = (ctx->prof_ev && ctx->prof_steps < ctx->prof_cap) ? ctx->prof_ev + (size_t)nev * ctx->prof_steps : nullptr;
    if (!ev && PLEN_FAN_MAX_N > 0 && ctx->n <= PLEN_FAN_MAX_N && ctx->n >= 2 * RANK_TILE) {
        // Cut the batch into two ranges of whole sort tiles on the context's private streams: the k_dyn of one range runs
        // under the k_solve of the other and each kernel's last partial wave is filled by the other range's work (+4-6 % from
        // 8,192 to 32,768 robots, +2 % at 65,536, +0.5 % at 131,072).  Fork / join with events on the caller's stream; robots
        // are independent, so the results are bit-identical to the single-stream order.
        size_t chunk = ((size_t)ctx->n + PLEN_FAN_RANGES - 1) / PLEN_FAN_RANGES;
        chunk = (chunk + RANK_TILE - 1) / RANK_TILE * RANK_TILE;
        CK(ctx, cudaEventRecord(ctx->fan_fork, st));
        int used = 0;
        for (size_t off = 0; off < (size_t)ctx->n; off += chunk, used++) {
            const size_t cnt = ((size_t)ctx->n - off < chunk) ? (size_t)ctx->n - off : chunk;
            cudaStream_t s = ctx->pipe[used];
            CK(ctx, cudaStreamWaitEvent(s, ctx->fan_fork, 0));
            launch_step_range(ctx, off, (int)cnt, actions_dev, obs_dev, reward_dev, done_dev, timeout_dev, terminal_obs_dev, s, nullptr, 0);
            CK(ctx, cudaEventRecord(ctx->fan_join[used], s));
            CK(ctx, cudaStreamWaitEvent(st, ctx->fan_join[used], 0));
        }
    } else {
        launch_step_range(ctx, 0, ctx->n, actions_dev, obs_dev, reward_dev, done_dev, timeout_dev, terminal_obs_dev, st, ev, nev);
    }
    if (ev) ctx->prof_steps++;
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, st));
    return PLEN_OK;
}

int plen_step_host(plen_ctx *ctx, const float *actions_host, float *obs_host, float *reward_host, uint8_t *done_host,
                   uint8_t *timeout_host) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    if (!actions_host || !obs_host || !reward_host || !done_host) return fail(ctx, PLEN_E_ARG, "plen_step_host: NULL buffer");
    const size_t n = ctx->n;
    CK(ctx, cudaSetDevice(ctx->device));
    // The batch is cut into up to PLEN_HOST_PIPE ranges (multiples of the 1024-robot sort tile), each on its own stream:
    // H2D of the range's actions -> its 13 kernels -> D2H of its obs / reward / done.  Robots are independent, so the
    // copies of one range overlap the kernels of the others and only the first H2D and the last D2H stay exposed.
    // How many ranges: measured per batch size (profiles/r2_ab_runs.txt, r2_host2: 1 / 2 / 3 / 4 ranges at 4,096 ... 1,048,576
    // robots).  Small batches lose more to short grids than they gain from overlapped copies (4,096: one range +6 % over four,
    // 16,384: two +8 %); at 65,536 robots and from 262,144 on four ranges win by ~1 %, around 131,072 two ranges of 65,536 are
    // 3.6 % faster than four of 32,768 (0.9 % of it is the merged solver that ranges <= PLEN_MERGE_MAX run, the rest the
    // finer split itself: r2_merge).  More than PLEN_HOST_PIPE ranges (8, 16 at 1,048,576 robots) are never better.
    int n_ranges = ctx->host_ranges;                   // dev knob PLEN_HOST_RANGES; 0 = by size
    if (n_ranges <= 0) n_ranges = n <= 8192 ? 1 : n <= 32768 ? 2 : n <= 98304 ? 4 : n <= 196608 ? 2 : PLEN_HOST_PIPE;
    // range boundaries (multiples of the sort tile): equal parts, or the weights of the dev knob PLEN_HOST_SPLIT ("1,3,3,1")
    size_t bound[2 * PLEN_HOST_PIPE + 1];
    int nb = 0;
    bound[0] = 0;
    // large batches on four ranges: a short first range (its H2D is the exposed one) -- 1 : 2 : 3 : 2 measured 0.3-1.5 % faster
    // than equal parts from 262,144 to 1,048,576 robots (r2_host5)
    static const int big_w[4] = {1, 2, 3, 2};
    const bool weighted = ctx->host_nw > 0 || (ctx->host_ranges <= 0 && n_ranges == 4 && n > 196608);
    const int nw = ctx->host_nw > 0 ? ctx->host_nw : 4;
    const int *wts = ctx->host_nw > 0 ? ctx->host_w : big_w;
    if (weighted) {
        int wsum = 0, acc = 0;
        for (int k = 0; k < nw; k++) wsum += wts[k];
        for (int k = 0; k < nw && bound[nb] < n; k++) {
            acc += wts[k];
            size_t b = (size_t)((double)n * acc / wsum);
            b = (b + RANK_TILE - 1) / RANK_TILE * RANK_TILE;
            if (b > n || k == nw - 1) b = n;
            if (b > bound[nb]) bound[++nb] = b;
        }
    } else {
        size_t chunk = (n + n_ranges - 1) / n_ranges;
        chunk = (chunk + RANK_TILE - 1) / RANK_TILE * RANK_TILE;
        for (size_t off = 0; off < n && nb < 2 * PLEN_HOST_PIPE; off += chunk) { bound[nb + 1] = (off + chunk < n) ? off + chunk : n; nb++; }
        bound[nb] = n;
    }
    int used = 0;
    for (; used < nb; used++) {
        const size_t off = bound[used], cnt = bound[used + 1] - off;
        cudaStream_t st = ctx->pipe[used % PLEN_HOST_PIPE];
        // ordering contract (plen_b200.h): this call runs on the context's private streams, so it first waits for whatever
        // the last stream-taking entry point (reset / step / set_state / set_env_scales / set_env_mass / set_env_latency /
        // tick) queued on the caller's stream
        CK(ctx, cudaStreamWaitEvent(st, ctx->last_work, 0));
        CK(ctx, cudaMemcpyAsync(ctx->d_act + off * PLEN_NJ, actions_host + off * PLEN_NJ, sizeof(float) * PLEN_NJ * cnt,
                                cudaMemcpyHostToDevice, st));
        launch_step_range(ctx, off, (int)cnt, ctx->d_act, ctx->d_obs, ctx->d_rew, ctx->d_done, ctx->d_tmo, nullptr, st, nullptr, 0);
        CK(ctx, cudaMemcpyAsync(obs_host + off * PLEN_OBS, ctx->d_obs + off * PLEN_OBS, sizeof(float) * PLEN_OBS * cnt,
                                cudaMemcpyDeviceToHost, st));
        CK(ctx, cudaMemcpyAsync(reward_host + off, ctx->d_rew + off, sizeof(float) * cnt, cudaMemcpyDeviceToHost, st));
        CK(ctx, cudaMemcpyAsync(done_host + off, ctx->d_done + off, cnt, cudaMemcpyDeviceToHost, st));
        if (timeout_host) CK(ctx, cudaMemcpyAsync(timeout_host + off, ctx->d_tmo + off, cnt, cudaMemcpyDeviceToHost, st));
    }
    CK(ctx, cudaGetLastError());
    for (int k = 0; k < used && k < PLEN_HOST_PIPE; k++) CK(ctx, cudaStreamSynchronize(ctx->pipe[k]));
    return PLEN_OK;
}

int plen_set_env_scales(plen_ctx *ctx, const float *friction_scale_dev, const float *motor_force_scale_dev,
                        const float *motor_gain_scale_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    k_set_scales<<<(ctx->n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ctx->d_scale, ctx->n, friction_scale_dev, motor_force_scale_dev,
                                                                       motor_gain_scale_dev, 0);
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_set_env_mass(plen_ctx *ctx, const float *mass_scale_dev, const float *payload_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t words = (size_t)MR_WORDS * ctx->n;
    const int init = !ctx->d_mass;          // the rows are allocated at the first call: a context that never sets them has none
    if (init) CK(ctx, cudaMalloc(&ctx->d_mass, sizeof(float) * words));
    k_set_mass<<<(unsigned)((words + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctx->d_mass, ctx->n, mass_scale_dev, payload_dev, init);
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_get_env_mass(plen_ctx *ctx, float *mass_scale_dev, float *payload_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t words = (size_t)MR_WORDS * ctx->n;
    k_get_mass<<<(unsigned)((words + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ctx->d_mass, ctx->n, mass_scale_dev, payload_dev);
    CK(ctx, cudaGetLastError());
    return ctx->d_mass ? 1 : 0;
}

int plen_set_env_latency(plen_ctx *ctx, const int32_t *ticks_dev, const float *history_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    const int init = !ctx->d_lat;           // the ring is allocated at the first call: a context that never sets it has none
    if (init) {
        cudaError_t e = cudaMalloc(&ctx->d_lat, sizeof(float) * LAT_WORDS * (size_t)ctx->n);
        if (e != cudaSuccess) {
            ctx->d_lat = nullptr;
            return fail(ctx, PLEN_E_CUDA, "plen_set_env_latency: cudaMalloc: %s", cudaGetErrorString(e));
        }
    }
    k_set_latency<<<(ctx->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d_scale, ctx->d_lat, ctx->d_state, ctx->d_tgt, ctx->n,
                                                                        PLEN_MAX_LATENCY_STEPS * ctx->cfg.substeps, ticks_dev,
                                                                        history_dev, init);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        if (init) { cudaFree(ctx->d_lat); ctx->d_lat = nullptr; }    // an unseeded ring must never be stepped with
        return fail(ctx, PLEN_E_CUDA, "plen_set_env_latency: k_set_latency: %s", cudaGetErrorString(e));
    }
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_get_env_latency(plen_ctx *ctx, int32_t *ticks_dev, float *history_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    k_get_latency<<<(ctx->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d_scale, ctx->d_lat, ctx->d_state, ctx->d_tgt, ctx->n,
                                                                        ticks_dev, history_dev);
    CK(ctx, cudaGetLastError());
    return ctx->d_lat ? 1 : 0;
}

int plen_get_manifold(plen_ctx *ctx, float *man_dev, void *stream) {
    if (!ctx || !man_dev) return fail(ctx, PLEN_E_ARG, "plen_get_manifold: bad arguments");
    if (!ctx->d_man) return fail(ctx, PLEN_E_STATE, "plen_get_manifold: the context was created with sole_manifold = 0");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(man_dev, ctx->d_man, sizeof(float) * PLEN_MAN_WORDS * (size_t)ctx->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_set_manifold(plen_ctx *ctx, const float *man_dev, void *stream) {
    if (!ctx || !man_dev) return fail(ctx, PLEN_E_ARG, "plen_set_manifold: bad arguments");
    if (!ctx->d_man) return fail(ctx, PLEN_E_STATE, "plen_set_manifold: the context was created with sole_manifold = 0");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(ctx->d_man, man_dev, sizeof(float) * PLEN_MAN_WORDS * (size_t)ctx->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_fault_count(plen_ctx *ctx, unsigned long long *count_host) {
    if (!ctx || !count_host) return fail(ctx, PLEN_E_ARG, "plen_fault_count: bad arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaDeviceSynchronize());
    CK(ctx, cudaMemcpy(count_host, ctx->d_faults, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return PLEN_OK;
}

int plen_get_state(plen_ctx *ctx, float *qpos_dev, float *qvel_dev, float *aux_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    k_get_state<<<(ctx->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d_state, ctx->n, qpos_dev, qvel_dev, aux_dev);
    CK(ctx, cudaGetLastError());
    return PLEN_OK;
}

int plen_set_state(plen_ctx *ctx, const float *qpos_dev, const float *qvel_dev, const float *aux_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    k_set_state<<<(ctx->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d_state, ctx->n, qpos_dev, qvel_dev, aux_dev);
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_tick(plen_ctx *ctx, const float *targets_dev, int n_ticks, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    if (n_ticks < 0) return fail(ctx, PLEN_E_ARG, "plen_tick: n_ticks < 0");
    CK(ctx, cudaSetDevice(ctx->device));
    if (targets_dev)
        CK(ctx, cudaMemcpyAsync(ctx->d_tgt, targets_dev, sizeof(float) * PLEN_NJ * (size_t)ctx->n, cudaMemcpyDeviceToDevice,
                                (cudaStream_t)stream));
    launch_ticks(ctx, ctx->d_state, ctx->n, nullptr, targets_dev ? ctx->d_tgt : nullptr, n_ticks, (cudaStream_t)stream);
    CK(ctx, cudaGetLastError());
    CK(ctx, mark_work(ctx, (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_debug_dynamics(plen_ctx *ctx, float *minv_dev, float *pos_dev, float *rot_dev, void *stream) {
    if (!ctx) return fail(nullptr, PLEN_E_ARG, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    launch_dyn(ctx, ctx->d_state, ctx->n, nullptr, nullptr, ctx->d_srec, ctx->d_key, minv_dev, pos_dev, rot_dev, ctx->d_scale, ctx->d_srx,
               nullptr /* diagnostics must not advance the manifolds */, ctx->d_mass, nullptr, 0, (cudaStream_t)stream);
    CK(ctx, cudaGetLastError());
    return PLEN_OK;
}

int plen_debug_records(plen_ctx *ctx, float *records_dev, void *stream) {
    if (!ctx || !records_dev) return fail(ctx, PLEN_E_ARG, "plen_debug_records: bad arguments");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(records_dev, ctx->d_state, sizeof(float) * PLEN_STATE_WORDS * (size_t)ctx->n, cudaMemcpyDeviceToDevice,
                            (cudaStream_t)stream));
    return PLEN_OK;
}

int plen_profile_enable(plen_ctx *ctx, int max_steps) {
    if (!ctx || max_steps <= 0) return fail(ctx, PLEN_E_ARG, "plen_profile_enable: bad arguments");
    if (ctx->prof_ev) return fail(ctx, PLEN_E_STATE, "plen_profile_enable: already enabled");
    CK(ctx, cudaSetDevice(ctx->device));
    const int nev = 2 * ctx->cfg.substeps + 2;
    ctx->prof_ev = (cudaEvent_t *)calloc((size_t)max_steps * nev, sizeof(cudaEvent_t));
    if (!ctx->prof_ev) return fail(ctx, PLEN_E_ARG, "out of host memory");
    for (int i = 0; i < max_steps * nev; i++) CK(ctx, cudaEventCreate(&ctx->prof_ev[i]));
    ctx->prof_cap = max_steps;
    ctx->prof_steps = 0;
    return PLEN_OK;
}

int plen_profile_read(plen_ctx *ctx, float *ms_dyn, float *ms_solve, float *ms_post, int *steps) {
    if (!ctx || !ctx->prof_ev) return fail(ctx, PLEN_E_STATE, "plen_profile_read: profiling is not enabled");
    CK(ctx, cudaSetDevice(ctx->device));
    const int nev = 2 * ctx->cfg.substeps + 2;
    double d = 0, s = 0, p = 0;
    for (int k = 0; k < ctx->prof_steps; k++) {
        cudaEvent_t *ev = ctx->prof_ev + (size_t)nev * k;
        CK(ctx, cudaEventSynchronize(ev[nev - 1]));
        float ms;
        for (int t = 0; t < ctx->cfg.substeps; t++) {
            CK(ctx, cudaEventElapsedTime(&ms, ev[2 * t], ev[2 * t + 1])); d += ms;
            CK(ctx, cudaEventElapsedTime(&ms, ev[2 * t + 1], ev[2 * t + 2])); s += ms;
        }
        CK(ctx, cudaEventElapsedTime(&ms, ev[nev - 2], ev[nev - 1])); p += ms;
    }
    if (ms_dyn) *ms_dyn = (float)d;
    if (ms_solve) *ms_solve = (float)s;
    if (ms_post) *ms_post = (float)p;
    if (steps) *steps = ctx->prof_steps;
    ctx->prof_steps = 0;
    return PLEN_OK;
}

int plen_gait_ik(int device, const double *params_dev, int n_gaits, double *traj_dev, double *bend_dev,
                 uint8_t *status_dev, void *stream) {
    if (!params_dev || !traj_dev || n_gaits <= 0) return fail(nullptr, PLEN_E_ARG, "plen_gait_ik: bad arguments");
    CK(nullptr, cudaSetDevice(device));
    k_gait_ik<<<(n_gaits + 127) / 128, 128, 0, (cudaStream_t)stream>>>(params_dev, n_gaits, traj_dev, bend_dev, status_dev);
    CK(nullptr, cudaGetLastError());
    return PLEN_OK;
}

int plen_measure_fp32_peak(int device, int mode, float *tflops, float *sm_mhz_hint) {
    if (!tflops || mode < 0 || mode > 1) return fail(nullptr, PLEN_E_ARG, "plen_measure_fp32_peak: bad arguments");
    CK(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(nullptr, cudaGetDeviceProperties(&prop, device));
    float *d_out = nullptr;
    CK(nullptr, cudaMalloc(&d_out, sizeof(float)));
    cudaEvent_t e0, e1;
    CK(nullptr, cudaEventCreate(&e0));
    CK(nullptr, cudaEventCreate(&e1));
    const int grid = prop.multiProcessorCount * 8, block = 256, iters = 4096;
    float best = 0.0f;
    for (int rep = 0; rep < 6; rep++) {        // first repetitions warm the clocks up; best of the rest
        CK(nullptr, cudaEventRecord(e0, 0));
        k_fp32_peak<<<grid, block>>>(d_out, iters, mode, 0.0f);
        CK(nullptr, cudaEventRecord(e1, 0));
        CK(nullptr, cudaEventSynchronize(e1));
        float ms = 0.0f;
        CK(nullptr, cudaEventElapsedTime(&ms, e0, e1));
        const double flop = 2.0 * 8.0 * 16.0 * (double)iters * (double)grid * (double)block;
        const float tf = (float)(flop / (ms * 1e-3) / 1e12);
        if (rep >= 2 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d_out);
    *tflops = best;
    if (sm_mhz_hint) *sm_mhz_hint = best * 1e12f / (2.0f * 128.0f * (float)prop.multiProcessorCount) / 1e6f;   // clock implied by 128 lanes/SM
    return PLEN_OK;
}

}  // extern "C"
