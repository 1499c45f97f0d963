// plen_device.cuh -- warp-per-robot PLEN dynamics: first half of a physics tick (k_dyn) (sm_100a device code).
//
// One warp owns one robot.  Lane l < 24 owns generalized velocity l (0..2 omega_world, 3..5 v_world, 6..23 joints);
// lane l >= 6 also owns body l-5 / joint l-6 (limb chains at lanes 6..11, 12..17, 18..20, 21..23); lanes 24..31
// own the 8 cached contact impulses.  Tree traversals become segmented warp scans over the limb chains.
//
// Per tick (replaces p.stepSimulation, plen_env.py:665-667; algorithm is ours, not Bullet's):
//   1. FK: local joint transforms -> prefix product along each chain -> world frames (origin = base position)
//   2. world-frame composite-rigid-body mass matrix M (suffix sums of 10-parameter inertias) and bias forces C
//      (prefix sums of twists / accelerations, suffix sums of body forces)
//   3. M^-1 by block elimination: 4 limb blocks inverted in parallel (Gauss-Jordan across lanes), 6x6 base Schur
//      complement inverted redundantly, M^-1 assembled column-major in shared memory
//   4. v* = v - dt M^-1 C;  sole-vertex contacts vs z = 0;  Y = M^-1 Jfoot^T and Lambda^-1 = Jfoot M^-1 Jfoot^T
//   5. the SOLVE RECORD: G = [M^-1_jj Y; Y^T Lambda^-1] and the scalars of every constraint row (limits, 18 servo rows,
//      per contact normal + spin + 2 roll + 2 lateral); flat ground => every contact row is a functional of the foot
//      twist with <= 3 non-zeros, so no per-row Jacobian storage exists at all
// plen_solve.cuh (k_solve) then runs the projected Gauss-Seidel, applies delta-v and integrates.
//
// The same source is compiled for the host by tests/emu (32 threads + barriers emulate the warp shuffles) so the
// CPU test suite can check this code against the float64 oracle without a GPU.  That emulation is test-only; the
// product library has no CPU path.
#pragma once

#include <math.h>
#include <stdint.h>

#include "../../include/plen_b200.h"

#ifndef PLEN_HOST_EMU
#define PLEN_DEV __device__ __forceinline__
#define PLEN_DEV_NOINLINE __device__ __noinline__
namespace plen {
PLEN_DEV int lane_id() { return threadIdx.x & 31; }
PLEN_DEV float shfl(float v, int src) { return __shfl_sync(0xffffffffu, v, src); }
// broadcast inside every aligned group of four lanes (src = 0..3): the source is an immediate of the SHFL, no lane arithmetic
PLEN_DEV float shfl4(float v, int src) { return __shfl_sync(0xffffffffu, v, src, 4); }
PLEN_DEV float shfl_up(float v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
PLEN_DEV float shfl_down(float v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
PLEN_DEV float shfl_xor(float v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
PLEN_DEV unsigned ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
PLEN_DEV unsigned redux_max(unsigned v) { return __reduce_max_sync(0xffffffffu, v); }
PLEN_DEV unsigned redux_or(unsigned v) { return __reduce_or_sync(0xffffffffu, v); }
PLEN_DEV void warp_sync() { __syncwarp(); }
PLEN_DEV float f_as_u_max(float v) { return __uint_as_float(redux_max(__float_as_uint(v))); }
PLEN_DEV void sincos_(float x, float *s, float *c) { sincosf(x, s, c); }
#ifndef PLEN_FAST_RCP
#define PLEN_FAST_RCP 1
#endif
// 1 / x as one MUFU.RCP (rcp.approx.ftz, <= 1 ulp: the same order as any fp32 rounding on this path) instead of the IEEE
// division, whose denormal / special-case slow path puts a CALL behind each of the ~20 reciprocals of a tick: -2 % of the
// step (PLEN_FAST_RCP = 0 restores the division)
PLEN_DEV float rcp_(float x) {
#if PLEN_FAST_RCP
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}
PLEN_DEV unsigned f_bits(float v) { return __float_as_uint(v); }
PLEN_DEV int lowest_bit(unsigned m) { return __ffs((int)m) - 1; }
PLEN_DEV int highest_bit(unsigned m) { return 31 - __clz((int)m); }
PLEN_DEV int popc_(unsigned m) { return __popc(m); }
}  // namespace plen
#endif

namespace plen {

// ---- model table rows (each row is 32 floats, one per lane), staged in shared memory per CTA
enum {
    T_RPJ = 0, T_PPJ = 9, T_AXIS = 12, T_COM = 15, T_MASS = 18, T_INERTIA = 19, T_LOWER = 25, T_UPPER = 26,
    T_CS = 27, T_CE = 28, T_ENVLO = 29, T_ENVHI = 30,
    // box collider b of the model in word b of a row (lane b tests box b against the ground): owning body lane, centre (3),
    // rotation (9, row major) and half extents (3) in the body frame, restitution factor
    T_BOX_LANE = 31, T_BOX_C = 32, T_BOX_R = 35, T_BOX_H = 44, T_BOX_REST = 47, T_ROWS = 48
};

// ---- per-env state record in HBM / smem: 96 words, word w = 32*k + lane
enum {
    W_U = 0,        // words 0..23: generalized velocity; 24..31: cached normal impulses lam_n[8]
    W_Q = 32,       // words 38..55: joint angles (lane 6..23)
    W_POS = 32,     // words 32..34: base position
    W_MAN = 35,     // manifold bits (int)
    W_EPRET = 36,   // episode return
    W_QUAT = 56,    // words 56..59: base quaternion xyzw
    W_CNT = 60, W_DS = 61, W_HIST = 62, W_EPT = 63,   // ints
    W_LAST = 64,    // 6
    W_SUMS = 70,    // 9
    W_ITERS = 79,   // PGS iterations of the last tick (diagnostic)
    W_SPARE = 80
};

struct DevConfig {
    float dt, inv_dt, gravity_z, motor_imp, kp_over_dt, one_minus_kd, linear_damping;
    float mu_lateral, mu_spinning, mu_rolling, restitution, rest_thresh, erp_contact_over_dt, erp_joint_over_dt;
    float linear_slop, warm, hull_margin, vmax, residual_threshold, mu_link;
    float foot_break[2];
    float foot_pts[2][4][3];
    float start_pos[3];
    int foot_lane[2];
    int substeps, reset_ticks, iterations, joint_act, max_episode_steps, auto_reset, link_contacts, n_boxes;
    // persistent sole manifold (plen_config.sole_manifold): hull vertices [2][PLEN_MAX_HULL][3] of the feet (device memory; the
    // warp-emulation harness points it at host memory), their counts
    int sole_manifold, n_hull[2];
    const float *hull;
    float support_tie;
};

// ---- solve record: per robot, per tick, written by k_dyn and consumed by k_solve (global memory, words)
// operational-space index i of x (32 slots): 0..17 joints, 18..23 right-foot twist, 24..25 unused, 26..31 left-foot twist;
// word i of a 32-word row holds entry i, so solver lane g = i >> 3 (four lanes per robot) owns entries 8 g .. 8 g + 7 and
// each foot's twist lives in ONE lane (lane 2: right, lane 3: left; component c at slot 2 + c of either).
// Servo / limit rows are kept in VELOCITY units (impulse times G_jj): joint columns of G and B are pre-divided by G_jj, so
// the row update needs no per-row multiply and its velocity change (the residual term) is the broadcast value itself.
enum {
    SR_G = 0,          // 30 columns (18 joints, 6 right-foot, 6 left-foot components) x 32 words (rows i) of G
    SR_B = 960,        // 6 rows x 32 words: base rows of M^-1 J^T in the same word order
    SR_MRHS = 1152, SR_MD = 1184, SR_LDIR = 1216, SR_LRHS = 1248, SR_VSTAR = 1280, SR_Q = 1312,   // 32 words each
    SR_CRHS = 1344, SR_CDINV = 1408, SR_CD = 1472,   // 64 words each: [contact slot q = 4 foot + k][solver lane g]
    SR_PT = 1536,      // 8 x (x, y, z, distance): k-th ACTIVE contact point of each foot, relative to the base origin
    SR_LAMC = 1568,    // 8 cached normal impulses, same slot order
    SR_BASE = 1576,    // v* of the base (6), base position (3), quaternion (4), manifold bits (1), friction / servo-force scale (2)
    SR_WORDS = 1600
};

// ---- extension record: per robot, per tick, written by k_dyn only for a robot whose link boxes touch the ground and read by
// the EXT instance of k_solve.  Up to PLEN_MAX_BOX_POINTS contact points (the deepest), three rows each (normal, lateral t1,
// lateral t2), every row as explicit vectors in the operational space x of the solve record:
//   Jx (32)  row velocity = Jx . x        Bx (32)  x += Bx * impulse        Bb (6)  base delta-v = Bb * impulse
// (a box sits on an arbitrary body, whose twist is NOT a slot of x; but the base twist is the right-foot twist minus the
// right leg's joint motion, so any body twist -- and with it any row -- is a linear functional of x: see box_rows below).
enum {
    XR_NX = 0,           // number of points (float)
    XR_ROWS = 16,        // row (3 q + r) at XR_ROWS + (3 q + r) * XR_ROW_WORDS
    XR_J = 0, XR_B = 32, XR_BB = 64, XR_RHS = 70, XR_DINV = 71, XR_D = 72, XR_ROW_WORDS = 80,
    XR_WORDS = XR_ROWS + 3 * PLEN_MAX_BOX_POINTS * XR_ROW_WORDS
};
// sort keys of a robot with nx = 1 .. PLEN_MAX_BOX_POINTS box contact points: PLEN_KEY_EXT + nx - 1, above every foot-only key
// (<= 124), so these robots lead every tile of k_rank, those with the most points first (a solver warp loops to the largest
// point count of its eight robots)
#define PLEN_KEY_EXT 125

// index (0..3) of the k-th set bit of a 4-bit mask, -1 if there are fewer
PLEN_DEV int nth_bit4(unsigned m, int k) {
    int r = -1, c = 0;
#pragma unroll
    for (int b = 0; b < 4; b++) {
        const bool on = (m >> b) & 1u;
        r = (on && c == k) ? b : r;
        c += on ? 1 : 0;
    }
    return r;
}

#ifndef PLEN_HOST_EMU
struct __align__(16) vec4 { float x, y, z, w; };
struct __align__(8) vec2 { float x, y; };
#define PLEN_ALIGN16 __align__(16)
#else
struct vec4 { float x, y, z, w; };
struct vec2 { float x, y; };
#define PLEN_ALIGN16
#endif

// Loads of data another kernel of the step produced (state records, solve records, targets, permutation, sort keys) go
// through plain coherent ld.global, never the non-coherent read-only path (LDG.E.CONSTANT) that `const __restrict__`
// pointers invite: plen_step_host runs ranges of the batch on several streams, so kernels of different ranges share an SM
// and its L1 while these buffers are rewritten tick after tick.  (ld.global.cg -- L2 only -- was measured 6 % slower.)
#ifndef PLEN_HOST_EMU
PLEN_DEV float gld(const float *p) {
    float v;
    asm("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
PLEN_DEV vec4 gld4(const float *p) {
    vec4 r;
    asm("ld.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
PLEN_DEV int gld_i(const int *p) {
    int v;
    asm("ld.global.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
PLEN_DEV int gld_u8(const uint8_t *p) {
    unsigned v;
    asm("ld.global.u8 %0, [%1];" : "=r"(v) : "l"(p));
    return (int)v;
}
#else
PLEN_DEV float gld(const float *p) { return *p; }
PLEN_DEV vec4 gld4(const float *p) { return *reinterpret_cast<const vec4 *>(p); }
PLEN_DEV int gld_i(const int *p) { return *p; }
PLEN_DEV int gld_u8(const uint8_t *p) { return *p; }
#endif

// six consecutive floats of a 32-byte-aligned row (tw / kk / gg rows of WarpScratch) as LDS.128 + LDS.64
PLEN_DEV void load6(const float *row, float (&o)[6]) {
    const vec4 a = *reinterpret_cast<const vec4 *>(row);
    const vec2 b = *reinterpret_cast<const vec2 *>(row + 4);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y;
}
// ... and the store: STS.128 + STS.64
PLEN_DEV void store6(float *row, float v0, float v1, float v2, float v3, float v4, float v5) {
    vec4 a; a.x = v0; a.y = v1; a.z = v2; a.w = v3;
    vec2 b; b.x = v4; b.y = v5;
    *reinterpret_cast<vec4 *>(row) = a;
    *reinterpret_cast<vec2 *>(row + 4) = b;
}

// per-warp shared scratch of k_dyn (floats); 16-byte aligned so that the 8-float rows can be read as vectors
struct PLEN_ALIGN16 WarpScratch {
    float st[96];
    float tw[24][8];      // joint twists s_j = [a(3), m(3)] about the base origin, world axes
    float kk[24][8];      // K rows = A_c M_c0, later Y_right = M^-1 Jfoot_right^T
    float gg[24][8];      // G rows = K S^-1, later Y_left
    float cb[32];         // bias forces C
    float minv[24][32];   // M^-1, [column j][lane l]
    float cp[8][4];       // contact point x,y,z (rel. base origin, on the inflated hull) and distance
    union {
        float lin[12][12];    // operational inverse inertia of the two feet, Lambda^-1 = Jfoot M^-1 Jfoot^T
        float red[32 * 21];   // Schur complement partial products (dead before lin is built)
    };
    float obs[32];
    float xp[PLEN_MAX_BOX_POINTS][8];   // selected box contact points: x y z (rel. base origin), depth, body lane, restitution factor
    float mn[2][28];      // sole_manifold: per foot local xyz of 4 points | plane xyz of 4 points | count | 3 spare
    float mlam[8];        // ... and the cached normal impulses of the 2 x 4 slots while the manifolds are updated
};

struct LaneState {
    float u;          // generalized velocity of this lane (0 for lanes >= 24)
    float q;          // joint angle (lanes 6..23)
    float tgt;        // servo target (lanes 6..23)
    float lam;        // cached normal impulse (lanes 24..31)
    float pos[3];     // base position (uniform)
    float quat[4];    // base orientation xyzw (uniform)
    unsigned man;     // manifold bits (uniform)
    int iters;        // PGS iterations of the last tick (diagnostic, uniform)
    float fric_s, motor_s, kp_s;   // per-robot scales of the friction coefficients, the servo force limit and the servo
                                   // gain (domain randomisation, plen_set_env_scales; 1 = the reference's constants)
    float mass_w;     // word `lane` of the robot's mass row (plen_set_env_mass; read by the MASS instance of tick_dynamics
                      // only): the mass scale of this lane's body (lanes 0, 6..23), the torso payload (lanes 24..27: m, x, y, z)
};

// per-robot mass row (plen_set_env_mass): 32 words, one per lane, so that a warp reads it with one 128-byte load
enum { MR_PAYLOAD = 24, MR_WORDS = 32 };

// per-robot command latency (plen_set_env_latency): the delay d in ticks is word SC_LATENCY of the robot's scale row (d_scale,
// [n][4], loaded by k_dyn anyway; plen_set_env_scales never writes that word), kept as a float holding an integer.  The
// command history is a ring of LAT_SLOTS 128-byte rows per robot ([n][LAT_WORDS]): the raw servo targets of the step whose
// episode counter is e sit in row e mod LAT_SLOTS, lanes 6..23 (the other lanes are unused).  Tick 0 of a step writes its
// row while the rows of the two steps before stay readable, so no row is ever copied.
enum { SC_LATENCY = 3, LAT_SLOTS = 3, LAT_WORDS = LAT_SLOTS * 32 };

PLEN_DEV void mat3_mul(const float *A, const float *B, float *C) {
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}
PLEN_DEV void mat3_vec(const float *A, const float *v, float *o) {
    o[0] = A[0] * v[0] + A[1] * v[1] + A[2] * v[2];
    o[1] = A[3] * v[0] + A[4] * v[1] + A[5] * v[2];
    o[2] = A[6] * v[0] + A[7] * v[1] + A[8] * v[2];
}
PLEN_DEV void cross(const float *a, const float *b, float *o) {
    o[0] = a[1] * b[2] - a[2] * b[1];
    o[1] = a[2] * b[0] - a[0] * b[2];
    o[2] = a[0] * b[1] - a[1] * b[0];
}
PLEN_DEV void quat_to_mat(const float *q, float *R) {
    const float x = q[0], y = q[1], z = q[2], w = q[3];
    R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
    R[3] = 2 * (x * y + w * z); R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - w * x);
    R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = 1 - 2 * (x * x + y * y);
}
PLEN_DEV float warp_sum(float v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += shfl_xor(v, m);
    return v;
}
PLEN_DEV void warp_sum2(float &a, float &b) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) { a += shfl_xor(a, m); b += shfl_xor(b, m); }
}

// Forward kinematics of the 19 body frames.  Outputs for this lane: Rw (world rotation), pw (frame origin relative
// to the base origin, world axes).  Lanes without a body (1..5, 24..31) get the base frame.
PLEN_DEV void forward_kinematics(const float *tab, int lane, float q, const float *quat, float *Rw, float *pw) {
    float R[9], p[3];
    {
        float s, c;
        sincos_(q, &s, &c);
        const float ax = tab[(T_AXIS + 0) * 32 + lane], ay = tab[(T_AXIS + 1) * 32 + lane], az = tab[(T_AXIS + 2) * 32 + lane];
        const float t = 1.0f - c;
        float Rq[9] = {t * ax * ax + c, t * ax * ay - s * az, t * ax * az + s * ay,
                       t * ax * ay + s * az, t * ay * ay + c, t * ay * az - s * ax,
                       t * ax * az - s * ay, t * ay * az + s * ax, t * az * az + c};
        float Rpj[9];
#pragma unroll
        for (int k = 0; k < 9; k++) Rpj[k] = tab[(T_RPJ + k) * 32 + lane];
        mat3_mul(Rpj, Rq, R);
#pragma unroll
        for (int k = 0; k < 3; k++) p[k] = tab[(T_PPJ + k) * 32 + lane];
    }
    const int cs = (int)tab[T_CS * 32 + lane];
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
        float Rp[9], pp[3];
#pragma unroll
        for (int k = 0; k < 9; k++) Rp[k] = shfl_up(R[k], d);
#pragma unroll
        for (int k = 0; k < 3; k++) pp[k] = shfl_up(p[k], d);
        if (lane - d >= cs) {
            float t[3], Rn[9];
            mat3_vec(Rp, p, t);
            p[0] = pp[0] + t[0]; p[1] = pp[1] + t[1]; p[2] = pp[2] + t[2];
            mat3_mul(Rp, R, Rn);
#pragma unroll
            for (int k = 0; k < 9; k++) R[k] = Rn[k];
        }
    }
    float R0[9];
    quat_to_mat(quat, R0);
    mat3_mul(R0, R, Rw);
    mat3_vec(R0, p, pw);
}

PLEN_DEV float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

// Contact-row Jacobian entry J and response entry B of this lane for row `type` of a contact at p (rel. base origin).
// a/m: this lane's twist masked to {base, the foot's leg}; Y: this lane's row of M^-1 Jfoot^T.
// Normal n = +z, tangents t1 = (0,-1,0), t2 = (1,0,0) (btPlaneSpace1 of +z).
PLEN_DEV void row_entries(int type, const float *a, const float *m, const float *Y, float px, float py, float pz,
                          float &J, float &B) {
    switch (type) {
        case 0: J = a[0] * py - a[1] * px + m[2]; B = Y[0] * py - Y[1] * px + Y[5]; break;          // normal
        case 1: J = a[2]; B = Y[2]; break;                                                           // spin about n
        case 2: J = -a[1]; B = -Y[1]; break;                                                         // roll about t1
        case 3: J = a[0]; B = Y[0]; break;                                                           // roll about t2
        case 4: J = a[0] * pz - a[2] * px - m[1]; B = Y[0] * pz - Y[2] * px - Y[4]; break;           // lateral t1
        default: J = a[1] * pz - a[2] * py + m[0]; B = Y[1] * pz - Y[2] * py + Y[3]; break;          // lateral t2
    }
}

// First half of a physics tick for the robot owned by this warp: dynamics + constraint set-up (k_dyn).
struct DebugOut { float *minv, *pos, *rot; };   // [24*24], [24*3], [24*9] of one env; all nullable

PLEN_DEV_NOINLINE void box_rows(const DevConfig &cfg, const float *tab, WarpScratch &ws, int lane, float vstar, int nx, float *srx);
PLEN_DEV_NOINLINE int box_points(const DevConfig &cfg, const float *tab, WarpScratch &ws, int lane, bool touch, float cz, float rz0,
                                 float rz1, float rz2, int bl, float R0, float R1, float R2, float R3, float R4, float R5, float R6,
                                 float R7, float R8, float p0, float p1, float p2);

PLEN_DEV_NOINLINE void manifold_merge(const DevConfig &cfg, float *mn, float *lam, const float *Rf, const float *pf, const float *pos,
                                      int f, int idx);

PLEN_DEV_NOINLINE unsigned sole_manifold_contacts(const DevConfig &cfg, WarpScratch &ws, int lane, float *man, float pos0, float pos1,
                                                  float pos2, float lam_in, float R0, float R1, float R2, float R3, float R4, float R5,
                                                  float R6, float R7, float R8, float p0, float p1, float p2);

// MASS = true: the robot's own body masses and torso payload (L.mass_w) replace the model table's inertial values; the
// false instance is the stock path and never reads L.mass_w.
template <bool MASS = false>
PLEN_DEV void tick_dynamics(const DevConfig &cfg, const float *tab, WarpScratch &ws, LaneState &L, int lane,
                            float *srec, uint8_t *sort_key, const DebugOut *dbg = nullptr, float *srx = nullptr,
                            float *man = nullptr) {
    const bool is_joint = lane >= 6 && lane < 24;
    const int cs = (int)tab[T_CS * 32 + lane], ce = (int)tab[T_CE * 32 + lane];
    float Rw[9], pw[3];
    forward_kinematics(tab, lane, L.q, L.quat, Rw, pw);

    // ---- joint twist s = [a; m] about the base origin (world axes); base lanes carry the identity columns
    //      (every index compile-time: a lane-indexed a[lane] = 1 would put a and m in local memory)
    float a[3], m[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { a[k] = (lane == k) ? 1.0f : 0.0f; m[k] = (lane == 3 + k) ? 1.0f : 0.0f; }
    if (is_joint) {
        float ax[3] = {tab[(T_AXIS + 0) * 32 + lane], tab[(T_AXIS + 1) * 32 + lane], tab[(T_AXIS + 2) * 32 + lane]};
        mat3_vec(Rw, ax, a);
        cross(pw, a, m);
    }
    if (lane < 24) {
        store6(ws.tw[lane], a[0], a[1], a[2], m[0], m[1], m[2]);
    }

    // ---- body inertia about the base origin, world axes: mass, h = m c, Ibar (xx yy zz xy xz yz)
    float mass = tab[T_MASS * 32 + lane];
    float h[3], Ib[6];
    {
        float com[3] = {tab[(T_COM + 0) * 32 + lane], tab[(T_COM + 1) * 32 + lane], tab[(T_COM + 2) * 32 + lane]};
        float c[3];
        mat3_vec(Rw, com, c);
        c[0] += pw[0]; c[1] += pw[1]; c[2] += pw[2];
        float ixx = tab[(T_INERTIA + 0) * 32 + lane], iyy = tab[(T_INERTIA + 1) * 32 + lane],
              izz = tab[(T_INERTIA + 2) * 32 + lane], ixy = tab[(T_INERTIA + 3) * 32 + lane],
              ixz = tab[(T_INERTIA + 4) * 32 + lane], iyz = tab[(T_INERTIA + 5) * 32 + lane];
        if (MASS) {
            // uniform density scaling of this lane's body: mass and rotational inertia times s, centre of mass unchanged
            // (lanes >= 24 hold payload words, not scales; their table mass is 0 like that of lanes 1..5)
            const float s = lane < MR_PAYLOAD ? L.mass_w : 1.0f;
            mass *= s; ixx *= s; iyy *= s; izz *= s; ixy *= s; ixz *= s; iyz *= s;
        }
        // Iw = Rw I Rw^T
        float T[9] = {Rw[0] * ixx + Rw[1] * ixy + Rw[2] * ixz, Rw[0] * ixy + Rw[1] * iyy + Rw[2] * iyz, Rw[0] * ixz + Rw[1] * iyz + Rw[2] * izz,
                      Rw[3] * ixx + Rw[4] * ixy + Rw[5] * ixz, Rw[3] * ixy + Rw[4] * iyy + Rw[5] * iyz, Rw[3] * ixz + Rw[4] * iyz + Rw[5] * izz,
                      Rw[6] * ixx + Rw[7] * ixy + Rw[8] * ixz, Rw[6] * ixy + Rw[7] * iyy + Rw[8] * iyz, Rw[6] * ixz + Rw[7] * iyz + Rw[8] * izz};
        const float cc = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
        Ib[0] = T[0] * Rw[0] + T[1] * Rw[1] + T[2] * Rw[2] + mass * (cc - c[0] * c[0]);
        Ib[1] = T[3] * Rw[3] + T[4] * Rw[4] + T[5] * Rw[5] + mass * (cc - c[1] * c[1]);
        Ib[2] = T[6] * Rw[6] + T[7] * Rw[7] + T[8] * Rw[8] + mass * (cc - c[2] * c[2]);
        Ib[3] = T[0] * Rw[3] + T[1] * Rw[4] + T[2] * Rw[5] - mass * c[0] * c[1];
        Ib[4] = T[0] * Rw[6] + T[1] * Rw[7] + T[2] * Rw[8] - mass * c[0] * c[2];
        Ib[5] = T[3] * Rw[6] + T[4] * Rw[7] + T[5] * Rw[8] - mass * c[1] * c[2];
        h[0] = mass * c[0]; h[1] = mass * c[1]; h[2] = mass * c[2];
        if (MASS) {
            // torso payload: a point mass m_p rigidly attached at r (torso body frame), added to lane 0's body with the same
            // expressions.  Skipped for m_p = 0, so that a unit row leaves every bit as the stock path computes it.
            const float mp = shfl(L.mass_w, MR_PAYLOAD);
            const float r[3] = {shfl(L.mass_w, MR_PAYLOAD + 1), shfl(L.mass_w, MR_PAYLOAD + 2), shfl(L.mass_w, MR_PAYLOAD + 3)};
            if (lane == 0 && mp != 0.0f) {
                float cp[3];
                mat3_vec(Rw, r, cp);
                cp[0] += pw[0]; cp[1] += pw[1]; cp[2] += pw[2];
                const float pp = cp[0] * cp[0] + cp[1] * cp[1] + cp[2] * cp[2];
                mass += mp;
                Ib[0] += mp * (pp - cp[0] * cp[0]);
                Ib[1] += mp * (pp - cp[1] * cp[1]);
                Ib[2] += mp * (pp - cp[2] * cp[2]);
                Ib[3] -= mp * cp[0] * cp[1];
                Ib[4] -= mp * cp[0] * cp[2];
                Ib[5] -= mp * cp[1] * cp[2];
                h[0] += mp * cp[0]; h[1] += mp * cp[1]; h[2] += mp * cp[2];
            }
        }
    }

    // ---- spatial velocity of this lane's body: V = V0 + sum_{ancestors} s_j qd_j
    float V0[6];
    load6(ws.st + W_U, V0);       // base velocity = u of lanes 0..5, still in the staged state record (two broadcast reads)
    float tv[6];   // own term s * u (joint lanes only)
#pragma unroll
    for (int k = 0; k < 3; k++) { tv[k] = is_joint ? a[k] * L.u : 0.0f; tv[3 + k] = is_joint ? m[k] * L.u : 0.0f; }
    float V[6];
#pragma unroll
    for (int k = 0; k < 6; k++) V[k] = tv[k];
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const float t = shfl_up(V[k], d);
            if (lane - d >= cs) V[k] += t;
        }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) V[k] += V0[k];

    // ---- velocity-product accelerations: ab = a0 + sum_{ancestors} V_j x s_j qd_j, a0 = [0; -w0 x v0 - g]
    float ab[6];
    {
        float t1[3], t2[3], t3[3];
        cross(V, tv, t1);          // w x t_ang
        cross(V, tv + 3, t2);      // w x t_lin
        cross(V + 3, tv, t3);      // v x t_ang
#pragma unroll
        for (int k = 0; k < 3; k++) { ab[k] = t1[k]; ab[3 + k] = t2[k] + t3[k]; }
#pragma unroll
        for (int d = 1; d < 8; d <<= 1) {
#pragma unroll
            for (int k = 0; k < 6; k++) {
                const float t = shfl_up(ab[k], d);
                if (lane - d >= cs) ab[k] += t;
            }
        }
        float wv[3];
        cross(V0, V0 + 3, wv);
        ab[3] -= wv[0]; ab[4] -= wv[1]; ab[5] -= wv[2] + cfg.gravity_z;
    }

    // ---- body net force F = I ab + V x* (I V)  (about the base origin)
    float F[6];
    {
        float IV[6], Ia[6], t[3], t2[3];
        // I x = [Ibar xa + h x xl ; m xl - h x xa]
        cross(h, V + 3, t);
        IV[0] = Ib[0] * V[0] + Ib[3] * V[1] + Ib[4] * V[2] + t[0];
        IV[1] = Ib[3] * V[0] + Ib[1] * V[1] + Ib[5] * V[2] + t[1];
        IV[2] = Ib[4] * V[0] + Ib[5] * V[1] + Ib[2] * V[2] + t[2];
        cross(h, V, t);
        IV[3] = mass * V[3] - t[0]; IV[4] = mass * V[4] - t[1]; IV[5] = mass * V[5] - t[2];
        cross(h, ab + 3, t);
        Ia[0] = Ib[0] * ab[0] + Ib[3] * ab[1] + Ib[4] * ab[2] + t[0];
        Ia[1] = Ib[3] * ab[0] + Ib[1] * ab[1] + Ib[5] * ab[2] + t[1];
        Ia[2] = Ib[4] * ab[0] + Ib[5] * ab[1] + Ib[2] * ab[2] + t[2];
        cross(h, ab, t);
        Ia[3] = mass * ab[3] - t[0]; Ia[4] = mass * ab[4] - t[1]; Ia[5] = mass * ab[5] - t[2];
        cross(V, IV, t);           // w x n
        cross(V + 3, IV + 3, t2);  // v x f
        F[0] = Ia[0] + t[0] + t2[0]; F[1] = Ia[1] + t[1] + t2[1]; F[2] = Ia[2] + t[2] + t2[2];
        cross(V, IV + 3, t);       // w x f
        F[3] = Ia[3] + t[0]; F[4] = Ia[4] + t[1]; F[5] = Ia[5] + t[2];
        if (cfg.linear_damping != 0.0f && mass > 0.0f) {
            // Bullet's multibody drag: f = -k m v_com (1 + |v_com|) at the com  (joint_act only, plen_env.py:472-481)
            float c[3] = {h[0] / mass, h[1] / mass, h[2] / mass}, vc[3], fd[3], nd[3];
            cross(V, c, t);
            vc[0] = V[3] + t[0]; vc[1] = V[4] + t[1]; vc[2] = V[5] + t[2];
            const float nv = sqrtf(vc[0] * vc[0] + vc[1] * vc[1] + vc[2] * vc[2]);
            const float k = cfg.linear_damping * mass * (1.0f + nv);
            fd[0] = -k * vc[0]; fd[1] = -k * vc[1]; fd[2] = -k * vc[2];
            cross(c, fd, nd);
            F[0] -= nd[0]; F[1] -= nd[1]; F[2] -= nd[2];
            F[3] -= fd[0]; F[4] -= fd[1]; F[5] -= fd[2];
        }
    }

    // ---- suffix sums along the chains: composite inertia (10 values) and subtree force (6 values)
    float mc = mass, hc[3] = {h[0], h[1], h[2]}, Ic[6] = {Ib[0], Ib[1], Ib[2], Ib[3], Ib[4], Ib[5]};
    float Fc[6] = {F[0], F[1], F[2], F[3], F[4], F[5]};
#pragma unroll
    for (int d = 1; d < 8; d <<= 1) {
        const bool take = is_joint && (lane + d <= ce);
        float t;
        t = shfl_down(mc, d); if (take) mc += t;
#pragma unroll
        for (int k = 0; k < 3; k++) { t = shfl_down(hc[k], d); if (take) hc[k] += t; }
#pragma unroll
        for (int k = 0; k < 6; k++) { t = shfl_down(Ic[k], d); if (take) Ic[k] += t; }
#pragma unroll
        for (int k = 0; k < 6; k++) { t = shfl_down(Fc[k], d); if (take) Fc[k] += t; }
    }
    // whole robot: torso (lane 0) + the four chain roots
    //      (one shared-memory gather: the <= 5 root lanes store their 16 composite values, every lane adds them up -- it used
    //      to be 16 full-warp butterfly reductions, 80 SHFL)
    float mt, ht[3], It[6], Ft[6];
    {
        const bool root = (lane == 0) || (is_joint && lane == cs);
        const unsigned roots = ballot(root);
        const int ord = popc_(roots & ((1u << lane) - 1u)), n_roots = popc_(roots);
        if (root) {
            float *dst = ws.red + 16 * ord;            // red is free until the Schur-complement products below
            dst[0] = mc; dst[1] = hc[0]; dst[2] = hc[1]; dst[3] = hc[2];
#pragma unroll
            for (int k = 0; k < 6; k++) { dst[4 + k] = Ic[k]; dst[10 + k] = Fc[k]; }
        }
        warp_sync();
        float acc[16];
#pragma unroll
        for (int v = 0; v < 16; v++) acc[v] = 0.0f;
        for (int r = 0; r < n_roots; r++) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const vec4 x = *reinterpret_cast<const vec4 *>(ws.red + 16 * r + 4 * q);
                acc[4 * q] += x.x; acc[4 * q + 1] += x.y; acc[4 * q + 2] += x.z; acc[4 * q + 3] += x.w;
            }
        }
        mt = acc[0]; ht[0] = acc[1]; ht[1] = acc[2]; ht[2] = acc[3];
#pragma unroll
        for (int k = 0; k < 6; k++) { It[k] = acc[4 + k]; Ft[k] = acc[10 + k]; }
        warp_sync();
    }

    // ---- bias force of this lane's coordinate and f = Ic s (column of M restricted to ancestors)
    float Cl = 0.0f, fM[6] = {0, 0, 0, 0, 0, 0};
    if (is_joint) {
        Cl = a[0] * Fc[0] + a[1] * Fc[1] + a[2] * Fc[2] + m[0] * Fc[3] + m[1] * Fc[4] + m[2] * Fc[5];
        float t[3];
        cross(hc, m, t);
        fM[0] = Ic[0] * a[0] + Ic[3] * a[1] + Ic[4] * a[2] + t[0];
        fM[1] = Ic[3] * a[0] + Ic[1] * a[1] + Ic[5] * a[2] + t[1];
        fM[2] = Ic[4] * a[0] + Ic[5] * a[1] + Ic[2] * a[2] + t[2];
        cross(hc, a, t);
        fM[3] = mc * m[0] - t[0]; fM[4] = mc * m[1] - t[1]; fM[5] = mc * m[2] - t[2];
    } else {
#pragma unroll
        for (int k = 0; k < 6; k++) Cl = (lane == k) ? Ft[k] : Cl;   // compile-time indices: Ft stays in registers
    }
    ws.cb[lane] = Cl;

    // ---- limb block rows: Mrow[d] = M[lane][cs+d], Krow = M[lane][0..5] = fM
    float Mrow[6], Krow[6];
    const int off = lane - cs;
    {
        // exchange f through shared memory (kk is free at this point)
        if (lane < 24) {
#pragma unroll
            for (int k = 0; k < 6; k++) ws.kk[lane][k] = fM[k];
        }
        warp_sync();
#pragma unroll
        for (int d = 0; d < 6; d++) {
            const int j = cs + d;
            float v = (d == off) ? 1.0f : 0.0f;   // identity padding for short chains / non-joint lanes
            if (is_joint && j <= ce) {
                float r6[6];
                if (d <= off) {  // ancestor-or-self j: M = s_j . f_lane
                    load6(ws.tw[j], r6);
                    v = r6[0] * fM[0] + r6[1] * fM[1] + r6[2] * fM[2] + r6[3] * fM[3] + r6[4] * fM[4] + r6[5] * fM[5];
                } else {         // descendant j: M = s_lane . f_j
                    load6(ws.kk[j], r6);
                    v = a[0] * r6[0] + a[1] * r6[1] + a[2] * r6[2] + m[0] * r6[3] + m[1] * r6[4] + m[2] * r6[5];
                }
            }
            Mrow[d] = v;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) Krow[k] = fM[k];
        warp_sync();
    }
    // Gauss-Jordan across the lanes of each chain: Mrow -> row of A_c = M_cc^-1, Krow -> row of K_c = A_c M_c0.
    // The pivot row of step k is published by lane cs + k in its own 12-word slot of red (free until the Schur products
    // below) and read back with three LDS.128 instead of twelve SHFL.  A slot is written once, so one warp_sync per step
    // suffices; the 48-byte slot stride keeps the four chains' pivot rows in distinct banks.
#pragma unroll
    for (int k = 0; k < 6; k++) {
        const bool act = is_joint && (cs + k <= ce);
        if (off == k) {
            float *dst = ws.red + 12 * lane;
            store6(dst, Mrow[0], Mrow[1], Mrow[2], Mrow[3], Mrow[4], Mrow[5]);
            store6(dst + 6, Krow[0], Krow[1], Krow[2], Krow[3], Krow[4], Krow[5]);
        }
        warp_sync();
        float pr[6], pk[6];
        {
            const float *srcp = ws.red + 12 * (act ? cs + k : 6 + k);   // idle lanes read a valid slot and ignore it
            const vec4 x0 = *reinterpret_cast<const vec4 *>(srcp), x1 = *reinterpret_cast<const vec4 *>(srcp + 4),
                       x2 = *reinterpret_cast<const vec4 *>(srcp + 8);
            pr[0] = x0.x; pr[1] = x0.y; pr[2] = x0.z; pr[3] = x0.w; pr[4] = x1.x; pr[5] = x1.y;
            pk[0] = x1.z; pk[1] = x1.w; pk[2] = x2.x; pk[3] = x2.y; pk[4] = x2.z; pk[5] = x2.w;
        }
        if (act) {
            const float inv = rcp_(pr[k]);
            if (off == k) {
#pragma unroll
                for (int d = 0; d < 6; d++) Mrow[d] = (d == k) ? inv : pr[d] * inv;
#pragma unroll
                for (int d = 0; d < 6; d++) Krow[d] = pk[d] * inv;
            } else {
                const float f = Mrow[k] * inv;
#pragma unroll
                for (int d = 0; d < 6; d++) Mrow[d] = (d == k) ? -f : Mrow[d] - f * pr[d];
#pragma unroll
                for (int d = 0; d < 6; d++) Krow[d] -= f * pk[d];
            }
        }
    }

    warp_sync();   // the last pivot rows are read before red is overwritten
    // ---- base Schur complement S = M00 - sum_l fM_l (x) K_l, via a conflict-free smem transpose-reduce
    {
        int idx = 0;
#pragma unroll
        for (int r = 0; r < 6; r++)
#pragma unroll
            for (int c = r; c < 6; c++) { ws.red[lane * 21 + idx] = is_joint ? fM[r] * Krow[c] : 0.0f; idx++; }
        warp_sync();
        if (lane < 21) {
            float s = 0.0f;
            for (int j = 6; j < 24; j++) s += ws.red[j * 21 + lane];
            ws.red[lane] = s;   // row 0 of red belongs to lane 0, which contributed zeros: safe to overwrite after sync
        }
    }
    // note: red[0..20] is written by lanes < 21 while other lanes may still read red[j*21 + lane] for j >= 6 only
    warp_sync();
    // ---- S^-1 by Gauss-Jordan ACROSS lanes 0..5 (lane r owns row r; lane k publishes the scaled pivot row of step k in
    //      kk[k], free until the K rows are stored below, and every lane reads it back as two broadcast LDS) instead of
    //      every lane inverting the full 6 x 6 redundantly: ~150 warp instructions instead of ~450.  Same elimination order
    //      and operations per entry as a serial in-place Gauss-Jordan without pivoting (S is SPD).
    float R[6];     // lanes 0..5: row `lane` of S, then of S^-1 (other lanes: scratch)
    {
        // M00 = [[Ibar, hx],[hx^T, m 1]] of the whole robot
        float M00[6][6] = {{It[0], It[3], It[4], 0.0f, -ht[2], ht[1]},
                           {It[3], It[1], It[5], ht[2], 0.0f, -ht[0]},
                           {It[4], It[5], It[2], -ht[1], ht[0], 0.0f},
                           {0.0f, ht[2], -ht[1], mt, 0.0f, 0.0f},
                           {-ht[2], 0.0f, ht[0], 0.0f, mt, 0.0f},
                           {ht[1], -ht[0], 0.0f, 0.0f, 0.0f, mt}};
        float S[6][6];
        int idx = 0;
#pragma unroll
        for (int r = 0; r < 6; r++)
#pragma unroll
            for (int c = r; c < 6; c++) {
                const float v = M00[r][c] - ws.red[idx];
                S[r][c] = v; S[c][r] = v; idx++;
            }
#pragma unroll
        for (int c = 0; c < 6; c++) {
            float v = S[0][c];
#pragma unroll
            for (int r = 1; r < 6; r++) v = (lane == r) ? S[r][c] : v;
            R[c] = v;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const float inv = rcp_(R[k]);
            float P[6];     // row k after scaling: [.. R[j] inv .., inv at j = k, ..]
            if (lane == k) {
#pragma unroll
                for (int j = 0; j < 6; j++) P[j] = (j == k) ? inv : R[j] * inv;
                store6(ws.kk[k], P[0], P[1], P[2], P[3], P[4], P[5]);
            }
            warp_sync();
            load6(ws.kk[k], P);
            const float f = R[k];
            const bool piv = lane == k;
#pragma unroll
            for (int j = 0; j < 6; j++) {
                const float elim = (j == k) ? -(f * P[k]) : R[j] - f * P[j];
                R[j] = piv ? P[j] : elim;
            }
        }
    }
    // S^-1 to every lane through shared memory (gg is free until the G rows are stored below)
    warp_sync();
    if (lane < 6) store6(ws.gg[lane], R[0], R[1], R[2], R[3], R[4], R[5]);
    warp_sync();
    // G = K S^-1
    float G[6];
    {
        float Si[6][6];
#pragma unroll
        for (int b = 0; b < 6; b++)
#pragma unroll
            for (int c = 0; c < 6; c++) Si[b][c] = ws.gg[b][c];
#pragma unroll
        for (int c = 0; c < 6; c++) {
            float s = 0.0f;
#pragma unroll
            for (int b = 0; b < 6; b++) s += Krow[b] * Si[b][c];
            G[c] = is_joint ? s : 0.0f;
        }
    }
    warp_sync();
    if (lane < 24) store6(ws.kk[lane], is_joint ? Krow[0] : 0.0f, is_joint ? Krow[1] : 0.0f, is_joint ? Krow[2] : 0.0f,
                          is_joint ? Krow[3] : 0.0f, is_joint ? Krow[4] : 0.0f, is_joint ? Krow[5] : 0.0f);
    warp_sync();
    // ---- assemble M^-1 (this lane's row), stored column-major so later reads are conflict free: lanes < 24 their row of
    //      the base columns (-G, or S^-1 on base lanes), joint lanes also the base rows of their own column (the transposed
    //      -G: one STS.128 + STS.64) and G . K_j (+ the limb block) in the joint columns
    if (lane < 24) {
#pragma unroll
        for (int k = 0; k < 6; k++) ws.minv[k][lane] = is_joint ? -G[k] : R[k];
        if (is_joint) store6(ws.minv[lane], -G[0], -G[1], -G[2], -G[3], -G[4], -G[5]);
#pragma unroll 6
        for (int j = 6; j < 24; j++) {
            float r6[6];
            load6(ws.kk[j], r6);
            const float s = G[0] * r6[0] + G[1] * r6[1] + G[2] * r6[2] + G[3] * r6[3] + G[4] * r6[4] + G[5] * r6[5];
            if (is_joint) ws.minv[j][lane] = s;
        }
        if (is_joint) {
#pragma unroll
            for (int d = 0; d < 6; d++)
                if (cs + d <= ce) ws.minv[cs + d][lane] += Mrow[d];
        }
    }
    warp_sync();

    if (dbg != nullptr && lane < 24) {
        if (dbg->minv) for (int j = 0; j < 24; j++) dbg->minv[lane * 24 + j] = ws.minv[j][lane];
        if (dbg->pos) for (int k = 0; k < 3; k++) dbg->pos[lane * 3 + k] = pw[k] + L.pos[k];
        if (dbg->rot) for (int k = 0; k < 9; k++) dbg->rot[lane * 9 + k] = Rw[k];
    }

    // ---- unconstrained velocity v* = clamp(v - dt M^-1 C)
    float vstar = 0.0f;
    if (lane < 24) {
        float acc = 0.0f;
        for (int j = 0; j < 24; j++) acc += ws.minv[j][lane] * ws.cb[j];
        vstar = clampf(L.u - cfg.dt * acc, -cfg.vmax, cfg.vmax);
    }

    // ---- contacts: sole vertices vs z = 0 at the start-of-tick pose; lanes 24..31 own one candidate point each
    unsigned man_new;
    if (cfg.sole_manifold && man != nullptr) {
        // persistent manifold per foot, out of line (an option: it must not cost the default path registers or fetches)
        man_new = sole_manifold_contacts(cfg, ws, lane, man, L.pos[0], L.pos[1], L.pos[2], L.lam, Rw[0], Rw[1], Rw[2], Rw[3], Rw[4],
                                         Rw[5], Rw[6], Rw[7], Rw[8], pw[0], pw[1], pw[2]);
        L.man = man_new;
        L.lam = (lane >= 24) ? ws.mlam[lane - 24] : L.lam;
    } else {
        const int i = lane - 24, f = (lane >= 28) ? 1 : 0;
        // the two foot lanes publish their frame (Rw, pw) in 16 words of kk each (free until the Y stash below); the contact
        // lanes read it back with three LDS.128 instead of twelve SHFL
        const int fw = (lane == cfg.foot_lane[0]) ? 0 : ((lane == cfg.foot_lane[1]) ? 1 : -1);
        if (fw >= 0) {
            vec4 *dst = reinterpret_cast<vec4 *>(&ws.kk[0][0] + 16 * fw);
            vec4 x;
            x.x = Rw[0]; x.y = Rw[1]; x.z = Rw[2]; x.w = Rw[3]; dst[0] = x;
            x.x = Rw[4]; x.y = Rw[5]; x.z = Rw[6]; x.w = Rw[7]; dst[1] = x;
            x.x = Rw[8]; x.y = pw[0]; x.z = pw[1]; x.w = pw[2]; dst[2] = x;
        }
        warp_sync();
        bool in = false;
        if (lane >= 24) {
            const vec4 *fr = reinterpret_cast<const vec4 *>(&ws.kk[0][0] + 16 * f);
            const vec4 x0 = fr[0], x1 = fr[1], x2 = fr[2];
            const float Rf[9] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w, x2.x}, pf[3] = {x2.y, x2.z, x2.w};
            const float *pt = cfg.foot_pts[f][i & 3];
            float w[3];
            mat3_vec(Rf, pt, w);
            w[0] += pf[0]; w[1] += pf[1]; w[2] += pf[2];
            const float dist = (L.pos[2] + w[2]) - cfg.hull_margin;
            in = dist <= cfg.foot_break[f];
            vec4 c4;
            c4.x = w[0]; c4.y = w[1]; c4.z = w[2] - cfg.hull_margin; c4.w = dist;
            *reinterpret_cast<vec4 *>(ws.cp[i]) = c4;
            const bool was = (L.man >> i) & 1u;
            if (!in || !was) L.lam = 0.0f;
        }
        man_new = ballot(in) >> 24;
        L.man = man_new;
    }
    warp_sync();

    // ---- ground contact of the link BOXES (every collider but the two foot hulls; SURVEY.md 8f-2): lane b tests box b.
    //      Hot path = one quick test per lane (lowest point of the box above the ground?) and a ballot; the rest is the rare
    //      branch.  Contact model (restates btBoxBoxDetector for a small box on the ground box of plane.urdf, as the oracle
    //      does): the incident face is the box face whose normal points most downward, its vertices that PENETRATE are the
    //      contact points; the PLEN_MAX_BOX_POINTS deepest of a robot are kept (ties: lower box, lower vertex) and enter the
    //      solver in (box, vertex) order.  No manifold hysteresis and no warm start for these points.
    int nx = 0;
    if (cfg.link_contacts && srx != nullptr) {
        const int bl = (int)tab[T_BOX_LANE * 32 + lane];
        const float r20 = shfl(Rw[6], bl), r21 = shfl(Rw[7], bl), r22 = shfl(Rw[8], bl), pz = shfl(pw[2], bl);
        float rz[3], az[3];      // z component of each box axis (world), and times its half extent
#pragma unroll
        for (int k = 0; k < 3; k++) {
            rz[k] = r20 * tab[(T_BOX_R + k) * 32 + lane] + r21 * tab[(T_BOX_R + 3 + k) * 32 + lane] + r22 * tab[(T_BOX_R + 6 + k) * 32 + lane];
            az[k] = rz[k] * tab[(T_BOX_H + k) * 32 + lane];
        }
        const float cz = L.pos[2] + pz + r20 * tab[(T_BOX_C + 0) * 32 + lane] + r21 * tab[(T_BOX_C + 1) * 32 + lane] +
                         r22 * tab[(T_BOX_C + 2) * 32 + lane];
        const bool touch = lane < cfg.n_boxes && cz - (fabsf(az[0]) + fabsf(az[1]) + fabsf(az[2])) <= 0.0f;
        // rare branch, kept out of line: k_dyn is an instruction-fetch-bound straight line (no_instruction stalls are 8-14 % of
        // its warp latency, profiles/r2_summary.md) and must not carry this code in the middle of its hot path
        if (ballot(touch))
            nx = box_points(cfg, tab, ws, lane, touch, cz, rz[0], rz[1], rz[2], bl, Rw[0], Rw[1], Rw[2], Rw[3], Rw[4], Rw[5], Rw[6],
                            Rw[7], Rw[8], pw[0], pw[1], pw[2]);
    }
    const bool ext = nx > 0;

    // ---- masked twists and operational columns Y_f = M^-1 Jfoot_f^T per foot with active contacts
    float Y[2][6], mb[6];     // mb: this lane's row of the base columns of M^-1, read once for both feet
#pragma unroll
    for (int k = 0; k < 6; k++) mb[k] = (man_new || ext) && lane < 24 ? ws.minv[k][lane] : 0.0f;
#pragma unroll
    for (int f = 0; f < 2; f++) {
        const int fl = cfg.foot_lane[f], fcs = fl - 5;
#pragma unroll
        for (int k = 0; k < 6; k++) Y[f][k] = 0.0f;
        // (a robot with box contacts always carries the right-foot twist: the box rows are expressed through it)
        if ((((man_new >> (4 * f)) & 0xFu) || (f == 0 && ext)) && lane < 24) {
#pragma unroll
            for (int k = 0; k < 6; k++) Y[f][k] = mb[k];
            for (int j = fcs; j <= fl; j++) {
                const float w = ws.minv[j][lane];
                float r6[6];
                load6(ws.tw[j], r6);
#pragma unroll
                for (int k = 0; k < 6; k++) Y[f][k] += w * r6[k];
            }
        }
    }

    // =====================================================================================================
    // Emit the SOLVE RECORD of this robot (global memory) for k_solve: everything the projected Gauss-Seidel needs,
    // in the 30-dimensional operational space  x = [18 joint velocities; right-foot twist (6); left-foot twist (6)].
    // Every constraint row of the tick is a functional of x: servo / limit rows read one joint velocity, the rows of
    // a contact point on foot f read the foot twist (flat ground => <= 3 non-zeros, known per row type).  With
    //   G = [ M^-1_jj  Y ; Y^T  Lambda^-1 ]   (30 x 30, symmetric),   Y = (M^-1 Jfoot^T) joint rows,
    // a row update with impulse delta adds (a combination of <= 3 columns of) G * delta to x.
    // =====================================================================================================
    // ---- servo rows (btMultiBodyJointMotor semantics): target velocity kp (q* - q)/dt + (1 - kd) v*, |impulse| <= f dt
    float m_dinv = 0.0f, m_rhs = 0.0f, l_rhs = 0.0f, l_dir = 0.0f;   // joint-limit row only when violated
    if (is_joint) {
        const float m_d = ws.minv[lane][lane];
        m_dinv = (m_d > 1.1920929e-7f) ? rcp_(m_d) : 0.0f;
        const float desired = cfg.kp_over_dt * L.kp_s * (L.tgt - L.q) + cfg.one_minus_kd * vstar;
        m_rhs = (m_dinv > 0.0f) ? (desired - vstar) : 0.0f;          // velocity units
        const float lo = tab[T_LOWER * 32 + lane], hi = tab[T_UPPER * 32 + lane];
        const float pen_lo = L.q - lo, pen_hi = hi - L.q;
        if (m_dinv > 0.0f) {
            if (pen_lo <= 0.0f) { l_dir = 1.0f; l_rhs = -pen_lo * cfg.erp_joint_over_dt - vstar; }
            else if (pen_hi <= 0.0f) { l_dir = -1.0f; l_rhs = -pen_hi * cfg.erp_joint_over_dt + vstar; }
        }
    }
    // ---- foot twists at v*: Vs_f = Jfoot_f v*;  Y stash;  Lambda^-1 = Jfoot M^-1 Jfoot^T (12 x 12)
    //      Vs is computed by lanes 0..11 (one twist component each: 12 terms from shared memory) and read back by the
    //      contact-row lanes through ws.st[W_SPARE ..]; it used to be twelve full-warp butterfly reductions (60 SHFL).
    ws.obs[lane] = vstar;                           // obs is free scratch in k_dyn (lanes >= 24 hold 0)
    if (lane < 24) {
        store6(ws.kk[lane], Y[0][0], Y[0][1], Y[0][2], Y[0][3], Y[0][4], Y[0][5]);
        store6(ws.gg[lane], Y[1][0], Y[1][1], Y[1][2], Y[1][3], Y[1][4], Y[1][5]);
    }
    warp_sync();
    if (man_new || ext) {
        if (lane < 12) {
            const int f = (lane >= 6) ? 1 : 0, k = lane - 6 * f, fl = cfg.foot_lane[f];
            float vb[6];                                // v* of the base: two broadcast reads
            load6(ws.obs, vb);
            float acc = 0.0f;
#pragma unroll
            for (int l = 0; l < 6; l++) acc += ws.tw[l][k] * vb[l];
#pragma unroll
            for (int l = 0; l < 6; l++) acc += ws.tw[fl - 5 + l][k] * ws.obs[fl - 5 + l];
            ws.st[W_SPARE + lane] = acc;
        }
        // Lambda^-1[fa*6+a][fb*6+b] = Y_fb[a][b] + sum_{j in leg fa} s_j[a] Y_fb[j][b], summed in leg order.
        // Lane fa*12 + col (lanes < 24) owns the six entries (fa*6 + a, col): Y_fb[j][b] is read once for all six, the twist
        // rows of leg fa as one broadcast row read per joint.  (It was 4.5 entries per lane with two scalar reads per term.)
        if (lane < 24) {
            const int fa = (lane >= 12) ? 1 : 0, col = lane - 12 * fa, fb = (col >= 6) ? 1 : 0, b6 = col - 6 * fb;
            const float(*Yb)[8] = fb ? ws.gg : ws.kk;
            const int j0 = cfg.foot_lane[fa] - 5;
            float acc[6];
#pragma unroll
            for (int a = 0; a < 6; a++) acc[a] = Yb[a][b6];
#pragma unroll
            for (int t = 0; t < 6; t++) {
                float s6[6];
                load6(ws.tw[j0 + t], s6);
                const float y = Yb[j0 + t][b6];
#pragma unroll
                for (int a = 0; a < 6; a++) acc[a] += s6[a] * y;
            }
#pragma unroll
            for (int a = 0; a < 6; a++) ws.lin[6 * fa + a][col] = acc[a];
        }
        warp_sync();
    }

    // ---- G (30 columns x 32 words) and B (6 rows x 32 words): word w of a column = entry i = w; joint columns are
    //      divided by their diagonal entry (velocity-unit servo rows, see the SR_ enum)
    {
        // Branch free: every lane reads its entries through ONE base pointer + a stride fixed per lane class (joint rows
        // from M^-1 / Y, foot-twist rows from Y^T / Lambda^-1, the two unused words zero), so the 30 column stores are
        // straight-line LDS -> (FMUL) -> STG with the loops fully unrolled.
        const int i = lane;
        const bool ij = i < 18, ic = (i >= 18 && i < 24) || i >= 26;
        const int fa = (i >= 26) ? 1 : 0, a6 = fa ? i - 26 : i - 18;
        const float(*Ya)[8] = fa ? ws.gg : ws.kk;
        float *G = srec + SR_G;
        ws.obs[lane] = m_dinv;                      // obs is free scratch in k_dyn; word 6 + c = 1 / G_cc of joint column c
        warp_sync();
        {
            const float *b1 = ij ? &ws.minv[6][6 + i] : (ic ? &Ya[6][a6] : &ws.cb[0]);
            const int st1 = ij ? 32 : (ic ? 8 : 0);
            const bool on1 = ij || ic;
            float sc[18];                               // the 18 broadcast scales as one LDS.64 + four LDS.128
            {
                const vec2 s2 = *reinterpret_cast<const vec2 *>(ws.obs + 6);
                sc[0] = s2.x; sc[1] = s2.y;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const vec4 s4 = *reinterpret_cast<const vec4 *>(ws.obs + 8 + 4 * q);
                    sc[2 + 4 * q] = s4.x; sc[3 + 4 * q] = s4.y; sc[4 + 4 * q] = s4.z; sc[5 + 4 * q] = s4.w;
                }
            }
#pragma unroll
            for (int c = 0; c < 18; c++) {
                const float v = b1[c * st1];
                G[c * 32 + lane] = on1 ? v * sc[c] : 0.0f;
            }
        }
        {
            // column c = 18 + 6 fb + b6:  joint rows Y_fb[6 + i][b6], twist rows Lambda^-1[fa 6 + a6][c - 18] when any
            // contact is active; six consecutive words per foot (the Lambda^-1 half of fb = 1 is only 8-byte aligned)
            const bool on2 = ij || (ic && (man_new || ext));
            const float *b2 = ij ? &ws.kk[6 + i][0] : (on2 ? &ws.lin[fa * 6 + a6][0] : &ws.cb[0]);
            const float *b2b = ij ? &ws.gg[6 + i][0] : b2 + 6;
            float v2[12];
            {
                float r6[6];
                load6(b2, r6);
#pragma unroll
                for (int k = 0; k < 6; k++) v2[k] = r6[k];
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    const vec2 x = *reinterpret_cast<const vec2 *>(b2b + 2 * k);
                    v2[6 + 2 * k] = x.x; v2[7 + 2 * k] = x.y;
                }
            }
#pragma unroll
            for (int c = 18; c < 30; c++) G[c * 32 + lane] = on2 ? v2[c - 18] : 0.0f;
        }
        // per-joint scalars in the same word order (entries >= 18 are zero)
        const int src = ij ? 6 + i : 0;
        const float s_rhs = shfl(m_rhs, src), s_dinv = shfl(m_dinv, src), s_ldir = shfl(l_dir, src),
                    s_lrhs = shfl(l_rhs, src), s_vs = shfl(vstar, src), s_q = shfl(L.q, src),
                    s_d = shfl(is_joint ? ws.minv[lane][lane] : 0.0f, src);
        float *Bm = srec + SR_B;
        {
            const float *b3 = ij ? &ws.minv[6 + i][0] : (ic ? &Ya[0][a6] : &ws.cb[0]);
            const int st3 = ij ? 1 : (ic ? 8 : 0);
            const float sc3 = ij ? s_dinv : (ic ? 1.0f : 0.0f);
#pragma unroll
            for (int k = 0; k < 6; k++) Bm[k * 32 + lane] = (ij || ic) ? b3[k * st3] * sc3 : 0.0f;
        }
        srec[SR_MRHS + lane] = ij ? s_rhs : 0.0f;
        srec[SR_MD + lane] = (ij && s_dinv > 0.0f) ? s_d : 0.0f;
        srec[SR_LDIR + lane] = ij ? s_ldir : 0.0f;
        srec[SR_LRHS + lane] = ij ? s_lrhs : 0.0f;
        srec[SR_VSTAR + lane] = ij ? s_vs : 0.0f;
        srec[SR_Q + lane] = ij ? s_q : 0.0f;
    }

    // ---- contact rows, COMPACTED per foot: slot q = 4 f + k is the k-th active point of foot f.  Word q*8+g of
    //      SR_CRHS / SR_CDINV / SR_CD belongs to solver lane g, which owns the row whose "own" twist component is g - 2:
    //      comp 0 wx: roll about t2   1 wy: roll about t1 (sign flipped)   2 wz: spin
    //           3 vx: lateral t2      4 vy: lateral t1 (sign flipped)      5 vz: normal
    //      (flipping the sign of a row with symmetric bounds leaves the Gauss-Seidel iterates unchanged)
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const int f = half, g = lane & 7, comp = g - 2;
        const int pb = nth_bit4((man_new >> (4 * f)) & 15u, lane >> 3);
        const int p = 4 * f + (pb < 0 ? 0 : pb);
        const bool valid = comp >= 0 && pb >= 0;
        float rhs = 0.0f, dinv = 0.0f, d = 0.0f;
        if (valid) {
            const float px = ws.cp[p][0], py = ws.cp[p][1], pz = ws.cp[p][2];
            int i0 = comp, i1 = comp, i2 = comp;
            float c0 = 1.0f, c1 = 0.0f, c2 = 0.0f;
            if (comp == 3) { i0 = 1; i1 = 2; i2 = 3; c0 = pz; c1 = -py; c2 = 1.0f; }
            else if (comp == 4) { i0 = 0; i1 = 2; i2 = 4; c0 = -pz; c1 = px; c2 = 1.0f; }
            else if (comp == 5) { i0 = 0; i1 = 1; i2 = 5; c0 = py; c1 = -px; c2 = 1.0f; }
            const int o = 6 * f;
            d = c0 * (c0 * ws.lin[o + i0][o + i0] + c1 * ws.lin[o + i0][o + i1] + c2 * ws.lin[o + i0][o + i2]) +
                c1 * (c0 * ws.lin[o + i1][o + i0] + c1 * ws.lin[o + i1][o + i1] + c2 * ws.lin[o + i1][o + i2]) +
                c2 * (c0 * ws.lin[o + i2][o + i0] + c1 * ws.lin[o + i2][o + i1] + c2 * ws.lin[o + i2][o + i2]);
            dinv = (d > 1.1920929e-7f) ? rcp_(d) : 0.0f;
            const float *vsf = &ws.st[W_SPARE + 6 * f];      // foot twist at v* (written above, before the Lambda^-1 sync)
            const float v0 = vsf[i0], v1 = vsf[i1], v2 = vsf[i2];
            const float rel = c0 * v0 + c1 * v1 + c2 * v2;
            if (comp == 5) {
                const float pdist = ws.cp[p][3] + cfg.linear_slop;
                float rest = (fabsf(rel) < cfg.rest_thresh) ? 0.0f : cfg.restitution * -rel;
                rest = fmaxf(rest, 0.0f);
                float velerr = rest - rel, poserr = 0.0f;
                if (pdist > 0.0f) velerr -= pdist * cfg.inv_dt; else poserr = -pdist * cfg.erp_contact_over_dt;
                rhs = (poserr + velerr) * dinv;
            } else {
                rhs = -rel * dinv;
                if (comp < 3) {
                    const float mu = (comp == 2) ? cfg.mu_spinning : cfg.mu_rolling;
                    if (!(mu > 0.0f)) { dinv = 0.0f; rhs = 0.0f; d = 0.0f; }   // row not created when its coefficient is 0
                }
            }
        }
        srec[SR_CRHS + 32 * half + lane] = rhs;
        srec[SR_CDINV + 32 * half + lane] = dinv;
        srec[SR_CD + 32 * half + lane] = d;
    }
    {
        const int q = lane >> 2, pb = nth_bit4((man_new >> (4 * (q >> 2))) & 15u, q & 3);
        srec[SR_PT + lane] = (pb >= 0) ? ws.cp[4 * (q >> 2) + pb][lane & 3] : 0.0f;
        const int q2 = lane & 7, pb2 = nth_bit4((man_new >> (4 * (q2 >> 2))) & 15u, q2 & 3);
        const float lc = shfl(L.lam, 24 + 4 * (q2 >> 2) + (pb2 < 0 ? 0 : pb2));
        if (lane >= 24) srec[SR_LAMC + q2] = (pb2 >= 0) ? lc : 0.0f;
    }
    if (lane < 6) srec[SR_BASE + lane] = vstar;
    // base pose from the staged state record (the copy L.pos / L.quat came from): a lane-indexed L.pos[lane] would put L in
    // local memory
    if (lane < 3) srec[SR_BASE + 6 + lane] = ws.st[W_POS + lane];
    if (lane < 4) srec[SR_BASE + 9 + lane] = ws.st[W_QUAT + lane];
    if (lane == 0) {
        srec[SR_BASE + 13] = (float)man_new;
        srec[SR_BASE + 14] = L.fric_s;            // k_solve scales mu_lateral / mu_spinning / mu_rolling ...
        srec[SR_BASE + 15] = L.motor_s;           // ... and the servo impulse bound of this robot
        // k_solve groups robots of similar contact load into the same warp (tile-local sort by this key)
        const int n0 = popc_(man_new & 15u), n1 = popc_((man_new >> 4) & 15u);
        if (sort_key) *sort_key = ext ? (uint8_t)(PLEN_KEY_EXT + nx - 1) : (uint8_t)((n0 > n1 ? n0 : n1) * 25 + n0 * 5 + n1);
    }
    warp_sync();
    if (ext) box_rows(cfg, tab, ws, lane, vstar, nx, srx);
}

// Persistent sole manifolds (plen_config.sole_manifold = 1; restates btConvexPlaneCollisionAlgorithm + btPersistentManifold as
// the oracle's manifold_mode 1 does): one new point per tick and foot = the hull's support vertex towards the ground, merged
// into a cache of <= 4 points; slot k of foot f is contact slot 4 f + k and its impulse travels with it.  The vertex search runs
// across the warp, the (scalar, short) cache update on lane 0.  Fills ws.cp, leaves the slots' cached impulses in ws.mlam,
// returns the manifold bits.  Not inlined: an option must not cost the default path registers or instruction fetches.
PLEN_DEV_NOINLINE unsigned sole_manifold_contacts(const DevConfig &cfg, WarpScratch &ws, int lane, float *man, float pos0, float pos1,
                                                  float pos2, float lam_in, float R0, float R1, float R2, float R3, float R4, float R5,
                                                  float R6, float R7, float R8, float p0, float p1, float p2) {
    const float Rw[9] = {R0, R1, R2, R3, R4, R5, R6, R7, R8}, pw[3] = {p0, p1, p2}, pos[3] = {pos0, pos1, pos2};
    unsigned man_new = 0;
    float lam_out = 0.0f;
    // Persistent manifold per foot (plen_config.sole_manifold = 1; restates btConvexPlaneCollisionAlgorithm +
    // btPersistentManifold as the oracle's manifold_mode 1 does): one new point per tick = the hull's support vertex
    // towards the ground, merged into a cache of <= 4 points; slot k of foot f is contact slot 4 f + k, its impulse travels
    // with it.  The search runs across the warp, the (scalar, short) cache updates on lanes 0 / 1 out of line.
    if (lane < 24) { ws.mn[0][lane] = man[lane]; ws.mn[1][lane] = man[24 + lane]; }
    if (lane < 2) ws.mn[lane][24] = man[48 + lane];
    if (lane >= 24) ws.mlam[lane - 24] = lam_in;
    warp_sync();
    // support vertices of both feet: every lane keeps the heights of its <= 8 vertices in registers (one pass over the list)
    int idx2[2];
#pragma unroll
    for (int f = 0; f < 2; f++) {
        const int src = cfg.foot_lane[f];
        const float r6 = shfl(Rw[6], src), r7 = shfl(Rw[7], src), r8 = shfl(Rw[8], src);
        const float *hv = cfg.hull + (size_t)f * PLEN_MAX_HULL * 3;
        const int nh = cfg.n_hull[f];
        float z[PLEN_MAX_HULL / 32];
        float zmin = 3.0e38f;
#pragma unroll
        for (int j = 0; j < PLEN_MAX_HULL / 32; j++) {
            const int i = lane + 32 * j;
            z[j] = 3.0e38f;
            if (i < nh) z[j] = r6 * hv[3 * i] + r7 * hv[3 * i + 1] + r8 * hv[3 * i + 2];
            zmin = fminf(zmin, z[j]);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) zmin = fminf(zmin, shfl_xor(zmin, d));
        // vertices within support_tie of the lowest are ties (a foot flat on the ground): the first of them in the list
        const float zlim = zmin + cfg.support_tie;
        int idx = 0x7fffffff;
#pragma unroll
        for (int j = PLEN_MAX_HULL / 32 - 1; j >= 0; j--)
            if (z[j] <= zlim && lane + 32 * j < nh) idx = lane + 32 * j;
        idx2[f] = 0x7fffffff - (int)redux_max((unsigned)(0x7fffffff - idx));       // the smallest index
    }
    {
        // the (scalar, short) cache updates of the two feet run side by side on lanes 0 and 1
        const int f = lane & 1, src = cfg.foot_lane[f];
        float Rf[9], pf[3];
#pragma unroll
        for (int k = 0; k < 9; k++) Rf[k] = shfl(Rw[k], src);
#pragma unroll
        for (int k = 0; k < 3; k++) pf[k] = shfl(pw[k], src);
        if (lane < 2) manifold_merge(cfg, ws.mn[f], ws.mlam + 4 * f, Rf, pf, pos, f, f ? idx2[1] : idx2[0]);
        warp_sync();
    }
    {
        const int i = lane - 24, f = (lane >= 28) ? 1 : 0, k = i & 3;
        const int src = cfg.foot_lane[f];
        float Rf[9], pf[3];
#pragma unroll
        for (int q = 0; q < 9; q++) Rf[q] = shfl(Rw[q], src);
#pragma unroll
        for (int q = 0; q < 3; q++) pf[q] = shfl(pw[q], src);
        bool in = false;
        if (lane >= 24) {
            in = k < (int)ws.mn[f][24];
            float w[3] = {0.0f, 0.0f, 0.0f};
            if (in) { mat3_vec(Rf, &ws.mn[f][3 * k], w); w[0] += pf[0]; w[1] += pf[1]; w[2] += pf[2]; }
            ws.cp[i][0] = w[0]; ws.cp[i][1] = w[1]; ws.cp[i][2] = w[2];
            ws.cp[i][3] = in ? (pos[2] + w[2]) - ws.mn[f][12 + 3 * k + 2] : 0.0f;
            lam_out = in ? ws.mlam[i] : 0.0f;
        }
        man_new = ballot(in) >> 24;
    }
    warp_sync();
    if (lane < 24) { man[lane] = ws.mn[0][lane]; man[24 + lane] = ws.mn[1][lane]; }
    if (lane < 2) man[48 + lane] = ws.mn[lane][24];
    warp_sync();
    if (lane >= 24) ws.mlam[lane - 24] = lam_out;
    warp_sync();
    return man_new;
}

// Cache update of one foot's persistent manifold (lane f for foot f; see sole_manifold_contacts).  mn: local xyz of 4 points | plane xyz of 4
// points | count; lam: the four cached impulses; Rf / pf: world rotation and origin (relative to the base origin) of the foot
// frame; pos: base position; idx: the hull's support vertex towards the ground.  Restates oracle/plen_oracle.c:manifold_update.
PLEN_DEV_NOINLINE void manifold_merge(const DevConfig &cfg, float *mn, float *lam, const float *Rf, const float *pf, const float *pos,
                                      int f, int idx) {
    float *loc = mn, *pln = mn + 12;
    int n = (int)mn[24];
    const float thr = cfg.foot_break[f];
    const float fx = pos[0] + pf[0], fy = pos[1] + pf[1], fz = pos[2] + pf[2];      // foot frame origin, world
    if (idx >= 0 && idx < cfg.n_hull[f]) {
        const float *v = cfg.hull + ((size_t)f * PLEN_MAX_HULL + idx) * 3;
        // point on the inflated hull: the vertex moved by the margin towards the ground (world -z = -(third row of Rf) locally)
        const float la[3] = {v[0] - cfg.hull_margin * Rf[6], v[1] - cfg.hull_margin * Rf[7], v[2] - cfg.hull_margin * Rf[8]};
        float t[3];
        mat3_vec(Rf, la, t);
        const float pa[3] = {fx + t[0], fy + t[1], fz + t[2]};
        const float dist = pa[2];
        if (dist < thr) {
            int slot = -1;
            float nearest = thr * thr;
            for (int k = 0; k < n; k++) {           // getCacheEntry
                const float e0 = loc[3 * k] - la[0], e1 = loc[3 * k + 1] - la[1], e2 = loc[3 * k + 2] - la[2];
                const float dd = e0 * e0 + e1 * e1 + e2 * e2;
                if (dd < nearest) { nearest = dd; slot = k; }
            }
            if (slot < 0) {
                if (n < 4) { slot = n; n = n + 1; lam[slot] = 0.0f; }
                else {                               // sortCachedPoints: keep the deepest, drop the one that leaves the largest area
                    int deepest = -1;
                    float maxpen = dist;
                    for (int k = 0; k < 4; k++) {
                        const float zk = fz + Rf[6] * loc[3 * k] + Rf[7] * loc[3 * k + 1] + Rf[8] * loc[3 * k + 2];
                        if (zk < maxpen) { deepest = k; maxpen = zk; }
                    }
                    float best = -1.0f;
                    slot = 0;
                    for (int k = 0; k < 4; k++) {
                        float res = 0.0f;
                        if (k != deepest) {
                            const int o0 = (k == 0) ? 1 : 0, o1 = (k <= 1) ? 2 : 1, o2 = (k <= 2) ? 3 : 2;
                            const float a[3] = {la[0] - loc[3 * o0], la[1] - loc[3 * o0 + 1], la[2] - loc[3 * o0 + 2]};
                            const float b[3] = {loc[3 * o2] - loc[3 * o1], loc[3 * o2 + 1] - loc[3 * o1 + 1], loc[3 * o2 + 2] - loc[3 * o1 + 2]};
                            float c[3];
                            cross(a, b, c);
                            res = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
                        }
                        if (res > best) { best = res; slot = k; }
                    }
                    lam[slot] = 0.0f;
                }
            }
            loc[3 * slot] = la[0]; loc[3 * slot + 1] = la[1]; loc[3 * slot + 2] = la[2];
            pln[3 * slot] = pa[0]; pln[3 * slot + 1] = pa[1]; pln[3 * slot + 2] = 0.0f;
        }
    }
    // refreshContactPoints, last to first
    for (int k = n - 1; k >= 0; k--) {
        float t[3];
        mat3_vec(Rf, loc + 3 * k, t);
        const float dist = (fz + t[2]) - pln[3 * k + 2];
        const float dx = pln[3 * k] - (fx + t[0]), dy = pln[3 * k + 1] - (fy + t[1]);
        if (dist > thr || dx * dx + dy * dy > thr * thr) {
            const int last = n - 1;
            if (k != last) {
                for (int c = 0; c < 3; c++) { loc[3 * k + c] = loc[3 * last + c]; pln[3 * k + c] = pln[3 * last + c]; }
                lam[k] = lam[last];
            }
            lam[last] = 0.0f;
            n = last;
        }
    }
    mn[24] = (float)n;
}

// Rare path of tick_dynamics, part 1: some link box of this robot touches the ground.  Lane b holds box b (touch, centre height
// cz, z components rz of its axes, owning body lane bl) and the world frame Rw / pw of its OWN body; selects the
// PLEN_MAX_BOX_POINTS deepest penetrating vertices of the robot, publishes them in ws.xp in (box, vertex) order and returns
// their number.  Not inlined (see the call site).
PLEN_DEV_NOINLINE int box_points(const DevConfig &cfg, const float *tab, WarpScratch &ws, int lane, bool touch, float cz, float rz0,
                                 float rz1, float rz2, int bl, float R0, float R1, float R2, float R3, float R4, float R5, float R6,
                                 float R7, float R8, float p0, float p1, float p2) {
    const float Rw[9] = {R0, R1, R2, R3, R4, R5, R6, R7, R8}, pw[3] = {p0, p1, p2};
    const float rz[3] = {rz0, rz1, rz2};
    float az[3];
#pragma unroll
    for (int k = 0; k < 3; k++) az[k] = rz[k] * tab[(T_BOX_H + k) * 32 + lane];
    int nx = 0;
    // incident face: axis ks most aligned with the ground normal (first maximum), walked towards the ground;
    // vertex v = (+-) along ki = ks + 1, (+-) along kj = ks + 2 (mod 3), bit 0 / bit 1 of v
    const int ks = (fabsf(rz[1]) > fabsf(rz[0])) ? ((fabsf(rz[2]) > fabsf(rz[1])) ? 2 : 1) : ((fabsf(rz[2]) > fabsf(rz[0])) ? 2 : 0);
    const float zs = (ks == 0) ? az[0] : ((ks == 1) ? az[1] : az[2]);
    const float zi = (ks == 0) ? az[1] : ((ks == 1) ? az[2] : az[0]);
    const float zj = (ks == 0) ? az[2] : ((ks == 1) ? az[0] : az[1]);
    float depth[4];
    unsigned cand = 0;
#pragma unroll
    for (int v = 0; v < 4; v++) {
        const float vz = cz - fabsf(zs) + ((v & 1) ? zi : -zi) + ((v & 2) ? zj : -zj);
        depth[v] = -vz;
        if (touch && depth[v] >= 0.0f) cand |= 1u << v;
    }
    unsigned mine = 0;
    for (int q = 0; q < PLEN_MAX_BOX_POINTS; q++) {
        float bd = -1.0f;
        int bv = 0;
#pragma unroll
        for (int v = 0; v < 4; v++)
            if (((cand & ~mine) >> v) & 1u) { if (depth[v] > bd) { bd = depth[v]; bv = v; } }
        const unsigned key = (bd >= 0.0f) ? f_bits(bd) + 1u : 0u;     // depth >= 0: the bit pattern orders like the value
        const unsigned best = redux_max(key);
        if (best == 0u) break;
        if (lane == lowest_bit(ballot(key == best))) mine |= 1u << bv;
        nx++;
    }
    if (nx) {
        // slots in (box, vertex) order; the owning lane publishes point, depth, body lane and restitution factor
        int below = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) below += popc_(ballot((mine >> b) & 1u) & ((1u << lane) - 1u));
        float Rb[9], pb[3];
#pragma unroll
        for (int k = 0; k < 9; k++) Rb[k] = shfl(Rw[k], bl);
#pragma unroll
        for (int k = 0; k < 3; k++) pb[k] = shfl(pw[k], bl);
        if (mine) {
            float ax[3][3], c[3];     // ax[k] = box axis k in world axes times its half extent; c = box centre rel. base origin
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const float h = tab[(T_BOX_H + k) * 32 + lane];
#pragma unroll
                for (int r = 0; r < 3; r++)
                    ax[k][r] = (Rb[3 * r] * tab[(T_BOX_R + k) * 32 + lane] + Rb[3 * r + 1] * tab[(T_BOX_R + 3 + k) * 32 + lane] +
                                Rb[3 * r + 2] * tab[(T_BOX_R + 6 + k) * 32 + lane]) * h;
            }
#pragma unroll
            for (int r = 0; r < 3; r++)
                c[r] = pb[r] + Rb[3 * r] * tab[(T_BOX_C + 0) * 32 + lane] + Rb[3 * r + 1] * tab[(T_BOX_C + 1) * 32 + lane] +
                       Rb[3 * r + 2] * tab[(T_BOX_C + 2) * 32 + lane];
            const float sg = (zs > 0.0f) ? -1.0f : 1.0f;
            int slot = below;
#pragma unroll
            for (int v = 0; v < 4; v++) {
                if (!((mine >> v) & 1u)) continue;
                const float si = (v & 1) ? 1.0f : -1.0f, sj = (v & 2) ? 1.0f : -1.0f;
#pragma unroll
                for (int r = 0; r < 3; r++) {
                    const float as_ = (ks == 0) ? ax[0][r] : ((ks == 1) ? ax[1][r] : ax[2][r]);
                    const float ai_ = (ks == 0) ? ax[1][r] : ((ks == 1) ? ax[2][r] : ax[0][r]);
                    const float aj_ = (ks == 0) ? ax[2][r] : ((ks == 1) ? ax[0][r] : ax[1][r]);
                    ws.xp[slot][r] = c[r] + sg * as_ + si * ai_ + sj * aj_;
                }
                ws.xp[slot][3] = depth[v];
                ws.xp[slot][4] = (float)bl;
                ws.xp[slot][5] = tab[T_BOX_REST * 32 + lane];
                slot++;
            }
        }
        warp_sync();
    }
    return nx;
}

// Rare path of tick_dynamics, part 2: the rows of the nx selected box contact points (ws.xp), as explicit operational-space vectors.
// For a unit impulse along direction d at point p of body b, with generalized Jacobian Jg (support: base lanes 0..5 and the
// chain of b) and response Bg = M^-1 Jg^T:
//   Jx: base twist = right-foot twist - sum_{j in right leg} s_j qd_j   =>   slots of the right-foot twist carry Jg_base,
//       a right-leg joint carries Jg_j - Jg_base . s_j, any other joint Jg_j
//   Bx = [Bg_joints; Jfoot_right Bg; Jfoot_left Bg],   Bb = Bg_base
// Scratch: ws.red (free after the solve record is out).  Not inlined: keeps the rare path's registers out of k_dyn's hot path.
PLEN_DEV_NOINLINE void box_rows(const DevConfig &cfg, const float *tab, WarpScratch &ws, int lane, float vstar, int nx, float *srx) {
    float *Jg = ws.red, *Bg = ws.red + 96;      // [3][32] each
    const int flR = cfg.foot_lane[0], flL = cfg.foot_lane[1];
    if (lane == 0) srx[XR_NX] = (float)nx;
    for (int q = 0; q < nx; q++) {
        const float px = ws.xp[q][0], py = ws.xp[q][1], pz = ws.xp[q][2], depth = ws.xp[q][3];
        const int bl = (int)ws.xp[q][4];
        const float restf = ws.xp[q][5];
        const int bcs = (int)tab[T_CS * 32 + bl];
        const bool sup = lane < 6 || (bl >= 6 && lane >= bcs && lane <= bl);
        float a[3] = {0, 0, 0}, m[3] = {0, 0, 0};
        if (lane < 24) {
#pragma unroll
            for (int k = 0; k < 3; k++) { a[k] = ws.tw[lane][k]; m[k] = ws.tw[lane][3 + k]; }
        }
        // r = 0: normal +z; r = 1: t1 = (0,-1,0); r = 2: t2 = (1,0,0)  (btPlaneSpace1 of +z, the oracle's order)
        float jg[3];
        jg[0] = a[0] * py - a[1] * px + m[2];
        jg[1] = a[0] * pz - a[2] * px - m[1];
        jg[2] = a[1] * pz - a[2] * py + m[0];
        warp_sync();
#pragma unroll
        for (int r = 0; r < 3; r++) { jg[r] = (sup && lane < 24) ? jg[r] : 0.0f; Jg[32 * r + lane] = jg[r]; }
        warp_sync();
        float bg[3] = {0, 0, 0};
        if (lane < 24) {
            for (int j = 0; j < 6; j++) {
                const float w = ws.minv[j][lane];
#pragma unroll
                for (int r = 0; r < 3; r++) bg[r] += w * Jg[32 * r + j];
            }
            if (bl >= 6)
                for (int j = bcs; j <= bl; j++) {
                    const float w = ws.minv[j][lane];
#pragma unroll
                    for (int r = 0; r < 3; r++) bg[r] += w * Jg[32 * r + j];
                }
        }
#pragma unroll
        for (int r = 0; r < 3; r++) Bg[32 * r + lane] = bg[r];
        warp_sync();
#pragma unroll
        for (int r = 0; r < 3; r++) {
            float d = jg[r] * bg[r], rel = jg[r] * vstar;
            warp_sum2(d, rel);
            const float dinv = (d > 1.1920929e-7f) ? rcp_(d) : 0.0f;
            float rhs;
            if (r == 0) {
                const float pdist = -depth + cfg.linear_slop;
                float rest = (fabsf(rel) < cfg.rest_thresh) ? 0.0f : cfg.restitution * restf * -rel;
                rest = fmaxf(rest, 0.0f);
                float velerr = rest - rel, poserr = 0.0f;
                if (pdist > 0.0f) velerr -= pdist * cfg.inv_dt; else poserr = -pdist * cfg.erp_contact_over_dt;
                rhs = (poserr + velerr) * dinv;
            } else {
                rhs = -rel * dinv;
            }
            // operational-space vectors, word i = lane
            const int i = lane;
            float jx = 0.0f, bx = 0.0f;
            const float *jr = Jg + 32 * r, *br = Bg + 32 * r;
            if (i < 18) {
                const int j = 6 + i;
                jx = jr[j];
                if (j >= flR - 5 && j <= flR) {
#pragma unroll
                    for (int k = 0; k < 6; k++) jx -= jr[k] * ws.tw[j][k];
                }
                bx = br[j];
            } else if (i < 24 || i >= 26) {
                const int c = (i < 24) ? i - 18 : i - 26, fl = (i < 24) ? flR : flL;
                jx = (i < 24) ? jr[c] : 0.0f;
                bx = br[c];
                for (int j = fl - 5; j <= fl; j++) bx += ws.tw[j][c] * br[j];
            }
            float *row = srx + XR_ROWS + (3 * q + r) * XR_ROW_WORDS;
            row[XR_J + lane] = jx;
            row[XR_B + lane] = bx;
            if (lane < 6) row[XR_BB + lane] = br[lane];
            if (lane == 0) { row[XR_RHS] = rhs; row[XR_DINV] = dinv; row[XR_D] = d; }
        }
    }
    warp_sync();
}

}  // namespace plen
