// plen_env.cuh -- env logic around the physics ticks: agent_to_env (before), observation -> done -> reward ->
// counters -> auto-reset (after), one warp per robot.  Restates PlenWalkEnv.step (plen_bullet/src/plen_bullet/plen_env.py
// :638-692) with the running-sum form of the joint histories (SURVEY.md Appendix C); citations inline.
#pragma once

#include "plen_device.cuh"

namespace plen {

// ---- state record <-> lane registers ---------------------------------------------------------------------------
// r0..r2: this lane's words lane, 32 + lane, 64 + lane of the record (already fetched, so the fetch can overlap other loads)
PLEN_DEV void unpack_record(float r0, float r1, float r2, WarpScratch &ws, LaneState &L, int lane);
PLEN_DEV void load_record(const float *rec, WarpScratch &ws, LaneState &L, int lane) {
    unpack_record(gld(rec + lane), gld(rec + 32 + lane), gld(rec + 64 + lane), ws, L, lane);
}
PLEN_DEV void unpack_record(float r0, float r1, float r2, WarpScratch &ws, LaneState &L, int lane) {
    ws.st[lane] = r0;
    ws.st[32 + lane] = r1;
    ws.st[64 + lane] = r2;
    warp_sync();
    L.u = (lane < 24) ? ws.st[W_U + lane] : 0.0f;
    L.lam = (lane >= 24) ? ws.st[W_U + lane] : 0.0f;
    L.q = (lane >= 6 && lane < 24) ? ws.st[W_Q + lane] : 0.0f;
    L.tgt = 0.0f;
#pragma unroll
    for (int k = 0; k < 3; k++) L.pos[k] = ws.st[W_POS + k];
#pragma unroll
    for (int k = 0; k < 4; k++) L.quat[k] = ws.st[W_QUAT + k];
    L.man = (unsigned)ws.st[W_MAN];
    L.iters = 0;
    L.fric_s = L.motor_s = L.kp_s = 1.0f;
}

PLEN_DEV void store_record(float *rec, WarpScratch &ws, const LaneState &L, int lane) {
    warp_sync();
    ws.st[W_U + lane] = (lane < 24) ? L.u : L.lam;
    if (lane >= 6 && lane < 24) ws.st[W_Q + lane] = L.q;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) ws.st[W_POS + k] = L.pos[k];
#pragma unroll
        for (int k = 0; k < 4; k++) ws.st[W_QUAT + k] = L.quat[k];
        ws.st[W_MAN] = (float)L.man;
    }
    warp_sync();
    rec[lane] = ws.st[lane];
    rec[32 + lane] = ws.st[32 + lane];
    rec[64 + lane] = ws.st[64 + lane];
}

// pybullet getEulerFromQuaternion (plen_env.py:799-800) incl. the +-0.99999 gimbal branches
PLEN_DEV void quat_to_euler(const float *q, float *rpy) {
    const float x = q[0], y = q[1], z = q[2], w = q[3];
    const float sarg = -2.0f * (x * z - w * y);
    if (sarg <= -0.99999f) { rpy[1] = -1.57079632679f; rpy[0] = 0.0f; rpy[2] = 2.0f * atan2f(x, -y); }
    else if (sarg >= 0.99999f) { rpy[1] = 1.57079632679f; rpy[0] = 0.0f; rpy[2] = 2.0f * atan2f(-x, y); }
    else {
        rpy[0] = atan2f(2.0f * (y * z + w * x), w * w - x * x - y * y + z * z);
        rpy[1] = asinf(sarg);
        rpy[2] = atan2f(2.0f * (x * y + w * z), w * w + x * x - y * y - z * z);
    }
}

// compute_observation (plen_env.py:768-822) into ws.obs[0..25]; no history side effects
PLEN_DEV void observe(WarpScratch &ws, const LaneState &L, int lane) {
    const float vx = shfl(L.u, 3);
    float rpy[3];
    quat_to_euler(L.quat, rpy);
    warp_sync();
    if (lane >= 6 && lane < 24) ws.obs[lane - 6] = L.q;                        // :807-814
    if (lane == 0) {
        ws.obs[18] = L.pos[2]; ws.obs[19] = vx; ws.obs[20] = rpy[0]; ws.obs[21] = rpy[1]; ws.obs[22] = rpy[2];
        ws.obs[23] = L.pos[1];
        ws.obs[24] = (L.man & 0x0Fu) ? 1.0f : 0.0f;                            // right foot, link 11, :784-790
        ws.obs[25] = (L.man & 0xF0u) ? 1.0f : 0.0f;                            // left foot, link 19, :774-782
    }
    warp_sync();
}

// post-reset snapshot: record (96) | observation (26, padded to 32) | sole manifolds (PLEN_MAN_WORDS)
#define PLEN_SNAP_MAN (PLEN_STATE_WORDS + 32)
#define PLEN_SNAP_WORDS (PLEN_SNAP_MAN + PLEN_MAN_WORDS)

struct StepIO {
    const float *action;      // [18] this env
    float *obs;               // [26]
    float *reward;            // scalar
    uint8_t *done, *timeout;  // scalars (timeout nullable)
    float *terminal_obs;      // [26] nullable
    const float *snapshot;    // [96 + 26] post-reset record and its observation
    unsigned long long *faults;   // device counter of numeric faults (nullable)
    float *man;               // this robot's persistent sole manifold (sole_manifold = 1), nullable: reset with the record
};

// env_ranges of plen_env.py:148-167 are kept in double so that the a = +-1 inset branch (plen_env.py:707-711) takes
// the same side as the reference's float64 arithmetic.
struct EnvRanges { double lo[18], hi[18]; };

// agent_to_env (plen_env.py:694-714), bypassed when joint_act (:652-654): servo target of joint j for action `act`
PLEN_DEV float agent_target(const DevConfig &cfg, const EnvRanges &rng, int j, float act) {
    if (cfg.joint_act) return act;
    const double lo = rng.lo[j], hi = rng.hi[j];
    const double mm = (hi - lo) / (1.0 - (-1.0));
    const double b = hi - (mm * 1.0);
    double y = mm * (double)act + b;
    if (y >= hi) y = hi - 0.001; else if (y <= lo) y = lo + 0.001;
    return (float)y;
}

// Per-robot command latency (plen_set_env_latency): tick k (0 <= k < S = substeps) of an env step applies the raw targets
// of the step s = ceil(max(d - k, 0) / S) steps back, s = 0, 1 or 2 for a delay of 0 <= d <= 2 S ticks.  ep_t is the
// robot's episode counter (steps since its last reset) at this step; a command from before that reset is the reset-pose
// hold target 0, returned as -1.
PLEN_DEV int latency_source(int d, int k, int S, int ep_t) {
    const int late = d - k;
    const int s = late > 0 ? (late + S - 1) / S : 0;
    return (s == 0 || s <= ep_t) ? s : -1;
}
// ring row (LAT_SLOTS rows per robot) of the targets s steps before the step with episode counter ep_t (0 <= s <= 2, ep_t >= 0)
PLEN_DEV int latency_slot(int ep_t, int s) { return (ep_t + LAT_SLOTS - s) % LAT_SLOTS; }

// Everything of PlenWalkEnv.step after the 4 physics ticks (:671-678) + TimeLimit + optional auto-reset (k_post).
PLEN_DEV void env_post(const DevConfig &cfg, const float *tab, WarpScratch &ws, LaneState &L, int lane,
                       const StepIO &io) {
    // ---- compute_observation (:768-871)
    observe(ws, L, lane);
    const float z = ws.obs[18], vx = ws.obs[19], roll = ws.obs[20], pitch = ws.obs[21], yaw = ws.obs[22], y = ws.obs[23];
    const bool Rc = ws.obs[24] != 0.0f, Lc = ws.obs[25] != 0.0f;
    // foot link orientation (getLinkState(...)[1], :1016, :1029): flat test |roll|,|pitch| <= 0.1
    bool flat = false;
    {
        float Rw[9], pw[3];
        forward_kinematics(tab, lane, L.q, L.quat, Rw, pw);
        const float sarg = -Rw[6];
        if (sarg > -0.99999f && sarg < 0.99999f)
            flat = fabsf(atan2f(Rw[7], Rw[8])) <= 0.1f && fabsf(asinf(sarg)) <= 0.1f;
    }
    const unsigned flat_bits = ballot(flat);
    const bool flatR = (flat_bits >> cfg.foot_lane[0]) & 1u, flatL = (flat_bits >> cfg.foot_lane[1]) & 1u;

    // joint-angle histories as running sums; pairs (JointStates[2],[8]), ([3],[9]), ([4],[10])  (:825-866)
    float cur[6];
    cur[0] = shfl(L.q, 8); cur[1] = shfl(L.q, 14); cur[2] = shfl(L.q, 9); cur[3] = shfl(L.q, 15);
    cur[4] = shfl(L.q, 10); cur[5] = shfl(L.q, 16);
    int cnt = (int)ws.st[W_CNT], ds = (int)ws.st[W_DS], hist = (int)ws.st[W_HIST], ept = (int)ws.st[W_EPT];
    float epret = ws.st[W_EPRET];
    float diff[6], sums[9];
    const bool first_pass = !(hist > 0);
#pragma unroll
    for (int k = 0; k < 6; k++) diff[k] = first_pass ? 0.0f : ws.st[W_LAST + k] - cur[k];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        sums[3 * k] = ws.st[W_SUMS + 3 * k] + cur[2 * k] * cur[2 * k + 1];
        sums[3 * k + 1] = ws.st[W_SUMS + 3 * k + 1] + cur[2 * k] * cur[2 * k];
        sums[3 * k + 2] = ws.st[W_SUMS + 3 * k + 2] + cur[2 * k + 1] * cur[2 * k + 1];
    }
    hist += 1;

    // ---- per-env numeric guard (SURVEY.md section 5; the reference has none): a robot whose physical state went
    //      non-finite is retired as a fall -- done, the dead penalty alone as its (finite) reward, forced reset from the
    //      snapshot whether or not auto_reset is on -- and counted (plen_fault_count).  A NaN REWARD out of the 0/0 cosine
    //      similarity of a finite state is reference behaviour (E5, plen_env.py:929-945) and is left alone.
    bool fin = isfinite(L.u) && isfinite(L.q);
    if (lane == 0) fin = fin && isfinite(L.pos[0] + L.pos[1] + L.pos[2] + L.quat[0] + L.quat[1] + L.quat[2] + L.quat[3]);
    const bool fault = ballot(!fin) != 0u;

    // ---- compute_done (:1072-1093), one-sided
    const bool dead = fault || (roll > 1.0471975511965976f) || (pitch > 1.0471975511965976f) || (z < 0.08f) || (y > 1.0f);

    // ---- compute_reward (:873-1070)
    float r = 0.0f;                                                        // alive_reward = 0 (:65)
    if (vx < 0.0f) r -= expf(vx * 3.0f); else r += (vx * 3.0f) * (vx * 3.0f);   // :885-889
    { const float hh = fabsf(0.160178937611f - z) * 40.0f; r -= hh * hh; }      // :894-895
    r -= y * y; r -= roll * roll; r -= 0.5f * pitch * pitch; r -= yaw * yaw;    // :901-907
    float jrew = 0.0f, jpen = 0.0f;
    if (cnt >= 80 && Rc) {                                                 // :913-923
        hist = 0; cnt = 0; ds = 0;
#pragma unroll
        for (int k = 0; k < 9; k++) sums[k] = 0.0f;
    } else if (cnt >= 120) {                                               // :924-925
        r -= 2.0f;
    } else if (cnt > 0) {                                                  // :926-968
#pragma unroll
        for (int k = 0; k < 3; k++) jrew += sums[3 * k] / (sqrtf(sums[3 * k + 1]) * sqrtf(sums[3 * k + 2]));
        jrew *= (1.0f / 3.0f);
        if (!first_pass) {
#pragma unroll
            for (int k = 0; k < 6; k++) jpen -= 1.0f / expf(fabsf(diff[k]));
            jpen *= 0.5f * (1.0f / 3.0f);
        }
    }
    r += jrew; r += jpen;                                                  // :972-973
    if (Lc) { const float aa = (cnt * 10.0f / 80.0f) - 5.0f; r += 0.5f * (1.0f - tanhf(aa * aa)); }   // :978-982
    if (cnt < 40) { if (Rc && !Lc) r += 0.1f; else if (!Rc) r -= 0.1f; }   // :988-994
    else if (cnt < 80) { if (Lc && !Rc) r += 0.1f; else if (!Lc) r -= 0.1f; }   // :995-1001
    if (Rc && Lc) { ds += 1; if (ds >= 16) r -= 2.0f; }                    // :1004-1007
    if (Lc && flatL) r += 0.1f;                                            // :1014-1023
    if (Rc && flatR) r += 0.1f;                                            // :1027-1036
    if (dead) r -= 100.0f;                                                 // :1057-1059
    if (fault) r = -100.0f;
    // ---- bookkeeping (:674-678) and the TimeLimit wrapper (:15-19)
    epret += r; ept += 1; cnt += 1;
    const bool timeout = !dead && (ept >= cfg.max_episode_steps);
    const bool done = dead || timeout;

    warp_sync();
    if (lane == 0) {
        ws.st[W_CNT] = (float)cnt; ws.st[W_DS] = (float)ds; ws.st[W_HIST] = (float)hist; ws.st[W_EPT] = (float)ept;
        ws.st[W_EPRET] = epret;
        *io.reward = r;
        *io.done = done ? 1 : 0;
        if (io.timeout) *io.timeout = timeout ? 1 : 0;
#ifndef PLEN_HOST_EMU
        if (fault && io.faults) atomicAdd(io.faults, 1ull);
#else
        if (fault && io.faults) *io.faults += 1ull;
#endif
    }
    if (lane < 6) ws.st[W_LAST + lane] = cur[lane];
    if (lane >= 6 && lane < 15) {
        float v = sums[0];
#pragma unroll
        for (int k = 1; k < 9; k++) v = (lane - 6 == k) ? sums[k] : v;
        ws.st[W_SUMS + (lane - 6)] = v;
    }
    warp_sync();
    if ((done && cfg.auto_reset) || fault) {
        // the reference caller resets after a terminal step (plen_td3.py:122-129); the reset is deterministic
        // (fixed pose + 8 ticks, plen_env.py:561-570) so the post-reset record is a constant snapshot
        if (io.terminal_obs && lane < 26) io.terminal_obs[lane] = fault ? io.snapshot[96 + lane] : ws.obs[lane];
        load_record(io.snapshot, ws, L, lane);
        if (lane < 26) io.obs[lane] = io.snapshot[96 + lane];
        if (io.man) {       // the manifolds of the post-reset snapshot sit behind its record and observation
            for (int w = lane; w < PLEN_MAN_WORDS; w += 32) io.man[w] = io.snapshot[PLEN_SNAP_MAN + w];
        }
    } else {
        if (lane < 26) io.obs[lane] = ws.obs[lane];
        if (done && io.terminal_obs && lane < 26) io.terminal_obs[lane] = ws.obs[lane];
    }
}

}  // namespace plen
