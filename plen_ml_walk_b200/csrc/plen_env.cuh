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

// post-reset snapshot: record (96) | observation (26, padded to 32) | sole manifolds (PLEN_MAN_WORDS).  The per-robot reset rows
// of plen_settle_env_resets / plen_set_env_resets have the same layout, one row per robot.
#define PLEN_SNAP_MAN (PLEN_STATE_WORDS + 32)
#define PLEN_SNAP_WORDS (PLEN_SNAP_MAN + PLEN_MAN_WORDS)

// Record of a robot teleported to base position (x, y, z) with heading yaw about world z, quaternion (0, 0, sin(yaw/2),
// cos(yaw/2)): zero joints, velocities, contact cache and bookkeeping (plen_env.py:561-565), before the settle ticks.
// init_record (plen_host_tables.h) is the case cfg.start_pos, yaw 0.  The half-angle sine and cosine are taken in double and
// rounded once, so that a host building the same quaternion in float64 gets the same float32 words.
PLEN_DEV void start_record(float x, float y, float z, float yaw, float *rec /* [96] */) {
    for (int w = 0; w < PLEN_STATE_WORDS; w++) rec[w] = 0.0f;
    rec[W_POS] = x; rec[W_POS + 1] = y; rec[W_POS + 2] = z;
    const double h = 0.5 * (double)yaw;
    rec[W_QUAT + 2] = (float)sin(h);
    rec[W_QUAT + 3] = (float)cos(h);
}

struct StepIO {
    const float *action;      // [18] this env
    float *obs;               // [26]
    float *reward;            // scalar
    uint8_t *done, *timeout;  // scalars (timeout nullable)
    float *terminal_obs;      // [26] nullable
    const float *snapshot;    // [96 + 26] post-reset record and its observation: the shared snapshot or the robot's own reset row
    unsigned long long *faults;   // device counter of numeric faults (nullable)
    float *man;               // this robot's persistent sole manifold (sole_manifold = 1), nullable: reset with the record
    // observation noise (plen_set_env_obs_noise; read by env_post<true> only)
    float *noise;             // [ON_WORDS] this robot's noise row
    float *clean_obs;         // [26] the noise-free obs
    float *clean_tobs;        // [26] the noise-free terminal obs, written where done
    unsigned long long nkey;  // obs_noise_base(seed, first_env_id + robot)
};

// ---- observation noise (plen_set_env_obs_noise) ------------------------------------------------------------------
// Noise row of a robot, ON_WORDS floats: sigma [24] | bias std beta [24] | bias b of the running episode [24] | flip p | draw
// counter (uint32 bits) | padding.  Continuous words w = 0..23 of an observation the agent receives become
//   clean_w + fmaf(sigma_w, n, b_w)   (passed through bit for bit where sigma_w == 0 and b_w == 0),
// contact flags w = 24, 25 become 1 - clean_w with probability p.  No clipping, no angle wrapping.  b_w = beta_w * n' is drawn
// at every reset of the robot and kept for its episode.  Draws are counter-based:
//   key(w, s) = mix64(seed ^ mix64(gid)) + (counter << 8) + (s << 5) + w       (uint64 arithmetic, gid = first_env_id + robot)
//   hash32(k) = mix64(k) >> 32,  mix64 = the splitmix64 finaliser (x += 0x9E3779B97F4A7C15, then the two xor-shift-multiplies
//               and the final x ^ (x >> 31))
//   n = sqrtf(-2 logf(u1)) * cospif(2 u2),  u1 = ((float)hash32(k) + 1) * 2.3283064e-10f,
//       u2 = (float)hash32(k ^ 0xA5A5A5A5DEADBEEF) * 2.3283064e-10f                  (the generator of plen_actor_forward)
//   flip where (uint64)hash32(k) < (uint64)((double)p * 2^32)                       (p = 0 never flips, p = 1 always)
// Streams s: the step's obs noise, its flips, the new episode's bias, the reset obs noise, its flips.  k_post draws with the
// counter and then increments it once; k_reset does the same once per robot it resets.
enum { ON_SIGMA = 0, ON_BETA = 24, ON_BIAS = 48, ON_FLIP = 72, ON_CTR = 73, ON_WORDS = 96 };
enum { NS_OBS = 0, NS_FLIP = 1, NS_BIAS = 2, NS_ROBS = 3, NS_RFLIP = 4 };

PLEN_DEV uint64_t mix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
PLEN_DEV uint32_t noise_hash32(uint64_t k) { return (uint32_t)(mix64(k) >> 32); }
PLEN_DEV uint64_t obs_noise_base(unsigned long long seed, long long gid) { return mix64(seed ^ mix64((uint64_t)gid)); }
PLEN_DEV uint64_t obs_noise_key(uint64_t base, unsigned ctr, int stream, int word) {
    return base + ((uint64_t)ctr << 8) + ((uint64_t)stream << 5) + (uint64_t)word;
}
// float with the given bit pattern (the inverse of f_bits): the draw counter travels in a float word of the noise row
#ifndef PLEN_HOST_EMU
PLEN_DEV float bits_f(unsigned u) { return __uint_as_float(u); }
#else
PLEN_DEV float bits_f(unsigned u) { float32_t_ f; std::memcpy(&f, &u, 4); return (float)f; }
#endif
PLEN_DEV float noise_u1(uint64_t k) { return ((float)noise_hash32(k) + 1.0f) * 2.3283064e-10f; }
PLEN_DEV float noise_u2(uint64_t k) { return (float)noise_hash32(k ^ 0xA5A5A5A5DEADBEEFull) * 2.3283064e-10f; }
PLEN_DEV float noise_normal(uint64_t k) {
    const float u1 = noise_u1(k), u2 = noise_u2(k);
#ifndef PLEN_HOST_EMU
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
#else   // the host has no cospif: libm in double, rounded to the build's precision
    return (float)(std::sqrt(-2.0 * std::log((double)u1)) * std::cos(3.14159265358979323846 * (double)(2.0f * u2)));
#endif
}
PLEN_DEV bool noise_flip(uint64_t k, float p) { return (uint64_t)noise_hash32(k) < (uint64_t)((double)p * 4294967296.0); }

// one observation word through the noise of its lane: a continuous word (lane < 24) with sigma, b and the Gaussian of stream
// s, a contact flag (lanes 24, 25) with flip probability p and stream s + 1
PLEN_DEV float obs_noise_word(float x, int lane, float sigma, float b, float p, uint64_t base, unsigned ctr, int s) {
    if (lane < 24) return (sigma == 0.0f && b == 0.0f) ? x : x + fmaf(sigma, noise_normal(obs_noise_key(base, ctr, s, lane)), b);
    return noise_flip(obs_noise_key(base, ctr, s + 1, lane), p) ? 1.0f - x : x;
}

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
// NOISE: observation noise at the obs / terminal_obs stores (io.noise), the clean words into io.clean_obs / io.clean_tobs;
// everything else -- reward, done, counters, the record -- is the stock computation on the true state.
template <bool NOISE = false>
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
    if constexpr (NOISE) {
        // this lane's noise parameters: sigma, b of the running episode and beta for words 0..23, p for the flags
        const float *nr = io.noise;
        const unsigned ctr = f_bits(nr[ON_CTR]);
        const float sigma = lane < 24 ? nr[ON_SIGMA + lane] : 0.0f, b = lane < 24 ? nr[ON_BIAS + lane] : 0.0f;
        const float beta = lane < 24 ? nr[ON_BETA + lane] : 0.0f, p = nr[ON_FLIP];
        const float x = lane < 26 ? ws.obs[lane] : 0.0f;
        if ((done && cfg.auto_reset) || fault) {
            const float tx = (lane < 26 && fault) ? io.snapshot[96 + lane] : x;
            if (lane < 26) {      // the finished episode's terminal observation carries its own bias
                io.clean_tobs[lane] = tx;
                if (io.terminal_obs) io.terminal_obs[lane] = obs_noise_word(tx, lane, sigma, b, p, io.nkey, ctr, NS_OBS);
            }
            load_record(io.snapshot, ws, L, lane);
            const float nb = lane < 24 ? beta * noise_normal(obs_noise_key(io.nkey, ctr, NS_BIAS, lane)) : 0.0f;
            if (lane < 26) {
                const float rx = io.snapshot[96 + lane];
                io.clean_obs[lane] = rx;
                io.obs[lane] = obs_noise_word(rx, lane, sigma, nb, p, io.nkey, ctr, NS_ROBS);
            }
            if (lane < 24) io.noise[ON_BIAS + lane] = nb;
            if (io.man) {
                for (int w = lane; w < PLEN_MAN_WORDS; w += 32) io.man[w] = io.snapshot[PLEN_SNAP_MAN + w];
            }
        } else if (lane < 26) {
            const float y = obs_noise_word(x, lane, sigma, b, p, io.nkey, ctr, NS_OBS);
            io.clean_obs[lane] = x;
            io.obs[lane] = y;
            if (done) {
                io.clean_tobs[lane] = x;
                if (io.terminal_obs) io.terminal_obs[lane] = y;
            }
        }
        warp_sync();      // every lane has read the counter
        if (lane == 0) io.noise[ON_CTR] = bits_f(ctr + 1u);
    } else if ((done && cfg.auto_reset) || fault) {
        // the reference caller resets after a terminal step (plen_td3.py:122-129); the reset is deterministic
        // (fixed pose + 8 ticks, plen_env.py:561-570) so the post-reset record is precomputed: the shared snapshot, or the
        // robot's own row settled under its parameters (plen_settle_env_resets)
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
