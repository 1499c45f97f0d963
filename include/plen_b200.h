/* plen_b200.h -- C ABI of the B200-native batched PLEN walking environment (libplen_b200.so).
 *
 * Drop-in boundary for the hot path of moribots/plen_ml_walk: the physics step behind
 * plen_bullet/src/plen_bullet/plen_env.py and the observation / reward / termination / auto-reset logic around
 * it.  In the reference that boundary is the in-process PyBullet C extension (module-global client 0); every entry
 * point below names the reference call(s) it replaces.  Plain pointers and sizes only -- no torch, no C++ types.
 *
 * Conventions
 *   - one ctx per GPU; calls on a ctx are stream-ordered, non-blocking (except *_host) and not re-entrant;
 *   - all *_dev pointers are device memory owned by the caller; the ctx owns the per-env state and model tables;
 *     no allocation happens inside plen_step;
 *   - every function returns 0 on success, a negative PLEN_E_* code otherwise; text via plen_last_error();
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - there is NO CPU fallback: without a CUDA device plen_create fails with PLEN_E_CUDA.
 *
 * Layouts (row-major, float32 unless noted)
 *   actions  [N,18]  agent space [-1,1] (or raw radians when config.joint_act), joint order plen_env.py:547-554
 *   obs      [N,26]  [q1..q18, z, vx, roll, pitch, yaw, y, right_contact, left_contact]   (plen_env.py:816-822)
 *   qpos     [N,25]  [pos xyz, quat xyzw, q1..q18]
 *   qvel     [N,24]  [v_lin world xyz, omega world xyz, qd1..qd18]
 *   aux      [N,PLEN_AUX_WORDS]  [lam_n[8], manifold bits, cnt, ds, hist_len, ep_t, last[6], sums[9], ep_ret]
 */
#ifndef PLEN_B200_H
#define PLEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLEN_LANES 24          /* 6 base velocity coordinates + 18 joints */
#define PLEN_NJ 18
#define PLEN_OBS 26
#define PLEN_QPOS 25
#define PLEN_QVEL 24
#define PLEN_AUX_WORDS 29
#define PLEN_STATE_WORDS 96    /* per-env state record in HBM: 3 x 128 B lines, one word per lane per line */
#define PLEN_MAX_BOXES 32      /* box colliders besides the two feet (plen.urdf: torso + 30 links): one per lane of a warp */
#define PLEN_MAX_BOX_POINTS 4  /* box-vs-ground contact points kept per robot and tick (the deepest ones) */
#define PLEN_MAX_HULL 256      /* convex-hull vertices of a foot collider (plen.urdf feet: 209 each) */
#define PLEN_BODIES 19         /* rigid bodies of the robot: the torso composite and the body each of the 18 joints moves */
#define PLEN_MAX_LATENCY_STEPS 2   /* command latency (plen_set_env_latency) <= PLEN_MAX_LATENCY_STEPS * substeps ticks */
#define PLEN_MAN_WORDS 52      /* per-robot persistent sole manifold (sole_manifold = 1): [foot][point][local xyz | plane xyz] = 48
                                  floats, the two point counts, 2 spare */

#define PLEN_OK 0
#define PLEN_E_ARG (-1)
#define PLEN_E_CUDA (-2)
#define PLEN_E_STATE (-3)

/* Per-lane articulation tables produced by the URDF loader (plen_ml_walk_b200/urdf_loader.py).
 * Replaces: p.loadURDF("plen.urdf", ...) (plen_env.py:312-315) + the dynamics overrides (plen_env.py:438-481). */
typedef struct {
    float R_pj[PLEN_LANES][9];     /* parent body frame -> joint frame at q = 0, row major (lanes 6..23) */
    float p_pj[PLEN_LANES][3];     /* joint origin in the parent body frame */
    float axis[PLEN_LANES][3];     /* joint axis in the body frame */
    float mass[PLEN_LANES];        /* lane 0 = torso composite; 1..5 unused */
    float com[PLEN_LANES][3];      /* centre of mass in the body frame */
    float inertia[PLEN_LANES][6];  /* xx yy zz xy xz yz about the com, body axes */
    float lower[PLEN_LANES], upper[PLEN_LANES];   /* joint limits (plen.urdf:1310 ...) */
    int32_t chain_start[PLEN_LANES];              /* first lane of the limb this lane belongs to */
    int32_t foot_lane[2];          /* [0] right foot (Bullet link 11), [1] left foot (link 19) */
    float foot_pts[2][4][3];       /* sole contact vertices in the foot body frame */
    float foot_break[2];           /* contact breaking threshold per foot */
    /* Box colliders of every link except the feet (plen.urdf:504-1274), for the ground contact of knees, hands, torso ...
     * (in Bullet every link collider hits plane.urdf; the reference's setCollisionFilterPair loops, plen_env.py:355-434,
     * only concern self-collision).  Bullet link order; pose in the frame of the body (lane) the link is folded into. */
    int32_t n_boxes;
    int32_t box_lane[PLEN_MAX_BOXES];      /* 0 = torso body, 6..23 = limb bodies */
    float box_center[PLEN_MAX_BOXES][3];
    float box_rot[PLEN_MAX_BOXES][9];      /* row major */
    float box_half[PLEN_MAX_BOXES][3];     /* half extents */
    float box_rest[PLEN_MAX_BOXES];        /* factor on config.restitution: 0 for the base link (its restitution stays 0:
                                              it is not in the changeDynamics loop, plen_env.py:476-481), 1 otherwise */
    /* Convex-hull vertices of the two foot colliders in the foot body frame (plen.urdf:1097, :1263 -> the STL meshes):
     * the support-vertex search of the persistent sole manifold (config.sole_manifold = 1) walks them. */
    int32_t n_hull[2];
    float foot_hull[2][PLEN_MAX_HULL][3];
} plen_model;

/* Every constant of the path; defaults = the reference literals (cited) or the PyBullet defaults they rely on. */
typedef struct {
    float dt;                  /* 1/240 s            plen_env.py:41 */
    int32_t substeps;          /* 4                  plen_env.py:40-42 */
    int32_t reset_ticks;       /* 8                  plen_env.py:569-570 */
    float gravity_z;           /* -9.81              plen_env.py:296 */
    float start_pos[3];        /* 0 0 0.158          plen_env.py:312 */
    float motor_max_force;     /* 0.15 N m           plen_env.py:753 */
    int32_t joint_act;         /* raw-radian actions plen_env.py:34, :652-654 */
    float linear_damping;      /* 0 | 0.1            plen_env.py:472-481 */
    float mu_lateral;          /* 0.8*0.8            plen_env.py:309, :444 */
    float mu_spinning;         /* 0.1*0.8            plen_env.py:445 */
    float mu_rolling;          /* (0.1|0.01)*0.8     plen_env.py:439-442 */
    float restitution;         /* 0.5*0.5            plen_env.py:309, :481 */
    double env_lo[PLEN_NJ], env_hi[PLEN_NJ];  /* env_ranges, plen_env.py:148-167 (double: the a=+-1 inset branch
                                                 must fall on the same side as the reference's float64) */
    int32_t max_episode_steps; /* 500                plen_env.py:15-19 */
    float motor_kp, motor_kd;  /* 0.1, 1.0  PyBullet POSITION_CONTROL defaults */
    int32_t solver_iterations; /* 50 */
    float residual_threshold;  /* 1e-7 */
    float erp_contact;         /* 0.08 */
    float erp_joint;           /* 0.2 */
    float linear_slop;         /* 1e-5 */
    float warmstart_factor;    /* 0.1 */
    float restitution_vel_threshold; /* 0.2 */
    float hull_margin;         /* 0.001 */
    float max_coord_velocity;  /* 100 */
    int32_t auto_reset;        /* 1: plen_step resets finished envs in the same launch (the reference leaves it to
                                  the caller, plen_td3.py:122-129) */
    int32_t link_contacts;     /* 1: the box colliders of the non-foot links collide with the ground (default); 0: soles only */
    float mu_link;             /* 0.5*0.8: URDF default lateral friction of a link x the plane's, plen_env.py:309 */
    int32_t sole_manifold;     /* how the sole contact points of a foot come into being.  0 (default): the four extreme sole
                                  corners, each in contact while within the breaking threshold of the ground -- the limiting set
                                  of Bullet's manifold reduction, present from the first tick.  1: as Bullet's
                                  btConvexPlaneCollisionAlgorithm + btPersistentManifold do it ([RECALL]): ONE new point per tick
                                  (the hull's support vertex towards the ground) merged into a cache of <= 4 points per foot
                                  (replace the nearest within the threshold / add / keep the deepest and the largest area), points
                                  that separated or drifted by more than the threshold dropped; impulses travel with the points.
                                  profiles/r2_physics_pin.md section 5: the shipped policy's mean return moves from -5 to +56
                                  against +68 in Bullet. */
    float support_tie;         /* sole_manifold = 1: hull vertices within this distance (m) of the lowest one count as equally
                                  low, and the first of them in the vertex list is the support vertex.  1e-7 (default): a foot flat
                                  on the ground -- the reset pose -- is an exact tie that rounding would decide, differently in
                                  float32 and in the float64 oracle; 0: plain first-minimum search */
} plen_config;

typedef struct plen_ctx plen_ctx;

const char *plen_version(void);

/* Fill `cfg` with the reference defaults (joint_act selects the trajectory_eval.py variant, plen_env.py:439-475). */
int plen_default_config(plen_config *cfg, int joint_act);

/* Replaces PlenWalkEnv.__init__ (plen_env.py:34-556): p.connect / loadURDF / changeDynamics.  Allocates the per-env
 * state for n_envs robots on CUDA device `device`, uploads the tables, and precomputes the post-reset snapshot
 * (the reference reset is deterministic: fixed pose + 8 ticks, plen_env.py:561-570).  NULL on failure
 * (plen_last_error(NULL) has the reason). */
plen_ctx *plen_create(const plen_config *cfg, const plen_model *model, int n_envs, int device);
void plen_destroy(plen_ctx *ctx);
const char *plen_last_error(const plen_ctx *ctx);
int plen_num_envs(const plen_ctx *ctx);
/* Kernels launched so far by plen_reset / plen_step / plen_step_host / plen_tick / plen_settle_env_resets on this context (13
 * per step and range: plen_step_host runs up to four ranges, plen_step of 2,048 robots or more runs two; a settle launches its
 * reset_ticks ticks over the whole batch plus 2); bench.py's gpu_launches reads it. */
unsigned long long plen_kernel_launches(const plen_ctx *ctx);

/* Replaces PlenWalkEnv.reset (plen_env.py:558-614) for the envs whose mask byte is non-zero (NULL = all): each restores the
 * post-reset snapshot, or its own row of the reset table once plen_settle_env_resets / plen_set_env_resets made one.
 * obs_dev may be NULL. */
int plen_reset(plen_ctx *ctx, const uint8_t *mask_dev, float *obs_dev, void *stream);

/* Replaces PlenWalkEnv.step (plen_env.py:638-692) + the TimeLimit wrapper (plen_env.py:15-19) for all N envs:
 * agent_to_env -> motor targets -> 4 ticks (contact, dynamics, PGS, integrate) -> observation -> done -> reward ->
 * counters -> optional auto-reset.  2*substeps+1 kernel launches on `stream` (k_dyn + k_solve per tick, then k_post),
 * no host synchronisation.
 *   obs_dev          [N,26] observation the agent acts on next (the reset observation where done && auto_reset)
 *   reward_dev       [N]
 *   done_dev         [N] uint8, dead || ep_t >= max_episode_steps
 *   timeout_dev      [N] uint8 (nullable), !dead && ep_t >= max_episode_steps (plen_td3.py:109-110 done_bool)
 *   terminal_obs_dev [N,26] (nullable) observation of the finished episode's last step, written where done */
int plen_step(plen_ctx *ctx, const float *actions_dev, float *obs_dev, float *reward_dev, uint8_t *done_dev,
              uint8_t *timeout_dev, float *terminal_obs_dev, void *stream);

/* Same call with HOST buffers (pinned memory recommended): H2D of the actions, the step, D2H of obs / reward / done,
 * and a stream synchronise.  This is the end-to-end path a PyBullet user would see.
 * Ordering contract: the call runs on the context's PRIVATE streams (the batch is pipelined in ranges).  It first waits
 * (cudaStreamWaitEvent) for the work the last plen_reset / plen_step / plen_set_state / plen_set_manifold / plen_set_env_scales /
 * plen_set_env_mass / plen_set_env_latency / plen_settle_env_resets / plen_set_env_resets / plen_clear_env_resets /
 * plen_set_env_obs_noise / plen_set_env_obs_noise_state / plen_clear_env_obs_noise / plen_tick call queued on its caller stream, so `plen_reset(...); plen_step_host(...)`
 * needs no synchronisation in between; it
 * returns after its own streams have drained, so whatever the caller queues next is ordered after it.  (Work the caller
 * queued on a stream WITHOUT going through this library -- e.g. a torch kernel still writing the state through
 * plen_set_state's source buffer -- is the caller's to order.) */
int plen_step_host(plen_ctx *ctx, const float *actions_host, float *obs_host, float *reward_host,
                   uint8_t *done_host, uint8_t *timeout_host);

/* Numeric guard (SURVEY.md section 5; the reference's Bullet env has none, its Gazebo twin shuts ROS down on a NaN
 * reward, robot_gazebo_env.py:180-185): a robot whose physical state is non-finite after a step is reported done with
 * reward -100 and reset from the snapshot (even when auto_reset is off).  Returns how many robots that has happened to
 * since plen_create; synchronises the device. */
int plen_fault_count(plen_ctx *ctx, unsigned long long *count_host);

/* Replaces getBasePositionAndOrientation / getJointStates / getBaseVelocity (plen_env.py:771-773) and
 * resetBasePositionAndOrientation / resetJointState (plen_env.py:561-565) for all envs; any pointer may be NULL. */
int plen_get_state(plen_ctx *ctx, float *qpos_dev, float *qvel_dev, float *aux_dev, void *stream);
int plen_set_state(plen_ctx *ctx, const float *qpos_dev, const float *qvel_dev, const float *aux_dev, void *stream);

/* The persistent sole manifolds (config.sole_manifold = 1; PLEN_E_STATE otherwise): [N,PLEN_MAN_WORDS] device floats, per robot
 * [foot 0|1][point 0..3][x y z of the point on the inflated hull in the foot frame | x y z of its partner on the plane, world]
 * followed by the two point counts (as floats).  The cached normal impulses of the points are words of the state record
 * (plen_get_state's aux).  Used by the teacher-forced parity tests and by snapshots. */
int plen_get_manifold(plen_ctx *ctx, float *man_dev, void *stream);
int plen_set_manifold(plen_ctx *ctx, const float *man_dev, void *stream);

/* Per-env domain randomisation (the reference lists it as future work, README.md:75-76; SURVEY.md 8f-3): scale factors of
 * the three foot friction coefficients (plen_env.py:309, 439-452), of the servo force limit (setJointMotorControlArray
 * forces=0.15, plen_env.py:753) and of the servo position gain (POSITION_CONTROL kp 0.1).  Arrays are [N] device floats;
 * NULL leaves a column as it is; every scale is 1 after plen_create.  Takes effect from the next tick.
 * Resets: a reset (explicit or auto) restores the ONE snapshot settled under unit scales at plen_create, whatever the robot's
 * own scales are -- unless plen_settle_env_resets has settled each robot's reset state under its own scales (call it after
 * the setters). */
int plen_set_env_scales(plen_ctx *ctx, const float *friction_scale_dev, const float *motor_force_scale_dev,
                        const float *motor_gain_scale_dev, void *stream);

/* Per-env mass randomisation (SURVEY.md 8f-3): a robot carrying a different battery, cables or a sensor board.
 *   mass_scale_dev [N,PLEN_BODIES]  factor on the mass AND the rotational inertia of each body (uniform density scaling, centre
 *                  of mass unchanged).  Body 0 is the torso composite; body 1 + j is the body moved by joint j (action order).
 *                  The URDF links folded into each body: PlenModel.body_links (plen_ml_walk_b200/urdf_loader.py).
 *   payload_dev    [N,4]  (m, x, y, z): a point mass of m kg without rotational inertia, rigidly attached at (x, y, z) in the
 *                  torso body frame (the frame of qpos's base pose).
 * NULL leaves a part as it is.  Until the first call every robot has scale 1 and payload 0, and the context holds no mass
 * table at all (the first call allocates 128 bytes per robot); a robot with scale 1 and payload 0 steps bit-identically to a
 * context that never called this.  Takes effect from the next tick.  Precondition: scales finite and > 0, m finite and >= 0,
 * x y z finite; a violation produces non-finite states, which the numeric guard retires (plen_fault_count).
 * Resets: as for plen_set_env_scales, a reset (explicit or auto) restores the ONE snapshot settled under the nominal model at
 * plen_create, and the robot's own masses apply from its first tick after that -- unless plen_settle_env_resets has settled
 * each robot's reset state under its own parameters. */
int plen_set_env_mass(plen_ctx *ctx, const float *mass_scale_dev, const float *payload_dev, void *stream);
/* The current values into [N,PLEN_BODIES] / [N,4] device buffers (either NULL to skip), stream-ordered.  Returns 1 when
 * plen_set_env_mass was ever called on this context, 0 when not (the buffers then receive 1 and 0), < 0 on error. */
int plen_get_env_mass(plen_ctx *ctx, float *mass_scale_dev, float *payload_dev, void *stream);

/* Per-env servo command latency (SURVEY.md 8f-3): the delay between sending a command and the servo acting on it.
 *   ticks_dev   [N] int32  delay d of each robot in physics ticks, 0 <= d <= PLEN_MAX_LATENCY_STEPS * substeps (0 .. 8 ticks,
 *               0 .. 33 ms at the default 240 Hz and 4 substeps); a value outside is clamped into that range.
 *   history_dev [N,2,PLEN_NJ]  the raw servo targets (radians) of the robot's last env step ([:,0]) and of the step before
 *               ([:,1]), relative to its current episode counter (set the state first); for snapshots that must continue
 *               a run bit for bit.
 * Tick k (0-based) of env step t applies the raw targets (after agent_to_env) of step t - s, s = ceil(max(d - k, 0) / substeps):
 * d = 0 is the stock behaviour, d = substeps applies the previous step's command for the whole step.  A command from before
 * the robot's last reset (explicit or auto) is the reset-pose hold target 0.  Every plen_step / plen_step_host records each
 * robot's targets once the history exists; plen_tick, plen_debug_dynamics and the reset snapshot settled at plen_create
 * neither apply nor record it.  NULL leaves a part as it is.  The first call allocates the history (384 bytes per robot;
 * until then the context holds none) and fills it with each robot's last servo targets, as if that command had been held,
 * so a robot switched to a delay mid-episode does not jump to 0; later calls only change what they are given.  Delays may
 * change between any two steps.  Takes effect from the next step. */
int plen_set_env_latency(plen_ctx *ctx, const int32_t *ticks_dev, const float *history_dev, void *stream);
/* The current delays [N] and history [N,2,PLEN_NJ] (same order as above) into device buffers (either NULL to skip),
 * stream-ordered.  Returns 1 when plen_set_env_latency was ever called on this context, 0 when not (the buffers then receive
 * 0 and each robot's last servo targets), < 0 on error. */
int plen_get_env_latency(plen_ctx *ctx, int32_t *ticks_dev, float *history_dev, void *stream);

/* Per-env reset states (no reference counterpart: the reference resets every robot to one pose, plen_env.py:558-574).
 * A context starts without a reset table: every reset restores the one snapshot settled at plen_create.  The first
 * plen_settle_env_resets or plen_set_env_resets call allocates one row per robot (720 bytes, plus 592 bytes of settle scratch),
 * filled with that snapshot; from then on every reset of robot e -- plen_reset, the auto-reset of plen_step / plen_step_host and
 * the numeric guard, including the terminal observation of a faulted robot -- restores row e: record, observation and sole
 * manifolds.  The running states are never touched by these calls; a new row applies from the robot's next reset.
 *
 * plen_settle_env_resets runs the reference's reset procedure for every robot under its CURRENT friction, force and gain
 * scales and mass rows: the robot at its start pose with joints, velocities, targets and contact cache zero and empty sole
 * manifolds, then config.reset_ticks ticks with hold target 0; the result becomes its row.
 *   start_dev [N,4] (x, y, z, yaw): base position in the world and heading about world z, quaternion (0, 0, sin(yaw/2),
 *             cos(yaw/2)); NULL = config.start_pos and yaw 0 for every robot (a nominal robot's row is then the snapshot bit
 *             for bit).  Precondition: finite values; a non-finite pose settles into a non-finite row, which the numeric
 *             guard retires at the robot's first step after a reset.
 * Command latency does not apply (the settle, like plen_tick and the snapshot settle, is raw physics); the command history
 * and its rule that a command from before the last reset is the hold target 0 stay as they are.  Call it after the setters
 * whose parameters the rows should reflect.  Launches reset_ticks physics ticks over the whole batch plus 2 kernels.
 *
 * plen_set_env_resets: user-supplied reset states in the layouts of plen_set_state (qpos [N,25], qvel [N,24],
 * aux [N,PLEN_AUX_WORDS]) and plen_set_manifold (man [N,PLEN_MAN_WORDS]; PLEN_E_STATE when config.sole_manifold = 0); NULL
 * leaves that part of every row as it is.  Each row's observation is computed from its record.
 * plen_get_env_resets: the rows into device buffers of the same layouts plus obs [N,26]; any pointer may be NULL (man needs
 * sole_manifold = 1, as above).  Returns 1 when the context has a table, 0 when not (every robot then receives the shared
 * snapshot), < 0 on error.
 * plen_clear_env_resets: synchronises `stream` and frees the table; the context is then exactly the stock path again. */
int plen_settle_env_resets(plen_ctx *ctx, const float *start_dev, void *stream);
int plen_set_env_resets(plen_ctx *ctx, const float *qpos_dev, const float *qvel_dev, const float *aux_dev, const float *man_dev,
                        void *stream);
int plen_get_env_resets(plen_ctx *ctx, float *qpos_dev, float *qvel_dev, float *aux_dev, float *obs_dev, float *man_dev,
                        void *stream);
int plen_clear_env_resets(plen_ctx *ctx, void *stream);

/* Per-env observation noise (SURVEY.md 8f-3, sensing side; the reference has none): the observations the library hands to the
 * agent -- obs of plen_step / plen_step_host / plen_reset and terminal_obs -- carry sensor noise.  Reward, done, timeout, the
 * gait counters, the state record and the physics keep using the true state.  For robot e, continuous words w = 0..23
 * (q1..q18, z, vx, roll, pitch, yaw, y) and the contact flags w = 24, 25:
 *   noisy_w = clean_w + fmaf(sigma_w, n, b_w)    n ~ N(0,1) fresh for every observation; where sigma_w == 0 and b_w == 0 the
 *                                               word is passed through bit for bit (-0.0 and NaN included).  No clipping, no
 *                                               angle wrapping: roll / pitch / yaw may leave [-pi, pi], z may go negative.
 *   b_w = beta_w * n'                           per-episode bias, drawn at every reset of the robot (plen_reset for the masked
 *                                               robots, the auto-reset, the numeric guard's forced reset) and constant for
 *                                               the episode: its reset observation, every observation and its terminal_obs
 *                                               carry it.
 *   flag -> 1 - flag                            independently per observation with probability p.
 * Draws are counter-based and stateless given a per-robot draw counter in device memory, which k_post increments once per step
 * and k_reset once per robot it resets -- so a CUDA graph that captures plen_step draws new noise on every replay.  With
 * gid = first_env_id + e, mix64 the splitmix64 finaliser (x += 0x9E3779B97F4A7C15; x = (x ^ x >> 30) * 0xBF58476D1CE4E5B9;
 * x = (x ^ x >> 27) * 0x94D049BB133111EB; x ^ x >> 31) and hash32(k) = mix64(k) >> 32, all in uint64:
 *   k  = mix64(seed ^ mix64(gid)) + (counter << 8) + (s << 5) + w
 *   n  = sqrtf(-2 logf(u1)) * cospif(2 u2),  u1 = ((float)hash32(k) + 1) * 2.3283064e-10f,
 *        u2 = (float)hash32(k ^ 0xA5A5A5A5DEADBEEF) * 2.3283064e-10f        (float32 arithmetic; plen_actor_forward's generator)
 *   flip where (uint64)hash32(k) < (uint64)((double)p * 2^32)
 * Streams s: 0 the step's observation noise (also its terminal_obs), 1 the step's flips, 2 the new episode's bias, 3 the
 * noise of a reset observation, 4 its flips.  The draws depend neither on a robot's position in the batch nor on how
 * plen_step / plen_step_host cut it into ranges: a sharded caller passes its shard's first global robot id as first_env_id
 * and gets the noise of one big context.
 *
 * plen_set_env_obs_noise: sigma_dev [N,24] (>= 0), bias_std_dev [N,24] beta (>= 0), flip_dev [N] p (in [0,1]) device floats;
 * NULL leaves a part as it is.  seed and first_env_id (>= 0, else PLEN_E_ARG) are set by every call; a captured graph keeps
 * the values of its capture.  The first call allocates the noise rows (384 bytes per robot) and two clean-observation buffers
 * (2 x 104 bytes per robot), zeroes every sigma, beta, p, bias and counter, and switches k_post to its noise instance;
 * episodes already running keep b = 0, so the bias applies from each robot's next reset.  Graphs captured before the first
 * call keep the stock kernel.  Precondition (not checked here, PlenVecEnv.set_obs_noise checks it): finite values in those
 * ranges; a NaN sigma makes NaN observations, a p outside [0,1] acts as 0 or 1.
 * plen_set_env_obs_noise_state: the running biases bias_dev [N,24] and draw counters counter_dev [N] (uint32), NULL leaves a
 * part as it is; for snapshots that must continue bit for bit.  PLEN_E_STATE without a table.
 * plen_get_env_obs_noise: the parameters, biases and counters into device buffers of the same layouts, seed and first_env_id
 * into host variables; any pointer may be NULL.  Returns 1 when the context has a table, 0 when not (the buffers then receive
 * zeros), < 0 on error.
 * plen_clear_env_obs_noise: synchronises `stream` and frees the table; the context is then exactly the stock path again.
 * plen_get_clean_obs: the noise-free observations [N,26] of the last step or reset (what a context without noise would have
 * written to obs) and the noise-free terminal observations [N,26] (written where a step reported done, whether or not that
 * step was given a terminal_obs buffer); either pointer may be NULL.  Both are zero until the first step or reset after the
 * first plen_set_env_obs_noise.  For asymmetric actor-critic training.  PLEN_E_STATE without a table. */
int plen_set_env_obs_noise(plen_ctx *ctx, const float *sigma_dev, const float *bias_std_dev, const float *flip_dev,
                           unsigned long long seed, long long first_env_id, void *stream);
int plen_set_env_obs_noise_state(plen_ctx *ctx, const float *bias_dev, const uint32_t *counter_dev, void *stream);
int plen_get_env_obs_noise(plen_ctx *ctx, float *sigma_dev, float *bias_std_dev, float *flip_dev, float *bias_dev,
                           uint32_t *counter_dev, unsigned long long *seed, long long *first_env_id, void *stream);
int plen_clear_env_obs_noise(plen_ctx *ctx, void *stream);
int plen_get_clean_obs(plen_ctx *ctx, float *obs_dev, float *terminal_obs_dev, void *stream);

/* Advance every env by n_ticks physics ticks with raw joint targets [N,18] (radians) and no env logic.
 * Replaces move_joints + p.stepSimulation (plen_env.py:746-753, :665-667); used by the parity tests. */
int plen_tick(plen_ctx *ctx, const float *targets_dev, int n_ticks, void *stream);

/* Diagnostics: per-env generalized inverse mass matrix M^-1 [N,24,24] in coordinates [omega_w, v_w, qd]
 * and world pose of the 19 body frames pos [N,24,3] / rot [N,24,9] (lanes 1..5 unused). */
int plen_debug_dynamics(plen_ctx *ctx, float *minv_dev, float *pos_dev, float *rot_dev, void *stream);

/* Diagnostics: raw copy of the per-env state records [N,PLEN_STATE_WORDS] (layout: csrc/plen_device.cuh, W_* words;
 * word 79 = PGS iterations of the last tick, the figure DESIGN.md's work accounting uses). */
int plen_debug_records(plen_ctx *ctx, float *records_dev, void *stream);

/* Per-kernel device timing of plen_step (measurement aid for bench.py, no reference counterpart): after
 * plen_profile_enable the next max_steps plen_step calls record CUDA events around their launches on the caller's
 * stream; plen_profile_read synchronises on them, returns the summed milliseconds of the dynamics (k_dyn), solver
 * (k_solve) and env-epilogue (k_post) kernels and the number of recorded steps, and re-arms the recorder. */
int plen_profile_enable(plen_ctx *ctx, int max_steps);
int plen_profile_read(plen_ctx *ctx, float *ms_dyn, float *ms_solve, float *ms_post, int *steps);

/* FP32 FMA-pipe peak of `device` measured with a register-resident FMA chain kernel (mode 0: scalar FFMA, mode 1:
 * packed FFMA2 = fma.rn.f32x2), best of 4 timed launches after 2 warm-up launches, CUDA events.  Measurement aid for
 * bench.py's FP32 roofline (MEASURED_PEAKS.json carries only HBM and bf16 figures); no reference counterpart.
 * sm_mhz_hint (nullable): the SM clock that figure implies at 128 FP32 lanes per SM. */
int plen_measure_fp32_peak(int device, int mode, float *tflops, float *sm_mhz_hint);

/* Sinewave gait + closed-form leg IK for n_gaits parameter sets in one launch.
 * Replaces TrajectoryGenerator.main (plen_bullet/src/plen_bullet/trajectory_generator.py:54-277) and the trajectory
 * assembly of trajectory_eval.py:180-261.
 * All arithmetic and buffers are float64 (the reference is numpy float64; tolerance 1e-6 rad).
 *   params_dev [n_gaits,5]  = height, stride, bend_distance, body_sway, fwd_bias (mm; defaults 30 30 10 5 10)
 *   traj_dev   [n_gaits,40,18] one gait cycle (20 right-forward + 20 left-forward rows) in action order, sign map applied
 *   bend_dev   [n_gaits,18]   the "bend_legs" pose
 *   status_dev [n_gaits] uint8 (nullable): 1 where the IK target was unreachable (reference raises ValueError,
 *              trajectory_generator.py:187-189); the row is then filled with NaN. */
int plen_gait_ik(int device, const double *params_dev, int n_gaits, double *traj_dev, double *bend_dev,
                 uint8_t *status_dev, void *stream);

/* ---- device-resident TD3 pieces (reference: plen_ros/src/plen_ros_helpers/td3.py, driven by plen_bullet/src/plen_td3.py)
 *
 * Replay ring: replaces ReplayBuffer (td3.py:122-193).  One transition = 72 floats [s 26 | a 18 | s' 26 | r | done];
 * `add` appends until `capacity` tuples are stored, then overwrites from index 0 upwards (td3.py:136-147), n tuples per
 * call; `sample` draws `batch` rows uniformly WITH replacement (td3.py:175) from a counter-based generator keyed by
 * `seed` (pass a fresh value per call) and returns not_done = 1 - done (td3.py:189-191).  index_dev (nullable) receives
 * the sampled rows.  All *_dev pointers are caller-owned device memory; calls are stream-ordered. */
typedef struct plen_replay plen_replay;
plen_replay *plen_replay_create(long long capacity, int device);
void plen_replay_destroy(plen_replay *rb);
long long plen_replay_size(const plen_replay *rb);
long long plen_replay_ptr(const plen_replay *rb);
const float *plen_replay_storage(const plen_replay *rb);       /* device pointer to [capacity][72] */
int plen_replay_add(plen_replay *rb, const float *state_dev, const float *action_dev, const float *next_state_dev,
                    const float *reward_dev, const uint8_t *done_dev, int n, void *stream);
int plen_replay_sample(plen_replay *rb, int batch, unsigned long long seed, float *state_dev, float *action_dev,
                       float *next_state_dev, float *reward_dev, float *not_done_dev, int *index_dev, void *stream);

/* Replaces Actor.forward / TD3Agent.select_action (td3.py:45-57, :243-257) for n observations in one launch:
 * action = max_action * tanh(W3 relu(W2 relu(W1 s + b1) + b2) + b3), weights in nn.Linear layout (row-major [out][in]:
 * w1 [256][26], w2 [256][256], w3 [18][256]), float32 throughout.  noise_std > 0 adds the exploration noise of
 * plen_td3.py:101-104 (N(0, noise_std), then clip to +-max_action), drawn from a counter-based generator keyed by seed. */
int plen_actor_forward(int device, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                       const float *b3, const float *obs_dev, int n, float max_action, float noise_std,
                       unsigned long long seed, float *action_dev, void *stream);
/* The same forward pass on the 5th-generation tensor cores (tcgen05.mma kind::f16: FP16 operands, FP32 accumulation in
 * TMEM; weights resident in shared memory, one persistent CTA per SM, 128 observations per tile).  Throughput path for
 * rollouts with large N (8-13x the fp32 kernel); FP16 operand rounding (2^-12 relative) moves an action by ~5e-4 on
 * average (bound tested), so plen_actor_forward stays the parity path.  Same arguments and noise stream. */
int plen_actor_forward_tc(int device, const float *w1, const float *b1, const float *w2, const float *b2, const float *w3,
                            const float *b3, const float *obs_dev, int n, float max_action, float noise_std,
                            unsigned long long seed, float *action_dev, void *stream);
int plen_actor_tc_timed_out(void);   /* diagnostic: 1 if a tensor-core actor launch ever abandoned an mbarrier wait */
const char *plen_td3_last_error(void);

/* ---- TD3 learner: replaces TD3Agent.train (td3.py:259-356) -- target Q with clipped policy noise, twin-critic MSE step,
 * delayed actor step through Q1, Polyak target updates -- with hand-written CUDA (strided fp32 GEMM with fused
 * bias / ReLU / tanh / mask / bias-gradient epilogues, fused Adam, fused target update); no cuBLAS, no autograd.
 *
 * Every network is ONE flat float32 vector in state_dict order (weight, bias per layer; nn.Linear layout [out][in]):
 *   actor  (PLEN_TD3_ACTOR_PARAMS):  fc1 [256][26] b[256] | fc2 [256][256] b[256] | fc3 [18][256] b[18]          td3.py:37-41
 *   critic (PLEN_TD3_CRITIC_PARAMS): fc1 [256][44] b | fc2 [256][256] b | fc3 [1][256] b[1] | fc4 | fc5 | fc6     td3.py:72-81
 * The gradient vectors have the same layouts; a data-parallel learner all-reduces critic_grad / actor_grad between
 * plen_td3_*_grads and plen_td3_adam (SURVEY.md 8e).  All pointers are caller-owned device memory. */
#define PLEN_TD3_ACTOR_PARAMS 77330
#define PLEN_TD3_CRITIC_PARAMS 155138
typedef struct plen_td3 plen_td3;
typedef struct plen_td3_hyper {
    float discount, tau, policy_noise, noise_clip, max_action;   /* td3.py:211-219: 0.99 0.005 0.2 0.5 1.0 */
    float lr, beta1, beta2, eps;                                 /* torch.optim.Adam(lr=3e-4), td3.py:226-233 */
    int policy_freq;                                             /* 2 */
} plen_td3_hyper;
typedef struct plen_td3_params {
    float *actor, *actor_target, *critic, *critic_target;        /* parameters */
    float *actor_m, *actor_v, *critic_m, *critic_v;              /* Adam exp_avg / exp_avg_sq */
    float *actor_grad, *critic_grad;                             /* gradients of the last *_grads call */
} plen_td3_params;
int plen_td3_default_hyper(plen_td3_hyper *h);
plen_td3 *plen_td3_create(int max_batch, int device);            /* workspace for minibatches of <= max_batch rows */
void plen_td3_destroy(plen_td3 *t);
long long plen_td3_launches(const plen_td3 *t);                  /* kernels launched so far (bench accounting) */
/* Precision of the learner's matrix products (td3.py:259-356 runs them in fp32 torch): 0 = FP32 CUDA cores, within 1e-5 of
 * torch (default, the parity path); 1 = for minibatches >= 512 every product that fills a 128-row tile (forward,
 * backward-data and backward-weight of the 256-wide layers and of fc1) runs on the 5th-generation tensor cores --
 * tcgen05.mma kind::tf32 with every operand split into two TF32 parts (3xTF32: A_lo B_hi + A_hi B_lo + A_hi B_hi, FP32
 * accumulation in TMEM), which keeps fp32-level accuracy (one-pass TF32 flips ReLU masks and moves hidden-layer gradients by
 * 2-5 %; measured).  Tested against float64 entry by entry: every product within 10x the FP32 kernel's error and 2^-19
 * relative to (|A| |B|)_mn (measured: 1.6-6.0x, at most 9.6e-7 on a B200); gradients within 1e-3 of autograd relative to
 * the largest entry of each tensor.  Below 512 rows the update is launch bound and stays on the FP32 path either way. */
int plen_td3_set_precision(plen_td3 *t, int tf32);
int plen_td3_tc_timed_out(void);     /* diagnostic: 1 if a tensor-core learner launch ever abandoned an mbarrier wait */
/* minibatch: drawn from the replay ring (uniform with replacement, td3.py:175) or given explicitly */
int plen_td3_sample(plen_td3 *t, plen_replay *rb, int batch, unsigned long long seed, void *stream);
int plen_td3_set_batch(plen_td3 *t, const float *state_dev, const float *action_dev, const float *next_state_dev,
                       const float *reward_dev, const float *not_done_dev, int batch, void *stream);
/* td3.py:303-333: critic_loss and d critic_loss / d critic parameters -> params->critic_grad.  noise_dev (nullable)
 * [batch,18] standard-normal samples for the target policy smoothing; NULL draws them from a counter-based generator
 * keyed by seed.  critic_loss_dev (nullable) receives the scalar loss. */
int plen_td3_critic_grads(plen_td3 *t, const plen_td3_params *p, const plen_td3_hyper *h, const float *noise_dev,
                          unsigned long long seed, float *critic_loss_dev, void *stream);
/* td3.py:342-346: actor_loss = -Q1(s, actor(s)).mean() and its gradient -> params->actor_grad */
int plen_td3_actor_grads(plen_td3 *t, const plen_td3_params *p, const plen_td3_hyper *h, float *actor_loss_dev, void *stream);
/* one torch.optim.Adam step (step = 1, 2, ...) over a flat parameter vector; one Polyak update target = tau p + (1 - tau) target */
int plen_td3_adam(float *param_dev, const float *grad_dev, float *m_dev, float *v_dev, int n, long long step,
                  const plen_td3_hyper *h, int device, void *stream);
int plen_td3_soft_update(float *target_dev, const float *source_dev, int n, float tau, int device, void *stream);
/* The whole TD3Agent.train call: sample (rb nullable: reuse the minibatch already set), critic step (Adam step number
 * critic_step), and when total_it % policy_freq == 0 the actor step (actor_step) and both target updates.
 * losses_dev (nullable) = [actor_loss, critic_loss]. */
int plen_td3_train(plen_td3 *t, const plen_td3_params *p, const plen_td3_hyper *h, plen_replay *rb, int batch,
                   long long total_it, long long critic_step, long long actor_step, unsigned long long seed,
                   float *losses_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif
