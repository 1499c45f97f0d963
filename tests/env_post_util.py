"""TEST-ONLY: constructed state families for env_post / k_post, the env epilogue of a step (plen_env.cuh), and the float64
references the CPU and GPU tests of it share.

With plen_config.substeps = 0 an env step runs no physics tick, so a step is env_post alone on the records the test wrote:
observation, one-sided done, the ordered reward sum, the gait counters, TimeLimit, the terminal observation, auto-reset
from the snapshot and the numeric guard.  Random rollouts kill a robot within a few steps and so never reach most of those
branches; the families below put robots on each of them, every robot with a label, and `branch_counts` checks from the
float64 reference's own decisions that each branch is still taken."""
import numpy as np

from emu_util import Emu, oracle_state_from_record

# state record layout (plen_device.cuh W_*)
W_U, W_LAM, W_POS, W_MAN, W_EPRET, W_J, W_QUAT = 0, 24, 32, 35, 36, 38, 56
W_CNT, W_DS, W_HIST, W_EPT, W_LAST, W_SUMS, W_ITERS, W_SPARE = 60, 61, 62, 63, 64, 70, 79, 80
# words env_post neither reads nor writes (a step that resets nobody returns them unchanged)
UNTOUCHED = [37, W_ITERS] + list(range(W_SPARE, 96))
# observation words that are copies of record words: joint angles, z, vx, y
OBS_COPY = [(k, W_J + k) for k in range(18)] + [(18, W_POS + 2), (19, 3), (23, W_POS + 1)]
# joint pairs of the gait histories: (JointStates[2],[8]), ([3],[9]), ([4],[10])
CUR_JOINTS = (2, 8, 3, 9, 4, 10)

MAX_EP = 500                     # plen_config.max_episode_steps the families are built for
PI3 = np.pi / 3
SARG_GIMBAL = 0.99999
NEAR_REL = 2e-5                  # decision thresholds: robots this close (relative) may be decided either way in float32
FAMILIES = ("gait", "double_support", "sums", "termination", "orientation", "foot_flat", "vx", "timeout", "faults")


def _euler_quat(roll, pitch, yaw):
    """xyzw quaternion of the ZYX Euler angles pybullet's getEulerFromQuaternion returns"""
    cr, sr, cp, sp, cy, sy = (f(a / 2) for a in (roll, pitch, yaw) for f in (np.cos, np.sin))
    return np.stack([sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy,
                     cr * cp * cy + sr * sp * sy], -1)


def _contact_bits(rng, n, right, left):
    """manifold bits: a random nonempty subset of the foot's four points where the flag is set (0x0F right, 0xF0 left)"""
    r = np.where(np.asarray(right, bool), rng.integers(1, 16, n), 0)
    l = np.where(np.asarray(left, bool), rng.integers(1, 16, n), 0)
    return (r | (l << 4)).astype(np.float32)


def _base(rng, n):
    """n alive, upright-ish robots with random velocities, joints, contacts, counters and history sums (float32 [n,96])"""
    rec = Emu().init_record(n)
    rec[:, 0:3] = rng.uniform(-0.5, 0.5, (n, 3))                    # omega
    rec[:, 3:6] = rng.uniform(-0.3, 0.3, (n, 3))                    # v (word 3: vx)
    rec[:, 6:24] = rng.uniform(-2.0, 2.0, (n, 18))                  # qd
    rec[:, W_LAM:W_LAM + 8] = rng.uniform(0.0, 0.1, (n, 8))
    rec[:, W_POS:W_POS + 3] = np.stack([rng.uniform(-0.1, 0.1, n), rng.uniform(-0.2, 0.2, n), rng.uniform(0.12, 0.2, n)], 1)
    rec[:, W_MAN] = rng.integers(0, 256, n)
    rec[:, W_EPRET] = rng.uniform(-50.0, 50.0, n)
    rec[:, W_J:W_J + 18] = rng.uniform(-0.4, 0.4, (n, 18))
    rec[:, W_QUAT:W_QUAT + 4] = _euler_quat(*rng.uniform(-0.15, 0.15, (3, n)))
    rec[:, W_CNT] = rng.integers(0, 131, n)
    rec[:, W_DS] = rng.integers(0, 21, n)
    rec[:, W_HIST] = np.where(rng.random(n) < 0.2, 0, rng.integers(1, 101, n))
    rec[:, W_EPT] = rng.integers(0, 451, n)
    rec[:, W_LAST:W_LAST + 6] = rng.uniform(-0.5, 0.5, (n, 6))
    nl, nr = rng.uniform(0.1, 20.0, (2, n, 3))
    rec[:, W_SUMS + 1:W_SUMS + 9:3], rec[:, W_SUMS + 2:W_SUMS + 9:3] = nl, nr
    rec[:, W_SUMS:W_SUMS + 9:3] = rng.uniform(-1.0, 1.0, (n, 3)) * np.sqrt(nl * nr)
    return rec


def _foot_euler(o, rec):
    """float64 foot (roll, pitch, yaw) x 2 of float32 records through the oracle's kinematics: [n,6], right foot first"""
    o.set_state(oracle_state_from_record(rec.astype(np.float64)))
    return np.stack([o.observe(e)[1] for e in range(rec.shape[0])])


def _fam_gait(rng):
    cnts = (0, 1, 39, 40, 41, 79, 80, 81, 119, 120, 121, 250)
    grid = [(c, r, l, h) for c in cnts for r in (0, 1) for l in (0, 1) for h in (0, 1) for _ in range(3)]
    c, r, l, h = np.array(grid).T
    n = len(grid)
    rec = _base(rng, n)
    rec[:, W_CNT] = c
    rec[:, W_MAN] = _contact_bits(rng, n, r, l)
    rec[:, W_HIST] = np.where(h == 1, rng.integers(1, 101, n), 0)
    return rec, ["gait:cnt=%d,R=%d,L=%d,hist%s" % (a, b, d, ">0" if e else "=0") for a, b, d, e in grid]


def _fam_double_support(rng):
    ds = np.repeat([0, 14, 15, 16, 17, 40], 40)
    n = len(ds)
    rec = _base(rng, n)
    rec[:, W_DS] = ds
    rec[:, W_MAN] = _contact_bits(rng, n, np.ones(n), np.ones(n))
    return rec, ["double_support:ds=%d,cnt=%d" % (d, c) for d, c in zip(ds, rec[:, W_CNT].astype(int))]


def _fam_sums(rng):
    kinds = np.repeat(["zero", "one_norm_zero", "negative_dot", "large", "subnormal", "subnormal_products"], 40)
    n = len(kinds)
    rec = _base(rng, n)
    rec[:, W_CNT] = rng.integers(1, 80, n)          # the cosine term runs: 0 < cnt < 80, no gait reset
    s = rec[:, W_SUMS:W_SUMS + 9].astype(np.float64)
    jl = [W_J + j for j in CUR_JOINTS[0::2]]
    jr = [W_J + j for j in CUR_JOINTS[1::2]]
    for i, k in enumerate(kinds):
        if k == "zero":                             # 0 / (0 * 0): NaN, as in the reference
            s[i] = 0.0
            rec[i, jl + jr] = 0.0
        elif k == "one_norm_zero":                  # one history of one pair all zero: 0 / (0 * |b|)
            p = rng.integers(0, 3)
            s[i, 3 * p] = s[i, 3 * p + 1] = 0.0
            rec[i, jl[p]] = 0.0
        elif k == "negative_dot":
            s[i, 0::3] = -np.abs(s[i, 0::3]) - 0.2 * np.sqrt(s[i, 1::3] * s[i, 2::3])
        elif k == "large":
            s[i] *= 1e4 / np.abs(s[i]).max()
        elif k == "subnormal":                      # every sum below FLT_MIN, joints of the pairs at 0
            s[i] *= rng.uniform(1e-39, 1e-38) / np.abs(s[i]).max()
            rec[i, jl + jr] = 0.0
        elif k == "subnormal_products":             # empty sums, joints ~1e-19: every product is subnormal
            s[i] = 0.0
            rec[i, jl + jr] = rng.choice([-1.0, 1.0], 6) * rng.uniform(3e-20, 1e-19, 6)
    rec[:, W_SUMS:W_SUMS + 9] = s
    return rec, ["sums:%s" % k for k in kinds]


def _fam_termination(rng):
    cases = []
    for q, t in (("roll", PI3), ("pitch", PI3), ("z", 0.08), ("y", 1.0)):
        for d in (-1e-3, 1e-3):
            cases += [(q, t + d, "%s=%s%+g" % (q, "pi/3" if q in ("roll", "pitch") else t, d))] * 40
        for d in (-1e-6, 1e-6):
            cases += [(q, t + d, "%s=%s%+g" % (q, "pi/3" if q in ("roll", "pitch") else t, d))] * 2
    cases += [("roll", -1.2, "roll=-1.2")] * 24 + [("pitch", -1.2, "pitch=-1.2")] * 24 + [("y", -1.5, "y=-1.5")] * 24
    n = len(cases)
    rec = _base(rng, n)
    for i, (q, v, _) in enumerate(cases):
        if q in ("roll", "pitch"):
            a = rng.uniform(-0.15, 0.15, 3)
            a[0 if q == "roll" else 1] = v
            rec[i, W_QUAT:W_QUAT + 4] = _euler_quat(*a)
        else:
            rec[i, W_POS + (2 if q == "z" else 1)] = v
    return rec, ["termination:" + c[2] for c in cases]


def _fam_orientation(rng):
    labels = []
    rows = []
    for _ in range(64):                                             # uniform on the unit sphere of quaternions
        q = rng.normal(size=4)
        rows.append(q / np.linalg.norm(q)); labels.append("orientation:random")
    for _ in range(48):                                             # the same rotations with w < 0
        q = _euler_quat(*rng.uniform(-0.6, 0.6, 3))
        rows.append(-q); labels.append("orientation:w<0")
    for _ in range(48):                                             # 1e-3 off unit length
        q = _euler_quat(*rng.uniform(-0.6, 0.6, 3))
        f = 1.0 + rng.choice([-1e-3, 1e-3])
        rows.append(q * f); labels.append("orientation:|q|=1%+g" % (f - 1))
    # sarg = -2 (xz - wy) = |q|^2 sin(pitch) at the gimbal cut +-0.99999.  A unit quaternion has |sarg| <= 1, within 1e-5 of the
    # cut on its gimbal side; the robots well outside it are 1e-4 .. 2e-4 off unit length, as integration leaves them
    for sgn in (-1.0, 1.0):
        for d, reps in ((2e-4, 16), (-5e-5, 16), (2e-6, 2), (-2e-6, 2)):
            for _ in range(reps):
                s = SARG_GIMBAL + d
                q = _euler_quat(rng.uniform(-3, 3), sgn * (np.pi / 2 if s >= 1.0 else np.arcsin(s)), rng.uniform(-3, 3))
                rows.append(q * np.sqrt(max(s, 1.0))); labels.append("orientation:sarg=%s(0.99999%+g)" % ("-" if sgn < 0 else "+", d))
    n = len(rows)
    rec = _base(rng, n)
    rec[:, W_QUAT:W_QUAT + 4] = np.array(rows)
    return rec, labels


# foot f (0 right, 1 left): the joint that turns the foot's roll and the one that turns its pitch (+1 rad each, near 0)
_FOOT_JOINTS = {0: (4, 5), 1: (10, 11)}
_FOOT_SIGN = {0: (1.0, 1.0), 1: (-1.0, 1.0)}


def _fam_foot_flat(rng):
    from oracle.oracle import PlenOracle
    cases = []
    for f in (0, 1):
        for comp in (0, 1):
            for side in ("inside", "outside"):
                for sgn in (-1.0, 1.0):
                    cases += [(f, comp, side, sgn, 1e-4)] * 12
                cases += [(f, comp, side, 1.0, 1e-6)]
    n = len(cases)
    rec = _base(rng, n)
    rec[:, W_QUAT:W_QUAT + 4] = _euler_quat(*rng.uniform(-0.02, 0.02, (3, n)))
    tgt = np.zeros((n, 2))
    for i, (f, comp, side, sgn, d) in enumerate(cases):
        tgt[i, comp] = sgn * (0.1 - d if side == "inside" else 0.1 + d)
        tgt[i, 1 - comp] = rng.uniform(-0.05, 0.05)
        rec[i, W_J + np.array(_FOOT_JOINTS[f])] = 0.0
    contact = np.array([[c[0] == 0, c[0] == 1] for c in cases])
    rec[:, W_MAN] = _contact_bits(rng, n, contact[:, 0] | (rng.random(n) < 0.5), contact[:, 1] | (rng.random(n) < 0.5))
    # Newton on the foot's (roll, pitch) joints, in float64 through the oracle's kinematics, then rounded to float32
    o = PlenOracle(n)
    cols = np.array([[W_J + j for j in _FOOT_JOINTS[c[0]]] for c in cases])
    rows = np.arange(n)[:, None]
    x = rec[rows, cols].astype(np.float64)
    fsel = np.array([[3 * c[0], 3 * c[0] + 1] for c in cases])
    for _ in range(6):
        r64 = rec.astype(np.float64)
        r64[rows, cols] = x
        e0 = _foot_euler(o, r64)[rows, fsel]
        jac = np.zeros((n, 2, 2))
        for k in range(2):
            r1 = r64.copy()
            r1[np.arange(n), cols[:, k]] += 1e-6
            jac[:, :, k] = (_foot_euler(o, r1)[rows, fsel] - e0) / 1e-6
        x -= np.linalg.solve(jac, (e0 - tgt)[:, :, None])[:, :, 0]
    rec[rows, cols] = x
    labels = ["foot_flat:%s %s %s 0.1 by %g%s" % ("R" if f == 0 else "L", ("roll", "pitch")[comp], side, d, " (-)" if sgn < 0 else "")
              for f, comp, side, sgn, d in cases]
    return rec, labels


def _fam_vx(rng):
    v = np.repeat(np.array([-2.0, -1e-3, -0.0, 0.0, 1e-3, 2.0], np.float32), 32)
    rec = _base(rng, len(v))
    rec[:, 3] = v
    return rec, ["vx:%+g" % x if x != 0 else "vx:%s0.0" % ("-" if np.signbit(x) else "+") for x in v]


def _fam_timeout(rng):
    grid = [(e, d) for e in (MAX_EP - 2, MAX_EP - 1, MAX_EP) for d in (0, 1) for _ in range(32)]
    n = len(grid)
    rec = _base(rng, n)
    rec[:, W_EPT] = [g[0] for g in grid]
    dead = np.array([g[1] for g in grid], bool)
    rec[dead, W_POS + 2] = 0.05
    return rec, ["timeout:ept=max%+d%s" % (e - MAX_EP, ",dead" if d else "") for e, d in grid]


def _fam_faults(rng):
    words = [("u", w) for w in range(24)] + [("q", W_J + k) for k in range(18)] + [("pos", W_POS + k) for k in range(3)] + \
            [("quat", W_QUAT + k) for k in range(4)]
    cases = [(g, w, v) for g, w in words for v in (np.nan, np.inf, -np.inf)] + \
            [("lam", W_LAM + k, np.nan) for k in range(8) for _ in range(3)]
    n = len(cases)
    rec = _base(rng, n)
    rec[::3, W_EPT] = MAX_EP - 1                    # a fault on the step that would time out is still a fall
    for i, (_, w, v) in enumerate(cases):
        rec[i, w] = v
    return rec, ["faults:%s word %d = %s" % (g, w, v) for g, w, v in cases]


def make_family(name, seed):
    """-> (records float32 [n,96], labels [n])"""
    rng = np.random.default_rng(seed)
    rec, labels = globals()["_fam_" + name](rng)
    return np.ascontiguousarray(rec, np.float32), np.array(labels)


def all_families(seed=0):
    """-> (records float32 [N,96], labels [N], family name [N]) of every family, in FAMILIES order"""
    out = [make_family(f, seed + i) for i, f in enumerate(FAMILIES)]
    return (np.concatenate([r for r, _ in out]), np.concatenate([l for _, l in out]),
            np.concatenate([[f] * len(l) for f, (_, l) in zip(FAMILIES, out)]))


# ---- float64 references
def record_to_state(rec):
    """float32 records [n,96] -> (qpos [n,25], qvel [n,24], aux [n,29]) for PlenVecEnv.set_state (layout: k_set_state)"""
    rec = np.asarray(rec, np.float32)
    qpos = np.concatenate([rec[:, W_POS:W_POS + 3], rec[:, W_QUAT:W_QUAT + 4], rec[:, W_J:W_J + 18]], 1)
    qvel = np.concatenate([rec[:, 3:6], rec[:, 0:3], rec[:, 6:24]], 1)
    aux = np.concatenate([rec[:, W_LAM:W_LAM + 8], rec[:, W_MAN:W_MAN + 1], rec[:, W_CNT:W_EPT + 1], rec[:, W_LAST:W_LAST + 6],
                          rec[:, W_SUMS:W_SUMS + 9], rec[:, W_EPRET:W_EPRET + 1]], 1)
    return qpos, qvel, aux


def faulted(rec):
    """robots whose velocities, joint angles, position or quaternion hold a non-finite word (the numeric guard's test)"""
    return ~(np.isfinite(rec[:, 0:24]).all(1) & np.isfinite(rec[:, W_J:W_J + 18]).all(1) &
             np.isfinite(rec[:, W_POS:W_POS + 3]).all(1) & np.isfinite(rec[:, W_QUAT:W_QUAT + 4]).all(1))


def quantities(rec):
    """float64 decisive quantities of float32 records: roll, pitch, yaw, z, y, vx, sarg [n] and the feet's Euler angles
    fe [n,6] (right foot first), from the oracle's observation and kinematics (NaN rows for faulted robots)"""
    from oracle.oracle import PlenOracle
    n = rec.shape[0]
    r64 = rec.astype(np.float64)
    ok = ~faulted(rec)
    o = PlenOracle(n)
    o.set_state(oracle_state_from_record(np.where(ok[:, None], r64, 0.0)))
    obs = np.full((n, 26), np.nan)
    fe = np.full((n, 6), np.nan)
    for e in np.where(ok)[0]:
        obs[e], fe[e] = o.observe(int(e))
    x, y, z, w = (r64[:, W_QUAT + k] for k in range(4))
    return dict(roll=obs[:, 20], pitch=obs[:, 21], yaw=obs[:, 22], z=obs[:, 18], y=obs[:, 23], vx=obs[:, 19],
                sarg=-2.0 * (x * z - w * y), fe=fe)


def near_threshold(q, rel=NEAR_REL):
    """robots whose float64 decisive quantity lies within `rel` (relative) of its threshold: roll and pitch against pi/3, z
    against 0.08, y against 1, each foot's roll and pitch against 0.1, sarg against +-0.99999"""
    with np.errstate(invalid="ignore"):
        m = (np.abs(q["roll"] - PI3) <= rel * PI3) | (np.abs(q["pitch"] - PI3) <= rel * PI3)
        m |= (np.abs(q["z"] - 0.08) <= rel * 0.08) | (np.abs(q["y"] - 1.0) <= rel)
        m |= (np.abs(np.abs(q["fe"][:, [0, 1, 3, 4]]) - 0.1) <= rel * 0.1).any(1)
        m |= np.abs(np.abs(q["sarg"]) - SARG_GIMBAL) <= rel * SARG_GIMBAL
    return m


def branch_counts(rec, q, reward, max_ep=MAX_EP):
    """How many robots take each branch of env_post, decided from the pre-step records, the float64 quantities q and the float64
    reference reward.  -> {branch: count}"""
    cnt, ds, hist, ept = (rec[:, w].astype(np.int64) for w in (W_CNT, W_DS, W_HIST, W_EPT))
    man = rec[:, W_MAN].astype(np.int64)
    R, L = (man & 0x0F) != 0, (man & 0xF0) != 0
    fault = faulted(rec)
    ok = ~fault
    reset = (cnt >= 80) & R
    ce = np.where(reset, 0, cnt)
    de = np.where(reset, 0, ds) + 1
    with np.errstate(invalid="ignore"):
        flat = (np.abs(q["fe"][:, [0, 3]]) <= 0.1) & (np.abs(q["fe"][:, [1, 4]]) <= 0.1)
        dead = (q["roll"] > PI3) | (q["pitch"] > PI3) | (q["z"] < 0.08) | (q["y"] > 1.0)
        b = {
            "gait_reset": reset, "cnt>=120": ~reset & (cnt >= 120), "cosine": ~reset & (cnt > 0) & (cnt < 120),
            "cosine+jpen": ~reset & (cnt > 0) & (cnt < 120) & (hist > 0), "cosine,first_pass": ~reset & (cnt > 0) & (cnt < 120) & (hist == 0),
            "nan_reward": np.isnan(reward),
            "tanh,cnt<40": L & (ce < 40), "tanh,cnt>=80": L & (ce >= 80),
            "sched<40:R only": (ce < 40) & R & ~L, "sched<40:no R": (ce < 40) & ~R, "sched<40:both": (ce < 40) & R & L,
            "sched<80:L only": (ce >= 40) & (ce < 80) & L & ~R, "sched<80:no L": (ce >= 40) & (ce < 80) & ~L,
            "sched<80:both": (ce >= 40) & (ce < 80) & L & R,
            "ds>=16": R & L & (de >= 16), "ds<16": R & L & (de < 16),
            "flat R": R & flat[:, 0], "tilted R": R & ~flat[:, 0], "flat L": L & flat[:, 1], "tilted L": L & ~flat[:, 1],
            "dead:roll": q["roll"] > PI3, "dead:pitch": q["pitch"] > PI3, "dead:z": q["z"] < 0.08, "dead:y": q["y"] > 1.0,
            "alive:roll<-1": ~dead & (q["roll"] < -1.0), "alive:pitch<-1": ~dead & (q["pitch"] < -1.0),
            "alive:y<-1": ~dead & (q["y"] < -1.0),
            "gimbal+": q["sarg"] >= SARG_GIMBAL, "gimbal-": q["sarg"] <= -SARG_GIMBAL,
            "near gimbal": (np.abs(q["sarg"]) > 0.9999) & (np.abs(q["sarg"]) < SARG_GIMBAL),
            "vx<0": q["vx"] < 0, "vx=0": q["vx"] == 0, "vx>0": q["vx"] > 0,
            "timeout": ok & ~dead & (ept + 1 >= max_ep), "dead at the limit": ok & dead & (ept + 1 >= max_ep),
            "one step before the limit": ok & (ept + 1 == max_ep - 1),
            "fault:u": ~np.isfinite(rec[:, 0:24]).all(1), "fault:q": ~np.isfinite(rec[:, W_J:W_J + 18]).all(1),
            "fault:pos": ~np.isfinite(rec[:, W_POS:W_POS + 3]).all(1), "fault:quat": ~np.isfinite(rec[:, W_QUAT:W_QUAT + 4]).all(1),
            "fault at ept=max-1": fault & (ept + 1 == max_ep), "lam_n NaN, no fault": ok & np.isnan(rec[:, W_LAM:W_LAM + 8]).any(1),
            "quat w<0": rec[:, W_QUAT + 3] < 0,
            "quat off unit": np.abs(np.linalg.norm(rec[:, W_QUAT:W_QUAT + 4].astype(np.float64), axis=1) - 1.0) > 5e-4,
        }
    for k in list(b):
        if not k.startswith("fault") and k != "lam_n NaN, no fault":
            b[k] = b[k] & ok
    return {k: int(v.sum()) for k, v in b.items()}


def check_coverage(counts, least=8):
    print("env_post branch coverage: " + ", ".join("%s %d" % kv for kv in counts.items()))
    thin = {k: v for k, v in counts.items() if v < least}
    assert not thin, "branches taken by fewer than %d robots: %s" % (least, thin)


# ---- running the step and comparing it
def snapshot_record(emu):
    """a post-reset snapshot for the warp emulation: [96 + 26] record (the unsettled start pose) and its observation"""
    snap = np.zeros(96 + 26, emu.real)
    snap[:96] = emu.init_record(1)[0]
    snap[96:] = emu.observe(snap[None, :96].copy())[0]
    return snap


def emu_post(emu, rec, snapshot, auto_reset=0, max_ep=MAX_EP):
    """env_post alone (substeps = 0) in the warp emulation -> dict(obs, reward, done, timeout, terminal_obs, rec) as float64"""
    emu.cfg.substeps, emu.cfg.auto_reset, emu.cfg.max_episode_steps = 0, int(auto_reset), int(max_ep)
    r = rec.astype(emu.real)
    obs, rew, done, tmo, tobs = emu.step(r, np.zeros((rec.shape[0], 18)), snapshot)
    return dict(obs=obs.astype(np.float64), reward=rew.astype(np.float64), done=done, timeout=tmo,
                terminal_obs=tobs.astype(np.float64), rec=r.astype(np.float64))


def oracle_post(rec, max_ep=MAX_EP):
    """PlenOracle.step with substeps = 0 on the same records (no auto-reset) -> dict(obs, reward, done, timeout, rec)"""
    from emu_util import record_from_oracle_state
    from oracle.oracle import PlenOracle
    n = rec.shape[0]
    o = PlenOracle(n)
    o.cfg.substeps, o.cfg.max_episode_steps = 0, int(max_ep)
    o.set_state(oracle_state_from_record(rec.astype(np.float64)))
    obs, rew, done, tmo = o.step(np.zeros((n, 18)))
    st = o.get_state()
    out = np.stack([record_from_oracle_state(st, e, np.float64) for e in range(n)])
    return dict(obs=obs, reward=rew, done=done, timeout=tmo, rec=out)


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, np.float32)).view(np.uint32)


def euler_bound(q, base):
    """per-robot bound [n,3] on the float32 Euler angles: `base` where the angles are well conditioned, plus 2e-7 / cos(pitch)
    towards the gimbal cut, where asin(sarg) and both atan2 of quantities of size cos(pitch) amplify the float32 error of
    sarg (measured on the host float32 build: 5.0e-6 at sarg = -0.99994, 2e-7 / cos(pitch) there is 1.8e-5)"""
    c = np.sqrt(np.clip(1.0 - np.minimum(q["sarg"] ** 2, 1.0), 0.0, None))
    return base + np.where(np.abs(q["sarg"]) < SARG_GIMBAL, 2e-7 / np.maximum(c, 1e-30), 0.0)[:, None] * np.ones((1, 3))


def step_mismatches(got, ref, rec, check, skip, reward_rel, ebound, sums_rel):
    """Robots (boolean masks [n] by check) where the step outputs `got` differ from the reference `ref` on records `rec` that
    were not reset.  check: robots compared at all; skip: robots near a decision threshold, left out of the checks that
    depend on one (done, timeout, Euler angles, reward, ep_ret); ebound [n,3]: bound on the Euler angles."""
    n = rec.shape[0]
    man = rec[:, W_MAN].astype(np.int64)
    exact = check & ~skip
    out = {}
    cw = [k for k, _ in OBS_COPY]
    out["copied obs words"] = (_bits(got["obs"][:, cw]) != _bits(rec[:, [w for _, w in OBS_COPY]])).any(1)
    out["contact flags"] = (got["obs"][:, 24] != ((man & 0x0F) != 0)) | (got["obs"][:, 25] != ((man & 0xF0) != 0))
    with np.errstate(invalid="ignore"):
        out["euler"] = ~(np.abs(got["obs"][:, 20:23] - ref["obs"][:, 20:23]) <= ebound).all(1) & exact
        out["done"] = (np.asarray(got["done"], bool) != np.asarray(ref["done"], bool)) & exact
        out["timeout"] = (np.asarray(got["timeout"], bool) != np.asarray(ref["timeout"], bool)) & exact
        out["reward NaN pattern"] = np.isnan(got["reward"]) != np.isnan(ref["reward"])
        rb = reward_rel * np.maximum(1.0, np.abs(ref["reward"]))
        out["reward"] = (np.abs(got["reward"] - ref["reward"]) > rb) & exact
        for name, w in (("cnt", W_CNT), ("ds", W_DS), ("hist", W_HIST), ("ept", W_EPT)):
            out[name] = got["rec"][:, w] != ref["rec"][:, w]
        out["last"] = (_bits(got["rec"][:, W_LAST:W_LAST + 6]) != _bits(ref["rec"][:, W_LAST:W_LAST + 6])).any(1)
        s0 = rec[:, W_SUMS:W_SUMS + 9].astype(np.float64)
        s1 = ref["rec"][:, W_SUMS:W_SUMS + 9]
        # relative to the larger of the old sum and the new one: the update old + a * b may cancel; 2^-148 for subnormal sums
        out["sums"] = ~(np.abs(got["rec"][:, W_SUMS:W_SUMS + 9] - s1) <= sums_rel * np.maximum(np.abs(s0), np.abs(s1)) + 2.0 ** -148).all(1)
        e1, e0 = ref["rec"][:, W_EPRET], got["rec"][:, W_EPRET]
        ulp = np.spacing(np.abs(e1).astype(np.float32)).astype(np.float64)
        out["ep_ret"] = ((np.isnan(e0) != np.isnan(e1)) | (np.abs(e0 - e1) > rb + ulp)) & exact
    return {k: v & check for k, v in out.items()}


def report(mism, labels, what):
    """assert that no mask of step_mismatches is set; the message names the first robots of each failing check by label"""
    bad = {k: labels[v][:4].tolist() + (["... %d robots" % v.sum()] if v.sum() > 4 else []) for k, v in mism.items() if v.any()}
    assert not bad, "%s: %s" % (what, bad)
