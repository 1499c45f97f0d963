"""TEST-ONLY numpy twin of the per-robot observation noise (plen_set_env_obs_noise, plen_env.cuh): the counter-based keys, the
hash bits, the float32 uniforms and flip decisions exactly, the Gaussians in float64 from those uniforms; the expected noisy
observations of a step or reset; and the warp-emulation harness (tests/emu/emu_obs_noise.cpp) that exports the device's
generator and env_post's noise instance."""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_util import _DEPS, ROOT, Emu

EMU_NOISE_SRC = os.path.join(ROOT, "tests", "emu", "emu_obs_noise.cpp")
EMU_NOISE_LIB = os.path.join(ROOT, "tests", "emu", "libplen_emu_obs_noise.so")

# noise row layout (plen_env.cuh ON_*) and draw streams (NS_*)
ON_SIGMA, ON_BETA, ON_BIAS, ON_FLIP, ON_CTR, ON_WORDS = 0, 24, 48, 72, 73, 96
NS_OBS, NS_FLIP, NS_BIAS, NS_ROBS, NS_RFLIP = 0, 1, 2, 3, 4
U32_SCALE = np.float32(2.3283064e-10)
XOR_U2 = np.uint64(0xA5A5A5A5DEADBEEF)
OBS_NAMES = ["q%d" % (j + 1) for j in range(18)] + ["z", "vx", "roll", "pitch", "yaw", "y", "right_contact", "left_contact"]


def mix64(x):
    """the splitmix64 finaliser, 64 bits; x: uint64 array"""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def hash32(k):
    return (mix64(k) >> np.uint64(32)).astype(np.uint32)


def base(seed, gid):
    """mix64(seed ^ mix64(gid)) per robot; gid: int array (first_env_id + robot)"""
    return mix64(np.uint64(seed) ^ mix64(np.asarray(gid, dtype=np.int64).astype(np.uint64)))


def key(seed, gid, ctr, stream, word):
    """uint64 keys, broadcast over the array arguments"""
    with np.errstate(over="ignore"):
        return (base(seed, gid) + (np.asarray(ctr, dtype=np.uint64) << np.uint64(8)) +
                (np.asarray(stream, dtype=np.uint64) << np.uint64(5)) + np.asarray(word, dtype=np.uint64))


def uniforms(k):
    """the float32 uniforms (u1 in (0, 1], u2 in [0, 1)) exactly as the kernels form them"""
    k = np.asarray(k, dtype=np.uint64)
    u1 = (hash32(k).astype(np.float32) + np.float32(1.0)) * U32_SCALE
    u2 = hash32(k ^ XOR_U2).astype(np.float32) * U32_SCALE
    return u1, u2


def normal(k):
    """float64 Box-Muller of the float32 uniforms: the device's sqrtf / logf / cospif differ from it by a few float32 ulps"""
    u1, u2 = uniforms(k)
    u1, u2 = u1.astype(np.float64), (np.float32(2.0) * u2).astype(np.float64)
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(np.pi * u2)


def flips(k, p):
    thr = (np.asarray(p, dtype=np.float32).astype(np.float64) * 4294967296.0).astype(np.uint64)
    return hash32(k).astype(np.uint64) < thr


def rows(n, sigma=0.0, beta=0.0, p=0.0, bias=0.0, counter=0):
    """noise rows [n, ON_WORDS] float32 with the given parameters (broadcast to [n,24] / [n])"""
    r = np.zeros((n, ON_WORDS), np.float32)
    r[:, ON_SIGMA:ON_SIGMA + 24] = np.broadcast_to(np.asarray(sigma, np.float32).reshape(-1, 24) if np.ndim(sigma) else sigma, (n, 24))
    r[:, ON_BETA:ON_BETA + 24] = np.broadcast_to(np.asarray(beta, np.float32).reshape(-1, 24) if np.ndim(beta) else beta, (n, 24))
    r[:, ON_BIAS:ON_BIAS + 24] = np.broadcast_to(np.asarray(bias, np.float32).reshape(-1, 24) if np.ndim(bias) else bias, (n, 24))
    r[:, ON_FLIP] = p
    r[:, ON_CTR] = np.broadcast_to(np.asarray(counter, np.uint32), (n,)).view(np.float32)
    return r


def counters(r):
    return np.ascontiguousarray(r[:, ON_CTR]).view(np.uint32)


def apply(clean, sigma, bias, p, seed, gid, ctr, stream):
    """expected noisy observations [n,26] (float64 noise: compare against float32 results within a bound) and the flip mask
    [n,2]: words 0..23 clean + sigma n + b (exactly clean where sigma == b == 0), flags flipped with stream + 1"""
    clean = np.asarray(clean, np.float32)
    n = clean.shape[0]
    w = np.arange(24)[None, :]
    g = np.asarray(gid)[:, None]
    c = np.asarray(ctr, np.uint64).reshape(-1, 1)
    z = normal(key(seed, g, c, stream, w))
    sigma, bias = np.asarray(sigma, np.float32), np.asarray(bias, np.float32)
    out = clean.astype(np.float64).copy()
    on = ~((sigma == 0) & (bias == 0))
    out[:, :24] = np.where(on, clean[:, :24].astype(np.float64) + sigma * z + bias, clean[:, :24])
    f = flips(key(seed, g, c, stream + 1, np.arange(24, 26)[None, :]), np.asarray(p).reshape(-1, 1))
    out[:, 24:] = np.where(f, 1.0 - clean[:, 24:].astype(np.float64), clean[:, 24:])
    return out, f


def new_bias(beta, seed, gid, ctr):
    """the bias [n,24] a reset with draw counter ctr gives the new episode, float64 (beta * n')"""
    return np.asarray(beta, np.float32) * normal(key(seed, np.asarray(gid)[:, None], np.asarray(ctr, np.uint64).reshape(-1, 1), NS_BIAS,
                                                    np.arange(24)[None, :]))


# ---- the emulation harness
def build_emu_obs_noise():
    deps = _DEPS + [EMU_NOISE_SRC]
    if os.path.exists(EMU_NOISE_LIB) and all(os.path.getmtime(EMU_NOISE_LIB) >= os.path.getmtime(d) for d in deps):
        return EMU_NOISE_LIB
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-pthread", "-fPIC", "-shared", "-ffp-contract=off",
                           "-I", ROOT, "-o", EMU_NOISE_LIB, EMU_NOISE_SRC])
    return EMU_NOISE_LIB


class EmuObsNoise(Emu):
    """float32 Emu whose library also exports the noise generator and env_post<true>"""

    def __init__(self, joint_act=False):
        super().__init__(joint_act=joint_act)
        self.L = C.CDLL(build_emu_obs_noise())
        assert self.L.emu_real_bytes() == 4
        self.L.emu_default_config(C.byref(self.cfg), int(joint_act))
        self.L.emu_noise_key.restype = C.c_uint64
        self.L.emu_noise_key.argtypes = [C.c_ulonglong, C.c_longlong, C.c_uint, C.c_int, C.c_int]

    def draws(self, k, p=None):
        """-> (hash32 uint32, u1 float32, u2 float32, normal float64, flip bool) of the device generator at keys k"""
        k = np.ascontiguousarray(k, dtype=np.uint64).ravel()
        n = k.size
        p = np.ascontiguousarray(np.broadcast_to(np.float32(0.5) if p is None else np.asarray(p, np.float32), (n,)))
        h = np.zeros(n, np.uint32)
        u1, u2, z, f = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n), np.zeros(n, np.uint8)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.L.emu_noise_draws(vp(k), vp(p), n, vp(h), vp(u1), vp(u2), vp(z), vp(f))
        return h, u1, u2, z, f.astype(bool)

    def key(self, seed, gid, ctr, stream, word):
        return int(self.L.emu_noise_key(seed, gid, ctr, stream, word))

    def step_noise(self, rec, actions, snapshot, noise_rows, seed, gid0=0):
        """emu_step with env_post<true>; noise_rows [n, ON_WORDS] float32 is updated in place.
        -> (obs, reward, done, timeout, terminal_obs, clean_obs, clean_terminal_obs)"""
        n = rec.shape[0]
        actions = np.ascontiguousarray(actions, dtype=np.float32).reshape(n, 18)
        obs, tobs, cobs, ctobs = (np.full((n, 26), np.float32(-7.0), np.float32) for _ in range(4))
        rew = np.zeros(n, np.float32)
        done, tmo = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
        assert noise_rows.dtype == np.float32 and noise_rows.flags.c_contiguous and noise_rows.shape == (n, ON_WORDS)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        self.L.emu_step_noise(C.byref(self.model), C.byref(self.cfg), vp(rec), vp(actions), n, vp(obs), vp(rew), vp(done),
                              vp(tmo), vp(tobs), vp(snapshot), vp(noise_rows), vp(cobs), vp(ctobs), C.c_ulonglong(seed),
                              C.c_longlong(gid0))
        return obs, rew, done.astype(bool), tmo.astype(bool), tobs, cobs, ctobs
