"""ctypes mirror of include/plen_b200.h (plen_model, plen_config) and the loader of libplen_b200.so.

The CUDA library is the only implementation: if it is missing or no CUDA device is present the import of the library
(or plen_create) raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .urdf_loader import MAX_BOXES, N_LANES, PlenModel

NJ = 18
HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libplen_b200.so")

STATE_WORDS = 96
AUX_WORDS = 29
MAX_HULL = 256
MAN_WORDS = 52          # PLEN_MAN_WORDS
BODIES = 19             # PLEN_BODIES
MAX_LATENCY_STEPS = 2   # PLEN_MAX_LATENCY_STEPS
OBS_DIM = 26
ACT_DIM = 18


class PlenModelC(C.Structure):
    _fields_ = [
        ("R_pj", (C.c_float * 9) * N_LANES), ("p_pj", (C.c_float * 3) * N_LANES), ("axis", (C.c_float * 3) * N_LANES),
        ("mass", C.c_float * N_LANES), ("com", (C.c_float * 3) * N_LANES), ("inertia", (C.c_float * 6) * N_LANES),
        ("lower", C.c_float * N_LANES), ("upper", C.c_float * N_LANES), ("chain_start", C.c_int32 * N_LANES),
        ("foot_lane", C.c_int32 * 2), ("foot_pts", ((C.c_float * 3) * 4) * 2), ("foot_break", C.c_float * 2),
        ("n_boxes", C.c_int32), ("box_lane", C.c_int32 * MAX_BOXES), ("box_center", (C.c_float * 3) * MAX_BOXES),
        ("box_rot", (C.c_float * 9) * MAX_BOXES), ("box_half", (C.c_float * 3) * MAX_BOXES), ("box_rest", C.c_float * MAX_BOXES),
        ("n_hull", C.c_int32 * 2), ("foot_hull", ((C.c_float * 3) * MAX_HULL) * 2),
    ]


class PlenConfigC(C.Structure):
    _fields_ = [
        ("dt", C.c_float), ("substeps", C.c_int32), ("reset_ticks", C.c_int32), ("gravity_z", C.c_float),
        ("start_pos", C.c_float * 3), ("motor_max_force", C.c_float), ("joint_act", C.c_int32),
        ("linear_damping", C.c_float), ("mu_lateral", C.c_float), ("mu_spinning", C.c_float),
        ("mu_rolling", C.c_float), ("restitution", C.c_float),
        ("env_lo", C.c_double * NJ), ("env_hi", C.c_double * NJ), ("max_episode_steps", C.c_int32),
        ("motor_kp", C.c_float), ("motor_kd", C.c_float), ("solver_iterations", C.c_int32),
        ("residual_threshold", C.c_float), ("erp_contact", C.c_float), ("erp_joint", C.c_float),
        ("linear_slop", C.c_float), ("warmstart_factor", C.c_float), ("restitution_vel_threshold", C.c_float),
        ("hull_margin", C.c_float), ("max_coord_velocity", C.c_float), ("auto_reset", C.c_int32),
        ("link_contacts", C.c_int32), ("mu_link", C.c_float), ("sole_manifold", C.c_int32), ("support_tie", C.c_float),
    ]


def model_to_c(model: PlenModel) -> PlenModelC:
    m = PlenModelC()
    for l in range(N_LANES):
        for k in range(9):
            m.R_pj[l][k] = float(model.R_pj[l].reshape(9)[k])
        for k in range(3):
            m.p_pj[l][k] = float(model.p_pj[l][k])
            m.axis[l][k] = float(model.axis[l][k])
            m.com[l][k] = float(model.com[l][k])
        for k in range(6):
            m.inertia[l][k] = float(model.inertia[l][k])
        m.mass[l] = float(model.mass[l])
        m.lower[l] = float(model.lower[l])
        m.upper[l] = float(model.upper[l])
        m.chain_start[l] = int(model.chain_start[l])
    for f in range(2):
        m.foot_lane[f] = int(model.foot_lane[f])
        m.foot_break[f] = float(model.foot_break[f])
        for p in range(4):
            for k in range(3):
                m.foot_pts[f][p][k] = float(model.foot_pts[f][p][k])
    for f in range(2):
        hull = model.foot_hull[f]
        m.n_hull[f] = min(len(hull), MAX_HULL)
        for i in range(m.n_hull[f]):
            for k in range(3):
                m.foot_hull[f][i][k] = float(hull[i][k])
    m.n_boxes = int(model.n_boxes)
    for b in range(int(model.n_boxes)):
        m.box_lane[b] = int(model.box_lane[b])
        m.box_rest[b] = float(model.box_rest[b])
        for k in range(3):
            m.box_center[b][k] = float(model.box_center[b][k])
            m.box_half[b][k] = float(model.box_half[b][k])
        for k in range(9):
            m.box_rot[b][k] = float(np.asarray(model.box_rot[b]).reshape(9)[k])
    return m


EXPORTS = (
    "plen_version", "plen_default_config", "plen_create", "plen_destroy", "plen_last_error", "plen_num_envs", "plen_kernel_launches",
    "plen_reset", "plen_step", "plen_step_host", "plen_fault_count", "plen_get_state", "plen_set_state", "plen_set_env_scales", "plen_set_env_mass", "plen_get_env_mass", "plen_set_env_latency", "plen_get_env_latency", "plen_get_manifold", "plen_set_manifold", "plen_tick",
    "plen_debug_dynamics", "plen_debug_records", "plen_gait_ik", "plen_profile_enable", "plen_profile_read", "plen_measure_fp32_peak",
    "plen_replay_create", "plen_replay_destroy", "plen_replay_size", "plen_replay_ptr", "plen_replay_storage",
    "plen_replay_add", "plen_replay_sample", "plen_actor_forward", "plen_actor_forward_tc", "plen_actor_tc_timed_out", "plen_td3_last_error", "plen_td3_set_precision", "plen_td3_tc_timed_out",
    "plen_td3_default_hyper", "plen_td3_create", "plen_td3_destroy", "plen_td3_launches", "plen_td3_sample",
    "plen_td3_set_batch", "plen_td3_critic_grads", "plen_td3_actor_grads", "plen_td3_adam", "plen_td3_soft_update",
    "plen_td3_train",
)

TD3_ACTOR_PARAMS, TD3_CRITIC_PARAMS = 77330, 155138


class PlenTd3HyperC(C.Structure):
    _fields_ = [("discount", C.c_float), ("tau", C.c_float), ("policy_noise", C.c_float), ("noise_clip", C.c_float),
                ("max_action", C.c_float), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("policy_freq", C.c_int32)]


class PlenTd3ParamsC(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("actor", "actor_target", "critic", "critic_target", "actor_m", "actor_v",
                                          "critic_m", "critic_v", "actor_grad", "critic_grad")]

_lib = None


def load_library(path: str = LIB_PATH):
    """dlopen libplen_b200.so and declare the prototypes of every symbol include/plen_b200.h exports."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(
            "libplen_b200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`python -m plen_ml_walk_b200.build`. There is no CPU fallback." % path)
    L = C.CDLL(path)
    vp, ip = C.c_void_p, C.c_int
    L.plen_version.restype = C.c_char_p
    L.plen_default_config.argtypes = [C.POINTER(PlenConfigC), ip]
    L.plen_create.argtypes = [C.POINTER(PlenConfigC), C.POINTER(PlenModelC), ip, ip]
    L.plen_create.restype = vp
    L.plen_destroy.argtypes = [vp]
    L.plen_destroy.restype = None
    L.plen_last_error.argtypes = [vp]
    L.plen_last_error.restype = C.c_char_p
    L.plen_num_envs.argtypes = [vp]
    L.plen_kernel_launches.argtypes = [vp]
    L.plen_kernel_launches.restype = C.c_ulonglong
    L.plen_reset.argtypes = [vp, vp, vp, vp]
    L.plen_step.argtypes = [vp] * 8
    L.plen_step_host.argtypes = [vp] * 6
    L.plen_fault_count.argtypes = [vp, C.POINTER(C.c_ulonglong)]
    L.plen_get_state.argtypes = [vp] * 5
    L.plen_set_state.argtypes = [vp] * 5
    L.plen_set_env_scales.argtypes = [vp] * 5
    L.plen_set_env_mass.argtypes = [vp] * 4
    L.plen_get_env_mass.argtypes = [vp] * 4
    L.plen_set_env_latency.argtypes = [vp] * 4
    L.plen_get_env_latency.argtypes = [vp] * 4
    L.plen_tick.argtypes = [vp, vp, ip, vp]
    L.plen_get_manifold.argtypes = [vp, vp, vp]
    L.plen_set_manifold.argtypes = [vp, vp, vp]
    L.plen_debug_dynamics.argtypes = [vp] * 5
    L.plen_debug_records.argtypes = [vp] * 3
    L.plen_profile_enable.argtypes = [vp, ip]
    L.plen_profile_read.argtypes = [vp] * 5
    ll, ull = C.c_longlong, C.c_ulonglong
    L.plen_replay_create.argtypes = [ll, ip]
    L.plen_replay_create.restype = vp
    L.plen_replay_destroy.argtypes = [vp]
    L.plen_replay_destroy.restype = None
    L.plen_replay_size.argtypes = [vp]
    L.plen_replay_size.restype = ll
    L.plen_replay_ptr.argtypes = [vp]
    L.plen_replay_ptr.restype = ll
    L.plen_replay_storage.argtypes = [vp]
    L.plen_replay_storage.restype = vp
    L.plen_replay_add.argtypes = [vp] * 6 + [ip, vp]
    L.plen_replay_sample.argtypes = [vp, ip, ull] + [vp] * 7
    L.plen_actor_forward.argtypes = [ip] + [vp] * 7 + [ip, C.c_float, C.c_float, ull, vp, vp]
    L.plen_actor_forward_tc.argtypes = [ip] + [vp] * 7 + [ip, C.c_float, C.c_float, ull, vp, vp]
    L.plen_td3_last_error.restype = C.c_char_p
    hp, pp = C.POINTER(PlenTd3HyperC), C.POINTER(PlenTd3ParamsC)
    L.plen_td3_default_hyper.argtypes = [hp]
    L.plen_td3_create.argtypes = [ip, ip]
    L.plen_td3_create.restype = vp
    L.plen_td3_destroy.argtypes = [vp]
    L.plen_td3_destroy.restype = None
    L.plen_td3_set_precision.argtypes = [vp, ip]
    L.plen_td3_launches.argtypes = [vp]
    L.plen_td3_launches.restype = ll
    L.plen_td3_sample.argtypes = [vp, vp, ip, ull, vp]
    L.plen_td3_set_batch.argtypes = [vp] * 6 + [ip, vp]
    L.plen_td3_critic_grads.argtypes = [vp, pp, hp, vp, ull, vp, vp]
    L.plen_td3_actor_grads.argtypes = [vp, pp, hp, vp, vp]
    L.plen_td3_adam.argtypes = [vp, vp, vp, vp, ip, ll, hp, ip, vp]
    L.plen_td3_soft_update.argtypes = [vp, vp, ip, C.c_float, ip, vp]
    L.plen_td3_train.argtypes = [vp, pp, hp, vp, ip, ll, ll, ll, ull, vp, vp]
    L.plen_gait_ik.argtypes = [ip, vp, ip, vp, vp, vp, vp]
    L.plen_measure_fp32_peak.argtypes = [ip, ip, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    _lib = L
    return L
