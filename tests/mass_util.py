"""TEST-ONLY helpers for the per-robot mass tables (plen_set_env_mass): the models a robot with body mass scales s [19] and a
torso payload (m, x, y, z) must be equivalent to, built independently of the device code.

  equivalent_tree   the oracle's 33-link tree with every URDF link of body b scaled by s_b and the payload folded into the base
                    link (new mass, new com, parallel-axis inertia).  The oracle stores a diagonal base inertia, so the payload
                    must sit on one of the base link's principal axes through its com (payload_on_base_axis).
  equivalent_model  the product's 19-body lane tables (PlenModel) with the same scaling and the payload folded into lane 0.
"""
import copy

import numpy as np

BODY_LANES = [0] + list(range(6, 24))     # body b of the [N,19] scale array lives on lane BODY_LANES[b]


def payload_on_base_axis(tree, m, axis, t):
    """(m, x, y, z): m kg at the base link's com shifted by t metres along body axis `axis` (0 x, 1 y, 2 z)."""
    r = np.array(tree["base_com"], dtype=np.float64)
    r[axis] += t
    return np.array([m, r[0], r[1], r[2]])


def _fold_point_mass(mass, com, inertia3x3, mp, r):
    """A body (mass, com, inertia about its com) plus a point mass mp at r -> the composite body."""
    M = mass + mp
    c = (mass * com + mp * r) / M
    d0, d1 = com - c, r - c
    I = inertia3x3 + mass * (d0 @ d0 * np.eye(3) - np.outer(d0, d0)) + mp * (d1 @ d1 * np.eye(3) - np.outer(d1, d1))
    return M, c, I


def equivalent_tree(tree, body_links, scale, payload):
    """tree: oracle.urdf_tree.load_tree(); body_links: PlenModel.body_links (24 lanes); scale [19]; payload [4]."""
    t = copy.deepcopy(tree)
    for b, lane in enumerate(BODY_LANES):
        s = float(scale[b])
        for name in body_links[lane]:
            if name == t["base_name"]:
                t["base_mass"] *= s
                t["base_inertia"] = [v * s for v in t["base_inertia"]]
            else:
                i = t["link_names"].index(name)
                t["mass"][i] *= s
                t["inertia"][i] = [v * s for v in t["inertia"][i]]
    mp, r = float(payload[0]), np.asarray(payload[1:4], dtype=np.float64)
    if mp != 0.0:
        M, c, I = _fold_point_mass(t["base_mass"], np.array(t["base_com"]), np.diag(t["base_inertia"]), mp, r)
        off = I - np.diag(np.diag(I))
        assert np.abs(off).max() <= 1e-12 * np.abs(I).max(), "payload off the base link's principal axes"
        t["base_mass"], t["base_com"], t["base_inertia"] = M, c.tolist(), np.diag(I).tolist()
    return t


def equivalent_model(model, scale, payload):
    """model: PlenModel; returns a copy whose lane tables hold the scaled bodies and the payload folded into lane 0."""
    m = copy.deepcopy(model)
    for b, lane in enumerate(BODY_LANES):
        m.mass[lane] *= float(scale[b])
        m.inertia[lane] = m.inertia[lane] * float(scale[b])
    mp, r = float(payload[0]), np.asarray(payload[1:4], dtype=np.float64)
    if mp != 0.0:
        xx, yy, zz, xy, xz, yz = m.inertia[0]
        I0 = np.array([[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]])
        M, c, I = _fold_point_mass(m.mass[0], np.array(m.com[0]), I0, mp, r)
        m.mass[0], m.com[0] = M, c
        m.inertia[0] = [I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[0, 2], I[1, 2]]
    m.total_mass = float(sum(m.mass[l] for l in BODY_LANES))
    return m
