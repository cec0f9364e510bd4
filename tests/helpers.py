"""Shared scene builders for the tests (the reference's test scenes re-expressed through the
host mirror pfc_b200.scenario)."""
import math

import numpy as np

import pfc_b200  # noqa: F401
from pfc_b200 import geometry as G
from pfc_b200 import scenario as S


def rot_x(a):
    c, s = math.cos(a), math.sin(a)
    return np.array([[1, 0, 0], [0, c, -s], [0, s, c]], dtype=float)


def rot_y(a):
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], dtype=float)


def rot_z(a):
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], dtype=float)


def angle_axis(theta, axis):
    a = np.asarray(axis, dtype=float)
    a = a / np.linalg.norm(a)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + math.sin(theta) * K + (1 - math.cos(theta)) * (K @ K)


def rotation_between(u, v):
    """Shortest-arc rotation taking direction u to direction v."""
    u = np.asarray(u, float) / np.linalg.norm(u)
    v = np.asarray(v, float) / np.linalg.norm(v)
    ax = np.cross(u, v)
    s, c = np.linalg.norm(ax), float(u @ v)
    if s < 1e-14:
        if c > 0:
            return np.eye(3)
        p = np.cross(u, [1.0, 0, 0])
        if np.linalg.norm(p) < 1e-8:
            p = np.cross(u, [0, 1.0, 0])
        return angle_axis(math.pi, p)
    return angle_axis(math.atan2(s, c), ax)


def rel_err(a, b):
    """SURVEY.md H7: || a - b ||_inf / max(|| b ||_inf, tiny) per 3-vector."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def wrench_rel_err(w, w_ref, floor=0.0):
    """max over the angular and linear halves; `floor` guards halves that are ~0 by symmetry."""
    w, w_ref = np.asarray(w, float).reshape(-1, 6), np.asarray(w_ref, float).reshape(-1, 6)
    worst = 0.0
    for a, b in zip(w, w_ref):
        for sl in (slice(0, 3), slice(3, 6)):
            den = max(np.max(np.abs(b[sl])), floor, 1e-300)
            worst = max(worst, float(np.max(np.abs(a[sl] - b[sl])) / den))
    return worst


# ---- reference scenes ------------------------------------------------------------------------------
def scene_boxes(backend=None, max_env=1, bristle=False):
    """test/boxes.jl:18-45 (config C1): plane + 4 boxes alternately rigid (tri) / compliant (tet).  bristle=True: the box_1-box_2 and
    box_3-box_4 instructions use bristle friction instead (12 more state entries), for tests of the paths bristle scenes take."""
    r = 0.05
    c_prop = S.ContactProperties(1.0e6)
    i_c, i_r = S.InertiaProperties(400.0), S.InertiaProperties(400.0, d=r)
    box = G.eMesh_box(r)
    m = S.MechanismScenario()
    id_plane = S.add_contact(m, "plane", G.as_tet_eMesh(G.eMesh_half_plane()), c_prop=c_prop)
    b1 = S.add_body_contact(m, "box_1", G.as_tri_eMesh(box), i_prop=i_r)
    b2 = S.add_body_contact(m, "box_2", G.as_tet_eMesh(box), i_prop=i_c, c_prop=c_prop)
    b3 = S.add_body_contact(m, "box_3", G.as_tri_eMesh(box), i_prop=i_r)
    b4 = S.add_body_contact(m, "box_4", G.as_tet_eMesh(box), i_prop=i_c, c_prop=c_prop)
    S.add_friction_regularize(m, id_plane, b1[2], mu_d=0.0, chi=2.2, n_quad_rule=2)
    add_12_34 = (lambda a, c: S.add_friction_bristle(m, a, c, mu_d=0.2, chi=0.2, k_bar=2.0e4, tau=0.05, n_quad_rule=2)) if bristle else (
        lambda a, c: S.add_friction_regularize(m, a, c, mu_d=0.2, chi=0.2, n_quad_rule=2))
    add_12_34(b1[2], b2[2])
    S.add_friction_regularize(m, b2[2], b3[2], mu_d=0.2, chi=0.2, n_quad_rule=2)
    add_12_34(b3[2], b4[2])
    S.finalize(m, backend, max_env)
    for k, b in enumerate((b1, b2, b3, b4)):
        S.set_state_spq(m, b[0], trans=(0.0, 0.0, (2 + 3 * k) * r), w=(0.0, 0.0, float(k + 1)))
    return m, (b1, b2, b3, b4)


def _tet_tet_scene(backend, n_env):
    """test/test_vol_vol.jl-style volumetric contact: plane + two compliant (tet) boxes; instructions plane-box_1 and box_1-box_2
    (regularized) and box_2-box_1 (bristle), so n_small = 3."""
    r = 0.05
    c_prop = S.ContactProperties(1.0e6)
    m = S.MechanismScenario()
    id_plane = S.add_contact(m, "plane", G.as_tet_eMesh(G.eMesh_half_plane()), c_prop=c_prop)
    b1 = S.add_body_contact(m, "box_1", G.as_tet_eMesh(G.eMesh_box(r)), i_prop=S.InertiaProperties(400.0), c_prop=c_prop)
    b2 = S.add_body_contact(m, "box_2", G.as_tet_eMesh(G.eMesh_box(r)), i_prop=S.InertiaProperties(400.0), c_prop=S.ContactProperties(3.0e6))
    S.add_friction_regularize(m, id_plane, b1[2], mu_d=0.0, chi=0.0, n_quad_rule=2)
    S.add_friction_regularize(m, b1[2], b2[2], mu_s=0.4, mu_d=0.3, chi=0.7, v_tol=1e-3, n_quad_rule=2)
    S.add_friction_bristle(m, b2[2], b1[2], mu_d=0.3, chi=0.3, k_bar=1.0e5, tau=0.02, n_quad_rule=1)
    S.finalize(m, backend, n_env)
    return m


def _sphere_scene(n_div_a=4, n_div_b=3, with_small=True):
    """Builder of a scene of curved meshes (a tri and a tet sphere against a tet ground sphere, plus a box on a plane with
    with_small=True): large-path or mid-size instructions depending on the subdivision levels."""
    def build(backend, n_env):
        m = S.MechanismScenario()
        sa, sb = G.eMesh_sphere(0.05, n_div_a), G.eMesh_sphere(0.06, n_div_b)
        ground = S.add_contact(m, "ground", G.as_tet_eMesh(sb), c_prop=S.ContactProperties(2.0e6))
        b1 = S.add_body_contact(m, "s_tri", G.as_tri_eMesh(sa), i_prop=S.InertiaProperties(400.0, d=0.01))
        b2 = S.add_body_contact(m, "s_tet", G.as_tet_eMesh(sa), i_prop=S.InertiaProperties(400.0), c_prop=S.ContactProperties(1.0e6))
        S.add_friction_regularize(m, b1[2], ground, mu_s=0.4, mu_d=0.3, chi=0.5, n_quad_rule=2)   # tri-tet, large
        S.add_friction_regularize(m, b2[2], ground, mu_d=0.3, chi=0.5, n_quad_rule=1)            # tet-tet, large
        S.add_friction_bristle(m, b1[2], b2[2], mu_d=0.4, k_bar=2.0e4, tau=0.05, n_quad_rule=2)  # tri-tet, large, bristle
        if with_small:
            box = S.add_body_contact(m, "box", G.as_tri_eMesh(G.eMesh_box(0.03)), i_prop=S.InertiaProperties(400.0, d=0.01))
            plane = S.add_contact(m, "plane", G.as_tet_eMesh(G.eMesh_half_plane()), c_prop=S.ContactProperties(1.0e6))
            S.add_friction_regularize(m, box[2], plane, mu_d=0.3, chi=0.5, n_quad_rule=2)        # small path in the same scene
        S.finalize(m, backend, n_env)
        return m
    return build


def _sphere_states(m, n_env, seed, with_small=True):
    """Seeded states of _sphere_scene: the spheres overlap the ground sphere (even environments) or each other (odd ones)."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n_env, S.num_x(m)))
    nq = m.nq
    for e in range(n_env):
        d1 = rng.standard_normal(3); d1 /= np.linalg.norm(d1)
        d2 = rng.standard_normal(3); d2 /= np.linalg.norm(d2)
        x[e, 0:3] = rng.uniform(-0.3, 0.3, 3)
        x[e, 3:6] = d1 * rng.uniform(0.095, 0.108)
        x[e, 6:9] = rng.uniform(-0.3, 0.3, 3)
        x[e, 9:12] = x[e, 3:6] + d2 * rng.uniform(0.085, 0.098) if e % 2 else d2 * rng.uniform(0.095, 0.108)
        if with_small:
            x[e, 12:15] = rng.uniform(-0.02, 0.02, 3)
            x[e, 15:18] = [rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), 0.03 - rng.uniform(0, 0.003)]
        x[e, nq:nq + m.nv] = rng.uniform(-1, 1, m.nv) * 0.3
        x[e, nq + m.nv:] = rng.uniform(-1, 1, 6) * 1e-4
    return x


def splitmix64(seed):
    state = seed & 0xFFFFFFFFFFFFFFFF

    def nxt():
        nonlocal state
        state = (state + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        z = state
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        z = z ^ (z >> 31)
        return (z >> 11) * (1.0 / 9007199254740992.0)

    return nxt


def boxes_env_states(m, n_env, r=0.05, start=0):
    """Config C3: randomized *settled-stack* states of the test/boxes.jl scene, env e seeded with
    splitmix64(0x5EED0000 + e).  Box k (1..4) sits at z = (2k-1) r minus a cumulative sink of
    U(0, 0.02) r per level, with xy jitter, a small tilt, a free yaw and random twists, so that
    every instruction has real contact work.  (SURVEY.md section 8d's formula keeps the 3 r drop
    spacing of boxes.jl:42-45, at which nothing touches and only the root SAT would run.)"""
    nq = m.nq
    X = np.zeros((n_env, S.num_x(m)))
    for e in range(n_env):
        u = splitmix64(0x5EED0000 + start + e)
        U = lambda lo, hi: lo + (hi - lo) * u()
        sink = 0.0
        for k in range(1, 5):
            b = m.bodies[k]
            sink += U(0.0, 0.02) * r
            xy = [U(-0.5, 0.5) * r, U(-0.5, 0.5) * r]
            z = (2 * k - 1) * r - sink
            mrp = [U(-0.005, 0.005), U(-0.005, 0.005), U(-0.2, 0.2)]
            om = [U(-1, 1) * k for _ in range(3)]
            vel = [U(-0.1, 0.1) for _ in range(3)]
            X[e, b.q0:b.q0 + 6] = mrp + xy + [z]
            X[e, nq + b.v0:nq + b.v0 + 6] = om + vel
        X[e, nq + m.nv:] = [U(-1e-4, 1e-4) for _ in range(6 * m.n_bristle)]
    return X


def kernel_grids(fn):
    """Runs fn() under torch.profiler and returns [(kernel name, grid x)] of every kernel launched on the device, in launch order:
    which template instance of a launcher ran, and with how many CTAs, is what the batch-shape tests assert.  fn must leave its
    work finished (it synchronises the device again here anyway)."""
    import json
    import os
    import tempfile

    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    finally:
        os.remove(path)
    ks = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return [(e["name"], int(e["args"]["grid"][0])) for e in ks]
