"""GPU tests of per-environment body parameters (pfc_set_body_params): with a table set, environment e of every calcXd!, Jacobian and
Radau entry point gives the bits of a context whose pfc_set_dynamics got row e (spatial inertias and gravity), evaluated on the same
batch.  Rows are physical: masses scaled 0.5-2x, centres of mass moved by up to 10 % of the box, second moments scaled per axis, gravity
tilted by up to 15 degrees and rescaled.

(The file name sorts after test_gpu_batch_shapes.py and test_gpu_jacobian_scale.py on purpose: their torch.profiler kernel lists lose the
first kernels of the profiled call once the process has run long enough -- 15 s more of any GPU work ahead of them is enough on a B200 --
and these tests take about that long.)"""
import numpy as np
import pytest
import torch

import pfc_b200  # noqa: F401
from helpers import _tet_tet_scene, boxes_env_states, scene_boxes
from pfc_b200 import capi, dynamics
from pfc_b200 import scenario as S
from test_gpu_contact_params import _Constants, _calcxd_device, _jacobian_device, _radau_run, _random_table, _same_row, _t

pytestmark = pytest.mark.gpu

PFC_E_ARG = -1
DEV = torch.device("cuda", 0)


def _body_inertias(m):
    """(tensor_I about the centre of mass, com, mass, mesh) of every floating body, as scenario.finalize builds them."""
    out = {}
    for k, b in enumerate(m.bodies):
        if b.joint is None:
            continue
        mesh = next(mc.mesh for mc in m.MeshCache if mc.body_id == k)
        out[k] = dynamics.make_inertia_info(mesh, b.i_prop)[:3] + (mesh,)
    return out


def _own_bodies(m, n_env):
    """The scene's own spatial inertias and gravity as a table."""
    H = np.zeros((len(m.bodies), 6, 6))
    for k, (I, com, mass, _) in _body_inertias(m).items():
        H[k] = dynamics.spatial_inertia(I, com, mass)
    return np.repeat(H[None], n_env, 0), np.repeat(np.asarray(m.gravity, dtype=np.float64)[None], n_env, 0)


def _random_bodies(m, n_env, seed):
    """Random physical rows: per floating body the mass times U(0.5, 2), the second moments about the centre of mass scaled per axis
    (so the inertia stays a rigid body's), the centre of mass moved by up to 10 % of the mesh's extent per axis; gravity tilted by up to
    15 degrees about a random horizontal-ish axis and its magnitude times U(0.8, 1.2).  World-attached rows are NaN (ignored)."""
    rng = np.random.default_rng(seed)
    H = np.full((n_env, len(m.bodies), 6, 6), np.nan)
    for k, (I, com, mass, mesh) in _body_inertias(m).items():
        ext = np.ptp(np.asarray(mesh.point, dtype=np.float64), axis=0)
        sigma = 0.5 * np.trace(I) * np.eye(3) - I   # int r r' dm about the centre of mass
        for e in range(n_env):
            ms = rng.uniform(0.5, 2.0)
            s = np.diag(rng.uniform(0.8, 1.25, 3))
            sig = ms * s @ sigma @ s
            Ie = np.trace(sig) * np.eye(3) - sig
            H[e, k] = dynamics.spatial_inertia(Ie, com + rng.uniform(-0.1, 0.1, 3) * ext, mass * ms)
    g0 = np.asarray(m.gravity, dtype=np.float64)
    g = np.zeros((n_env, 3))
    for e in range(n_env):
        axis = np.cross(g0, rng.normal(size=3))
        axis /= np.linalg.norm(axis)
        a = np.deg2rad(rng.uniform(0.0, 15.0))
        K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        R = np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K
        g[e] = rng.uniform(0.8, 1.2) * R @ g0
    return H, g


def _with_row(m, H, g, e):
    """m's backend after pfc_set_dynamics got row e (world-attached rows are ignored, so zeros stand in for their NaN)."""
    m.backend.set_dynamics(np.nan_to_num(H[e]), g[e])
    return m


def _dual6_device(ctx, x, seed):
    n_env, nx = x.shape
    xd = _t(x)
    xdot7 = torch.zeros((n_env, nx, 7), dtype=torch.float64, device=DEV)
    np_ = torch.zeros((n_env, ctx.n_ins), dtype=torch.int64, device=DEV)
    fl = torch.zeros((n_env, ctx.n_ins), dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    ctx.calcxd_dual6_device(n_env, xd.data_ptr(), None, seed, xdot7.data_ptr(), np_.data_ptr(), fl.data_ptr())
    ctx.sync()
    return dict(xdot7=xdot7.cpu().numpy(), n_pairs=np_.cpu().numpy(), flags=fl.cpu().numpy())


def _dynamics_entry_points(ctx, x, dual=True):
    """Every dynamics entry point of ctx on the batch x, host and device: name -> dict of outputs."""
    out = dict(calcxd_host=ctx.calcxd_f64(x), calcxd_device=_calcxd_device(ctx, x), jac_host=ctx.calcxd_jacobian(x),
               jac_device=_jacobian_device(ctx, x))
    if dual:
        for seed in range(0, x.shape[1], 6):
            out[f"dual6_host_{seed}"] = ctx.calcxd_dual6(x, seed)
            out[f"dual6_device_{seed}"] = _dual6_device(ctx, x, seed)
    return out


def _keys(name):
    if name.startswith("dual6"):
        return ("xdot7", "n_pairs", "flags")
    if name.startswith("jac"):
        return ("jac", "xdot", "n_pairs", "flags")
    return ("xdot", "n_pairs", "flags")


def _check_scene(build, x, envs, seed, dual=True):
    """Table context against one context per sampled environment whose pfc_set_dynamics got its row, bit for bit; the table changes
    x_dot of at least 90 % of the environments."""
    n_env = x.shape[0]
    m = build(capi.Context(0))
    ctx = m.backend
    H, g = _random_bodies(m, n_env, seed)
    base = _dynamics_entry_points(ctx, x, dual)
    ctx.set_body_params(H, g)
    got = _dynamics_entry_points(ctx, x, dual)
    changed = np.mean([not np.array_equal(base["calcxd_device"]["xdot"][e], got["calcxd_device"]["xdot"][e]) for e in range(n_env)])
    assert changed >= 0.9, changed
    for a, b in (("calcxd_host", "calcxd_device"), ("jac_host", "jac_device")):
        _same_row(got[a], got[b], slice(None), _keys(a))
    for e in envs:
        ref = _dynamics_entry_points(_with_row(build(capi.Context(0)), H, g, e).backend, x, dual)
        for name in got:
            _same_row(got[name], ref[name], e, _keys(name))


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_boxes_every_dynamics_entry_point_per_environment():
    """boxes.jl at 8 n_sm + 1 environments: pfc_calcxd_f64, every seed chunk of pfc_calcxd_dual6 and pfc_calcxd_jacobian, host and device."""
    n_sm = _n_sm()
    n_env = 8 * n_sm + 1
    m0, _ = scene_boxes(None)
    x = boxes_env_states(m0, n_env)
    _check_scene(lambda be: scene_boxes(be, max_env=n_env)[0], x, [0, 1, 4 * n_sm, 6 * n_sm + 7, 8 * n_sm], seed=41)


def test_tet_tet_and_bristle_scenes_per_environment():
    """The tet-tet scene (three small problems per environment: narrow tiles hold neighbours' problems, which calcXd! does not mind) and
    boxes.jl with bristle friction: calcXd! and its Jacobian."""
    from test_gpu_batch_shapes import _tet_tet_states
    n_env = 101
    x = _tet_tet_states(_tet_tet_scene(None, 1), n_env, 5)
    _check_scene(lambda be: _tet_tet_scene(be, n_env), x, [0, 37, 100], seed=42, dual=False)
    n_env = 300
    m0, _ = scene_boxes(None, bristle=True)
    x = boxes_env_states(m0, n_env)
    _check_scene(lambda be: scene_boxes(be, max_env=n_env, bristle=True)[0], x, [0, 150, 299], seed=43, dual=False)


def _check_radau(build, x0, H, g, envs, P=None, ebar=None, n_step=10):
    knots = np.array([0.012, 0.02, 0.03, 0.04])
    m = build(capi.Context(0))
    tau = np.random.default_rng(47).uniform(-2.0, 2.0, (len(knots), x0.shape[0], m.nv))
    if P is not None:
        m.backend.set_contact_params(P)
    m.backend.set_body_params(H, g)
    steps, ro, dev_steps, dev_ro = _radau_run(m.backend, x0, n_step, knots, tau)
    for a, b in zip(steps, dev_steps):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)
    for u, v in zip(ro, dev_ro):
        assert np.array_equal(u, v)
    assert (ro[3][:, 0] == len(knots)).all()
    for e in envs:
        be = capi.Context(0) if P is None else _Constants(capi.Context(0), ebar[e], P[e])
        mr = _with_row(build(be), H, g, e)
        r_steps, r_ro, _, _ = _radau_run(mr.backend, x0, n_step, knots, tau)
        for a, b in zip(steps, r_steps):
            for u, v in zip(a, b):
                assert np.array_equal(u[e], v[e]), e
        x, t, x_knot, st = ro
        rx, rt, rk, rs = r_ro
        assert np.array_equal(x[e], rx[e]) and np.array_equal(t[e], rt[e]) and np.array_equal(x_knot[:, e], rk[:, e]) and np.array_equal(st[e], rs[e])
    return steps, ro


def test_radau_step_and_rollout_per_environment():
    """64 boxes.jl environments with distinct rows: 10 pfc_radau_step calls and a 4-knot pfc_radau_rollout with a tau_ext schedule.
    Sampled environments equal a context built with their row (x, t, h_taken, x_knot, stats bit for bit); host = device entry points."""
    n_env = 64
    build = lambda be: scene_boxes(be, max_env=n_env)[0]
    m = build(None)
    x0 = boxes_env_states(m, n_env)
    H, g = _random_bodies(m, n_env, 44)
    _check_radau(build, x0, H, g, (0, 17, 63))


def test_contact_and_body_tables_together():
    """A contact table and a body table at once equal a context built with both rows: calcXd! and a roll-out."""
    n_env = 64
    build = lambda be: scene_boxes(be, max_env=n_env)[0]
    m = build(capi.Context(0))
    x0 = boxes_env_states(m, n_env)
    P, ebar = _random_table(m, n_env, 45)
    H, g = _random_bodies(m, n_env, 46)
    m.backend.set_contact_params(P)
    m.backend.set_body_params(H, g)
    got = _calcxd_device(m.backend, x0)
    for e in (0, 31, 63):
        mr = _with_row(build(_Constants(capi.Context(0), ebar[e], P[e])), H, g, e)
        _same_row(got, _calcxd_device(mr.backend, x0), e, ("xdot", "n_pairs", "flags"))
    _check_radau(build, x0, H, g, (5, 40), P=P, ebar=ebar, n_step=2)


def test_own_values_change_nothing():
    """A table of the scene's own inertias and gravity gives the bits of no table: 4096 environments through pfc_calcxd_f64_device,
    pfc_calcxd_jacobian_device and a short roll-out."""
    n_env = 4096
    m, _ = scene_boxes(capi.Context(0), max_env=n_env)
    x = boxes_env_states(m, n_env)
    H, g = _own_bodies(m, n_env)

    def run():
        out = dict(xd=_calcxd_device(m.backend, x), jac=_jacobian_device(m.backend, x))
        m.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        out["ro"] = m.backend.radau_rollout(x, np.zeros(n_env), [0.003])
        return out
    a = run()
    m.backend.set_body_params(H, g)
    b = run()
    for k in ("xdot", "n_pairs", "flags"):
        assert np.array_equal(a["xd"][k], b["xd"][k])
    for k in ("jac", "xdot", "n_pairs", "flags"):
        assert np.array_equal(a["jac"][k], b["jac"][k])
    for u, v in zip(a["ro"], b["ro"]):
        assert np.array_equal(u, v)


def test_argument_errors_keep_the_table():
    """Each rejected call returns PFC_E_ARG and leaves the table in force; entry points that read it require its n_env, the others do not;
    pfc_set_dynamics, pfc_set_bodies and n_env = 0 clear it."""
    L = capi.lib()
    n_env = 8
    c0 = capi.Context(0)
    assert L.pfc_set_body_params(c0._h, 0, None, None) == PFC_E_ARG                       # before pfc_set_dynamics
    m, _ = scene_boxes(capi.Context(0), max_env=n_env)
    c = m.backend
    x = boxes_env_states(m, n_env)
    H, g = _random_bodies(m, n_env, 48)
    own, own4 = _calcxd_device(c, x)["xdot"], c.calcxd_f64(x[:4])["xdot"]
    c.set_body_params(H, g)
    want = c.calcxd_f64(x)["xdot"]
    assert not np.array_equal(want, own)
    k = next(k for k, b in enumerate(m.bodies) if b.joint is not None)
    bad = []
    big_H, big_g = np.concatenate([H, H], 0), np.concatenate([g, g], 0)
    bad.append(lambda: L.pfc_set_body_params(c._h, n_env + 1, big_H.ctypes.data, big_g.ctypes.data))   # n_env > max_env
    bad.append(lambda: L.pfc_set_body_params(c._h, -1, H.ctypes.data, g.ctypes.data))
    bad.append(lambda: L.pfc_set_body_params(c._h, n_env, None, g.ctypes.data))
    bad.append(lambda: L.pfc_set_body_params(c._h, n_env, H.ctypes.data, None))
    Hn = H.copy(); Hn[3, k, 1, 4] = np.nan
    gn = g.copy(); gn[5, 2] = np.inf
    Hs = H.copy(); Hs[3, k, 0, 1] += 1e-3 * Hs[3, k, 0, 0]                                  # not symmetric
    Hp = H.copy(); Hp[3, k, 3:, 3:] *= -1.0                                                 # negative mass: not positive definite
    for Hx, gx in ((Hn, g), (H, gn), (Hs, g), (Hp, g)):
        bad.append(lambda Hx=Hx, gx=gx: L.pfc_set_body_params(c._h, n_env, Hx.ctypes.data, gx.ctypes.data))
    for call in bad:
        assert call() == PFC_E_ARG
        assert np.array_equal(c.calcxd_f64(x)["xdot"], want)
    for Hx in (Hs, Hp):
        L.pfc_set_body_params(c._h, n_env, Hx.ctypes.data, g.ctypes.data)
        assert f"environment 3, body {k}".encode() in L.pfc_last_error()
    # rows of world-attached bodies are ignored (their NaN included)
    assert np.isnan(H[:, 0]).all()
    # batch size: the entry points that read the table refuse another n_env, the evaluations that do not read it accept one
    for call in (lambda: c.calcxd_f64(x[:4]), lambda: c.calcxd_jacobian(x[:4]), lambda: c.calcxd_dual6(x[:4], 0), lambda: c.radau_init(4)):
        with pytest.raises(capi.PfcError) as ei:
            call()
        assert ei.value.code == PFC_E_ARG
    assert b"body-parameter table" in L.pfc_last_error()
    c.eval_state_f64(x[:4])
    X, tw, _ = S.boundary_arrays(m, x[:4])
    c.eval_f64(X, tw, None)
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    c.set_body_params(H[:4], g[:4])
    for call in (lambda: c.radau_step(x, np.zeros(n_env)), lambda: c.radau_rollout(x, np.zeros(n_env), [0.01])):
        with pytest.raises(capi.PfcError) as ei:
            call()
        assert ei.value.code == PFC_E_ARG
    # pfc_set_dynamics clears the table: any batch size again, its own values
    H_own, g_own = _own_bodies(m, 1)
    c.set_dynamics(H_own[0], g_own[0])
    assert np.array_equal(c.calcxd_f64(x)["xdot"], own)
    assert np.array_equal(c.calcxd_f64(x[:4])["xdot"], own4)
    # so does pfc_set_bodies (scenario.finalize's description of the same mechanism)
    c.set_body_params(H, g)
    pose = np.array([np.concatenate([b.pose_R.reshape(9), b.pose_t]) for b in m.bodies])
    c.set_bodies([0 if b.joint is None else 1 for b in m.bodies], [b.q0 for b in m.bodies], [b.v0 for b in m.bodies],
                 [mc.body_id for mc in m.MeshCache], m.nq, m.nv, pose=pose)
    assert np.array_equal(c.calcxd_f64(x[:4])["xdot"], own4)
    # and n_env = 0
    c.set_body_params(H, g)
    assert np.array_equal(c.calcxd_f64(x)["xdot"], want)
    c.set_body_params(None)
    assert np.array_equal(c.calcxd_f64(x[:4])["xdot"], own4)
