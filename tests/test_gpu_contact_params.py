"""GPU tests of per-environment contact parameters (pfc_set_contact_params): with a table set, environment e of every evaluation gives the
bits of a context whose scene was built with row e's values (Ebar per tetrahedral mesh, chi and the friction parameters per instruction).
The reference for environment e is always the SAME batch of states evaluated by such a context, so no test relies on batch invariance of
the evaluation itself."""
import numpy as np
import pytest
import torch

import pfc_b200  # noqa: F401
from helpers import _sphere_scene, _sphere_states, _tet_tet_scene, boxes_env_states, scene_boxes, wrench_rel_err
from oracle import orc
from pfc_b200 import capi, scenes
from pfc_b200 import scenario as S

pytestmark = pytest.mark.gpu

PFC_E_ARG = -1
DEV = torch.device("cuda", 0)


class _Constants:
    """A backend (capi.Context or the oracle) whose scene is built with one row of contact constants instead of the scenario's own:
    ebar[mesh] for every mesh, row[ins] = (chi, Ebar_1, Ebar_2, q0..q4) for every instruction (the layout of pfc_set_contact_params)."""

    def __init__(self, inner, ebar, row):
        self._inner, self._ebar, self._row, self._n_mesh, self._n_ins = inner, ebar, row, 0, 0

    def add_mesh(self, kind, xyz, idx, eps, Ebar, tree):
        e = float(self._ebar[self._n_mesh])
        self._n_mesh += 1
        return self._inner.add_mesh(kind, xyz, idx, eps, e, tree)

    def add_instruction(self, mesh_1, mesh_2, chi, model, params, n_quad_rule):
        r = self._row[self._n_ins]
        self._n_ins += 1
        return self._inner.add_instruction(mesh_1, mesh_2, float(r[0]), model, [float(v) for v in r[3:3 + len(params)]], n_quad_rule)

    def __getattr__(self, name):
        return getattr(self._inner, name)


def _own_table(m, n_env):
    """The scene's own constants as a table (and per-mesh Ebar)."""
    ebar = np.array([mc.c_prop.E_bar if mc.mesh.is_tet else 0.0 for mc in m.MeshCache])
    P = np.zeros((len(m.ContactInstructions), 8))
    for k, ci in enumerate(m.ContactInstructions):
        q = ci.friction_model.params()
        P[k, :3] = [ci.chi, ebar[ci.id_1], ebar[ci.id_2]]
        P[k, 3:3 + len(q)] = q
    return np.repeat(P[None], n_env, 0), np.repeat(ebar[None], n_env, 0)


def _random_table(m, n_env, seed):
    """Random constants over ranges that change the contact: Ebar per tetrahedral mesh, chi and friction parameters per instruction.
    Entries the model ignores (Ebar_1 of a triangle mesh_1, q3 / q4 of a regularized instruction) are NaN."""
    rng = np.random.default_rng(seed)
    n_mesh, ins = len(m.MeshCache), m.ContactInstructions
    ebar = np.zeros((n_env, n_mesh))
    for i, mc in enumerate(m.MeshCache):
        if mc.mesh.is_tet:
            ebar[:, i] = mc.c_prop.E_bar * rng.uniform(0.3, 3.0, n_env)
    P = np.full((n_env, len(ins), 8), np.nan)
    for k, ci in enumerate(ins):
        P[:, k, 0] = rng.uniform(0.0, 3.0, n_env)
        P[:, k, 1] = ebar[:, ci.id_1] if m.MeshCache[ci.id_1].mesh.is_tet else np.nan
        P[:, k, 2] = ebar[:, ci.id_2]
        mu_d = rng.uniform(0.05, 0.6, n_env)
        mu_s = mu_d * rng.uniform(1.0, 1.6, n_env)
        if ci.friction_model.model == 0:
            P[:, k, 3:6] = np.stack([mu_s, mu_d, rng.uniform(2e-3, 3e-2, n_env)], 1)
        else:
            P[:, k, 3:8] = np.stack([rng.uniform(0.01, 0.1, n_env), rng.uniform(5e3, 5e4, n_env), mu_s, mu_d, rng.uniform(5e-4, 2e-3, n_env)], 1)
    return P, ebar


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV) if a is not None else None


def _eval_device(ctx, X, tw, s=None):
    n_env, n_ins = X.shape[0], ctx.n_ins
    nb = ctx.n_bristle
    Xd, twd, sd_in = _t(X), _t(tw), _t(np.asarray(s).reshape(n_env, nb, 6)) if nb else None
    w = torch.full((n_env, n_ins, 6), float("nan"), dtype=torch.float64, device=DEV)
    sd = torch.full((n_env, nb, 6), float("nan"), dtype=torch.float64, device=DEV) if nb else None
    np_ = torch.full((n_env, n_ins), -1, dtype=torch.int64, device=DEV)
    fl = torch.zeros((n_env, n_ins), dtype=torch.int32, device=DEV)
    p = lambda t: None if t is None else t.data_ptr()
    torch.cuda.synchronize()
    ctx.eval_f64_device(n_env, p(Xd), p(twd), p(sd_in), p(w), p(sd), p(np_), p(fl))
    ctx.sync()
    return dict(wrench=w.cpu().numpy(), sdot=sd.cpu().numpy() if nb else None, n_pairs=np_.cpu().numpy(), flags=fl.cpu().numpy())


def _calcxd_device(ctx, x):
    n_env, nx = x.shape
    xd = _t(x)
    xdot = torch.zeros((n_env, nx), dtype=torch.float64, device=DEV)
    np_ = torch.zeros((n_env, ctx.n_ins), dtype=torch.int64, device=DEV)
    fl = torch.zeros((n_env, ctx.n_ins), dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    ctx.calcxd_f64_device(n_env, xd.data_ptr(), None, xdot.data_ptr(), np_.data_ptr(), fl.data_ptr())
    ctx.sync()
    return dict(xdot=xdot.cpu().numpy(), n_pairs=np_.cpu().numpy(), flags=fl.cpu().numpy())


def _jacobian_device(ctx, x):
    n_env, nx = x.shape
    xd = _t(x)
    jac = torch.full((n_env, nx, nx), float("nan"), dtype=torch.float64, device=DEV)
    xdot = torch.full((n_env, nx), float("nan"), dtype=torch.float64, device=DEV)
    np_ = torch.zeros((n_env, ctx.n_ins), dtype=torch.int64, device=DEV)
    fl = torch.zeros((n_env, ctx.n_ins), dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    ctx.calcxd_jacobian_device(n_env, xd.data_ptr(), None, jac.data_ptr(), xdot.data_ptr(), np_.data_ptr(), fl.data_ptr())
    ctx.sync()
    return dict(jac=jac.cpu().numpy(), xdot=xdot.cpu().numpy(), n_pairs=np_.cpu().numpy(), flags=fl.cpu().numpy())


def _same_row(a, b, e, keys):
    for k in keys:
        if a[k] is None:
            assert b[k] is None
            continue
        assert np.array_equal(a[k][e], b[k][e]), (k, e)


def _entry_points(m, ctx, x, with_state=True):
    """Every evaluation entry point of ctx (a backend of scenario m) on the batch x: name -> dict of outputs."""
    X, tw, s = S.boundary_arrays(m, x)
    out = dict(eval_device=_eval_device(ctx, X, tw, s), eval_host=ctx.eval_f64(X, tw, s))
    if with_state:
        out["state"] = ctx.eval_state_f64(x)
        out["calcxd"] = _calcxd_device(ctx, x)
        out["jacobian"] = _jacobian_device(ctx, x)
    return out


_KEYS = dict(eval_device=("wrench", "sdot", "n_pairs", "flags"), eval_host=("wrench", "sdot", "n_pairs", "flags"),
             state=("f_generalized", "sdot", "n_pairs", "flags"), calcxd=("xdot", "n_pairs", "flags"), jacobian=("jac", "xdot", "n_pairs", "flags"))


def _tile_neighbours(e, per_env, n_env, tile=4):
    """The environments whose problems share a narrow tile (4 problems) with environment e's, when every environment has per_env small
    problems."""
    lo, hi = (e * per_env) // tile, ((e + 1) * per_env - 1) // tile
    return range((lo * tile) // per_env, min(n_env - 1, (hi * tile + tile - 1) // per_env) + 1)


def _check_scene(build, x, envs, seed, with_state=True, min_changed=0.9, tile_share=None):
    """Table context against one reference context per sampled environment, through every entry point, bit for bit.

    tile_share = small problems per environment, for scenes whose narrow tiles (4 problems) hold problems of neighbouring environments.
    The tile kernel's sums of a problem depend, in the last bits, on where its items fall among the tile's other items, so on the clip
    results of those neighbours -- with or without a table.  The environments that share a tile with a sampled one then carry its row, so
    that its tiles are the same in both contexts."""
    n_env = x.shape[0]
    m = build(capi.Context(0))
    ctx = m.backend
    P, ebar = _random_table(m, n_env, seed)
    if tile_share:
        for e in envs:
            for n in _tile_neighbours(e, tile_share, n_env):
                P[n], ebar[n] = P[e], ebar[e]
    base = _entry_points(m, ctx, x, with_state)
    ctx.set_contact_params(P)
    got = _entry_points(m, ctx, x, with_state)
    # not vacuous: the table changes the contact of most environments
    w0, w1 = base["eval_device"]["wrench"], got["eval_device"]["wrench"]
    changed = np.mean([not np.array_equal(w0[e], w1[e]) for e in range(n_env)])
    assert changed >= min_changed, changed
    for e in envs:
        mr = build(_Constants(capi.Context(0), ebar[e], P[e]))
        ref = _entry_points(mr, mr.backend, x, with_state)
        for name, keys in _KEYS.items():
            if name in got:
                _same_row(got[name], ref[name], e, keys)
    return m, ctx, P, ebar


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_boxes_every_entry_point_per_environment():
    """boxes.jl at 8 n_sm + 1 environments (the narrow tile kernel's ticket path runs): environments of the first tile, ticket-only tiles
    and the last tile equal a context built with their row, through pfc_eval_f64[_device], pfc_eval_state_f64, pfc_calcxd_f64_device and
    pfc_calcxd_jacobian_device; the traction dump of pfc_get_traction follows the table too."""
    n_sm = _n_sm()
    n_env = 8 * n_sm + 1
    m0, _ = scene_boxes(None)
    x = boxes_env_states(m0, n_env)
    build = lambda be: scene_boxes(be, max_env=n_env)[0]
    envs = [0, 1, 4 * n_sm, 6 * n_sm + 7, 8 * n_sm]
    m, ctx, P, ebar = _check_scene(build, x, envs, seed=11)
    X, tw, _ = S.boundary_arrays(m, x)
    ctx.eval_f64(X, tw, None, keep=True)
    for e in (0, 8 * n_sm):
        mr = build(_Constants(capi.Context(0), ebar[e], P[e]))
        mr.backend.eval_f64(X, tw, None, keep=True)
        for k in range(ctx.n_ins):
            t = ctx.get_traction(e, k)
            assert len(t) > 0 and np.array_equal(t, mr.backend.get_traction(e, k)), (e, k)


def test_tet_tet_scene_per_environment():
    """Plane + two compliant boxes: tet-tet instructions (Ebar_1 enters the pressure plane and the normal) and a bristle one.  Three small
    problems per environment, so narrow tiles hold problems of neighbouring environments (see _check_scene)."""
    from test_gpu_batch_shapes import _tet_tet_states
    n_env = 101
    m0 = _tet_tet_scene(None, 1)
    x = _tet_tet_states(m0, n_env, 5)
    build = lambda be: _tet_tet_scene(be, n_env)
    m, ctx, P, _ = _check_scene(build, x, [0, 37, 100], seed=12, tile_share=3)
    # every environment its own row: an environment whose tiles hold neighbours with other rows matches its reference to rounding
    P, ebar = _random_table(m, n_env, 13)
    ctx.set_contact_params(P)
    X, tw, s = S.boundary_arrays(m, x)
    got = _eval_device(ctx, X, tw, s)
    for e in (37, 38, 51):
        mr = build(_Constants(capi.Context(0), ebar[e], P[e]))
        ref = _eval_device(mr.backend, X, tw, s)
        _same_row(got, ref, e, ("sdot", "n_pairs", "flags"))
        assert wrench_rel_err(got["wrench"][e], ref["wrench"][e], floor=1e-6) <= 1e-12, e
    k = next(k for k, ci in enumerate(m.ContactInstructions) if m.MeshCache[ci.id_1].mesh.is_tet)
    Q = P.copy()
    Q[5, k, 1] = np.nan   # Ebar_1 of a tetrahedral mesh_1 is used: rejected
    assert capi.lib().pfc_set_contact_params(ctx._h, n_env, Q.ctypes.data) == PFC_E_ARG


def test_bristle_boxes_per_environment():
    """boxes.jl with bristle friction: per-environment tau, k_bar, mu_s, mu_d and magic; s-dot bit for bit."""
    n_env = 300
    m0, _ = scene_boxes(None, bristle=True)
    x = boxes_env_states(m0, n_env)
    _check_scene(lambda be: scene_boxes(be, max_env=n_env, bristle=True)[0], x, [0, 150, 299], seed=13)


@pytest.mark.parametrize("scene,mid_leaves", [("c4", None), ("spheres", None), ("spheres", "0")])
def test_large_and_mid_path_scenes_per_environment(monkeypatch, scene, mid_leaves):
    """3 environments of scene_c4_sphere_on_slab(24, 27) (large path), and of coarse spheres whose instructions (one of them bristle)
    take the mid-size path, or the large path with PFC_MID_LEAVES=0."""
    if mid_leaves is not None:
        monkeypatch.setenv("PFC_MID_LEAVES", mid_leaves)
    if scene == "c4":
        m0, x0 = scenes.scene_c4_sphere_on_slab(24, 27)
        x = np.repeat(x0[None], 3, 0)
        x[1, 5] -= 0.001
        x[2, 5] += 0.0015
        x[2, m0.nq:m0.nq + 3] += 0.3

        def build(be):   # the one scenario, attached to another backend each time
            S.attach_backend(m0, be, 3)
            return m0
        min_changed = 1.0
    else:
        build = _sphere_scene(2, 2)
        x = _sphere_states(build(None, 3), 3, 41)
        build = (lambda b: lambda be: b(be, 3))(build)
        min_changed = 0.6
    _check_scene(build, x, [0, 1, 2], seed=14, min_changed=min_changed)


def test_oracle_with_each_row():
    """3 boxes.jl environments against the CPU oracle built with their rows, within 1e-9."""
    n_env = 3
    m0, _ = scene_boxes(None)
    x = boxes_env_states(m0, n_env)
    m, _ = scene_boxes(capi.Context(0), max_env=n_env)
    P, ebar = _random_table(m, n_env, 15)
    m.backend.set_contact_params(P)
    X, tw, _ = S.boundary_arrays(m, x)
    g = m.backend.eval_f64(X, tw, None)
    for e in range(n_env):
        mo, _ = scene_boxes(_Constants(orc.OracleContext(), ebar[e], P[e]))
        c = mo.backend.eval_f64(X[e:e + 1], tw[e:e + 1], None)
        assert np.array_equal(g["n_pairs"][e], c["n_pairs"][0]) and np.array_equal(g["flags"][e], c["flags"][0])
        assert wrench_rel_err(g["wrench"][e], c["wrench"][0], floor=1e-6) <= 1e-9


def _radau_run(ctx, x0, n_step, knots, tau):
    """From (x0, t = 0) and a fresh pfc_radau_init each: n_step steps, and a roll-out through knots with the tau schedule; through the
    host entry points, then through the device ones."""
    n_env = x0.shape[0]
    ctx.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x, t = x0.copy(), np.zeros(n_env)
    steps = []
    for _ in range(n_step):
        x, t, h, st = ctx.radau_step(x, t)
        steps.append((x.copy(), t.copy(), h.copy(), st.copy()))
    ctx.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    ro = ctx.radau_rollout(x0, np.zeros(n_env), knots, tau)
    ctx.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    xd, td = _t(x0), torch.zeros(n_env, dtype=torch.float64, device=DEV)
    hd = torch.zeros(n_env, dtype=torch.float64, device=DEV)
    sd = torch.zeros((n_env, 4), dtype=torch.int32, device=DEV)
    dev_steps = []
    for _ in range(n_step):
        ctx.radau_step_device(n_env, xd.data_ptr(), None, td.data_ptr(), hd.data_ptr(), sd.data_ptr())
        ctx.sync()
        dev_steps.append((xd.cpu().numpy(), td.cpu().numpy(), hd.cpu().numpy(), sd.cpu().numpy()))
    ctx.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    xd, td = _t(x0), torch.zeros(n_env, dtype=torch.float64, device=DEV)
    taud = _t(tau)
    xk = torch.zeros((len(knots), n_env, x0.shape[1]), dtype=torch.float64, device=DEV)
    ctx.radau_rollout_device(n_env, knots, 1000, xd.data_ptr(), taud.data_ptr(), td.data_ptr(), xk.data_ptr(), sd.data_ptr())
    ctx.sync()
    dev_ro = (xd.cpu().numpy(), td.cpu().numpy(), xk.cpu().numpy(), sd.cpu().numpy())
    return steps, ro, dev_steps, dev_ro


def test_radau_step_and_rollout_per_environment():
    """64 boxes.jl environments with distinct rows: 10 pfc_radau_step calls, and a 4-knot pfc_radau_rollout with a tau_ext schedule.
    Sampled environments equal a context built with their row (x, t, h_taken, x_knot, stats bit for bit); host = device entry points."""
    n_env = 64
    build = lambda be: scene_boxes(be, max_env=n_env)[0]
    m = build(capi.Context(0))
    x0 = boxes_env_states(m, n_env)
    P, ebar = _random_table(m, n_env, 16)
    knots = np.array([0.012, 0.02, 0.03, 0.04])
    tau = np.random.default_rng(17).uniform(-2.0, 2.0, (len(knots), n_env, m.nv))
    m.backend.set_contact_params(P)
    steps, ro, dev_steps, dev_ro = _radau_run(m.backend, x0, 10, knots, tau)
    for a, b in zip(steps, dev_steps):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)
    for u, v in zip(ro, dev_ro):
        assert np.array_equal(u, v)
    assert (ro[3][:, 0] == len(knots)).all()
    for e in (0, 17, 63):
        mr = build(_Constants(capi.Context(0), ebar[e], P[e]))
        r_steps, r_ro, _, _ = _radau_run(mr.backend, x0, 10, knots, tau)
        for a, b in zip(steps, r_steps):
            for u, v in zip(a, b):
                assert np.array_equal(u[e], v[e]), e
        x, t, x_knot, st = ro
        rx, rt, rk, rs = r_ro
        assert np.array_equal(x[e], rx[e]) and np.array_equal(t[e], rt[e]) and np.array_equal(x_knot[:, e], rk[:, e]) and np.array_equal(st[e], rs[e])


def test_own_values_change_nothing():
    """A table holding the scene's own values gives the bits of no table: 4096 environments through pfc_eval_f64_device,
    pfc_calcxd_jacobian_device and a short roll-out."""
    n_env = 4096
    m, _ = scene_boxes(capi.Context(0), max_env=n_env)
    x = boxes_env_states(m, n_env)
    X, tw, _ = S.boundary_arrays(m, x)
    P, _ = _own_table(m, n_env)

    def run():
        out = dict(ev=_eval_device(m.backend, X, tw), jac=_jacobian_device(m.backend, x))
        m.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        out["ro"] = m.backend.radau_rollout(x, np.zeros(n_env), [0.003])
        return out
    a = run()
    m.backend.set_contact_params(P)
    b = run()
    for k in ("wrench", "n_pairs", "flags"):
        assert np.array_equal(a["ev"][k], b["ev"][k])
    for k in ("jac", "xdot", "n_pairs", "flags"):
        assert np.array_equal(a["jac"][k], b["jac"][k])
    for u, v in zip(a["ro"], b["ro"]):
        assert np.array_equal(u, v)


@pytest.mark.parametrize("scene", ["boxes_host", "bristle_device"])
def test_graph_caches_follow_the_table(scene):
    """Calls that replay a captured CUDA graph: the small host call of boxes.jl (pfc_eval_f64, packed copies) and the bristle scene's
    device evaluation.  Three evaluations without a table (the third is a replay), then a table, the same table with other values
    (same buffer), and no table again: every result equals its reference."""
    n_env = 16
    bristle = scene == "bristle_device"
    build = lambda be: scene_boxes(be, max_env=n_env, bristle=bristle)[0]
    m = build(capi.Context(0))
    x = boxes_env_states(m, n_env)
    X, tw, s = S.boundary_arrays(m, x)
    ev = (lambda mm: _eval_device(mm.backend, X, tw, s)) if bristle else (lambda mm: mm.backend.eval_f64(X, tw, None))
    keys = ("wrench", "sdot", "n_pairs", "flags")
    first = [ev(m) for _ in range(3)]
    for o in first[1:]:
        _same_row(o, first[0], slice(None), keys)
    for seed in (21, 22):
        P, ebar = _random_table(m, n_env, seed)
        m.backend.set_contact_params(P)
        for _ in range(3):
            got = ev(m)
        for e in (0, n_env - 1):
            ref = ev(build(_Constants(capi.Context(0), ebar[e], P[e])))
            _same_row(got, ref, e, keys)
        assert not np.array_equal(got["wrench"], first[0]["wrench"])
    m.backend.set_contact_params(None)
    for _ in range(2):
        _same_row(ev(m), first[0], slice(None), keys)


def test_argument_errors_keep_the_table():
    """Each rejected call returns PFC_E_ARG and leaves the table in force; n_env mismatches at evaluation and at the Radau entry points;
    the sharded entry points refuse a context that holds a table."""
    L = capi.lib()
    n_env = 8
    c0 = capi.Context(0)
    assert L.pfc_set_contact_params(c0._h, 0, None) == PFC_E_ARG          # before pfc_finalize
    m, _ = scene_boxes(capi.Context(0), max_env=n_env)
    c = m.backend
    x = boxes_env_states(m, n_env)
    X, tw, _ = S.boundary_arrays(m, x)
    P, ebar = _random_table(m, n_env, 31)
    assert np.isnan(P).any()   # the entries no model uses (Ebar_1 of a triangle mesh_1, q3 / q4 of a regularized instruction) are NaN
    c.set_contact_params(P)
    want = c.eval_f64(X, tw, None)
    bad = []
    big = np.concatenate([P, P], 0)
    bad.append(lambda: L.pfc_set_contact_params(c._h, n_env + 1, big.ctypes.data))   # n_env > max_env
    bad.append(lambda: L.pfc_set_contact_params(c._h, -1, P.ctypes.data))
    bad.append(lambda: L.pfc_set_contact_params(c._h, n_env, None))                  # NULL params
    for (k, j, v) in [(0, 0, np.nan), (1, 2, np.inf), (2, 3, np.nan), (3, 5, -np.inf)]:   # chi, Ebar_2, mu_s, v_c
        Q = P.copy()
        Q[3, k, j] = v
        bad.append(lambda Q=Q: L.pfc_set_contact_params(c._h, n_env, Q.ctypes.data))
    for call in bad:
        assert call() == PFC_E_ARG
        got = c.eval_f64(X, tw, None)
        assert np.array_equal(got["wrench"], want["wrench"])
    # batch size
    with pytest.raises(capi.PfcError) as ei:
        c.eval_f64(X[:4], tw[:4], None)
    assert ei.value.code == PFC_E_ARG
    with pytest.raises(capi.PfcError) as ei:
        c.calcxd_f64(x[:4])
    assert ei.value.code == PFC_E_ARG
    with pytest.raises(capi.PfcError) as ei:
        c.radau_init(4)
    assert ei.value.code == PFC_E_ARG
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    c.set_contact_params(P[:4])
    with pytest.raises(capi.PfcError) as ei:
        c.radau_step(x, np.zeros(n_env))
    assert ei.value.code == PFC_E_ARG
    with pytest.raises(capi.PfcError) as ei:
        c.radau_rollout(x, np.zeros(n_env), [0.01])
    assert ei.value.code == PFC_E_ARG
    # sharded entry points
    d = torch.zeros(1024, dtype=torch.float64, device=DEV)
    assert L.pfc_eval_sharded_begin(c._h, 4, d.data_ptr(), d.data_ptr(), None, d.data_ptr(), None, d.data_ptr(), d.data_ptr()) == PFC_E_ARG
    assert b"contact parameters" in L.pfc_last_error()
    assert L.pfc_eval_sharded_f64_device(c._h, 4, d.data_ptr(), d.data_ptr(), None, d.data_ptr(), None, d.data_ptr(), d.data_ptr()) == PFC_E_ARG
    assert b"contact parameters" in L.pfc_last_error()
    # cleared: any batch size again, the scene's own values
    c.set_contact_params(None)
    m2, _ = scene_boxes(capi.Context(0), max_env=n_env)
    assert np.array_equal(c.eval_f64(X[:4], tw[:4], None)["wrench"], m2.backend.eval_f64(X[:4], tw[:4], None)["wrench"])
