"""GPU tests of continuous affine state feedback (pfc_set_feedback): with a table set, calcXd! of environment e uses
tau = tau_ext[e] + K[seg][e] (x_ref[seg][e] - x[e][:nq + nv]) at every state it evaluates, and the Jacobian entry points add -H^-1 K in the
[q; v] columns of the v_dot rows.  Covered: the term itself against H^-1 K (x_ref - x) (with and without a body table), a K = 0 table
against no table bit for bit, the Jacobian and its Dual<6> chunks (bristle scene included), roll-outs against rollout_radau over the CPU
oracle with one feedback wrapper per interval, roll-out equalities bit for bit, a PD lift of the top box of boxes.jl (moderate and stiff
gains), and argument errors.

(The file name sorts after test_gpu_batch_shapes.py and test_gpu_jacobian_scale.py on purpose: their torch.profiler kernel lists lose the
first kernels of the profiled call once the process has run long enough, and these tests take about 40 s on a B200.)"""
import numpy as np
import pytest
import torch

import pfc_b200  # noqa: F401
from helpers import boxes_env_states, scene_boxes
from oracle import orc
from pfc_b200 import capi
from pfc_b200 import dynamics as D
from pfc_b200 import scenario as S
from test_gpu_contact_params import _Constants, _calcxd_device, _radau_run, _random_table, _same_row, _t
from test_gpu_per_env_body_params import _dynamics_entry_points, _keys, _random_bodies, _with_row
from test_gpu_radau_rollout import _boxes_states, _compare_knots, _mirror_rollout

pytestmark = pytest.mark.gpu

PFC_E_ARG = -1
DEV = torch.device("cuda", 0)


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _floating(m):
    return [(k, b) for k, b in enumerate(m.bodies) if b.joint is not None]


def _random_feedback(m, x, n_seg, seed, scale=50.0):
    """Dense random gains K[seg][env][nv][nq + nv] ~ U(-scale, scale) and references x_ref = x[:, :nq + nv] + U(-0.05, 0.05)."""
    rng = np.random.default_rng(seed)
    n_env, nc = x.shape[0], m.nq + m.nv
    K = rng.uniform(-scale, scale, (n_seg, n_env, m.nv, nc))
    xr = x[None, :, :nc] + rng.uniform(-0.05, 0.05, (n_seg, n_env, nc))
    return K, xr


def _hinv(m, H=None):
    """H^-1 [env or None][body] of the floating bodies: FloatingBodyDynamics' (the scene's own) or of a body table H[env][body]."""
    if H is None:
        return D.FloatingBodyDynamics(m).Hinv
    return {k: np.linalg.inv(H[:, k]) for k, _ in _floating(m)}


def _check_term(m, x, base, got, K, xr, Hinv, per_env):
    """The table's x_dot minus the no-table x_dot: H^-1 K (x_ref - x) in the v_dot rows (1e-12 of the larger of the term and the row's
    value), the q_dot and s_dot rows bit for bit."""
    nq, nv, nc = m.nq, m.nv, m.nq + m.nv
    assert np.array_equal(base[:, :nq], got[:, :nq]) and np.array_equal(base[:, nc:], got[:, nc:])
    u = np.einsum("eij,ej->ei", K[0], xr[0] - x[:, :nc])
    for k, b in _floating(m):
        Hi = Hinv[k]
        want = np.einsum("eij,ej->ei", Hi, u[:, b.v0:b.v0 + 6]) if per_env else u[:, b.v0:b.v0 + 6] @ Hi.T
        rows = slice(nq + b.v0, nq + b.v0 + 6)
        diff = got[:, rows] - base[:, rows]
        den = np.maximum(np.abs(want).max(axis=1), np.abs(got[:, rows]).max(axis=1))
        assert (np.abs(diff - want).max(axis=1) <= 1e-12 * den).all(), k


def test_the_feedback_term():
    """boxes.jl at 8 n_sm + 1 environments, random K and x_ref, tau_ext NULL and not: the term is H^-1 K (x_ref - x) per body, host and
    device entry points agree bit for bit; again with a body table (H^-1 of the environment's row)."""
    n_env = 8 * _n_sm() + 1
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    x = boxes_env_states(m, n_env)
    K, xr = _random_feedback(m, x, 1, 1)
    tau = np.random.default_rng(2).uniform(-1.0, 1.0, (n_env, m.nv))
    for H, g in ((None, None), _random_bodies(m, n_env, 3)):
        c.set_feedback(None)
        if H is not None:
            c.set_body_params(H, g)
        for tau_ext in (None, tau):
            base = c.calcxd_f64(x, tau_ext)["xdot"]
            c.set_feedback(K, xr)
            got = c.calcxd_f64(x, tau_ext)
            _check_term(m, x, base, got["xdot"], K, xr, _hinv(m, H), H is not None)
            if tau_ext is None:
                _same_row(got, _calcxd_device(c, x), slice(None), ("xdot", "n_pairs", "flags"))
            c.set_feedback(None)


def _radau_all(c, x0, knots, tau):
    steps, ro, dev_steps, dev_ro = _radau_run(c, x0, 3, knots, tau)
    for a, b in zip(steps, dev_steps):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)
    for u, v in zip(ro, dev_ro):
        assert np.array_equal(u, v)
    return steps, ro, c.radau_step_info()[2]


def test_zero_gains_change_nothing():
    """A K = 0 table (x_ref random) gives the bits of no table: pfc_calcxd_f64, every chunk of pfc_calcxd_dual6 and pfc_calcxd_jacobian
    (host and device), Radau steps and a 4-knot roll-out; one more launch per calcXd! and the same host synchronisations per roll-out."""
    n_env = 64
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    x0 = boxes_env_states(m, n_env)
    knots = np.array([0.012, 0.02, 0.03, 0.04])
    tau = np.random.default_rng(4).uniform(-2.0, 2.0, (len(knots), n_env, m.nv))
    K, xr = _random_feedback(m, x0, len(knots), 5)

    def launches_of_calcxd():
        n0 = c.launch_count()
        _calcxd_device(c, x0)
        return c.launch_count() - n0
    base, l0 = _dynamics_entry_points(c, x0), launches_of_calcxd()
    steps0, ro0, syncs0 = _radau_all(c, x0, knots, tau)
    c.set_feedback(np.zeros_like(K), xr)
    got, l1 = _dynamics_entry_points(c, x0), launches_of_calcxd()
    steps1, ro1, syncs1 = _radau_all(c, x0, knots, tau)
    for name in base:
        _same_row(base[name], got[name], slice(None), _keys(name))
    for a, b in zip(steps0, steps1):
        for u, v in zip(a, b):
            assert np.array_equal(u, v)
    for u, v in zip(ro0, ro1):
        assert np.array_equal(u, v)
    assert l1 == l0 + 1 and syncs1 == syncs0


@pytest.mark.parametrize("bristle", [False, True])
def test_jacobian_gains_minus_hinv_k(bristle):
    """With a table the Jacobian is the no-table Jacobian plus -H^-1 K in the [q; v] columns of the v_dot rows (1e-12), unchanged bit for
    bit elsewhere (bristle columns included); the whole Jacobian equals its pfc_calcxd_dual6 chunks bit for bit, host and device."""
    n_env = 40
    m = scene_boxes(capi.Context(0), max_env=n_env, bristle=bristle)[0]
    c = m.backend
    x = boxes_env_states(m, n_env)
    nq, nc, nx = m.nq, m.nq + m.nv, S.num_x(m)
    K, xr = _random_feedback(m, x, 1, 6)
    base = c.calcxd_jacobian(x)["jac"]
    c.set_feedback(K, xr)
    got = _dynamics_entry_points(c, x)
    jac = got["jac_host"]["jac"]
    _same_row(got["jac_host"], got["jac_device"], slice(None), _keys("jac"))
    Hinv = _hinv(m)
    mask = np.zeros((nx, nx), bool)
    for k, b in _floating(m):
        rows = slice(nq + b.v0, nq + b.v0 + 6)
        want = -np.einsum("ij,ejc->eic", Hinv[k], K[0][:, b.v0:b.v0 + 6])
        diff = jac[:, rows, :nc] - base[:, rows, :nc]
        den = np.maximum(np.abs(want).max(axis=(1, 2)), np.abs(jac[:, rows, :nc]).max(axis=(1, 2)))
        assert (np.abs(diff - want).max(axis=(1, 2)) <= 1e-12 * den).all(), k
        mask[rows, :nc] = True
    assert np.array_equal(jac[:, ~mask], base[:, ~mask])
    for seed in range(0, nx, 6):
        for name in (f"dual6_host_{seed}", f"dual6_device_{seed}"):
            x7 = got[name]["xdot7"]
            w = min(6, nx - seed)
            assert np.array_equal(x7[:, :, 1:1 + w], jac[:, :, seed:seed + w]), (name, seed)
            if seed == 0:   # x_dot is the value part of the first pass
                assert np.array_equal(x7[:, :, 0], got["jac_host"]["xdot"]), name


class _FeedbackDynamics:
    """FloatingBodyDynamics over the CPU oracle with H^-1 (tau + K (x_ref - x)) added to v_dot and -H^-1 K to its Jacobian chunks."""

    def __init__(self, m, tau, K, xr):
        self.base, self.m = D.FloatingBodyDynamics(m), m
        self.tau, self.K, self.xr, self.nc = tau, K, xr, m.nq + m.nv

    def _add(self, xx, x):
        f = self.tau + self.K @ (self.xr - x[:self.nc])
        for k, b in _floating(self.m):
            xx[self.m.nq + b.v0:self.m.nq + b.v0 + 6] += self.base.Hinv[k] @ f[b.v0:b.v0 + 6]

    def de(self, xx, x, t=0.0):
        self.base.de(xx, x, t)
        self._add(xx, x)

    def de_jacobian_chunk(self, x, i0, i1, t=0.0):
        xx, cols = self.base.de_jacobian_chunk(x, i0, i1, t)
        self._add(xx, x)
        for k, b in _floating(self.m):
            for d, j in enumerate(range(i0, i1)):
                if j < self.nc:
                    cols[self.m.nq + b.v0:self.m.nq + b.v0 + 6, d] -= self.base.Hinv[k] @ self.K[b.v0:b.v0 + 6, j]
        return xx, cols


def _pd_gains(m, x, w_n, zeta, bodies=None):
    """K[env][nv][nq + nv] of a PD law per floating body (all, or the listed ones) toward x_ref with v_ref = 0: tau = H (w_n^2 dq - 2 zeta
    w_n v), dq in the body frame (4 x the MRP difference, R' x the translation difference at the state x)."""
    n_env = x.shape[0]
    K = np.zeros((n_env, m.nv, m.nq + m.nv))
    dyn = D.FloatingBodyDynamics(m)
    for k, b in _floating(m):
        if bodies is not None and k not in bodies:
            continue
        for e in range(n_env):
            R = S.mrp_to_rotation(x[e, b.q0:b.q0 + 3])
            A = np.zeros((6, m.nq + m.nv))
            A[:3, b.q0:b.q0 + 3] = 4.0 * w_n ** 2 * np.eye(3)
            A[3:, b.q0 + 3:b.q0 + 6] = w_n ** 2 * R.T
            A[:, m.nq + b.v0:m.nq + b.v0 + 6] = 2.0 * zeta * w_n * np.eye(6)   # K (x_ref - x) = -2 zeta w_n v
            K[e, b.v0:b.v0 + 6] = dyn.H[k] @ A
    return K


def test_rollout_follows_the_oracle_backed_mirror():
    """boxes.jl, 6 environments, 4 knots, per-interval PD-like gains (stiffness and references change per interval) and a tau_ext
    schedule: per environment the same stats as rollout_radau over FloatingBodyDynamics (CPU oracle) wrapped with the interval's feedback,
    and x at every knot within 1e-7 per 3-vector."""
    n_env, h_max, knots = 6, 0.05, [0.01, 0.025, 0.05, 0.1]
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    x0 = _boxes_states(m, n_env)
    rng = np.random.default_rng(7)
    nc = m.nq + m.nv
    K = np.stack([_pd_gains(m, x0, w, 0.7) for w in (3.0, 6.0, 4.0, 8.0)]) * rng.uniform(0.8, 1.2, (len(knots), n_env, 1, 1))
    xr = x0[None, :, :nc] + rng.uniform(-0.01, 0.01, (len(knots), n_env, nc))
    tau = rng.uniform(-0.5, 0.5, (len(knots), n_env, m.nv))
    m.backend.set_feedback(K, xr)
    m.backend.radau_init(n_env, 2, 1.0e-4, h_max, 1.0e-16)
    _, t, x_knot, stats = m.backend.radau_rollout(x0, np.zeros(n_env), knots, tau)
    assert (t == knots[-1]).all() and (stats[:, 0] == len(knots)).all()
    m_cpu = scene_boxes(orc.OracleContext())[0]
    for e in range(n_env):
        dyn = [_FeedbackDynamics(m_cpu, tau[k, e], K[k, e], xr[k, e]) for k in range(len(knots))]
        ref, _, st_ref = _mirror_rollout(m_cpu, dyn, x0[e], 0.0, knots, h_max)
        assert stats[e].tolist() == st_ref, (e, stats[e], st_ref)
        _compare_knots(x_knot[:, e], ref, 1e-7)


def test_rollout_equalities_bit_for_bit():
    """128 boxes.jl environments, 4 knots, a 4-segment table of PD gains (w_n 3-8 rad/s, scaled per environment) and a tau schedule:
      * the 4-knot roll-out equals 4 one-knot roll-outs, each after pfc_set_feedback of its segment alone;
      * an n_seg = 1 table equals an n_seg = 4 table of identical segments;
      * the host and device roll-outs agree, and so do set_feedback and set_feedback_device;
      * environments alone equal themselves in the batch;
      * contact, body and feedback tables together give environment e the bits of a context with row e of each."""
    n_env = 128
    knots = np.array([0.01, 0.02, 0.035, 0.05])
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    x0 = _boxes_states(m, n_env)
    rng = np.random.default_rng(8)
    K = np.stack([_pd_gains(m, x0, w, 0.7) for w in (3.0, 6.0, 4.0, 8.0)]) * rng.uniform(0.8, 1.2, (len(knots), n_env, 1, 1))
    xr = x0[None, :, :m.nq + m.nv] + rng.uniform(-0.01, 0.01, (len(knots), n_env, m.nq + m.nv))
    tau = np.random.default_rng(9).uniform(-1.0, 1.0, (len(knots), n_env, m.nv))

    def rollout(ctx, x, t, kn, ta):
        return ctx.radau_rollout(x, t, kn, ta)
    c.set_feedback(K, xr)
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    xa, ta, xka, sa = rollout(c, x0, np.zeros(n_env), knots, tau)
    assert (sa[:, 0] == len(knots)).all()
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x, t, s_sum = x0.copy(), np.zeros(n_env), np.zeros_like(sa)
    for k in range(len(knots)):
        c.set_feedback(K[k:k + 1], xr[k:k + 1])
        x, t, xk, sk = rollout(c, x, t, knots[k:k + 1], tau[k:k + 1])
        assert np.array_equal(xk[0], xka[k]) and np.array_equal(x, xka[k]), k
        s_sum += sk
    assert np.array_equal(s_sum, sa)
    # one segment for every interval
    Kc = np.repeat(K[:1], len(knots), 0)
    xrc = np.repeat(xr[:1], len(knots), 0)
    outs = []
    for Kx, xx in ((K[:1], xr[:1]), (Kc, xrc)):
        c.set_feedback(Kx, xx)
        c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        outs.append(rollout(c, x0, np.zeros(n_env), knots, tau))
    for u, v in zip(*outs):
        assert np.array_equal(u, v)
    # host and device: entry points and the way the table was set
    c.set_feedback(_t(K), _t(xr))
    steps, ro, dev_steps, dev_ro = _radau_run(c, x0, 2, knots, tau)
    for u, v in zip(ro, dev_ro):
        assert np.array_equal(u, v)
    for u, v in zip(ro, (xa, ta, xka, sa)):
        assert np.array_equal(u, v)
    # alone
    for e in (0, 5, 77):
        c1 = scene_boxes(capi.Context(0), max_env=1)[0].backend
        c1.set_feedback(K[:, e:e + 1], xr[:, e:e + 1])
        c1.radau_init(1, 2, 1.0e-4, 0.05, 1.0e-16)
        xe, te, xke, se = rollout(c1, x0[e:e + 1], np.zeros(1), knots, tau[:, e:e + 1])
        assert np.array_equal(xke[:, 0], xka[:, e]) and np.array_equal(se[0], sa[e]) and te[0] == ta[e], e
    # three tables at once
    P, ebar = _random_table(m, n_env, 10)
    H, g = _random_bodies(m, n_env, 11)
    c.set_contact_params(P)
    c.set_body_params(H, g)
    c.set_feedback(K, xr)
    got = _calcxd_device(c, x0)
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    ro = rollout(c, x0, np.zeros(n_env), knots, tau)
    build = lambda be: scene_boxes(be, max_env=n_env)[0]
    for e in (3, 64):
        mr = _with_row(build(_Constants(capi.Context(0), ebar[e], P[e])), H, g, e)
        mr.backend.set_feedback(np.repeat(K[:, e:e + 1], n_env, 1), np.repeat(xr[:, e:e + 1], n_env, 1))
        _same_row(got, _calcxd_device(mr.backend, x0), e, ("xdot", "n_pairs", "flags"))
        mr.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
        r_ro = rollout(mr.backend, x0, np.zeros(n_env), knots, tau)
        for u, v in zip(ro, r_ro):
            assert np.array_equal(u[:, e] if u.ndim == 3 else u[e], v[:, e] if v.ndim == 3 else v[e]), e


def _lift(w_n, with_feedback, n_knot=20, t_end=2.0):
    """The top box of a boxes.jl stack at rest, held by a gravity-compensating tau_ext and a PD law (w_n, zeta = 1, one segment) to a
    target 5 cm above its start: (x_ref, x at t_end, stats)."""
    m = scene_boxes(capi.Context(0), max_env=1)[0]
    c = m.backend
    x0 = boxes_env_states(m, 1)
    x0[:, m.nq:] = 0.0
    top, b = _floating(m)[-1]
    xr = x0[:, :m.nq + m.nv].copy()
    xr[0, b.q0 + 5] += 0.05
    R = S.mrp_to_rotation(x0[0, b.q0:b.q0 + 3])
    tau = np.zeros((n_knot, 1, m.nv))
    tau[:, 0, b.v0:b.v0 + 6] = -D.FloatingBodyDynamics(m).H[top] @ np.concatenate([np.zeros(3), R.T @ np.asarray(m.gravity, dtype=np.float64)])
    if with_feedback:
        c.set_feedback(_pd_gains(m, x0, w_n, 1.0, bodies=[top])[None], xr[None])
    c.radau_init(1, 2, 1.0e-4, 0.05, 1.0e-16)
    knots = np.linspace(t_end / n_knot, t_end, n_knot)
    x, t, _, stats = c.radau_rollout(x0, np.zeros(1), knots, tau if with_feedback else None, max_steps=100000)
    assert t[0] == t_end, (t, stats)
    return m, b, xr[0], x[0], stats[0]


def test_pd_lift_of_the_top_box():
    """w_n = 20 rad/s: after 2 s the top box sits within 1e-3 m and 1e-3 m/s of the target.  w_n = 1000 rad/s (stiff): the roll-out
    finishes with at most 2x the rejected attempts of the run without feedback (the first measured run, on a B200: 63 with feedback, 76
    without; 316 and 357 accepted steps), which a Jacobian without the controller's -H^-1 K would not allow at these step sizes."""
    m, b, xr, x, st = _lift(20.0, True)
    err_p = np.abs(x[b.q0 + 3:b.q0 + 6] - xr[b.q0 + 3:b.q0 + 6]).max()
    err_v = np.abs(x[m.nq + b.v0 + 3:m.nq + b.v0 + 6]).max()
    print(f"w_n = 20: position error {err_p:.3e} m, velocity {err_v:.3e} m/s, stats {st.tolist()}")
    assert err_p <= 1e-3 and err_v <= 1e-3
    _, _, _, _, st_free = _lift(1000.0, False)
    _, _, _, _, st_stiff = _lift(1000.0, True)
    print(f"w_n = 1000: stats {st_stiff.tolist()}, without feedback {st_free.tolist()}")
    assert st_stiff[2] <= 2 * max(st_free[2], 5)


def test_argument_errors_keep_the_table():
    """Each rejected pfc_set_feedback[_device] returns PFC_E_ARG and leaves the table in force; a roll-out with a bad n_seg and every
    reading entry point with another n_env are refused; pfc_set_dynamics, pfc_set_bodies and n_env = 0 clear the table."""
    L = capi.lib()
    n_env = 8
    c0 = capi.Context(0)
    assert L.pfc_set_feedback(c0._h, 0, 1, None, None) == PFC_E_ARG                       # before pfc_set_dynamics
    m = scene_boxes(capi.Context(0), max_env=n_env)[0]
    c = m.backend
    x = boxes_env_states(m, n_env)
    own, own4 = c.calcxd_f64(x)["xdot"], c.calcxd_f64(x[:4])["xdot"]
    K = np.stack([_pd_gains(m, x, w, 0.7) for w in (4.0, 6.0)])
    xr = x[None, :, :m.nq + m.nv] + np.random.default_rng(12).uniform(-0.01, 0.01, (2, n_env, m.nq + m.nv))
    c.set_feedback(K, xr)
    want = c.calcxd_f64(x)["xdot"]
    assert not np.array_equal(want, own)
    Kd, xrd = _t(K), _t(xr)
    big_K, big_x = np.concatenate([K, K], 1), np.concatenate([xr, xr], 1)
    bad = []
    for f, KK, XX, bK, bX in ((L.pfc_set_feedback, K.ctypes.data, xr.ctypes.data, big_K.ctypes.data, big_x.ctypes.data),
                              (L.pfc_set_feedback_device, Kd.data_ptr(), xrd.data_ptr(), _t(big_K).data_ptr(), _t(big_x).data_ptr())):
        bad.append(lambda f=f, bK=bK, bX=bX: f(c._h, n_env + 1, 2, bK, bX))   # n_env > max_env
        bad.append(lambda f=f, KK=KK, XX=XX: f(c._h, -1, 2, KK, XX))
        bad.append(lambda f=f, KK=KK, XX=XX: f(c._h, n_env, 0, KK, XX))
        bad.append(lambda f=f, XX=XX: f(c._h, n_env, 2, None, XX))
        bad.append(lambda f=f, KK=KK: f(c._h, n_env, 2, KK, None))
    Kn = K.copy(); Kn[1, 3, 2, 7] = np.nan
    xn = xr.copy(); xn[0, 5, 1] = np.inf
    for Kx, xx in ((Kn, xr), (K, xn)):
        bad.append(lambda Kx=Kx, xx=xx: L.pfc_set_feedback(c._h, n_env, 2, Kx.ctypes.data, xx.ctypes.data))
        Kt, xt = _t(Kx), _t(xx)
        bad.append(lambda Kt=Kt, xt=xt: L.pfc_set_feedback_device(c._h, n_env, 2, Kt.data_ptr(), xt.data_ptr()))
    for call in bad:
        assert call() == PFC_E_ARG
        assert np.array_equal(c.calcxd_f64(x)["xdot"], want)
    # a roll-out whose knots are neither 1 nor n_seg: refused, nothing written
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    with pytest.raises(capi.PfcError) as ei:
        c.radau_rollout(x, np.zeros(n_env), [0.01, 0.02, 0.03])
    assert ei.value.code == PFC_E_ARG and b"segments" in L.pfc_last_error()
    xd, td = _t(x), torch.zeros(n_env, dtype=torch.float64, device=DEV)
    torch.cuda.synchronize()
    with pytest.raises(capi.PfcError):
        c.radau_rollout_device(n_env, [0.01, 0.02, 0.03], 1000, xd.data_ptr(), None, td.data_ptr(), None, None)
    assert np.array_equal(xd.cpu().numpy(), x) and not td.cpu().numpy().any()
    c.radau_rollout(x, np.zeros(n_env), [0.01, 0.02])
    # batch size: every entry point that reads the table refuses another n_env, the others accept it
    x4 = x[:4]
    x4d = _t(x4)
    o4 = torch.zeros((4, x.shape[1]), dtype=torch.float64, device=DEV)
    o7 = torch.zeros((4, x.shape[1], 7), dtype=torch.float64, device=DEV)
    oj = torch.zeros((4, x.shape[1], x.shape[1]), dtype=torch.float64, device=DEV)
    np4 = torch.zeros((4, c.n_ins), dtype=torch.int64, device=DEV)
    fl4 = torch.zeros((4, c.n_ins), dtype=torch.int32, device=DEV)
    reading = [lambda: c.calcxd_f64(x4), lambda: c.calcxd_jacobian(x4), lambda: c.calcxd_dual6(x4, 0), lambda: c.radau_init(4),
               lambda: c.calcxd_f64_device(4, x4d.data_ptr(), None, o4.data_ptr(), np4.data_ptr(), fl4.data_ptr()),
               lambda: c.calcxd_dual6_device(4, x4d.data_ptr(), None, 0, o7.data_ptr(), np4.data_ptr(), fl4.data_ptr()),
               lambda: c.calcxd_jacobian_device(4, x4d.data_ptr(), None, oj.data_ptr(), None, np4.data_ptr(), fl4.data_ptr())]
    for call in reading:
        with pytest.raises(capi.PfcError) as ei:
            call()
        assert ei.value.code == PFC_E_ARG and b"feedback table" in L.pfc_last_error()
    c.eval_state_f64(x4)
    X, tw, _ = S.boundary_arrays(m, x4)
    c.eval_f64(X, tw, None)
    c.set_feedback(K[:, :4], xr[:, :4])
    for call in (lambda: c.radau_step(x, np.zeros(n_env)), lambda: c.radau_rollout(x, np.zeros(n_env), [0.01]),
                 lambda: c.radau_step_device(n_env, xd.data_ptr(), None, td.data_ptr(), _t(np.zeros(n_env)).data_ptr(), None)):
        with pytest.raises(capi.PfcError) as ei:
            call()
        assert ei.value.code == PFC_E_ARG
    # pfc_set_dynamics clears the table
    c.set_feedback(K, xr)
    dyn = D.FloatingBodyDynamics(m)
    Hs = np.zeros((len(m.bodies), 6, 6))
    for k, _ in _floating(m):
        Hs[k] = dyn.H[k]
    c.set_dynamics(Hs, m.gravity)
    assert np.array_equal(c.calcxd_f64(x)["xdot"], own) and np.array_equal(c.calcxd_f64(x4)["xdot"], own4)
    # so does pfc_set_bodies
    c.set_feedback(K, xr)
    pose = np.array([np.concatenate([b.pose_R.reshape(9), b.pose_t]) for b in m.bodies])
    c.set_bodies([0 if b.joint is None else 1 for b in m.bodies], [b.q0 for b in m.bodies], [b.v0 for b in m.bodies],
                 [mc.body_id for mc in m.MeshCache], m.nq, m.nv, pose=pose)
    assert np.array_equal(c.calcxd_f64(x4)["xdot"], own4)
    # and n_env = 0
    c.set_feedback(K, xr)
    assert np.array_equal(c.calcxd_f64(x)["xdot"], want)
    c.set_feedback(None)
    assert np.array_equal(c.calcxd_f64(x4)["xdot"], own4)
