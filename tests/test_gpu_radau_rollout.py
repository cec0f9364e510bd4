"""GPU tests of the batched Radau roll-out through shared knot times (pfc_radau_rollout[_device]): against the single-scene mirror
radau.rollout_radau, for the equalities the knot rules promise (K knots = K one-knot calls, batch invariance, determinism, host entry
point = device entry point), on a large-path scene, and for the argument errors, the step budget and the error returns."""
import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import boxes_env_states, scene_boxes
from oracle import orc
from pfc_b200 import dynamics as D
from pfc_b200 import radau as R
from pfc_b200 import scenario as S
from test_gpu_radau_step import _TauDynamics

pytestmark = pytest.mark.gpu

PFC_E_ARG, PFC_E_STEP = -1, -6


def _ctx():
    from pfc_b200 import capi
    return capi.Context(0)


def _mirror_rollout(m, dyn, x0, t0, knots, h_max, max_steps=1000):
    """rollout_radau for one environment; dyn is one ODE object or one per interval."""
    rr = R.makeRadauIntegrator(dyn[0] if isinstance(dyn, list) else dyn, S.num_x(m), 1.0e-16, 2, 6)
    rr.step.h_max = h_max
    x_knot, x, t, stats = R.rollout_radau(rr, x0, t0, knots, de=dyn if isinstance(dyn, list) else None, max_steps=max_steps,
                                          after_step=lambda x: D.principal_value(m, x))
    return x_knot, t, stats


def _compare_knots(x_knot, ref, tol):
    """x_knot [K, NX] of one environment against the mirror's, per 3-vector relative to its own size (as _compare_with_mirror)."""
    assert np.isnan(x_knot).all(axis=1).tolist() == np.isnan(ref).all(axis=1).tolist()
    for k in range(ref.shape[0]):
        x = ref[k]
        if np.isnan(x).any():
            continue
        scale = np.abs(x).max()
        for i in range(0, x.shape[0], 3):
            den = max(np.abs(x[i:i + 3]).max(), 1e-6 * scale)
            assert np.abs(x_knot[k, i:i + 3] - x[i:i + 3]).max() <= tol * den, (k, i)


def _boxes_states(m, n_env):
    """boxes_env_states with the reference's drop (0), a settled stack at rest (1) and the drop 0.5 m higher (5), as the step tests use."""
    x0 = boxes_env_states(m, n_env)
    x0[0] = S.get_state(m)
    x0[1, m.nq:] = 0.0
    x0[5] = S.get_state(m)
    for b in m.bodies:
        if b.joint is not None:
            x0[5, b.q0 + 5] += 0.5
    return x0


def test_rollout_follows_the_oracle_backed_mirror():
    """boxes.jl, 6 environments from t = 0 through knots 0.01 / 0.025 / 0.05 / 0.1, h_max = 0.05: per environment the same knots, steps,
    rejected attempts and stage evaluations as rollout_radau over the CPU oracle, and x at every knot within 1e-7 per 3-vector."""
    n_env, h_max, knots = 6, 0.05, [0.01, 0.025, 0.05, 0.1]
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    x0 = _boxes_states(m, n_env)
    from pfc_b200.radau_batched import DeviceBatchedRadau
    dr = DeviceBatchedRadau(m, n_env, h_max=h_max)
    x_knot, stats = dr.rollout(x0, knots)
    x_knot, stats, t = x_knot.cpu().numpy(), stats.cpu().numpy(), dr.t.cpu().numpy()
    assert (t == 0.1).all() and (stats[:, 0] == 4).all()
    m_cpu = scene_boxes(orc.OracleContext())[0]
    for e in range(n_env):
        ref, t_ref, st_ref = _mirror_rollout(m_cpu, D.FloatingBodyDynamics(m_cpu), x0[e], 0.0, knots, h_max)
        assert stats[e].tolist() == st_ref, (e, stats[e], st_ref)
        _compare_knots(x_knot[:, e], ref, 1e-7)


def test_rollout_bristle_scene_with_a_tau_schedule():
    """Bristle boxes (n_x = 60), 8 environments, a random tau_ext per interval: against rollout_radau over calcxd_f64 / calcxd_dual6 with
    the interval's tau.  The knots stay within the first 0.01 s: later, the bristles' stick-slip transitions under this schedule amplify
    rounding so much that a 1e-15 relative change of x0 alone moves the mirror's states by 3e-7 at 0.025 s and changes its step decisions
    by 0.05 s (measured on a B200), so no comparison with a second implementation is meaningful there."""
    n_env, h_max, knots = 8, 0.05, [0.003, 0.006, 0.01]
    m = scene_boxes(_ctx(), max_env=3 * n_env, bristle=True)[0]
    x0 = boxes_env_states(m, n_env)
    tau = np.random.default_rng(11).uniform(-1, 1, (len(knots), n_env, m.nv))
    m.backend.radau_init(n_env, 2, 1.0e-4, h_max, 1.0e-16)
    _, t, x_knot, stats = m.backend.radau_rollout(x0, np.zeros(n_env), knots, tau)
    assert (t == knots[-1]).all()
    for e in range(n_env):
        ref, _, st_ref = _mirror_rollout(m, [_TauDynamics(m, tau[k, e]) for k in range(len(knots))], x0[e], 0.0, knots, h_max)
        assert stats[e].tolist() == st_ref, (e, stats[e], st_ref)
        _compare_knots(x_knot[:, e], ref, 1e-7)


def test_rollout_large_path_scene():
    """The tet-tet sphere on slab (one LARGE-path instruction, n_x = 12) at a generic pose, through three knots, against rollout_radau on
    the device backend."""
    from pfc_b200 import scenes
    m, x = scenes.scene_c4_sphere_on_slab(24, 27, backend=_ctx())
    x = x.copy()
    x[0:3] = [0.011, -0.017, 0.023]
    x[3:6] = [0.0123, -0.0071, 0.0451]
    knots = [0.002, 0.005, 0.011]
    m.backend.radau_init(1, 2, 1.0e-4, 0.01, 1.0e-16)
    _, t, x_knot, stats = m.backend.radau_rollout(x[None, :], np.zeros(1), knots)
    ref, t_ref, st_ref = _mirror_rollout(m, D.FloatingBodyDynamics(m, device=True), x, 0.0, knots, 0.01)
    assert t[0] == t_ref == knots[-1]
    assert stats[0].tolist() == st_ref
    _compare_knots(x_knot[:, 0], ref, 1e-7)


class _Prepared:
    """A boxes.jl context whose controllers have taken n_warm ordinary steps from x0, so the environments start the roll-out at different
    times, with different h and rules.  Deterministic: two of them are in the same state bit for bit."""

    def __init__(self, x0, n_warm):
        import torch
        from pfc_b200.radau_batched import DeviceBatchedRadau
        self.m = scene_boxes(_ctx(), max_env=3 * x0.shape[0])[0]
        self.dr = DeviceBatchedRadau(self.m, x0.shape[0], h_max=0.05)
        with torch.cuda.stream(self.dr.stream):
            x = torch.as_tensor(x0).to(self.dr.dev)
            self.warm_rejected = np.zeros(x0.shape[0], dtype=np.int64)
            for _ in range(n_warm):
                x, _ = self.dr.step(x)
                self.warm_rejected += self.dr.stats[:, 2].cpu().numpy()
            self.x = x

    def rollout(self, knots, tau, max_steps=1000):
        x_knot, stats = self.dr.rollout(self.x, knots, tau, max_steps)
        return x_knot.cpu().numpy(), stats.cpu().numpy(), self.dr.t.cpu().numpy()

    def next_step(self, x):
        """One more ordinary step from x: (x, t, h_taken, stats) -- shows the controller state the roll-out left behind."""
        import torch
        with torch.cuda.stream(self.dr.stream):
            xn, h = self.dr.step(torch.as_tensor(x).to(self.dr.dev))
            return xn.cpu().numpy(), self.dr.t.cpu().numpy(), h.cpu().numpy(), self.dr.stats.cpu().numpy()


def test_rollout_equalities_bit_for_bit():
    """1000 boxes.jl environments after 12 ordinary steps (start times, h and rules all differ; the raised drop is on rule 2), four knots
    and a random tau schedule:
      * two runs are identical;
      * the 4-knot roll-out equals 4 one-knot roll-outs, and the step after it too;
      * the host entry point equals the device entry point;
      * environments alone (n_env = 1; one that retried among them) equal themselves in the batch."""
    n_env, n_warm = 1000, 12
    m0 = scene_boxes(_ctx(), max_env=3)[0]
    x0 = _boxes_states(m0, n_env)
    a = _Prepared(x0, n_warm)
    t_start = a.dr.t.cpu().numpy()
    assert len(np.unique(t_start)) > 10
    base = float(t_start.max()) + 0.01
    knots = [base, base + 0.015, base + 0.04, base + 0.09]
    tau = np.random.default_rng(5).uniform(-1, 1, (len(knots), n_env, m0.nv))
    xa, sa, ta = a.rollout(knots, tau)
    assert (sa[:, 0] == len(knots)).all() and (ta == knots[-1]).all()
    retried = np.nonzero((sa[:, 2] > 0) | (a.warm_rejected > 0))[0]
    assert len(retried) > 0
    after_a = a.next_step(xa[-1])

    b = _Prepared(x0, n_warm)
    xb, sb, tb = b.rollout(knots, tau)
    assert np.array_equal(xa, xb, equal_nan=True) and np.array_equal(sa, sb) and np.array_equal(ta, tb)

    c = _Prepared(x0, n_warm)
    s_sum = np.zeros_like(sa)
    for k in range(len(knots)):
        xk, sk, tk = c.rollout(knots[k:k + 1], tau[k:k + 1])
        c.x = xk[0]
        assert np.array_equal(xk[0], xa[k]), k
        assert (tk == knots[k]).all()
        s_sum += sk
    assert np.array_equal(s_sum, sa)
    for u, v in zip(c.next_step(xa[-1]), after_a):
        assert np.array_equal(u, v)

    d = _Prepared(x0, n_warm)
    xd, td, xkd, sd = d.m.backend.radau_rollout(d.x.cpu().numpy(), d.dr.t.cpu().numpy(), knots, tau)
    assert np.array_equal(xkd, xa) and np.array_equal(sd, sa) and np.array_equal(td, ta) and np.array_equal(xd, xa[-1])

    for e in sorted({0, 1, 5, int(retried[0]), n_env - 1}):
        alone = _Prepared(x0[e:e + 1].copy(), n_warm)
        assert alone.dr.t.cpu().numpy()[0] == t_start[e]
        xe, se, te = alone.rollout(knots, tau[:, e:e + 1])
        assert np.array_equal(xe[:, 0], xa[:, e]) and np.array_equal(se[0], sa[e]) and te[0] == ta[e], e


def test_rollout_max_steps_and_step_after_rollout():
    """max_steps = 3 toward far knots: every environment stops after 3 steps short of knot 0, all x_knot rows NaN.  With start times
    that let some environments reach knot 0 within the budget but not knot 1, exactly the unreached rows are NaN.  pfc_radau_step after a roll-out continues from
    the controller state the roll-out left: 2 steps equal a roll-out toward a knot beyond the horizon with max_steps = 2."""
    n_env = 64
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    c = m.backend
    x0 = _boxes_states(m, n_env)
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x, t, x_knot, stats = c.radau_rollout(x0, np.zeros(n_env), [0.5, 1.0], max_steps=3)
    assert (stats[:, 0] == 0).all() and (stats[:, 1] == 3).all()
    assert np.isnan(x_knot).all()
    assert (t > 0).all() and (t < 0.5).all()

    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    t0 = np.where(np.arange(n_env) % 2 == 1, 0.0029, 0.0)   # odd environments start h0 short of knot 0
    _, _, x_knot, stats = c.radau_rollout(x0, t0, [0.003, 0.2], max_steps=3)
    reached = stats[:, 0]
    assert (reached[0::2] == 0).all() and (reached[1::2] == 1).any(), reached
    for e in range(n_env):
        assert not np.isnan(x_knot[:reached[e], e]).any() and np.isnan(x_knot[reached[e]:, e]).all(), e

    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x1, t1, _, _ = c.radau_rollout(x0, np.zeros(n_env), [0.02])
    for _ in range(2):
        x1, t1, _, _ = c.radau_step(x1, t1)
    m2 = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    m2.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x2, t2, _, _ = m2.backend.radau_rollout(x0, np.zeros(n_env), [0.02])
    x2, t2, x_knot, stats = m2.backend.radau_rollout(x2, t2, [1.0e3], max_steps=2)
    assert (stats[:, 1] == 2).all() and np.isnan(x_knot).all()
    assert np.array_equal(x1, x2) and np.array_equal(t1, t2)


def test_rollout_arguments_and_errors():
    """Bad knot arrays, max_steps < 1, a differing n_env and an environment less than h_min before knot 0 return PFC_E_ARG and leave
    x, t, x_knot, stats and the controllers untouched; tol_newton = 0 returns PFC_E_STEP; n_env = 0 is a no-op."""
    import torch
    from pfc_b200 import capi
    L = capi.lib()
    n_env = 4
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    c = m.backend
    x0 = boxes_env_states(m, n_env)
    nx = x0.shape[1]
    with pytest.raises(capi.PfcError) as ei:          # before pfc_radau_init
        c.radau_rollout(x0, np.zeros(n_env), [0.01])
    assert ei.value.code == PFC_E_ARG
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    dev = torch.device("cuda", 0)
    x = torch.as_tensor(x0).to(dev)
    t = torch.tensor([0.0, 0.0, 0.005, 0.0], dtype=torch.float64, device=dev)
    x_knot = torch.full((3, n_env, nx), 7.0, dtype=torch.float64, device=dev)
    stats = torch.full((n_env, 4), 9, dtype=torch.int32, device=dev)
    saved = [v.clone() for v in (x, t, x_knot, stats)]
    torch.cuda.synchronize()   # the library's stream does not wait for torch's default stream
    bad = [([0.01, 0.02, 0.02], 100), ([0.01, float("nan"), 0.03], 100), ([0.01, 0.02, 0.02 + 5e-9], 100), ([0.03, 0.02, 0.04], 100),
           ([0.01, 0.02, float("inf")], 100), ([0.01, 0.02, 0.03], 0),
           ([0.005 + 5e-9, 0.02, 0.03], 100)]                      # environment 2 starts at 0.005: less than h_min before knot 0
    for knots, max_steps in bad:
        with pytest.raises(capi.PfcError) as ei:
            c.radau_rollout_device(n_env, knots, max_steps, x.data_ptr(), None, t.data_ptr(), x_knot.data_ptr(), stats.data_ptr())
        assert ei.value.code == PFC_E_ARG, knots
        torch.cuda.synchronize()
        for u, v in zip((x, t, x_knot, stats), saved):
            assert torch.equal(u, v), knots
    assert L.pfc_radau_rollout_device(c._h, n_env, 0, np.zeros(1), 100, x.data_ptr(), None, t.data_ptr(), None, None) == PFC_E_ARG
    assert L.pfc_radau_rollout(c._h, n_env, 1, np.array([0.01]), 100, None, None, None, None, None) == PFC_E_ARG   # NULL buffers
    with pytest.raises(capi.PfcError) as ei:          # n_env differs from init's
        c.radau_rollout(x0[:2], np.zeros(2), [0.01])
    assert ei.value.code == PFC_E_ARG
    # the failed calls changed no controller: the roll-out now equals one on a fresh context
    got = c.radau_rollout(x0, np.zeros(n_env), [0.01, 0.02])
    m2 = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    m2.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    want = m2.backend.radau_rollout(x0, np.zeros(n_env), [0.01, 0.02])
    for u, v in zip(got, want):
        assert np.array_equal(u, v)
    # tol_newton = 0: no attempt converges, h falls by 10 per round until it is below h_min
    c.radau_init(n_env, 2, 1.0e-4, 0.05, 0.0)
    with pytest.raises(capi.PfcError) as ei:
        c.radau_rollout(x0, np.zeros(n_env), [0.01])
    assert ei.value.code == PFC_E_STEP and "time step is too small, something is wrong" in str(ei.value)
    c.radau_init(0, 2, 1.0e-4, 0.05, 1.0e-16)
    assert L.pfc_radau_rollout_device(c._h, 0, 1, np.array([0.01]), 100, None, None, None, None, None) == 0
