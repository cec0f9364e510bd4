"""GPU tests of the batched adaptive Radau IIA step behind the C ABI (pfc_radau_init / pfc_radau_step[_device]): the Newton iteration,
error estimate and step-size / order control in CUDA kernels, against the single-scene mirror of the reference's integrator (radau.py),
against the torch-driven BatchedRadau, and for batch invariance, host / device entry-point equality and the error returns."""
import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import boxes_env_states, scene_boxes
from oracle import orc
from pfc_b200 import dynamics as D
from pfc_b200 import radau as R
from pfc_b200 import scenario as S

pytestmark = pytest.mark.gpu


def _ctx():
    from pfc_b200 import capi
    return capi.Context(0)


class _TauDynamics:
    """calcXd! on the device with a constant tau_ext, through the single-environment entry points (calcxd_f64 / calcxd_dual6)."""

    def __init__(self, m, tau):
        self.m, self.tau = m, np.asarray(tau, dtype=np.float64)[None, :]

    def de(self, xx, x, t=0.0):
        xx[:] = self.m.backend.calcxd_f64(x, self.tau)["xdot"][0]

    def de_jacobian_chunk(self, x, i0, i1, t=0.0):
        xd7 = self.m.backend.calcxd_dual6(x, i0, self.tau)["xdot7"][0]
        return xd7[:, 0].copy(), xd7[:, 1:1 + (i1 - i0)].copy()


def _mirror(m, dyn, x0, n_steps, h_max):
    """radau.py one environment at a time: per step (h, t, x after principal_value!, stage evaluations of the step)."""
    rr = R.makeRadauIntegrator(dyn, S.num_x(m), 1.0e-16, 2, 6)
    rr.step.h_max = h_max
    x, t, out = np.array(x0, dtype=np.float64), 0.0, []
    for _ in range(n_steps):
        n0 = rr.n_de_float
        h, x, t = R.solveRadau(rr, x, t)
        D.principal_value(m, x)
        out.append((h, t, x.copy(), rr.n_de_float - n0))
    return out


def _run_device(m, x0, n_steps, h_max, tau=None):
    """pfc_radau_step_device for the batch: per step (x, t, h_taken, stats) on the host."""
    import torch
    from pfc_b200.radau_batched import DeviceBatchedRadau
    n_env = x0.shape[0]
    dr = DeviceBatchedRadau(m, n_env, h_max=h_max)
    steps = []
    with torch.cuda.stream(dr.stream):
        x = torch.as_tensor(x0).to(dr.dev)
        tau_t = None if tau is None else torch.as_tensor(tau).to(dr.dev)
        for _ in range(n_steps):
            x, h = dr.step(x, tau_t)
            steps.append((x.cpu().numpy().copy(), dr.t.cpu().numpy().copy(), h.cpu().numpy().copy(), dr.stats.cpu().numpy().copy()))
    return steps


def _compare_with_mirror(steps, ref, e, tol):
    for k, (h, t, x, n_eval) in enumerate(ref):
        xb, tb, hb, sb = steps[k]
        assert sb[e, 3] == n_eval, (e, k, sb[e], n_eval)
        assert abs(hb[e] - h) <= tol * h, (e, k, hb[e], h)
        assert abs(tb[e] - t) <= tol * t, (e, k)
        scale = np.abs(x).max()
        for i in range(0, x.shape[0], 3):
            den = max(np.abs(x[i:i + 3]).max(), 1e-6 * scale)
            assert np.abs(xb[e, i:i + 3] - x[i:i + 3]).max() <= tol * den, (e, k, i)


def test_radau_step_follows_the_oracle_backed_single_scene_integrator():
    """boxes.jl, 6 environments (the reference's drop, a settled stack at rest, random settled stacks, and the drop 0.5 m higher), 25
    steps, h_max = 0.05: per environment and step the same stage-evaluation count as radau.py over the CPU oracle, h and t within 1e-7,
    states within 1e-7 per 3-vector.  The run has rejected attempts and steps accepted on rule 2 (3 stages): the order only rises after
    10 accepted steps in a row, which the contact states never reach within 25 steps; the higher drop reaches it in free flight and
    takes steps 11-15 on rule 2 before its first contact.  (Not 0.3 m: there a rule-2 attempt stalls with residuals equal to 4 digits,
    and where the growth test r_k-2 < r_k-1 < r_k first fires is decided by rounding, so the oracle and the device differ in it.)"""
    n_env, n_steps, h_max = 6, 25, 0.05
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    x0[0] = S.get_state(m)
    x0[1, m.nq:] = 0.0
    x0[5] = S.get_state(m)
    for b in m.bodies:
        if b.joint is not None:
            x0[5, b.q0 + 5] += 0.5
    steps = _run_device(m, x0, n_steps, h_max)
    stats = np.array([s[3] for s in steps])   # [step][env][4]
    assert (stats[:, :, 2] > 0).any(), "no rejected attempt in the run"
    assert (stats[:, :, 0] == 3).any(), "no step accepted on rule 2"
    m_cpu = scene_boxes(orc.OracleContext())[0]
    for e in range(n_env):
        ref = _mirror(m_cpu, D.FloatingBodyDynamics(m_cpu), x0[e], n_steps, h_max)
        _compare_with_mirror(steps, ref, e, 1e-7)


def test_radau_step_agrees_with_batched_radau():
    """256 settled-stack environments, 10 steps: h_taken and the states after every step within 1e-9 of the torch-driven BatchedRadau
    (a different decision would show as a factor 0.1 or 2 in h)."""
    import torch
    from pfc_b200.radau_batched import BatchedRadau
    n_env, n_steps = 256, 10
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    steps = _run_device(m, x0, n_steps, 0.05)
    br = BatchedRadau(m, n_env, h_max=0.05)
    with torch.cuda.stream(br.stream):
        x = torch.as_tensor(x0).to(br.dev)
        for k in range(n_steps):
            x, h = br.step(x)
            xb, hb = x.cpu().numpy(), h.cpu().numpy()
            xd, _, hd, _ = steps[k]
            assert np.abs(hd - hb).max() <= 1e-9 * hb.max(), k
            scale = np.abs(xb).max(axis=1, keepdims=True)
            v_ref, v_dev = xb.reshape(n_env, -1, 3), xd.reshape(n_env, -1, 3)
            den = np.maximum(np.abs(v_ref).max(axis=2), 1e-6 * scale)
            assert (np.abs(v_dev - v_ref).max(axis=2) <= 1e-9 * den).all(), k


def test_radau_step_is_batch_invariant_and_deterministic():
    """1000 mixed environments, 8 steps, twice: identical bits.  Four of them (one that retried) alone (n_env = 1): identical x, t,
    h_taken and stats."""
    n_env, n_steps = 1000, 8
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    x0[0] = S.get_state(m)
    x0[1, m.nq:] = 0.0
    a = _run_device(m, x0, n_steps, 0.05)
    b = _run_device(m, x0, n_steps, 0.05)
    for sa, sb in zip(a, b):
        for u, v in zip(sa, sb):
            assert np.array_equal(u, v)
    retried = np.nonzero(np.array([s[3][:, 2] for s in a]).max(axis=0) > 0)[0]
    assert len(retried) > 0
    picks = sorted({0, 1, int(retried[0]), n_env - 1})
    for e in picks:
        alone = _run_device(m, x0[e:e + 1].copy(), n_steps, 0.05)
        for k in range(n_steps):
            for u, v in zip(a[k], alone[k]):
                assert np.array_equal(u[e:e + 1], v), (e, k)


def test_radau_step_bristle_scene_with_tau_ext():
    """Bristle boxes (n_x = 60: MRPs and bristle states), 16 environments, 10 steps, random constant tau_ext: against radau.py over an
    in-test de that hands the same tau to calcxd_f64 / calcxd_dual6."""
    n_env, n_steps, h_max = 16, 10, 0.05
    m = scene_boxes(_ctx(), max_env=3 * n_env, bristle=True)[0]
    assert S.num_x(m) == 60
    x0 = boxes_env_states(m, n_env)
    tau = np.random.default_rng(7).uniform(-1, 1, (n_env, m.nv))
    steps = _run_device(m, x0, n_steps, h_max, tau)
    for e in range(n_env):
        ref = _mirror(m, _TauDynamics(m, tau[e]), x0[e], n_steps, h_max)
        _compare_with_mirror(steps, ref, e, 1e-7)


def test_radau_step_large_path_scene():
    """The tet-tet sphere on slab (one LARGE-path instruction, n_x = 12) at a generic pose, 5 steps, against radau.py on the device
    backend."""
    from pfc_b200 import scenes
    m, x = scenes.scene_c4_sphere_on_slab(24, 27, backend=_ctx())
    x = x.copy()
    x[0:3] = [0.011, -0.017, 0.023]
    x[3:6] = [0.0123, -0.0071, 0.0451]
    steps = _run_device(m, x[None, :].copy(), 5, 0.01)
    ref = _mirror(m, D.FloatingBodyDynamics(m, device=True), x, 5, 0.01)
    _compare_with_mirror(steps, ref, 0, 1e-7)


def test_radau_step_host_entry_point_equals_device_entry_point():
    n_env, n_steps = 64, 4
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    x0 = boxes_env_states(m, n_env)
    tau = np.random.default_rng(3).uniform(-1, 1, (n_env, m.nv))
    dev = _run_device(m, x0, n_steps, 0.05, tau)
    m.backend.radau_init(n_env, 2, 1.0e-4, 0.05, 1.0e-16)
    x, t = x0.copy(), np.zeros(n_env)
    for k in range(n_steps):
        x, t, h, stats = m.backend.radau_step(x, t, tau)
        for u, v in zip((x, t, h, stats), dev[k]):
            assert np.array_equal(u, v), k


def test_radau_step_arguments_and_errors():
    from pfc_b200 import capi
    L = capi.lib()
    bare = _ctx()
    n_env = 4
    m = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    c = m.backend
    x0 = boxes_env_states(m, n_env)
    PFC_E_ARG, PFC_E_STEP = -1, -6
    # before pfc_set_dynamics / before pfc_radau_init
    assert L.pfc_radau_init(bare._h, 4, 2, 1e-4, 0.01, 1e-16) == PFC_E_ARG
    with pytest.raises(capi.PfcError) as ei:
        c.radau_step(x0, np.zeros(n_env))
    assert ei.value.code == PFC_E_ARG
    # bad init arguments
    for args in ((n_env, 0, 1e-4, 0.01, 1e-16), (n_env, 4, 1e-4, 0.01, 1e-16), (n_env, 2, float("nan"), 0.01, 1e-16), (n_env, 2, -1e-4, 0.01, 1e-16),
                 (n_env, 2, 1e-4, float("inf"), 1e-16), (n_env, 2, 1e-4, 0.0, 1e-16), (n_env, 2, 1e-4, 0.01, -1.0), (-1, 2, 1e-4, 0.01, 1e-16)):
        with pytest.raises(capi.PfcError) as ei:
            c.radau_init(*args)
        assert ei.value.code == PFC_E_ARG, args
    c.radau_init(n_env, 2, 1e-4, 0.05, 1e-16)
    with pytest.raises(capi.PfcError) as ei:      # n_env differs from init's
        c.radau_step(x0[:2], np.zeros(2))
    assert ei.value.code == PFC_E_ARG
    assert L.pfc_radau_step_device(c._h, n_env, None, None, None, None, None) == PFC_E_ARG   # NULL buffers
    assert L.pfc_radau_step(c._h, n_env, None, None, None, None, None) == PFC_E_ARG
    # n_env == 0 is a no-op
    c.radau_init(0, 2, 1e-4, 0.05, 1e-16)
    assert L.pfc_radau_step_device(c._h, 0, None, None, None, None, None) == 0
    # tol_newton = 0: no attempt converges, h falls by 10 per round until it is below h_min
    c.radau_init(n_env, 2, 1e-4, 0.05, 0.0)
    with pytest.raises(capi.PfcError) as ei:
        c.radau_step(x0, np.zeros(n_env))
    assert ei.value.code == PFC_E_STEP and "time step is too small, something is wrong" in str(ei.value)
    # the same context, re-initialised, steps exactly like a fresh one
    c.radau_init(n_env, 2, 1e-4, 0.05, 1e-16)
    got = c.radau_step(x0, np.zeros(n_env))
    m2 = scene_boxes(_ctx(), max_env=3 * n_env)[0]
    m2.backend.radau_init(n_env, 2, 1e-4, 0.05, 1e-16)
    want = m2.backend.radau_step(x0, np.zeros(n_env))
    for u, v in zip(got, want):
        assert np.array_equal(u, v)
