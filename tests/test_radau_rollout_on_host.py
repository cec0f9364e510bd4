"""CPU-only: the knot rules of the device roll-out (radau_knot_begin / radau_knot_end in csrc/pfc_radau_step.cuh) compiled for the host
with g++ around the same per-environment step arithmetic that tests/test_radau_step_on_host.py drives, through knot sequences on the
reference's exponential-decay and Robertson problems: the step sizes, rules, Newton iterations and states follow radau.rollout_radau
(pfc_b200/radau.py), every knot is hit exactly, no step leaves a remainder below h_min, and knots beyond the horizon change nothing."""
import os
import subprocess

import numpy as np
import pytest

import pfc_b200  # noqa: F401
from pfc_b200 import radau as R
from test_radau_step_on_host import CSRC, HARNESS, _Linear, _Robertson

H_MIN = 1.0e-8

# the problems, the Jacobians and the complex inverse of the step harness; a roll-out main instead of its fixed number of steps
MAIN = r"""
int main(int argc, char** argv) {
    problem = std::atoi(argv[1]);
    const int rule0 = std::atoi(argv[2]), max_rule = std::atoi(argv[3]);
    const double h0 = std::atof(argv[4]), h_max = std::atof(argv[5]), t0 = std::atof(argv[6]);
    const int max_steps = std::atoi(argv[7]), K = argc - 8;
    std::vector<double> knots(K);
    for (int k = 0; k < K; ++k) knots[k] = std::strtod(argv[8 + k], nullptr);
    nx = problem == 0 ? 4 : 3;
    std::vector<double> x0(nx, 0.0);
    if (problem == 0) for (double& v : x0) v = 1.0; else x0[0] = 1.0;
    RadauEnv e;
    radau_env_reset(e, h0);
    e.rule = rule0;
    const int S = kRadauMaxStage;
    std::vector<double> J(nx * nx), xx0(nx), X(S * nx), F(S * nx), st(S * nx), ar(S * nx), ai(S * nx), br(S * nx), bi(S * nx), inv(S * 2 * nx * nx);
    double t = t0;
    int k_knot = 0;
    for (int step = 0; k_knot < K && step < max_steps; ++step) {
        const double T = knots[k_knot];
        const double h_save = radau_knot_begin(e, t, T);
        jac(x0.data(), J.data());
        f(x0.data(), xx0.data());
        for (;;) {
            const RadauTableData& Tb = kRadauTables[e.rule - 1];
            const int s = Tb.s;
            const double h = e.h, h_inv = 1.0 / h;
            for (int i = 0; i < s; ++i) {
                std::vector<cd> C(nx * nx);
                const cd sh = cd(h_inv * Tb.lam_re[i], h_inv * Tb.lam_im[i]);
                for (int a = 0; a < nx * nx; ++a) C[a] = -J[a] + ((a / nx == a % nx) ? sh : cd(0.0));
                inverse(C, &inv[i * 2 * nx * nx]);
            }
            radau_attempt_begin(e);
            for (int i = 0; i < s; ++i) for (int n = 0; n < nx; ++n) X[i * nx + n] = x0[n];
            for (int k = 1;; ++k) {
                for (int i = 0; i < s; ++i) f(&X[i * nx], &F[i * nx]);
                for (int id = 0; id < s * nx; ++id) st[id] = radau_store(Tb, h, id / nx, id % nx, nx, x0.data(), X.data(), F.data());
                double residual = 0.0;
                for (int i = 0; i < s; ++i) { double a = 0.0; for (int n = 0; n < nx; ++n) a = a + st[i * nx + n] * st[i * nx + n]; residual += a; }
                for (int id = 0; id < s * nx; ++id) radau_ew(Tb, h_inv, id / nx, id % nx, nx, st.data(), &ar[id], &ai[id]);
                for (int id = 0; id < s * nx; ++id) { const int i = id / nx; radau_matvec_row(&inv[i * 2 * nx * nx], nx, id % nx, &ar[i * nx], &ai[i * nx], &br[id], &bi[id]); }
                unsigned mask = 0;
                for (int id = 0; id < s * nx; ++id) { st[id] = radau_update(Tb, id / nx, id % nx, nx, br.data(), bi.data()); if (std::fabs(st[id]) > 1.0e1) mask |= 1u << (id / nx); }
                const int first = mask ? __builtin_ctz(mask) : s;
                for (int id = 0; id < first * nx; ++id) X[id] = X[id] - st[id];
                e.n_evals += s;
                const int d = radau_newton_decide(e, k, residual, mask != 0, 1.0e-16);
                if (d == kRadauConverged) {
                    for (int n = 0; n < nx; ++n) ar[n] = radau_err_d(Tb, h, n, nx, xx0.data(), F.data());
                    double a = 0.0;
                    for (int r = 0; r < nx; ++r) a = a + radau_err_term(inv.data(), nx, r, ar.data(), X[(s - 1) * nx + r], x0[r]);
                    e.err_norm = std::sqrt(a / nx);
                }
                if (d != kRadauIterate) break;
            }
            const int k_iter = e.k_iter, exit_flag = e.exit_flag;
            double h_taken = 0.0;
            const int rc = radau_control(e, max_rule, h_max, &h_taken);
            std::printf("attempt %d %d %d %.17g\n", s, k_iter, exit_flag, e.h);
            if (rc < 0) { std::printf("error %d\n", rc); return 1; }
            if (rc == kRadauAccepted) {
                for (int n = 0; n < nx; ++n) x0[n] = X[(s - 1) * nx + n];
                double t_new = 0.0;
                const bool hit = radau_knot_end(e, t, T, h_taken, h_save, &t_new);
                t = t_new;
                k_knot += hit;
                std::printf("step %.17g %.17g %d %.17g", h_taken, t, int(hit), T);
                for (int n = 0; n < nx; ++n) std::printf(" %.17g", x0[n]);
                std::printf("\n");
                break;
            }
        }
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    d = tmp_path_factory.mktemp("radau_rollout_host")
    cpp, exe = d / "radau_rollout_host.cpp", d / "radau_rollout_host"
    cpp.write_text(HARNESS[:HARNESS.index("int main(")] + MAIN)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-I", CSRC, "-o", str(exe), str(cpp)])

    def run(problem, rule0, max_rule, h0, h_max, t0, max_steps, knots):
        args = [problem, rule0, max_rule, h0, h_max, repr(float(t0)), max_steps] + [repr(float(v)) for v in knots]
        out = subprocess.run([str(exe), *map(str, args)], capture_output=True, text=True, check=True).stdout.split("\n")
        attempts = [tuple(float(v) for v in ln.split()[1:]) for ln in out if ln.startswith("attempt")]
        steps = [[float(v) for v in ln.split()[1:]] for ln in out if ln.startswith("step")]
        return attempts, steps   # step: h_taken, t after, knot hit, knot aimed at, x
    return run


def _python_rollout(de, x0, rule0, NR, h0, h_max, t0, max_steps, knots, monkeypatch):
    attempts = []
    orig_rule = R._update_rule

    def rec_rule(rr):
        attempts.append((rr.current_table().n_stage, rr.rule.k_iter, rr.step.exit_flag, rr.step.h))
        orig_rule(rr)
    monkeypatch.setattr(R, "_update_rule", rec_rule)
    rr = R.makeRadauIntegrator(de, x0, 1.0e-16, NR, 6)
    R.update_h(rr, h0)
    rr.rule.s = rule0
    rr.step.h_max = h_max
    record = []
    x_knot, x, t, stats = R.rollout_radau(rr, x0, t0, knots, max_steps=max_steps, record=record)
    return attempts, record, x_knot, stats


def _check_against_mirror(host, py, knots):
    (ha, hs), (pa, rec, x_knot, stats) = host, py
    assert len(ha) == len(pa) and len(hs) == len(rec)
    for a, b in zip(ha, pa):
        assert a[:3] == tuple(float(v) for v in b[:3]), (a, b)      # stages, Newton iterations, exit flag
        assert abs(a[3] - b[3]) <= 1e-12 * b[3], (a, b)
    for a, (h, t, x, _) in zip(hs, rec):
        assert abs(a[0] - h) <= 1e-12 * h and abs(a[1] - t) <= 1e-12 * abs(t), (a, h, t)
        assert np.abs(np.array(a[4:]) - x).max() <= 1e-12 * max(np.abs(x).max(), 1.0)
    # every knot is hit exactly, by both; no step ends within h_min of the knot it aims at
    hits = [a for a in hs if a[2] == 1.0]
    assert len(hits) == stats[0]
    for a in hs:
        assert a[1] == a[3] if a[2] == 1.0 else a[3] - a[1] >= H_MIN, a
    assert [a[1] for a in hits] == [float(v) for v in knots[:len(hits)]]
    t_py = [t for (h, t, x, _) in rec]
    assert all(t in t_py for t in knots[:stats[0]])
    for k in range(stats[0]):
        assert not np.isnan(x_knot[k]).any()
    assert np.isnan(x_knot[stats[0]:]).all()


def test_exponential_decay_through_knots(harness, monkeypatch):
    """Rule 3, h_max = 0.01: knots closer than h (a knot step shorter than the proposal), a gap of 2 h_min, and a knot that an ordinary
    step would miss by less than h_min."""
    knots = [0.013, 0.02, 0.02000002, 0.0350000001, 0.05, 0.1]
    host = harness(0, 3, 3, 1.0e-3, 0.01, 0.0, 1000, knots)
    py = _python_rollout(_Linear(), np.ones(4), 3, 3, 1.0e-3, 0.01, 0.0, 1000, knots, monkeypatch)
    _check_against_mirror(host, py, knots)
    assert py[3][0] == len(knots)
    assert abs(np.exp(-0.1) - py[2][-1][0]) < 1e-6


def test_robertson_through_knots(harness, monkeypatch):
    """Rule 2, no h_max, from t0 = 1e-5: the step size grows by 2 per step between knots and is cut back at each; the rule rises."""
    knots = [1.0e-3, 2.5e-3, 0.01, 0.1, 0.4]
    host = harness(1, 1, 2, 1.0e-4, "inf", 1.0e-5, 1000, knots)
    py = _python_rollout(_Robertson(), np.array([1.0, 0.0, 0.0]), 1, 2, 1.0e-4, np.inf, 1.0e-5, 1000, knots, monkeypatch)
    _check_against_mirror(host, py, knots)
    assert py[3][0] == len(knots)
    assert 3 in [a[0] for a in py[0]], "no attempt on rule 2"


def test_max_steps_stops_short_of_the_knots(harness, monkeypatch):
    knots = [0.05, 0.1, 0.2]
    host = harness(0, 1, 2, 1.0e-3, 0.01, 0.0, 7, knots)
    py = _python_rollout(_Linear(), np.ones(4), 1, 2, 1.0e-3, 0.01, 0.0, 7, knots, monkeypatch)
    _check_against_mirror(host, py, knots)
    assert py[3][1] == 7 and py[3][0] == 0
    assert np.isnan(py[2]).all()


@pytest.mark.parametrize("problem", [0, 1])
def test_knots_beyond_the_horizon_change_no_step(harness, monkeypatch, problem):
    """A knot far ahead: the roll-out takes solveRadau's steps, bit for bit in radau.py and within the usual bound in the header."""
    de, x0, rule0, NR, h0, h_max, n = ((_Linear(), np.ones(4), 3, 3, 0.2, 0.01, 5) if problem == 0 else
                                       (_Robertson(), np.array([1.0, 0.0, 0.0]), 2, 2, 1.0e-4, np.inf, 12))
    knots = [1.0e6]
    host = harness(problem, rule0, NR, h0, "inf" if h_max == np.inf else h_max, 0.0, n, knots)
    py = _python_rollout(de, x0, rule0, NR, h0, h_max, 0.0, n, knots, monkeypatch)
    _check_against_mirror(host, py, knots)
    rr = R.makeRadauIntegrator(de, x0, 1.0e-16, NR, 6)
    R.update_h(rr, h0)
    rr.rule.s = rule0
    rr.step.h_max = h_max
    x, t = np.array(x0, dtype=np.float64), 0.0
    for h_r, t_r, x_r, _ in py[1]:
        h, x, t = R.solveRadau(rr, x, t)
        assert h == h_r and t == t_r and np.array_equal(x, x_r)


def test_rollout_radau_rejects_bad_knots():
    rr = R.makeRadauIntegrator(_Linear(), np.ones(4), 1.0e-16, 2, 6)
    for t0, knots in ((0.0, []), (0.0, [0.1, 0.1]), (0.0, [0.1, 0.1 + 1e-9]), (0.0, [float("nan")]), (0.0, [0.2, 0.1]), (0.1, [0.1 + 5e-9]),
                      (0.0, [0.1, float("inf")])):
        with pytest.raises(ValueError):
            R.rollout_radau(rr, np.ones(4), t0, knots)
