"""CPU-only: the per-environment arithmetic of the device Radau step (csrc/pfc_radau_step.cuh, with the Butcher data of
csrc/pfc_radau_tables.h) compiled for the host with g++ and driven the way radau_newton_kernel / radau_controller_kernel drive it, on the
reference's own integrator tests (test/test_radau/basic_test.jl, test_robertson.jl): the known answers hold, and the step sizes, rules,
Newton-iteration counts and states follow radau.solveRadau (pfc_b200/radau.py) on the same problems."""
import os
import re
import subprocess

import numpy as np
import pytest

import pfc_b200  # noqa: F401
from pfc_b200 import radau as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pressurefieldcontact.jl_b200", "csrc")

HARNESS = r"""
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <vector>
#define PFC_HOST_CHECK 1
#include "pfc_radau_step.cuh"
using namespace pfc;
using cd = std::complex<double>;

static int problem = 0;   // 0: exponential decay x' = -x (n = 4), 1: Robertson (n = 3)
static int nx = 0;
static void f(const double* x, double* xx) {
    if (problem == 0) { for (int i = 0; i < nx; ++i) xx[i] = -1.0 * x[i]; return; }
    const double y1 = x[0], y2 = x[1], y3 = x[2];
    xx[0] = -0.04 * y1 + 1.0e4 * y2 * y3;
    xx[1] = 0.04 * y1 - 1.0e4 * y2 * y3 - 3.0e7 * y2 * y2;
    xx[2] = 3.0e7 * y2 * y2;
}
static void jac(const double* x, double* J) {   // J[i][j] = d xx_i / d x_j
    for (int i = 0; i < nx * nx; ++i) J[i] = 0.0;
    if (problem == 0) { for (int i = 0; i < nx; ++i) J[i * nx + i] = -1.0; return; }
    const double y2 = x[1], y3 = x[2];
    J[0] = -0.04; J[1] = 1.0e4 * y3; J[2] = 1.0e4 * y2;
    J[3] = 0.04; J[4] = -1.0e4 * y3 - 6.0e7 * y2; J[5] = -1.0e4 * y2;
    J[6] = 0.0; J[7] = 6.0e7 * y2; J[8] = 0.0;
}
// plain Gauss-Jordan with partial pivoting; interleaved (re, im) row-major output like launch_radau_inv_c
static void inverse(std::vector<cd> A, double* out) {
    std::vector<cd> I(nx * nx, 0.0);
    for (int i = 0; i < nx; ++i) I[i * nx + i] = 1.0;
    for (int k = 0; k < nx; ++k) {
        int p = k;
        for (int i = k + 1; i < nx; ++i) if (std::abs(A[i * nx + k]) > std::abs(A[p * nx + k])) p = i;
        for (int j = 0; j < nx; ++j) { std::swap(A[k * nx + j], A[p * nx + j]); std::swap(I[k * nx + j], I[p * nx + j]); }
        const cd d = 1.0 / A[k * nx + k];
        for (int j = 0; j < nx; ++j) { A[k * nx + j] *= d; I[k * nx + j] *= d; }
        for (int i = 0; i < nx; ++i) {
            if (i == k) continue;
            const cd m = A[i * nx + k];
            for (int j = 0; j < nx; ++j) { A[i * nx + j] -= m * A[k * nx + j]; I[i * nx + j] -= m * I[k * nx + j]; }
        }
    }
    for (int i = 0; i < nx * nx; ++i) { out[2 * i] = I[i].real(); out[2 * i + 1] = I[i].imag(); }
}

int main(int argc, char** argv) {
    problem = std::atoi(argv[1]);
    const int n_steps = std::atoi(argv[2]), rule0 = std::atoi(argv[3]), max_rule = std::atoi(argv[4]);
    const double h0 = std::atof(argv[5]), h_max = std::atof(argv[6]);
    nx = problem == 0 ? 4 : 3;
    std::vector<double> x0(nx, 0.0);
    if (problem == 0) for (double& v : x0) v = 1.0; else x0[0] = 1.0;
    RadauEnv e;
    radau_env_reset(e, h0);
    e.rule = rule0;
    const int S = kRadauMaxStage;
    std::vector<double> J(nx * nx), xx0(nx), X(S * nx), F(S * nx), st(S * nx), ar(S * nx), ai(S * nx), br(S * nx), bi(S * nx), inv(S * 2 * nx * nx);
    double t = 0.0;
    for (int step = 0; step < n_steps; ++step) {
        jac(x0.data(), J.data());
        f(x0.data(), xx0.data());
        for (;;) {
            const RadauTableData& T = kRadauTables[e.rule - 1];
            const int s = T.s;
            const double h = e.h, h_inv = 1.0 / h;
            for (int i = 0; i < s; ++i) {
                std::vector<cd> C(nx * nx);
                const cd sh = cd(h_inv * T.lam_re[i], h_inv * T.lam_im[i]);
                for (int a = 0; a < nx * nx; ++a) C[a] = -J[a] + ((a / nx == a % nx) ? sh : cd(0.0));
                inverse(C, &inv[i * 2 * nx * nx]);
            }
            radau_attempt_begin(e);
            for (int i = 0; i < s; ++i) for (int n = 0; n < nx; ++n) X[i * nx + n] = x0[n];
            for (int k = 1;; ++k) {
                for (int i = 0; i < s; ++i) f(&X[i * nx], &F[i * nx]);
                for (int id = 0; id < s * nx; ++id) st[id] = radau_store(T, h, id / nx, id % nx, nx, x0.data(), X.data(), F.data());
                double residual = 0.0;
                for (int i = 0; i < s; ++i) { double a = 0.0; for (int n = 0; n < nx; ++n) a = a + st[i * nx + n] * st[i * nx + n]; residual += a; }
                for (int id = 0; id < s * nx; ++id) radau_ew(T, h_inv, id / nx, id % nx, nx, st.data(), &ar[id], &ai[id]);
                for (int id = 0; id < s * nx; ++id) { const int i = id / nx; radau_matvec_row(&inv[i * 2 * nx * nx], nx, id % nx, &ar[i * nx], &ai[i * nx], &br[id], &bi[id]); }
                unsigned mask = 0;
                for (int id = 0; id < s * nx; ++id) { st[id] = radau_update(T, id / nx, id % nx, nx, br.data(), bi.data()); if (std::fabs(st[id]) > 1.0e1) mask |= 1u << (id / nx); }
                const int first = mask ? __builtin_ctz(mask) : s;
                for (int id = 0; id < first * nx; ++id) X[id] = X[id] - st[id];
                e.n_evals += s;
                const int d = radau_newton_decide(e, k, residual, mask != 0, 1.0e-16);
                if (d == kRadauConverged) {
                    for (int n = 0; n < nx; ++n) ar[n] = radau_err_d(T, h, n, nx, xx0.data(), F.data());
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
                t += h_taken;
                std::printf("step %.17g %.17g", h_taken, t);
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
    d = tmp_path_factory.mktemp("radau_host")
    cpp, exe = d / "radau_host.cpp", d / "radau_host"
    cpp.write_text(HARNESS)
    # -ffp-contract=off: nvcc may contract a * b + c on the device; these tests bound the host build against radau.py, not bits
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-I", CSRC, "-o", str(exe), str(cpp)])

    def run(*args):
        out = subprocess.run([str(exe), *map(str, args)], capture_output=True, text=True, check=True).stdout.split("\n")
        attempts = [tuple(float(v) for v in ln.split()[1:]) for ln in out if ln.startswith("attempt")]
        steps = [np.array([float(v) for v in ln.split()[1:]]) for ln in out if ln.startswith("step")]
        return attempts, steps
    return run


def test_radau_tables_header_matches_the_generator():
    txt = open(os.path.join(CSRC, "pfc_radau_tables.h")).read()
    body = txt[txt.index("kRadauTables[kRadauMaxRule] = {"):]
    for n in (1, 2, 3):
        t = R.radau_table(n)
        block = body.split("// rule %d" % n)[1].split("// rule")[0]
        vals = [float.fromhex(v) for v in re.findall(r"-?0x[0-9a-fA-F.]+p[+-]\d+", block)]
        S = 5

        def pad_m(M):
            out = np.zeros((S, S))
            out[:M.shape[0], :M.shape[1]] = M
            return out.ravel()

        def pad_v(v):
            out = np.zeros(S)
            out[:len(v)] = v
            return out
        want = np.concatenate([pad_m(t.A), pad_v(t.c), pad_v(t.lam.real), pad_v(t.lam.imag), pad_m(t.T.real), pad_m(t.T.imag),
                               pad_m(t.Tinv.real), pad_m(t.Tinv.imag), pad_v(t.b_hat), [t.b_hat_0]])
        got = np.array(vals)
        assert got.shape == want.shape, n
        assert (np.abs(got - want) <= 2 * np.spacing(np.abs(want))).all(), n


class _Linear:   # test/test_radau/basic_test.jl
    def de(self, xx, x, t=0.0):
        xx[:] = -1.0 * x

    def de_jacobian_chunk(self, x, i0, i1, t=0.0):
        xx = -1.0 * np.asarray(x, dtype=np.float64)
        return xx, -np.eye(len(x))[:, i0:i1]


class _Robertson:   # test/test_radau/test_robertson.jl, with the analytic Jacobian the harness uses
    def de(self, xx, x, t=0.0):
        y1, y2, y3 = x
        xx[0] = -0.04 * y1 + 1.0e4 * y2 * y3
        xx[1] = 0.04 * y1 - 1.0e4 * y2 * y3 - 3.0e7 * y2 * y2
        xx[2] = 3.0e7 * y2 * y2

    def de_jacobian_chunk(self, x, i0, i1, t=0.0):
        xx = np.zeros(3)
        self.de(xx, x)
        _, y2, y3 = x
        J = np.array([[-0.04, 1.0e4 * y3, 1.0e4 * y2], [0.04, -1.0e4 * y3 - 6.0e7 * y2, -1.0e4 * y2], [0.0, 6.0e7 * y2, 0.0]])
        return xx, J[:, i0:i1]


def _python_run(de, x0, n_steps, rule0, NR, h0, h_max, monkeypatch):
    """radau.solveRadau with every attempt recorded as (stages, Newton iterations, exit flag, h after the controller)."""
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
    x, t, steps = np.array(x0, dtype=np.float64), 0.0, []
    for _ in range(n_steps):
        h, x, t = R.solveRadau(rr, x, t)
        steps.append(np.r_[h, t, x])
    return attempts, steps


def _same_run(host, py):
    (ha, hs), (pa, ps) = host, py
    assert len(ha) == len(pa) and len(hs) == len(ps)
    for a, b in zip(ha, pa):
        assert a[:3] == tuple(float(v) for v in b[:3]), (a, b)      # stages, Newton iterations, exit flag
        assert abs(a[3] - b[3]) <= 1e-12 * b[3], (a, b)
    for a, b in zip(hs, ps):
        assert np.abs(a - b).max() <= 1e-12 * max(np.abs(b).max(), 1.0), (a, b)


def test_exponential_decay_rule_3(harness, monkeypatch):
    attempts, steps = harness(0, 1, 3, 3, 0.2, 0.01)
    assert attempts[0][0] == 5 and len(steps) == 1
    assert abs(np.exp(-0.2) - steps[0][2]) < 1e-8 * np.exp(-0.2)
    _same_run((attempts, steps), _python_run(_Linear(), np.ones(4), 1, 3, 3, 0.2, 0.01, monkeypatch))


def test_robertson_rule_2(harness, monkeypatch):
    attempts, steps = harness(1, 10, 2, 2, 1.0e-4, "inf")
    y2 = steps[-1][3]
    assert 3.45e-5 < y2 < 3.7e-5
    assert steps[-1][1] == pytest.approx(1.0e-4 * (2 ** 10 - 1), rel=1e-12)
    _same_run((attempts, steps), _python_run(_Robertson(), np.array([1.0, 0.0, 0.0]), 10, 2, 2, 1.0e-4, np.inf, monkeypatch))
