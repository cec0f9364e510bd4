"""radau.py -- host-side mirror of the reference's adaptive Radau IIA integrator (the CALLER of the
contact-wrench path; SURVEY.md section 8f rank 4).  It exists so that the device path can be driven
exactly the way the reference drives it -- `rr.de_object.de(xx, x, de_object, t)` with Float64 vectors
for the stage evaluations and with Dual-6 chunks for the Jacobian -- and so that "state parity over N
Radau steps" (BASELINE.json configs[0..1]) can be measured between the CUDA path and the CPU oracle.

Follows /root/reference/src/radau:
  RadauTable / RadauStep / RadauRule / RadauIntegrator ... radau_struct.jl:1-118
  calcJacobian! / seed_indices! / write_indices! ......... radau_functions.jl:1-36
  updateFX! / calcEw! / updateInvC! / updateStageX! ...... radau_functions.jl:62-125
  solveRadau / solveRadau_inner / simple_newton! ......... radau_solve.jl:1-99
  calc_x_hat_minus_x / calc_x_err_norm / update_h! / update_rule! ... adaptive.jl:1-85
  makeRadauIntegrator ..................................... radau_utilities.jl:10-17

The Butcher data the reference reads from src/radau/table/*_rule/*.txt (A, c, lambda, T, inv_T, b_hat)
are mathematical constants of the Radau IIA family and are GENERATED here from their definitions
(collocation at the right Radau nodes; eigen-decomposition of inv(A); embedded weights of Hairer &
Wanner eq. IV.8.17 with b_hat_0 = 1 / real eigenvalue): radau_table().  The eigenvector scaling of T is
not unique; T only ever appears as the pair (T, inv_T), so the iteration is unchanged up to rounding.

Differences from the reference, on purpose:
  * the ODE is any object with  de(xx, x, t)  (Float64 in, Float64 out) and
    de_jacobian_chunk(x, i0, i1, t) -> (xx0, d xx / d x[i0:i1])  -- the Dual-N evaluation of one chunk
    (value + partials), which is what ForwardDiff's seeded call returns (radau_functions.jl:8-10);
    objects without it get a complex-step / central-difference fallback (tests only);
  * the reference re-enters solveRadau_inner WITHOUT passing t after a failed step (radau_solve.jl:27,
    so a retry evaluates the stages at t = 0); here the retry keeps t (only matters for time-dependent de).
"""
from __future__ import annotations

import numpy as np

__all__ = ["radau_table", "RadauTable", "RadauStep", "RadauRule", "RadauIntegrator", "makeRadauIntegrator", "solveRadau", "calcJacobian",
           "update_h", "radau_rule_to_stage", "integrate_radau", "rollout_radau"]


def radau_rule_to_stage(n: int) -> int:   # load_table_from_file.jl:2
    return 2 * n - 1


def _radau_nodes(s: int) -> np.ndarray:
    """Right Radau nodes on (0, 1]: roots of d^(s-1)/dx^(s-1) [x^(s-1) (x - 1)^s]."""
    p = np.polynomial.Polynomial([0.0, 1.0]) ** (s - 1) * np.polynomial.Polynomial([-1.0, 1.0]) ** s
    for _ in range(s - 1):
        p = p.deriv()
    c = np.sort(np.real(p.roots()))
    # Newton polish in extended precision is not needed for s <= 5 at double accuracy; two steps tighten the last ulps
    d = p.deriv()
    for _ in range(3):
        c = c - p(c) / d(c)
    c[-1] = 1.0
    return c


class RadauTable:
    """radau_struct.jl:43-62 -- A, c, lambda, T, inv_T, b_hat, b_hat_0 of the s-stage Radau IIA method."""

    def __init__(self, n_rule: int):
        if not (1 <= n_rule <= 6):
            raise ValueError(f"RadauIIA rule {n_rule} not implemented")
        s = radau_rule_to_stage(n_rule)
        c = _radau_nodes(s)
        # collocation: sum_j A_ij c_j^(k-1) = c_i^k / k, k = 1..s
        V = np.vander(c, s, increasing=True)                      # V[j, k-1] = c_j^(k-1)
        rhs = np.stack([c ** k / k for k in range(1, s + 1)], axis=1)
        A = np.linalg.solve(V.T, rhs.T).T
        lam, T = np.linalg.eig(np.linalg.inv(A))
        # order: the real eigenvalue first, then conjugate pairs by increasing |imaginary part|,
        # the positive one first (the order of the reference's files)
        order = sorted(range(s), key=lambda i: (abs(lam[i].imag) > 1e-12, round(abs(lam[i].imag), 9), -lam[i].imag))
        lam, T = lam[order].astype(np.complex128), T[:, order].astype(np.complex128)
        lam[0] = lam[0].real
        T[:, 0] = T[:, 0].real
        Tinv = np.linalg.inv(T)
        b_hat_0 = 1.0 / lam[0].real
        # embedded weights: b_hat_0 [k == 1] + sum_i b_hat_i c_i^(k-1) = 1 / k, k = 1..s
        r = np.array([1.0 / k for k in range(1, s + 1)])
        r[0] -= b_hat_0
        b_hat = np.linalg.solve(V.T, r)
        self.n_stage, self.A, self.c, self.lam, self.T, self.Tinv, self.b_hat, self.b_hat_0 = s, A, c, lam, T, Tinv, b_hat, b_hat_0

    @property
    def b(self):
        return self.A[-1]


_TABLES: dict = {}


def radau_table(n_rule: int) -> RadauTable:
    if n_rule not in _TABLES:
        _TABLES[n_rule] = RadauTable(n_rule)
    return _TABLES[n_rule]


class RadauStep:   # radau_struct.jl:64-81
    def __init__(self, h=1.0e-4, tol_a=1.0e-4, tol_r=1.0e-4, tol_newton=1.0e-16):
        self.h, self.h_inv, self.tol_a, self.tol_r, self.tol_newton = h, 1.0 / h, tol_a, tol_r, tol_newton
        self.h_prev, self.x_err_norm, self.x_err_norm_next = -9999.0, -9999.0, -9999.0
        self.h_max, self.h_min, self.exit_flag = 0.01, 1.0e-8, -9999


class RadauRule:   # radau_struct.jl:83-95
    def __init__(self, NR: int):
        self.s, self.n_increase_cooldown, self.theta, self.theta_prev = 1, 10, -9999.0, -9999.0
        self.k_iter, self.k_iter_max, self.Psi_k, self.max_rule = -9999, 15, 9999.0, NR


class RadauIntegrator:   # radau_struct.jl:108-125
    def __init__(self, de_object, NX: int, tol: float = 1.0e-16, NR: int = 2, NC: int = 6):
        self.de_object, self.NX, self.NC, self.NR = de_object, NX, NC, NR
        self.table = [radau_table(k) for k in range(1, NR + 1)]
        self.step, self.rule = RadauStep(tol_newton=tol), RadauRule(NR)
        n = radau_rule_to_stage(NR)
        self.neg_J = np.zeros((NX, NX))
        self.xx_0 = np.zeros(NX)
        self.X_stage = [np.zeros(NX) for _ in range(n)]
        self.F_X_stage = [np.zeros(NX) for _ in range(n)]
        self.inv_C_stage = [np.zeros((NX, NX), dtype=np.complex128) for _ in range(n)]
        self.n_de_float = 0     # Float64 evaluations of de (stage evaluations)
        self.n_de_chunk = 0     # Dual-NC evaluations of de (Jacobian chunks)
        self.n_rejected = 0     # attempts that did not converge

    def current_table(self) -> RadauTable:
        return self.table[self.rule.s - 1]


def makeRadauIntegrator(de_object, x_or_N, tol: float = 1.0e-16, NR: int = 2, NC: int = 6) -> RadauIntegrator:   # radau_utilities.jl:10-17
    NX = int(x_or_N) if np.isscalar(x_or_N) else len(x_or_N)
    return RadauIntegrator(de_object, NX, tol, NR, NC)


def update_h(rr: RadauIntegrator, h_new: float) -> None:   # adaptive.jl:52-57
    if not (0.0 < h_new < np.inf):
        raise RuntimeError(f"unacceptable h: {h_new}")
    rr.step.h_prev, rr.step.h, rr.step.h_inv = rr.step.h, h_new, 1.0 / h_new


def _chunk_fallback(de_object, x, i0, i1, t):
    """d xx / d x[i0:i1] for objects that only provide de(): complex step when de is complex-safe, else central differences."""
    n = len(x)
    xx0 = np.zeros(n)
    de_object.de(xx0, x, t)
    cols = np.zeros((n, i1 - i0))
    for d, j in enumerate(range(i0, i1)):
        try:
            xc = x.astype(np.complex128)
            xc[j] += 1e-30j
            out = np.zeros(n, dtype=np.complex128)
            de_object.de(out, xc, t)
            cols[:, d] = out.imag / 1e-30
        except (TypeError, ValueError):
            hh = 1e-6 * max(1.0, abs(x[j]))
            xp, xm, fp, fm = x.copy(), x.copy(), np.zeros(n), np.zeros(n)
            xp[j] += hh
            xm[j] -= hh
            de_object.de(fp, xp, t)
            de_object.de(fm, xm, t)
            cols[:, d] = (fp - fm) / (2 * hh)
    return xx0, cols


def calcJacobian(rr: RadauIntegrator, x0: np.ndarray, t: float) -> None:
    """radau_functions.jl:1-14: ceil(NX / NC) seeded evaluations; each fills xx_0 and NC columns of -J."""
    NX, NC = rr.NX, rr.NC
    for i0 in range(0, NX, NC):
        i1 = min(i0 + NC, NX)
        if hasattr(rr.de_object, "de_jacobian_chunk"):
            xx0, cols = rr.de_object.de_jacobian_chunk(x0, i0, i1, t)
        else:
            xx0, cols = _chunk_fallback(rr.de_object, x0, i0, i1, t)
        rr.n_de_chunk += 1
        rr.xx_0[:] = xx0
        rr.neg_J[:, i0:i1] = -cols


def _update_inv_C(rr, table):   # radau_functions.jl:88-99 (getrf + getri)
    eye = np.eye(rr.NX)
    for i in range(table.n_stage):
        rr.inv_C_stage[i] = np.linalg.inv(rr.neg_J.astype(np.complex128) + (rr.step.h_inv * table.lam[i]) * eye)


def _update_FX(rr, table, t):   # radau_functions.jl:62-68
    for i in range(table.n_stage):
        rr.de_object.de(rr.F_X_stage[i], rr.X_stage[i], table.c[i] * rr.step.h + t)
        rr.n_de_float += 1


def _calc_Ew(rr, table, x0, Ew):   # radau_functions.jl:70-86
    residual = 0.0
    s, h = table.n_stage, rr.step.h
    for i in range(s):
        store = rr.X_stage[i] - x0
        for j in range(s):
            store = store + (-h * table.A[i, j]) * rr.F_X_stage[j]
        residual += float(store @ store)
        for j in range(s):
            Ew[j] += (rr.step.h_inv * table.lam[j] * table.Tinv[j, i]) * store
    return residual


def _update_stage_X(rr, table, Ew):   # radau_functions.jl:101-125
    s = table.n_stage
    dZ = [np.zeros(rr.NX, dtype=np.complex128) for _ in range(s)]
    for i in range(s):
        sc = rr.inv_C_stage[i] @ Ew[i]
        for j in range(s):
            dZ[j] += table.T[j, i] * sc
    for i in range(s):
        upd = dZ[i].real
        if 1.0e1 < np.max(np.abs(upd)):
            return True
        rr.X_stage[i] -= upd
    return False


def _update_x_err_norm(rr, table, x0):   # adaptive.jl:1-36
    st, s, h = rr.step, table.n_stage, rr.step.h
    st.x_err_norm = st.x_err_norm_next
    d = (table.b_hat_0 * h) * rr.xx_0
    for k in range(s):
        d = d + ((table.b_hat[k] - table.A[s - 1, k]) * h) * rr.F_X_stage[k]
    x_err = (rr.inv_C_stage[0] @ d).real
    x_final = rr.X_stage[s - 1]
    sc = st.tol_a + np.maximum(np.abs(x_final), np.abs(x0)) * st.tol_r
    st.x_err_norm_next = float(np.sqrt(np.sum((x_err / sc) ** 2) / rr.NX))


def _simple_newton(rr, x0, table, t):   # radau_solve.jl:36-99
    _update_inv_C(rr, table)
    s = table.n_stage
    for i in range(s):
        rr.X_stage[i][:] = x0
    res_vec = [np.inf, np.inf, np.inf]
    for k_iter in range(1, rr.rule.k_iter_max + 1):
        rr.rule.k_iter = k_iter
        Ew = [np.zeros(rr.NX, dtype=np.complex128) for _ in range(s)]
        _update_FX(rr, table, t)
        residual = _calc_Ew(rr, table, x0, Ew)
        if _update_stage_X(rr, table, Ew):
            rr.step.exit_flag = 3
            return
        if residual < rr.step.tol_newton:
            rr.step.exit_flag = 0
            _update_x_err_norm(rr, table, x0)
            return
        if k_iter != 1:
            rr.rule.theta_prev = rr.rule.theta
            rr.rule.theta = np.sqrt(residual)
            rr.rule.Psi_k = np.sqrt(rr.rule.theta_prev * rr.rule.theta)
        else:
            rr.rule.theta = np.sqrt(residual)
            rr.rule.Psi_k = rr.rule.theta
        res_vec = [residual, res_vec[0], res_vec[1]]
        if res_vec[2] < res_vec[1] < res_vec[0]:
            rr.step.exit_flag = 3
            return
    rr.step.exit_flag = 1


def _calc_and_update_h(rr, table):   # adaptive.jl:38-50
    if rr.step.exit_flag == 0:
        two_k = 2 * rr.rule.k_iter_max
        fac = 0.9 * (two_k + 1) / (two_k + rr.rule.k_iter)
        with np.errstate(divide="ignore"):
            h_new = fac * rr.step.h * (1.0 / rr.step.x_err_norm_next) ** (1.0 / (1 + table.n_stage))
    else:
        h_new = rr.step.h * 0.1
    update_h(rr, min(rr.step.h_max, 2 * rr.step.h, h_new))


def _update_rule(rr):   # adaptive.jl:59-85
    if rr.step.exit_flag == 0:
        rr.rule.n_increase_cooldown -= 1
        if rr.rule.n_increase_cooldown < 1 and rr.rule.Psi_k < 0.1:
            rr.rule.s = min(rr.rule.s + 1, rr.rule.max_rule)
    else:
        rr.rule.n_increase_cooldown = 10
        rr.rule.s = max(rr.rule.s - 1, 1)


def solveRadau(rr: RadauIntegrator, x0: np.ndarray, t: float = 0.0):
    """radau_solve.jl:1-34: one accepted step.  Returns (h taken, x_final, t + h)."""
    x0 = np.asarray(x0, dtype=np.float64)
    calcJacobian(rr, x0, t)
    while True:
        table = rr.current_table()
        _simple_newton(rr, x0, table, t)
        _calc_and_update_h(rr, table)
        _update_rule(rr)
        if rr.step.exit_flag == 0:
            return rr.step.h_prev, rr.X_stage[table.n_stage - 1] * 1.0, t + rr.step.h_prev
        rr.n_rejected += 1
        if rr.step.h < rr.step.h_min:
            raise RuntimeError("time step is too small, something is wrong")


def integrate_radau(rr: RadauIntegrator, x0, t_final: float = 1.0, max_steps: int = 1000, after_step=None):
    """integrate_scenario_radau (src/example_integrator.jl:1-41) without the discrete controller: returns (times, states).
    after_step(x) is the reference's principal_value!(mech_scen, x) hook."""
    x = np.array(x0, dtype=np.float64)
    ts, xs, t = [0.0], [x.copy()], 0.0
    for _ in range(max_steps):
        h, x, _ = solveRadau(rr, x, t)
        if after_step is not None:
            after_step(x)
        t += h
        ts.append(t)
        xs.append(x.copy())
        if t_final < t:
            break
    return np.array(ts), np.array(xs)


def rollout_radau(rr: RadauIntegrator, x0, t0: float, t_knots, de=None, max_steps: int = 1000, after_step=None, record=None):
    """x0 at t0 through the knot times t_knots (strictly increasing, gaps and t_knots[0] - t0 at least h_min), one scene: the mirror of
    pfc_radau_rollout.  de (optional) holds one ODE object per interval (t_knots[k-1], t_knots[k]], e.g. one per tau_ext of a control
    sequence; rr.de_object otherwise.  The controller state of rr carries over from earlier steps and into later ones.

    A step toward knot T from t is a knot step of exactly T - t when h >= (T - t) - h_min, so no ordinary step leaves less than h_min to
    the knot.  A rejected knot step retries with a smaller, ordinary h.  Once the knot step is accepted, t = T exactly, x goes to
    x_knot[k], and a controller proposal of at least the knot step's h is raised back to the h the knot step replaced.
    after_step(x) is principal_value!; record (a list) gets (h_taken, t, x, stage evaluations) per accepted step.
    Returns (x_knot [K, NX] with NaN rows for knots not reached within max_steps, x, t, stats = [knots, steps, rejected, evaluations])."""
    t_knots = np.asarray(t_knots, dtype=np.float64).reshape(-1)
    h_min = rr.step.h_min
    if len(t_knots) == 0 or not np.isfinite(t_knots).all() or not (np.diff(t_knots) >= h_min).all() or not (t_knots[0] - t0 >= h_min):
        raise ValueError("knot times must be finite and increase by at least h_min, from t0 on")
    x = np.array(x0, dtype=np.float64)
    t = float(t0)
    x_knot = np.full((len(t_knots), len(x)), np.nan)
    stats = [0, 0, 0, 0]
    k = 0
    while k < len(t_knots) and stats[1] < max_steps:
        if de is not None:
            rr.de_object = de[k]
        T = float(t_knots[k])
        rem = T - t
        h_save = 0.0
        if rr.step.h >= rem - h_min:
            h_save = rr.step.h
            rr.step.h, rr.step.h_inv = rem, 1.0 / rem
        n_eval, n_rej = rr.n_de_float, rr.n_rejected
        h_taken, x, _ = solveRadau(rr, x, t)
        if after_step is not None:
            after_step(x)
        stats[1] += 1
        stats[2] += rr.n_rejected - n_rej
        stats[3] += rr.n_de_float - n_eval
        if h_save > 0.0 and h_taken == rem:
            t = T
            x_knot[k] = x
            k += 1
            stats[0] += 1
            if rr.step.h >= h_taken and h_save > rr.step.h:
                rr.step.h, rr.step.h_inv = h_save, 1.0 / h_save
        else:
            t = t + h_taken
        if record is not None:
            record.append((h_taken, t, x.copy(), rr.n_de_float - n_eval))
    return x_knot, x, t, stats
