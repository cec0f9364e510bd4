// pfc_radau_step.cuh -- the per-environment arithmetic of the reference's adaptive Radau IIA step (src/radau: radau_solve.jl, radau_functions.jl,
// adaptive.jl; restated one scene at a time in pfc_b200/radau.py, which is the specification followed here line by line).
//
// Every function computes ONE output element (or the scalar decisions of one environment) in a fixed order: the device kernels
// (pfc_radau.cu) deal the elements to threads, a host build (-DPFC_HOST_CHECK, tests/test_radau_step_on_host.py) loops over them.  Nothing
// here depends on which thread, CTA or batch computes an element, so the step of an environment is the same bits whatever the batch.
//
// Layouts (one environment): x0[n_x]; stage vectors X / F / store [stage][n_x]; complex vectors as separate re / im arrays [stage][n_x];
// invC [n_x][n_x] complex, row-major, interleaved (re, im) -- what launch_radau_inv_c writes.
#pragma once

#ifndef PFC_HOST_CHECK
#include <cuda_runtime.h>
#endif
#include <math.h>

#include "pfc_radau_tables.h"

#ifdef PFC_HOST_CHECK
#define PFC_RHD inline
#else
#define PFC_RHD __host__ __device__ __forceinline__
#endif

namespace pfc {

// the reference's constants (RadauStep / RadauRule, radau_struct.jl:64-95)
constexpr double kRadauTolA = 1.0e-4, kRadauTolR = 1.0e-4, kRadauHMin = 1.0e-8;
constexpr int kRadauKIterMax = 15;

// controller state of one environment; Psi persists across attempts and steps, the rest belongs to the current attempt
struct RadauEnv {
    double h, Psi, theta, res[3], err_norm, t;
    int rule, cooldown, k_iter, exit_flag;   // exit_flag: 0 converged, 1 iteration limit, 3 diverged / residuals growing (radau_solve.jl)
    int pending, active, n_rejected, n_evals;
};

PFC_RHD void radau_env_reset(RadauEnv& e, double h0) {   // RadauStep / RadauRule initial state
    e.h = h0; e.Psi = 9999.0; e.theta = -9999.0; e.res[0] = e.res[1] = e.res[2] = INFINITY; e.err_norm = -9999.0; e.t = 0.0;
    e.rule = 1; e.cooldown = 10; e.k_iter = 0; e.exit_flag = 1; e.pending = 0; e.active = 0; e.n_rejected = 0; e.n_evals = 0;
}

PFC_RHD void radau_attempt_begin(RadauEnv& e) {   // simple_newton! entry: res_vec = [Inf, Inf, Inf]
    e.k_iter = 0; e.exit_flag = 1; e.active = 1; e.res[0] = e.res[1] = e.res[2] = INFINITY;
}

// calcEw! (radau.py _calc_Ew): store_i[n] = X_i[n] - x0[n] + sum_j (-h A_ij) F_j[n]
PFC_RHD double radau_store(const RadauTableData& T, double h, int i, int n, int nx, const double* x0, const double* X, const double* F) {
    double v = X[i * nx + n] - x0[n];
    for (int j = 0; j < T.s; ++j) v = v + (-h * T.A[i][j]) * F[j * nx + n];
    return v;
}

// Ew_j[n] = sum_i (h^-1 lambda_j Tinv_ji) store_i[n]
PFC_RHD void radau_ew(const RadauTableData& T, double h_inv, int j, int n, int nx, const double* store, double* re, double* im) {
    const double a = h_inv * T.lam_re[j], b = h_inv * T.lam_im[j];
    double r = 0.0, q = 0.0;
    for (int i = 0; i < T.s; ++i) {
        const double cr = a * T.Tinv_re[j][i] - b * T.Tinv_im[j][i], ci = a * T.Tinv_im[j][i] + b * T.Tinv_re[j][i];
        const double st = store[i * nx + n];
        r = r + cr * st;
        q = q + ci * st;
    }
    *re = r; *im = q;
}

// row r of invC v (complex), summed in column order
PFC_RHD void radau_matvec_row(const double* invC, int nx, int r, const double* v_re, const double* v_im, double* re, double* im) {
    const double* row = invC + 2 * (long long)r * nx;
    double a = 0.0, b = 0.0;
    for (int k = 0; k < nx; ++k) {
        const double mr = row[2 * k], mi = row[2 * k + 1];
        a = a + (mr * v_re[k] - mi * v_im[k]);
        b = b + (mr * v_im[k] + mi * v_re[k]);
    }
    *re = a; *im = b;
}

// updateStageX! (radau.py _update_stage_X): the update of stage j is Re(sum_i T_ji sc_i[n])
PFC_RHD double radau_update(const RadauTableData& T, int j, int n, int nx, const double* sc_re, const double* sc_im) {
    double v = 0.0;
    for (int i = 0; i < T.s; ++i) v = v + (T.T_re[j][i] * sc_re[i * nx + n] - T.T_im[j][i] * sc_im[i * nx + n]);
    return v;
}

// update_x_err_norm! (adaptive.jl:1-36): d[n] = b_hat_0 h xx_0[n] + sum_k (b_hat_k - A_{s-1,k}) h F_k[n] ...
PFC_RHD double radau_err_d(const RadauTableData& T, double h, int n, int nx, const double* xx0, const double* F) {
    double v = (T.b_hat_0 * h) * xx0[n];
    for (int k = 0; k < T.s; ++k) v = v + ((T.b_hat[k] - T.A[T.s - 1][k]) * h) * F[k * nx + n];
    return v;
}
// ... and the squared scaled error of row r: (Re(invC_0 d)[r] / (tol_a + max(|x_final[r]|, |x0[r]|) tol_r))^2
PFC_RHD double radau_err_term(const double* invC0, int nx, int r, const double* d, double x_final_r, double x0_r) {
    const double* row = invC0 + 2 * (long long)r * nx;
    double a = 0.0;
    for (int k = 0; k < nx; ++k) a = a + row[2 * k] * d[k];
    const double sc = kRadauTolA + fmax(fabs(x_final_r), fabs(x0_r)) * kRadauTolR;
    const double q = a / sc;
    return q * q;
}

enum { kRadauIterate = 0, kRadauConverged = 1, kRadauDone = 2 };

// simple_newton! after the stage update of iteration k (radau.py _simple_newton): diverged = some stage's update exceeded 10.  Returns
// kRadauConverged (the caller then computes the error norm), kRadauDone (exit_flag 3 or 1) or kRadauIterate.
PFC_RHD int radau_newton_decide(RadauEnv& e, int k, double residual, bool diverged, double tol_newton) {
    e.k_iter = k;
    if (diverged) { e.exit_flag = 3; return kRadauDone; }
    if (residual < tol_newton) { e.exit_flag = 0; return kRadauConverged; }
    if (k != 1) {
        const double theta_prev = e.theta;
        e.theta = sqrt(residual);
        e.Psi = sqrt(theta_prev * e.theta);
    } else {
        e.theta = sqrt(residual);
        e.Psi = e.theta;
    }
    e.res[2] = e.res[1]; e.res[1] = e.res[0]; e.res[0] = residual;
    if (e.res[2] < e.res[1] && e.res[1] < e.res[0]) { e.exit_flag = 3; return kRadauDone; }
    if (k == kRadauKIterMax) { e.exit_flag = 1; return kRadauDone; }
    return kRadauIterate;
}

enum { kRadauAccepted = 0, kRadauRetry = 1, kRadauBadH = -1, kRadauHTooSmall = -2 };

// calc_and_update_h! + update_rule! (adaptive.jl:38-85) after an attempt on n_stage stages; *h_taken = the step's h on acceptance.
PFC_RHD int radau_control(RadauEnv& e, int max_rule, double h_max, double* h_taken) {
    const int s = 2 * e.rule - 1;
    double h_new;
    if (e.exit_flag == 0) {
        const int two_k = 2 * kRadauKIterMax;
        const double fac = 0.9 * (two_k + 1) / (two_k + e.k_iter);
        h_new = fac * e.h * pow(1.0 / e.err_norm, 1.0 / (1 + s));
    } else {
        h_new = e.h * 0.1;
    }
    double m = h_max;                 // Python's min(h_max, 2 h, h_new): the first of the smallest, a NaN h_new is never taken
    if (2 * e.h < m) m = 2 * e.h;
    if (h_new < m) m = h_new;
    if (!(0.0 < m && m < INFINITY)) return kRadauBadH;
    const double h_prev = e.h;
    e.h = m;
    if (e.exit_flag == 0) {
        e.cooldown -= 1;
        if (e.cooldown < 1 && e.Psi < 0.1) e.rule = e.rule + 1 < max_rule ? e.rule + 1 : max_rule;
        *h_taken = h_prev;
        return kRadauAccepted;
    }
    e.cooldown = 10;
    e.rule = e.rule - 1 > 1 ? e.rule - 1 : 1;
    return e.h < kRadauHMin ? kRadauHTooSmall : kRadauRetry;
}

// Roll-outs through knot times (radau.py rollout_radau).  Before a step toward knot T from t: if h would end within h_min of T (or past
// it), the step is a knot step of exactly T - t, so no ordinary step leaves a remainder below h_min.  Returns h_save, the h the controller
// had (0 for an ordinary step).
PFC_RHD double radau_knot_begin(RadauEnv& e, double t, double T) {
    const double rem = T - t;
    if (e.h >= rem - kRadauHMin) {
        const double h_save = e.h;
        e.h = rem;
        return h_save;
    }
    return 0.0;
}

// After the accepted step of h_taken from t: true when it was the knot step (a rejected knot step is retried with a smaller, ordinary h).
// *t_new is then T exactly, and a proposal of at least h_taken is raised back to h_save, so a short knot step does not shrink the next
// ordinary one.  Otherwise *t_new = t + h_taken, as after any step.
PFC_RHD bool radau_knot_end(RadauEnv& e, double t, double T, double h_taken, double h_save, double* t_new) {
    if (h_save > 0.0 && h_taken == T - t) {
        *t_new = T;
        if (e.h >= h_taken && h_save > e.h) e.h = h_save;
        return true;
    }
    *t_new = t + h_taken;
    return false;
}

}  // namespace pfc
