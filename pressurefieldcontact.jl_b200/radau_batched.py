"""radau_batched.py -- the reference's adaptive Radau IIA integrator (src/radau, mirrored one scene at a time in radau.py)
advanced for a whole BATCH of independent environments with every array resident on the GPU (SURVEY.md section 8f rank 4:
"batched Radau step: stage evals already batched by the kernels; add batched complex LU and the Newton / step controller").

What runs where
  * stage evaluations F(X_stage): pfc_calcxd_f64_device  -- calcXd! for n_env x n_stage states in ONE launch sequence
  * Jacobian: one call of pfc_calcxd_jacobian_device -- all ceil(NX / 6) Dual-6 chunks of all environments (calcJacobian!)
  * (h^-1 lambda_i I - J)^-1 for every environment and stage: pfc_radau_inv_c_device, one CTA per matrix, Gauss-Jordan with partial
    pivoting in shared memory (the reference calls LAPACK getrf / getri here, radau_functions.jl:88-99; batched cuSOLVER through
    torch.linalg.inv took 17.6 ms for 4096 48 x 48 matrices)
  * the Newton iteration, error estimate, step-size and order control: per-environment state vectors and masks, torch ops on the
    library's stream (radau_solve.jl:36-99, adaptive.jl) -- every environment follows exactly the decision sequence the
    single-scene integrator would take for it; environments that fail a step retry with their own smaller h while the others wait.

DeviceBatchedRadau is the same integrator behind the library's C ABI (pfc_radau_init / pfc_radau_step_device): the Newton iteration,
error estimate and step-size / order control run in CUDA kernels, and the host only reads how many stage states are still active once per
Newton iteration.  It has BatchedRadau's interface (step, integrate, t) so that the tests and scripts/run_batched_radau.py drive both,
and rollout(): every environment through shared knot times with a piecewise-constant tau_ext (pfc_radau_rollout_device).

BatchedRadau is caller-side code (the reference's is Julia); it exists to drive the device path end to end the way
integrate_scenario_radau does and to measure batched roll-out throughput.
"""
from __future__ import annotations

import numpy as np
import torch

from . import radau as R
from . import scenario as S

__all__ = ["BatchedRadau", "DeviceBatchedRadau"]


class BatchedRadau:
    def __init__(self, m, n_env: int, device_index: int = 0, NR: int = 2, tol_newton: float = 1.0e-16, h0: float = 1.0e-4, h_max: float = 0.01):
        if not getattr(m, "device_dynamics", False):
            raise RuntimeError("BatchedRadau needs a CUDA backend with pfc_set_dynamics (floating bodies with InertiaProperties)")
        self.m, self.ctx, self.E, self.NX, self.NR = m, m.backend, n_env, S.num_x(m), NR
        self.dev = torch.device("cuda", device_index)
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)
        f64, c128 = torch.float64, torch.complex128
        self.tab = []
        for k in range(1, NR + 1):
            t = R.radau_table(k)
            self.tab.append(dict(s=t.n_stage, A=torch.tensor(t.A, dtype=f64, device=self.dev), lam=torch.tensor(t.lam, dtype=c128, device=self.dev),
                                 T=torch.tensor(t.T, dtype=c128, device=self.dev), Tinv=torch.tensor(t.Tinv, dtype=c128, device=self.dev),
                                 b_hat=torch.tensor(t.b_hat, dtype=f64, device=self.dev), b_hat_0=float(t.b_hat_0)))
        with torch.cuda.stream(self.stream):
            E = n_env
            self.h = torch.full((E,), h0, dtype=f64, device=self.dev)
            self.rule = torch.ones(E, dtype=torch.int64, device=self.dev)
            self.cooldown = torch.full((E,), 10, dtype=torch.int64, device=self.dev)
            self.Psi = torch.full((E,), 9999.0, dtype=f64, device=self.dev)
            self.t = torch.zeros(E, dtype=f64, device=self.dev)
            self.eye = torch.eye(self.NX, dtype=c128, device=self.dev)
            self.info = torch.zeros(1, dtype=torch.int32, device=self.dev)   # bit 0: a pivot vanished in some inversion
        self.tol_newton, self.tol_a, self.tol_r, self.h_max, self.h_min, self.k_iter_max = tol_newton, 1.0e-4, 1.0e-4, h_max, 1.0e-8, 15
        self.n_ins = self.ctx.n_ins
        self.mrp_cols = torch.tensor([b.q0 for b in m.bodies if isinstance(b.joint, S.SPQuatFloating)], dtype=torch.int64, device=self.dev)
        self.n_calcxd_states = 0     # states pushed through pfc_calcxd_f64_device
        self.n_chunk_states = 0      # (state, chunk) pairs pushed through pfc_calcxd_jacobian_device
        self.n_attempts = 0

    # ---- device entry points ------------------------------------------------------------------------------------------
    def _calcxd(self, X: torch.Tensor) -> torch.Tensor:
        n = X.shape[0]
        X = X.contiguous()
        out = torch.zeros_like(X)
        npairs = torch.empty((n, self.n_ins), dtype=torch.int64, device=self.dev)
        flags = torch.empty((n, self.n_ins), dtype=torch.int32, device=self.dev)
        self.ctx.calcxd_f64_device(n, X.data_ptr(), None, out.data_ptr(), npairs.data_ptr(), flags.data_ptr())
        self.n_calcxd_states += n
        self._last_flags = flags
        return out

    def _jacobian(self, x0: torch.Tensor):
        """calcJacobian! (radau_functions.jl:1-14) for every environment: (xx_0 [E, NX], -J [E, NX, NX])."""
        E, NX = x0.shape
        x0 = x0.contiguous()
        jac = torch.empty((E, NX, NX), dtype=torch.float64, device=self.dev)
        xx0 = torch.empty((E, NX), dtype=torch.float64, device=self.dev)
        npairs = torch.empty((E, self.n_ins), dtype=torch.int64, device=self.dev)
        flags = torch.empty((E, self.n_ins), dtype=torch.int32, device=self.dev)
        # one call: Float64 kinematics + broad phase once, every seed chunk side by side in the Dual kernels (pfc_calcxd_jacobian_device)
        self.ctx.calcxd_jacobian_device(E, x0.data_ptr(), None, jac.data_ptr(), xx0.data_ptr(), npairs.data_ptr(), flags.data_ptr())
        self.n_chunk_states += E * ((NX + 5) // 6)
        return xx0, jac.neg_()

    # ---- one Newton attempt for the environments idx, all on rule `rule` -----------------------------------------------------
    def _newton(self, rule: int, idx: torch.Tensor, x0: torch.Tensor, xx_0: torch.Tensor, negJ: torch.Tensor):
        tab = self.tab[rule - 1]
        s, n, NX = tab["s"], idx.numel(), self.NX
        h = self.h[idx]
        hinv = 1.0 / h
        # updateInvC!: (h^-1 lambda_i I - J)^-1 for every environment of the group and every stage, one CTA per matrix (pfc_radau.cu)
        idx32 = idx.to(torch.int32).contiguous()
        invC = []
        for i in range(s):
            shift = torch.view_as_real((hinv * tab["lam"][i]).to(torch.complex128)).contiguous()
            out = torch.empty((n, NX, NX), dtype=torch.complex128, device=self.dev)
            self.ctx.radau_inv_c_device(n, NX, negJ.data_ptr(), shift.data_ptr(), idx32.data_ptr(), out.data_ptr(), self.info.data_ptr())
            invC.append(out)
        x0s = x0[idx]
        X = [x0s.clone() for _ in range(s)]
        active = torch.ones(n, dtype=torch.bool, device=self.dev)
        exit_flag = torch.full((n,), 1, dtype=torch.int64, device=self.dev)          # 1 = iteration limit unless decided earlier
        k_rec = torch.full((n,), self.k_iter_max, dtype=torch.int64, device=self.dev)
        err_norm = torch.full((n,), float("inf"), dtype=torch.float64, device=self.dev)
        theta = torch.zeros(n, dtype=torch.float64, device=self.dev)
        Psi = self.Psi[idx].clone()
        res_hist = torch.full((n, 3), float("inf"), dtype=torch.float64, device=self.dev)
        for k_iter in range(1, self.k_iter_max + 1):
            F = self._calcxd(torch.cat(X, dim=0)).view(s, n, NX)
            residual = torch.zeros(n, dtype=torch.float64, device=self.dev)
            Ew = [torch.zeros((n, NX), dtype=torch.complex128, device=self.dev) for _ in range(s)]
            for i in range(s):
                store = X[i] - x0s
                for j in range(s):
                    store = store + (-h * tab["A"][i, j])[:, None] * F[j]
                residual = residual + (store * store).sum(dim=1)
                for j in range(s):
                    Ew[j] = Ew[j] + (hinv * tab["lam"][j] * tab["Tinv"][j, i])[:, None] * store
            dZ = [torch.zeros((n, NX), dtype=torch.complex128, device=self.dev) for _ in range(s)]
            for i in range(s):
                sc = torch.bmm(invC[i], Ew[i].unsqueeze(2)).squeeze(2)
                for j in range(s):
                    dZ[j] = dZ[j] + tab["T"][j, i] * sc
            upd = [dZ[i].real for i in range(s)]
            # updateStageX!: stages are updated in order and the step is abandoned at the first stage whose update exceeds 10
            diverged = torch.zeros(n, dtype=torch.bool, device=self.dev)
            for i in range(s):
                diverged = diverged | (upd[i].abs().amax(dim=1) > 1.0e1)
                ok = active & ~diverged
                X[i] = torch.where(ok[:, None], X[i] - upd[i], X[i])
            newly = active & diverged
            exit_flag = torch.where(newly, torch.full_like(exit_flag, 3), exit_flag)
            active = active & ~diverged
            conv = active & (residual < self.tol_newton)
            if bool(conv.any()):
                # update_x_err_norm! (adaptive.jl:1-36) with this iteration's F_X_stage
                d = (tab["b_hat_0"] * h)[:, None] * xx_0[idx]
                for k in range(s):
                    d = d + ((tab["b_hat"][k] - tab["A"][s - 1, k]) * h)[:, None] * F[k]
                x_err = torch.bmm(invC[0], d.to(torch.complex128).unsqueeze(2)).squeeze(2).real
                sc_k = self.tol_a + torch.maximum(X[s - 1].abs(), x0s.abs()) * self.tol_r
                e = torch.sqrt(((x_err / sc_k) ** 2).sum(dim=1) / NX)
                err_norm = torch.where(conv, e, err_norm)
                exit_flag = torch.where(conv, torch.zeros_like(exit_flag), exit_flag)
                k_rec = torch.where(conv, torch.full_like(k_rec, k_iter), k_rec)
                active = active & ~conv
            root = torch.sqrt(residual)
            if k_iter != 1:
                Psi = torch.where(active, torch.sqrt(theta * root), Psi)
            else:
                Psi = torch.where(active, root, Psi)
            theta = torch.where(active, root, theta)
            res_hist = torch.where(active[:, None], torch.stack([residual, res_hist[:, 0], res_hist[:, 1]], dim=1), res_hist)
            growing = active & (res_hist[:, 2] < res_hist[:, 1]) & (res_hist[:, 1] < res_hist[:, 0])
            exit_flag = torch.where(growing, torch.full_like(exit_flag, 3), exit_flag)
            active = active & ~growing
            if not bool(active.any()):
                break
        return X[s - 1], exit_flag, k_rec, err_norm, Psi

    # ---- one accepted step for every environment ---------------------------------------------------------------------------
    def step(self, x0: torch.Tensor):
        """solveRadau (radau_solve.jl:1-34) for the batch: returns (x_final [E, NX], h_taken [E]); self.t advances by h_taken."""
        with torch.cuda.stream(self.stream):
            E = self.E
            xx_0, negJ = self._jacobian(x0)
            x_final = x0.clone()
            h_taken = torch.zeros(E, dtype=torch.float64, device=self.dev)
            pending = torch.ones(E, dtype=torch.bool, device=self.dev)
            while bool(pending.any()):
                self.n_attempts += 1
                for rule in range(1, self.NR + 1):
                    idx = torch.nonzero(pending & (self.rule == rule)).squeeze(1)
                    if idx.numel() == 0:
                        continue
                    s = self.tab[rule - 1]["s"]
                    xf, exit_flag, k_rec, err_norm, Psi = self._newton(rule, idx, x0, xx_0, negJ)
                    ok = exit_flag == 0
                    h = self.h[idx]
                    # calc_and_update_h! (adaptive.jl:38-57)
                    fac = 0.9 * (2 * self.k_iter_max + 1) / (2 * self.k_iter_max + k_rec.to(torch.float64))
                    h_good = fac * h * (1.0 / err_norm) ** (1.0 / (1 + s))
                    h_new = torch.where(ok, h_good, h * 0.1)
                    h_new = torch.minimum(torch.minimum(torch.full_like(h, self.h_max), 2 * h), h_new)
                    if not bool(((h_new > 0) & torch.isfinite(h_new)).all()):
                        raise RuntimeError("unacceptable h")
                    self.h[idx] = h_new
                    # update_rule! (adaptive.jl:59-85)
                    cd = torch.where(ok, self.cooldown[idx] - 1, torch.full_like(k_rec, 10))
                    r = self.rule[idx]
                    up = ok & (cd < 1) & (Psi < 0.1)
                    r_new = torch.where(ok, torch.where(up, torch.clamp(r + 1, max=self.NR), r), torch.clamp(r - 1, min=1))
                    self.cooldown[idx], self.rule[idx], self.Psi[idx] = cd, r_new, Psi
                    acc = idx[ok]
                    x_final[acc] = xf[ok]
                    h_taken[acc] = h[ok]
                    pending[acc] = False
                    if bool((~ok & (h_new < self.h_min)).any()):
                        raise RuntimeError("time step is too small, something is wrong")
            # principal_value!: MRPs with |p|^2 > 1 move to the shadow set
            for q0 in self.mrp_cols.tolist():
                p = x_final[:, q0:q0 + 3]
                n2 = (p * p).sum(dim=1, keepdim=True)
                x_final[:, q0:q0 + 3] = torch.where(n2 > 1.0, -p / n2, p)
            self.t = self.t + h_taken
            return x_final, h_taken

    def integrate(self, x0, n_steps: int):
        """n_steps accepted steps for every environment; returns (times [n_steps + 1, E], states [n_steps + 1, E, NX]) on the host."""
        with torch.cuda.stream(self.stream):     # every copy is ordered on the library's stream
            x = torch.as_tensor(np.asarray(x0, dtype=np.float64)).to(self.dev).reshape(self.E, self.NX)
            ts, xs = [self.t.cpu().numpy().copy()], [x.cpu().numpy().copy()]
            for _ in range(n_steps):
                x, _ = self.step(x)
                ts.append(self.t.cpu().numpy().copy())
                xs.append(x.cpu().numpy().copy())
        return np.array(ts), np.array(xs)


class DeviceBatchedRadau:
    """The batched adaptive Radau step of pfc_radau_step_device: same step(x0) -> (x_final, h_taken) / integrate(x0, n_steps) / t as
    BatchedRadau, over torch tensors on the library's stream.  tau_ext [E, nv] (or None) is held constant over each step."""

    def __init__(self, m, n_env: int, device_index: int = 0, NR: int = 2, tol_newton: float = 1.0e-16, h0: float = 1.0e-4, h_max: float = 0.01):
        if not getattr(m, "device_dynamics", False):
            raise RuntimeError("DeviceBatchedRadau needs a CUDA backend with pfc_set_dynamics (floating bodies with InertiaProperties)")
        self.m, self.ctx, self.E, self.NX, self.NR = m, m.backend, n_env, S.num_x(m), NR
        self.dev = torch.device("cuda", device_index)
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)
        self.ctx.radau_init(n_env, NR, h0, h_max, tol_newton)
        with torch.cuda.stream(self.stream):
            self.t = torch.zeros(n_env, dtype=torch.float64, device=self.dev)
            self.stats = torch.zeros((n_env, 4), dtype=torch.int32, device=self.dev)

    def step(self, x0: torch.Tensor, tau_ext: torch.Tensor = None):
        """solveRadau for the batch: returns (x_final [E, NX], h_taken [E]); self.t advances by h_taken; self.stats [E, 4] as pfc_radau_step."""
        with torch.cuda.stream(self.stream):
            x = x0.to(device=self.dev, dtype=torch.float64).contiguous().clone()
            tau = None if tau_ext is None else tau_ext.to(device=self.dev, dtype=torch.float64).contiguous()
            t = self.t.clone()
            h_taken = torch.zeros(self.E, dtype=torch.float64, device=self.dev)
            self.ctx.radau_step_device(self.E, x.data_ptr(), None if tau is None else tau.data_ptr(), t.data_ptr(), h_taken.data_ptr(),
                                       self.stats.data_ptr())
            self.t = t
            return x, h_taken

    def integrate(self, x0, n_steps: int, tau_ext=None):
        """n_steps accepted steps for every environment; returns (times [n_steps + 1, E], states [n_steps + 1, E, NX]) on the host."""
        with torch.cuda.stream(self.stream):
            x = torch.as_tensor(np.asarray(x0, dtype=np.float64)).to(self.dev).reshape(self.E, self.NX)
            tau = None if tau_ext is None else torch.as_tensor(np.asarray(tau_ext, dtype=np.float64)).to(self.dev)
            ts, xs = [self.t.cpu().numpy().copy()], [x.cpu().numpy().copy()]
            for _ in range(n_steps):
                x, _ = self.step(x, tau)
                ts.append(self.t.cpu().numpy().copy())
                xs.append(x.cpu().numpy().copy())
        return np.array(ts), np.array(xs)

    def rollout(self, x0, t_knots, tau=None, max_steps: int = 1000):
        """pfc_radau_rollout_device: every environment from x0 [E, NX] at self.t through the absolute knot times t_knots [K], with tau
        [K, E, nv] (or None) acting on (t_knots[k-1], t_knots[k]].  Returns (x_knot [K, E, NX] with NaN rows for knots an environment did
        not reach within max_steps, stats [E, 4] = knots reached, accepted steps, rejected attempts, stage evaluations), torch tensors on
        the device; self.t advances to where each environment stopped."""
        t_knots = np.asarray(t_knots, dtype=np.float64).reshape(-1)
        with torch.cuda.stream(self.stream):
            x = torch.as_tensor(x0).to(device=self.dev, dtype=torch.float64).reshape(self.E, self.NX).contiguous().clone()
            tau_t = None if tau is None else torch.as_tensor(tau).to(device=self.dev, dtype=torch.float64).contiguous()
            t = self.t.clone()
            x_knot = torch.empty((len(t_knots), self.E, self.NX), dtype=torch.float64, device=self.dev)
            stats = torch.zeros((self.E, 4), dtype=torch.int32, device=self.dev)
            self.ctx.radau_rollout_device(self.E, t_knots, max_steps, x.data_ptr(), None if tau_t is None else tau_t.data_ptr(), t.data_ptr(),
                                          x_knot.data_ptr(), stats.data_ptr())
            self.t = t
            return x_knot, stats
