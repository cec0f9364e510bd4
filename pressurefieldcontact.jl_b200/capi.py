"""ctypes binding of libpfc_b200.so -- the same symbols a Julia ``ccall`` shim binds (INTEGRATION.md).

There is no CPU fallback: if the CUDA library is missing this module raises at load time.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpfc_b200.so")
_LIB = None

_d = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32 = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i64 = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_vp = C.c_void_p

# every symbol include/pfc.h declares
SYMBOLS = [
    "pfc_create", "pfc_destroy", "pfc_add_mesh", "pfc_add_instruction", "pfc_finalize", "pfc_set_contact_params", "pfc_eval_f64", "pfc_eval_f64_device",
    "pfc_eval_dual6", "pfc_set_debug", "pfc_get_pairs", "pfc_get_traction", "pfc_set_shard", "pfc_eval_sharded_begin", "pfc_eval_sharded_partials", "pfc_eval_sharded_step", "pfc_sync", "pfc_stream",
    "pfc_set_bodies", "pfc_eval_state_f64", "pfc_eval_state_f64_device", "pfc_get_boundary", "pfc_set_dynamics", "pfc_calcxd_f64", "pfc_calcxd_f64_device", "pfc_calcxd_dual6", "pfc_calcxd_dual6_device", "pfc_calcxd_jacobian", "pfc_calcxd_jacobian_device", "pfc_radau_inv_c_device", "pfc_radau_init", "pfc_radau_step", "pfc_radau_step_device", "pfc_radau_rollout", "pfc_radau_rollout_device", "pfc_radau_step_info", "pfc_refit_mesh", "pfc_launch_count", "pfc_counters", "pfc_measure_fp64_peak", "pfc_set_timing", "pfc_kernel_times", "pfc_last_error", "pfc_version",
    "pfc_comm_unique_id", "pfc_comm_init_rank", "pfc_eval_sharded_f64_device", "pfc_group_create", "pfc_group_destroy", "pfc_group_size", "pfc_group_ctx",
    "pfc_group_add_mesh", "pfc_group_add_instruction", "pfc_group_finalize", "pfc_group_eval_f64",
]


class PfcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pfc error {code}: {msg}")
        self.code = code


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback for the contact-wrench path)")
        L = C.CDLL(LIB_PATH)
        L.pfc_create.argtypes = [C.c_int, C.POINTER(_vp)]
        L.pfc_destroy.argtypes = [_vp]
        L.pfc_add_mesh.argtypes = [_vp, C.c_int, C.c_int64, _d, C.c_int64, _i32, _vp, C.c_double, C.c_int64, _d, _d, _d, _i32, _i32, _i32,
                                   C.POINTER(C.c_int)]
        L.pfc_add_instruction.argtypes = [_vp, C.c_int, C.c_int, C.c_double, C.c_int, _d, C.c_int, C.POINTER(C.c_int)]
        L.pfc_finalize.argtypes = [_vp, C.c_int64]
        L.pfc_set_contact_params.argtypes = [_vp, C.c_int64, _vp]
        L.pfc_eval_f64.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_eval_f64_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_eval_dual6.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_set_debug.argtypes = [_vp, C.c_int]
        L.pfc_get_pairs.argtypes = [_vp, C.c_int64, C.c_int, _vp, C.c_int64, C.POINTER(C.c_int64)]
        L.pfc_get_traction.argtypes = [_vp, C.c_int64, C.c_int, _vp, C.c_int64, C.POINTER(C.c_int64)]
        L.pfc_set_shard.argtypes = [_vp, C.c_int, C.c_int]
        L.pfc_eval_sharded_begin.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_eval_sharded_partials.argtypes = [_vp, C.POINTER(_vp), C.POINTER(C.c_int64)]
        L.pfc_eval_sharded_step.argtypes = [_vp, C.POINTER(C.c_int)]
        L.pfc_set_bodies.argtypes = [_vp, C.c_int, _i32, _i32, _i32, _vp, _i32, C.c_int, C.c_int]
        L.pfc_eval_state_f64.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_eval_state_f64_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_get_boundary.argtypes = [_vp, C.c_int64, _vp, _vp, _vp]
        L.pfc_set_dynamics.argtypes = [_vp, C.c_int, _d, _d]
        L.pfc_calcxd_f64.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_calcxd_f64_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_calcxd_dual6.argtypes = [_vp, C.c_int64, _vp, _vp, C.c_int, _vp, _vp, _vp]
        L.pfc_calcxd_dual6_device.argtypes = [_vp, C.c_int64, _vp, _vp, C.c_int, _vp, _vp, _vp]
        L.pfc_calcxd_jacobian.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_calcxd_jacobian_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_refit_mesh.argtypes = [_vp, C.c_int, C.c_int64, _d]
        L.pfc_radau_inv_c_device.argtypes = [_vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, _vp]
        L.pfc_radau_init.argtypes = [_vp, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double]
        L.pfc_radau_step.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_radau_step_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_radau_rollout.argtypes = [_vp, C.c_int64, C.c_int, _d, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_radau_rollout_device.argtypes = [_vp, C.c_int64, C.c_int, _d, C.c_int64, _vp, _vp, _vp, _vp, _vp]
        L.pfc_radau_step_info.argtypes = [_vp, _vp, _vp]
        L.pfc_comm_unique_id.argtypes = [_vp]
        L.pfc_comm_init_rank.argtypes = [_vp, _vp, C.c_int, C.c_int]
        L.pfc_eval_sharded_f64_device.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_group_create.argtypes = [C.c_int, _i32, C.POINTER(_vp)]
        L.pfc_group_destroy.argtypes = [_vp]
        L.pfc_group_size.argtypes = [_vp]
        L.pfc_group_ctx.argtypes = [_vp, C.c_int]
        L.pfc_group_ctx.restype = _vp
        L.pfc_group_add_mesh.argtypes = [_vp, C.c_int, C.c_int64, _d, C.c_int64, _i32, _vp, C.c_double, C.c_int64, _d, _d, _d, _i32, _i32, _i32,
                                         C.POINTER(C.c_int)]
        L.pfc_group_add_instruction.argtypes = [_vp, C.c_int, C.c_int, C.c_double, C.c_int, _d, C.c_int, C.POINTER(C.c_int)]
        L.pfc_group_finalize.argtypes = [_vp, C.c_int64]
        L.pfc_group_eval_f64.argtypes = [_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
        L.pfc_sync.argtypes = [_vp]
        L.pfc_stream.argtypes = [_vp]
        L.pfc_stream.restype = _vp
        L.pfc_launch_count.argtypes = [_vp]
        L.pfc_launch_count.restype = C.c_int64
        L.pfc_counters.argtypes = [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.pfc_measure_fp64_peak.argtypes = [_vp, C.POINTER(C.c_double)]
        L.pfc_set_timing.argtypes = [_vp, C.c_int]
        L.pfc_kernel_times.argtypes = [_vp, C.POINTER(C.c_double), C.c_int]
        L.pfc_last_error.restype = C.c_char_p
        L.pfc_version.restype = C.c_char_p
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise PfcError(rc, lib().pfc_last_error().decode())


def _a(x, dt=np.float64):
    return np.ascontiguousarray(x, dtype=dt)


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


class Context:
    """One scene on one GPU.  Same protocol as the scenario backends: add_mesh, add_instruction,
    finalize, eval_f64, eval_dual6, get_pairs, get_traction."""

    name = "cuda"

    def __init__(self, device: int = 0):
        self._h = _vp()
        _check(lib().pfc_create(device, C.byref(self._h)))
        self.device = device
        self.n_ins = 0
        self.n_bristle = 0

    def close(self):
        if self._h:
            lib().pfc_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- scene ---------------------------------------------------------------------------------------
    def add_mesh(self, kind, xyz, idx, eps, Ebar, tree) -> int:
        xyz = _a(xyz).reshape(-1, 3)
        idx = _a(idx, np.int32)
        eps_a = None if eps is None else _a(eps)
        out = C.c_int(-1)
        _check(lib().pfc_add_mesh(self._h, kind, len(xyz), xyz, len(idx), idx, _p(eps_a), float(Ebar or 0.0), tree.n_node, _a(tree.c), _a(tree.e),
                                  _a(tree.R), _a(tree.left, np.int32), _a(tree.right, np.int32), _a(tree.leaf_id, np.int32), C.byref(out)))
        return out.value

    def add_instruction(self, mesh_1, mesh_2, chi, model, params, n_quad_rule) -> int:
        out = C.c_int(-1)
        _check(lib().pfc_add_instruction(self._h, mesh_1, mesh_2, float(chi), model, _a(params), n_quad_rule, C.byref(out)))
        self.n_ins = out.value + 1
        if model == 1:
            self.n_bristle += 1
        return out.value

    def finalize(self, max_env: int = 1):
        _check(lib().pfc_finalize(self._h, max_env))

    def set_contact_params(self, params):
        """Per-environment contact parameters: params[env][ins][8] = (chi, Ebar_1, Ebar_2, q0..q4), q = (mu_s, mu_d, v_c, -, -) for a
        regularized instruction and (tau, k_bar, mu_s, mu_d, magic) for a bristle one; None clears the table (pfc_set_contact_params)."""
        if params is None:
            _check(lib().pfc_set_contact_params(self._h, 0, None))
            return
        p = _a(params)
        if p.ndim != 3 or p.shape[1:] != (self.n_ins, 8):
            raise ValueError(f"params must have shape [n_env, {self.n_ins}, 8], got {p.shape}")
        _check(lib().pfc_set_contact_params(self._h, p.shape[0], _p(p)))

    def set_debug(self, keep_pairs: bool = True):
        _check(lib().pfc_set_debug(self._h, int(keep_pairs)))

    def set_shard(self, rank: int, world: int):
        _check(lib().pfc_set_shard(self._h, rank, world))

    # ---- evaluation ----------------------------------------------------------------------------------
    def eval_f64(self, X, twist, s=None, keep=False, out=None):
        """Host arrays in, host arrays out (copies inside the call)."""
        if keep:
            self.set_debug(True)
        X = _a(X).reshape(-1, self.n_ins, 16)
        n_env = X.shape[0]
        twist = _a(twist).reshape(n_env, self.n_ins, 6)
        nb = self.n_bristle
        s_a = _a(s).reshape(n_env, nb, 6) if nb else None
        if out is None:
            out = dict(wrench=np.zeros((n_env, self.n_ins, 6)), sdot=np.zeros((n_env, nb, 6)) if nb else None,
                       n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_eval_f64(self._h, n_env, _p(X), _p(twist), _p(s_a), _p(out["wrench"]), _p(out["sdot"]), _p(out["n_pairs"]),
                                  _p(out["flags"])))
        return out

    def eval_f64_ptr(self, n_env, X, twist, s, wrench, sdot, n_pairs, flags):
        """Host pointers given as integers (e.g. pinned torch tensors' data_ptr())."""
        _check(lib().pfc_eval_f64(self._h, n_env, X, twist, s, wrench, sdot, n_pairs, flags))

    def eval_f64_device(self, n_env, X, twist, s, wrench, sdot, n_pairs, flags):
        """Device pointers given as integers; asynchronous on self.stream."""
        _check(lib().pfc_eval_f64_device(self._h, n_env, X, twist, s, wrench, sdot, n_pairs, flags))

    # ---- state-level entry points: kinematics prologue and J' w epilogue on the device ---------------------
    def set_bodies(self, joint_type, q0, v0, mesh_body, nq, nv, pose=None):
        """joint_type[b]: 0 = world-attached, 1 = SPQuatFloating; pose: [n_body][12] (R row-major, t) or None."""
        jt, q0a, v0a, mb = _a(joint_type, np.int32), _a(q0, np.int32), _a(v0, np.int32), _a(mesh_body, np.int32)
        pose_a = None if pose is None else _a(pose).reshape(len(jt), 12)
        _check(lib().pfc_set_bodies(self._h, len(jt), jt, q0a, v0a, _p(pose_a), mb, int(nq), int(nv)))
        self.nq, self.nv = int(nq), int(nv)

    def eval_state_f64(self, x):
        """x[env][nq + nv + 6 n_bristle] (host) -> dict(f_generalized[env][nv], sdot, n_pairs, flags)."""
        x = _a(x)
        x = x.reshape(-1, self.nq + self.nv + 6 * self.n_bristle)
        n_env, nb = x.shape[0], self.n_bristle
        out = dict(f_generalized=np.zeros((n_env, self.nv)), sdot=np.zeros((n_env, nb, 6)) if nb else None,
                   n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_eval_state_f64(self._h, n_env, _p(x), _p(out["f_generalized"]), _p(out["sdot"]), _p(out["n_pairs"]), _p(out["flags"])))
        return out

    def eval_state_f64_ptr(self, n_env, x, f_generalized, sdot, n_pairs, flags):
        """Host pointers given as integers (pinned buffers)."""
        _check(lib().pfc_eval_state_f64(self._h, n_env, x, f_generalized, sdot, n_pairs, flags))

    def eval_state_f64_device(self, n_env, x, f_generalized, sdot, n_pairs, flags):
        """Device pointers given as integers; asynchronous on self.stream."""
        _check(lib().pfc_eval_state_f64_device(self._h, n_env, x, f_generalized, sdot, n_pairs, flags))

    # ---- calcXd! on the device (floating-body scenes) ----------------------------------------------------------------
    def set_dynamics(self, spatial_inertia, gravity):
        """spatial_inertia[n_body][6][6] about the body origins in the body frames ([angular; linear]); gravity[3] in the world."""
        H = _a(spatial_inertia).reshape(-1, 36)
        _check(lib().pfc_set_dynamics(self._h, H.shape[0], H, _a(gravity).reshape(3)))

    def calcxd_f64(self, x, tau_ext=None):
        """x[env][n_x] (host) -> dict(xdot[env][n_x], n_pairs, flags)."""
        nx = self.nq + self.nv + 6 * self.n_bristle
        x = _a(x).reshape(-1, nx)
        n_env = x.shape[0]
        tau = None if tau_ext is None else _a(tau_ext).reshape(n_env, self.nv)
        out = dict(xdot=np.zeros((n_env, nx)), n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_calcxd_f64(self._h, n_env, _p(x), _p(tau), _p(out["xdot"]), _p(out["n_pairs"]), _p(out["flags"])))
        return out

    def calcxd_dual6(self, x, seed_start, tau_ext=None):
        """Jacobian chunk of calcXd!: x[env][n_x] (host), seeds on x[seed_start : seed_start + 6] -> dict(xdot7[env][n_x][7], n_pairs, flags)."""
        nx = self.nq + self.nv + 6 * self.n_bristle
        x = _a(x).reshape(-1, nx)
        n_env = x.shape[0]
        tau = None if tau_ext is None else _a(tau_ext).reshape(n_env, self.nv)
        out = dict(xdot7=np.zeros((n_env, nx, 7)), n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_calcxd_dual6(self._h, n_env, _p(x), _p(tau), int(seed_start), _p(out["xdot7"]), _p(out["n_pairs"]), _p(out["flags"])))
        return out

    def calcxd_dual6_device(self, n_env, x, tau_ext, seed_start, xdot7, n_pairs, flags):
        """Device pointers given as integers; asynchronous on self.stream."""
        _check(lib().pfc_calcxd_dual6_device(self._h, n_env, x, tau_ext, int(seed_start), xdot7, n_pairs, flags))

    def calcxd_jacobian(self, x, tau_ext=None):
        """The whole Jacobian of calcXd! in one call: x[env][n_x] (host) -> dict(jac[env][n_x][n_x] = d xdot_i / d x_j, xdot, n_pairs, flags)."""
        nx = self.nq + self.nv + 6 * self.n_bristle
        x = _a(x).reshape(-1, nx)
        n_env = x.shape[0]
        tau = None if tau_ext is None else _a(tau_ext).reshape(n_env, self.nv)
        out = dict(jac=np.zeros((n_env, nx, nx)), xdot=np.zeros((n_env, nx)), n_pairs=np.zeros((n_env, self.n_ins), np.int64),
                   flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_calcxd_jacobian(self._h, n_env, _p(x), _p(tau), _p(out["jac"]), _p(out["xdot"]), _p(out["n_pairs"]), _p(out["flags"])))
        return out

    def calcxd_jacobian_device(self, n_env, x, tau_ext, jac, xdot, n_pairs, flags):
        """Device pointers given as integers (tau_ext / xdot may be None); asynchronous on self.stream."""
        _check(lib().pfc_calcxd_jacobian_device(self._h, n_env, x, tau_ext, jac, xdot, n_pairs, flags))

    def refit_mesh(self, mesh_id: int, xyz):
        """New vertex positions for mesh `mesh_id` (same connectivity): primitive records and every box of its tree are refitted on the device."""
        xyz = _a(xyz).reshape(-1, 3)
        _check(lib().pfc_refit_mesh(self._h, int(mesh_id), xyz.shape[0], xyz))

    def radau_inv_c_device(self, n_mat, n, neg_J, shift, index, inv_c, info=None):
        """Batched updateInvC!: device pointers given as integers; asynchronous on self.stream."""
        _check(lib().pfc_radau_inv_c_device(self._h, n_mat, n, neg_J, shift, index, inv_c, info))

    def radau_init(self, n_env, max_rule=2, h0=1.0e-4, h_max=0.01, tol_newton=1.0e-16):
        """Resets the batched Radau controller of n_env environments (h = h0, rule 1) and sizes its buffers."""
        _check(lib().pfc_radau_init(self._h, int(n_env), int(max_rule), float(h0), float(h_max), float(tol_newton)))

    def radau_step(self, x, t, tau_ext=None):
        """One accepted Radau step of every environment: host arrays in -> (x [env][n_x], t [env], h_taken [env], stats [env][4])."""
        nx = self.nq + self.nv + 6 * self.n_bristle
        x = _a(x).reshape(-1, nx).copy()
        n_env = x.shape[0]
        t = _a(t).reshape(n_env).copy()
        tau = None if tau_ext is None else _a(tau_ext).reshape(n_env, self.nv)
        h = np.zeros(n_env)
        stats = np.zeros((n_env, 4), np.int32)
        _check(lib().pfc_radau_step(self._h, n_env, _p(x), _p(tau), _p(t), _p(h), _p(stats)))
        return x, t, h, stats

    def radau_step_device(self, n_env, x, tau_ext, t, h_taken, stats):
        """Device pointers given as integers (tau_ext / stats may be None); on self.stream."""
        _check(lib().pfc_radau_step_device(self._h, n_env, x, tau_ext, t, h_taken, stats))

    def radau_rollout(self, x, t, t_knot, tau_ext=None, max_steps=1000):
        """Every environment through the knot times t_knot [n_knot] (host arrays): tau_ext [n_knot][env][nv] or None ->
        (x [env][n_x], t [env], x_knot [n_knot][env][n_x] (NaN rows for knots not reached), stats [env][4])."""
        nx = self.nq + self.nv + 6 * self.n_bristle
        x = _a(x).reshape(-1, nx).copy()
        n_env = x.shape[0]
        t = _a(t).reshape(n_env).copy()
        t_knot = _a(t_knot).reshape(-1)
        tau = None if tau_ext is None else _a(tau_ext).reshape(t_knot.shape[0], n_env, self.nv)
        x_knot = np.zeros((t_knot.shape[0], n_env, nx))
        stats = np.zeros((n_env, 4), np.int32)
        _check(lib().pfc_radau_rollout(self._h, n_env, t_knot.shape[0], t_knot, int(max_steps), _p(x), _p(tau), _p(t), _p(x_knot), _p(stats)))
        return x, t, x_knot, stats

    def radau_rollout_device(self, n_env, t_knot, max_steps, x, tau_ext, t, x_knot, stats):
        """t_knot is a host array; the rest are device pointers given as integers (tau_ext / x_knot / stats may be None); on self.stream."""
        t_knot = _a(t_knot).reshape(-1)
        _check(lib().pfc_radau_rollout_device(self._h, n_env, t_knot.shape[0], t_knot, int(max_steps), x, tau_ext, t, x_knot, stats))

    def radau_step_info(self):
        """(ms [Jacobian, stage evaluations, inverses, Newton + controller] -- needs set_timing(True) --, rounds, host synchronisations)
        of the last Radau step or roll-out (sums over its steps)."""
        ms = np.zeros(4)
        counts = np.zeros(2, np.int64)
        _check(lib().pfc_radau_step_info(self._h, _p(ms), _p(counts)))
        return ms, int(counts[0]), int(counts[1])

    def calcxd_f64_device(self, n_env, x, tau_ext, xdot, n_pairs, flags):
        """Device pointers given as integers; asynchronous on self.stream."""
        _check(lib().pfc_calcxd_f64_device(self._h, n_env, x, tau_ext, xdot, n_pairs, flags))

    def get_boundary(self, n_env):
        """(X_r2_r1, twist_r2, wrench_r2) of the last evaluation as computed / consumed on the device."""
        X, tw, w = np.zeros((n_env, self.n_ins, 16)), np.zeros((n_env, self.n_ins, 6)), np.zeros((n_env, self.n_ins, 6))
        _check(lib().pfc_get_boundary(self._h, n_env, _p(X), _p(tw), _p(w)))
        return X, tw, w

    def eval_sharded_begin(self, n_env, X, twist, s, wrench, sdot, n_pairs, flags):
        """Device pointers (integers).  See INTEGRATION.md for the protocol."""
        _check(lib().pfc_eval_sharded_begin(self._h, n_env, X, twist, s, wrench, sdot, n_pairs, flags))

    def eval_sharded_partials(self):
        ptr, n = _vp(), C.c_int64(0)
        _check(lib().pfc_eval_sharded_partials(self._h, C.byref(ptr), C.byref(n)))
        return (ptr.value or 0), n.value

    def eval_sharded_step(self) -> bool:
        more = C.c_int(0)
        _check(lib().pfc_eval_sharded_step(self._h, C.byref(more)))
        return bool(more.value)

    # ---- library-owned exchange (one process per GPU) ------------------------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        _check(lib().pfc_comm_unique_id(C.cast(buf, _vp)))
        return buf.raw

    def comm_init_rank(self, unique_id: bytes, rank: int, world: int):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        _check(lib().pfc_comm_init_rank(self._h, C.cast(buf, _vp), rank, world))

    def eval_sharded_f64_device(self, n_env, X, twist, s, wrench, sdot, n_pairs, flags):
        """Device pointers; this rank's share of the evaluation, the all-gather of the partial sums and their application, on self.stream."""
        _check(lib().pfc_eval_sharded_f64_device(self._h, n_env, X, twist, s, wrench, sdot, n_pairs, flags))

    def eval_dual6(self, X_bp, X7, twist7, s7=None):
        n_env = _a(X7).reshape(-1, self.n_ins, 16, 7).shape[0]
        X7 = _a(X7).reshape(n_env, self.n_ins, 16, 7)
        X_bp_a = None if X_bp is None else _a(X_bp).reshape(n_env, self.n_ins, 16)
        twist7 = _a(twist7).reshape(n_env, self.n_ins, 6, 7)
        nb = self.n_bristle
        s_a = _a(s7).reshape(n_env, nb, 6, 7) if nb else None
        out = dict(wrench=np.zeros((n_env, self.n_ins, 6, 7)), sdot=np.zeros((n_env, nb, 6, 7)) if nb else None,
                   n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_eval_dual6(self._h, n_env, _p(X_bp_a), _p(X7), _p(twist7), _p(s_a), _p(out["wrench"]), _p(out["sdot"]),
                                    _p(out["n_pairs"]), _p(out["flags"])))
        return out

    # ---- debug / parity --------------------------------------------------------------------------------
    def get_pairs(self, env: int, ins: int) -> np.ndarray:
        n = C.c_int64(0)
        _check(lib().pfc_get_pairs(self._h, env, ins, None, 0, C.byref(n)))
        out = np.zeros((max(n.value, 1), 2), np.int32)
        _check(lib().pfc_get_pairs(self._h, env, ins, _p(out), n.value, C.byref(n)))
        return out[:n.value]

    def get_traction(self, env: int, ins: int, cap: int = 1 << 16) -> np.ndarray:
        n = C.c_int64(0)
        out = np.zeros((cap, 8))
        _check(lib().pfc_get_traction(self._h, env, ins, _p(out), cap, C.byref(n)))
        return out[:min(n.value, cap)].copy()

    # ---- plumbing ------------------------------------------------------------------------------------
    def sync(self):
        _check(lib().pfc_sync(self._h))

    @property
    def stream(self) -> int:
        return int(lib().pfc_stream(self._h) or 0)

    def launch_count(self) -> int:
        return int(lib().pfc_launch_count(self._h))

    def measure_fp64_peak(self) -> float:
        v = C.c_double(0.0)
        _check(lib().pfc_measure_fp64_peak(self._h, C.byref(v)))
        return v.value

    def set_timing(self, on: bool = True):
        _check(lib().pfc_set_timing(self._h, int(on)))

    def kernel_times(self):
        """(broad_ms, narrow_ms) of the last evaluation (needs set_timing(True))."""
        ms = (C.c_double * 4)()
        _check(lib().pfc_kernel_times(self._h, ms, 4))
        return ms[0], ms[1]

    def counters(self):
        a, b = C.c_int64(0), C.c_int64(0)
        _check(lib().pfc_counters(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value


class Group:
    """pfc_group: one process, one context per listed GPU, one library-owned NCCL communicator; the scene is described once and
    pfc_group_eval_f64 splits the large instructions' candidate-pair lists over the devices (same add_mesh / add_instruction /
    finalize / eval_f64 surface as Context, so scenario.attach_backend works on it)."""
    name = "cuda-group"

    def __init__(self, devices):
        self._h = _vp()
        dev = _a(list(devices), np.int32)
        _check(lib().pfc_group_create(len(dev), dev, C.byref(self._h)))
        self.n_ins = 0
        self.n_bristle = 0
        self.size = int(lib().pfc_group_size(self._h))

    def close(self):
        if self._h:
            lib().pfc_group_destroy(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def add_mesh(self, kind, xyz, idx, eps, Ebar, tree) -> int:
        xyz = _a(xyz).reshape(-1, 3)
        idx = _a(idx, np.int32)
        eps_a = None if eps is None else _a(eps)
        out = C.c_int(-1)
        _check(lib().pfc_group_add_mesh(self._h, kind, len(xyz), xyz, len(idx), idx, _p(eps_a), float(Ebar or 0.0), tree.n_node, _a(tree.c), _a(tree.e),
                                        _a(tree.R), _a(tree.left, np.int32), _a(tree.right, np.int32), _a(tree.leaf_id, np.int32), C.byref(out)))
        return out.value

    def add_instruction(self, mesh_1, mesh_2, chi, model, params, n_quad_rule) -> int:
        out = C.c_int(-1)
        _check(lib().pfc_group_add_instruction(self._h, mesh_1, mesh_2, float(chi), model, _a(params), n_quad_rule, C.byref(out)))
        self.n_ins = out.value + 1
        if model == 1:
            self.n_bristle += 1
        return out.value

    def finalize(self, max_env: int = 1):
        _check(lib().pfc_group_finalize(self._h, max_env))

    def eval_f64(self, X, twist, s=None, keep=False, out=None):
        X = _a(X).reshape(-1, self.n_ins, 16)
        n_env = X.shape[0]
        twist = _a(twist).reshape(n_env, self.n_ins, 6)
        nb = self.n_bristle
        s_a = _a(s).reshape(n_env, nb, 6) if nb else None
        if out is None:
            out = dict(wrench=np.zeros((n_env, self.n_ins, 6)), sdot=np.zeros((n_env, nb, 6)) if nb else None,
                       n_pairs=np.zeros((n_env, self.n_ins), np.int64), flags=np.zeros((n_env, self.n_ins), np.int32))
        _check(lib().pfc_group_eval_f64(self._h, n_env, _p(X), _p(twist), _p(s_a), _p(out["wrench"]), _p(out["sdot"]), _p(out["n_pairs"]), _p(out["flags"])))
        return out
