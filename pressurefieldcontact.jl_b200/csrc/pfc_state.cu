// pfc_state.cu -- device-side prologue / epilogue / rigid-body dynamics of the contact-wrench evaluation for scenes whose
// bodies are world-attached or float on SPQuatFloating joints (SURVEY.md section 8f, ranks 1 and 2; config C3 is such a scene).
//
//   prologue  state x = [q; v; s] per environment  ->  x_r2_r1 (4x4), twist of r2 w.r.t. r1 in r2, bristle state s
//             (what refreshBodyBodyTransform! / refreshBodyBodyCache! compute through RigidBodyDynamics:
//             /root/reference/src/contact_algorithms_non_friction.jl:103-134; joint layout q = [MRP(3); trans(3)],
//             v = [omega(3); vel(3)] in the body frame: src/mechanism_scenario.jl:247-256)
//   epilogue  per-instruction wrench (about the r2 origin, in r2, on body 2)  ->  f_generalized += J' w on body 2,
//             -= J' w on body 1 (addGeneralizedForcesThirdLaw!, :267-286); every thread owns one body's six
//             velocity coordinates and adds its instructions in instruction order, so the sums are reproducible.
//   dynamics  calcXd! (:18-38): J' w as above, v_dot = H^-1 (f + tau_ext - v x* (H v)) + [0; R' g], q_dot, s_dot.
// Everything is templated on the scalar T in {double, Dual<6>}: the Dual instantiation is the reference's Jacobian mode
// (calcXd! on Vector{Dual{Nothing,Float64,6}}, src/radau/radau_functions.jl:2-26) with the seeds placed on x[seed0 .. seed0 + 6).
// With these kernels a batched evaluation takes the raw states and returns generalized forces or x_dot (and its Jacobian
// chunk): the host does no kinematics and moves 3.3x fewer bytes per environment.
#include "pfc_launch.h"
#include "pfc_math.cuh"

namespace pfc {

namespace {

typedef Dual<6> D6;

template <class T> struct Frame { T R[9]; T t[3]; T ang[3]; T lin[3]; };   // transform_to_root, twist_wrt_world (about the world origin)

// state entry j as a scalar of mode T: Dual mode seeds d x[j] / d x[seed0 + k] = [j == seed0 + k]
template <class T> struct StateRead;
template <> struct StateRead<double> {
    const double* x; int seed0;
    PFC_D double operator()(int j) const { return x[j]; }
};
template <> struct StateRead<D6> {
    const double* x; int seed0;
    PFC_D D6 operator()(int j) const {
        D6 r(x[j]);
        const int k = j - seed0;
#pragma unroll
        for (int i = 0; i < 6; ++i) r.p[i] = (i == k) ? 1.0 : 0.0;
        return r;
    }
};
PFC_D void store_scalar(double* p, long long i, double v) { p[i] = v; }
PFC_D void store_scalar(double* p, long long i, const D6& v) {
    p[7 * i] = v.v;
#pragma unroll
    for (int k = 0; k < 6; ++k) p[7 * i + 1 + k] = v.p[k];
}
PFC_D double load_scalar(const double* p, long long i, double*) { return p[i]; }
PFC_D D6 load_scalar(const double* p, long long i, D6*) {
    D6 r; r.v = p[7 * i];
#pragma unroll
    for (int k = 0; k < 6; ++k) r.p[k] = p[7 * i + 1 + k];
    return r;
}

// SPQuat / modified Rodrigues parameters -> rotation matrix (Rotations.jl: q = ((1 - a2) / (1 + a2), 2 p / (1 + a2)))
template <class T> PFC_D void mrp_to_rot(const T* p, T* R) {
    const T a2 = p[0] * p[0] + p[1] * p[1] + p[2] * p[2];
    const T inv = 1.0 / (a2 + 1.0);
    const T w = (1.0 - a2) * inv, x = 2.0 * p[0] * inv, y = 2.0 * p[1] * inv, z = 2.0 * p[2] * inv;
    R[0] = 1.0 - 2.0 * (y * y + z * z); R[1] = 2.0 * (x * y - w * z); R[2] = 2.0 * (x * z + w * y);
    R[3] = 2.0 * (x * y + w * z); R[4] = 1.0 - 2.0 * (x * x + z * z); R[5] = 2.0 * (y * z - w * x);
    R[6] = 2.0 * (x * z - w * y); R[7] = 2.0 * (y * z + w * x); R[8] = 1.0 - 2.0 * (x * x + y * y);
}

template <class A, class B, class C> PFC_D void mat_vec(const A* R, const B* v, C* out) {
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = R[3 * i] * v[0] + R[3 * i + 1] * v[1] + R[3 * i + 2] * v[2];
}
template <class A, class B, class C> PFC_D void mat_t_vec(const A* R, const B* v, C* out) {
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = R[i] * v[0] + R[3 + i] * v[1] + R[6 + i] * v[2];
}
template <class A, class B, class C> PFC_D void cross3(const A* a, const B* b, C* out) {
    out[0] = a[1] * b[2] - a[2] * b[1]; out[1] = a[2] * b[0] - a[0] * b[2]; out[2] = a[0] * b[1] - a[1] * b[0];
}

// x_env: reader of this environment's state (q at 0, v at nq)
template <class T> PFC_D void body_frame(const BodyDev& b, const StateRead<T>& xr, int nq, Frame<T>& f, bool with_twist) {
    if (b.joint == 0) {   // world-attached
#pragma unroll
        for (int i = 0; i < 9; ++i) f.R[i] = T((i % 4 == 0) ? 1.0 : 0.0);
#pragma unroll
        for (int i = 0; i < 3; ++i) { f.t[i] = T(0.0); f.ang[i] = T(0.0); f.lin[i] = T(0.0); }
        return;
    }
    T p[3] = {xr(b.q0), xr(b.q0 + 1), xr(b.q0 + 2)};
    T Rj[9];
    mrp_to_rot(p, Rj);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) f.R[3 * i + j] = b.pose_R[3 * i] * Rj[j] + b.pose_R[3 * i + 1] * Rj[3 + j] + b.pose_R[3 * i + 2] * Rj[6 + j];
    T tj[3] = {xr(b.q0 + 3), xr(b.q0 + 4), xr(b.q0 + 5)};
    mat_vec(b.pose_R, tj, f.t);
#pragma unroll
    for (int i = 0; i < 3; ++i) f.t[i] = f.t[i] + b.pose_t[i];
    if (with_twist) {
        const T om[3] = {xr(nq + b.v0), xr(nq + b.v0 + 1), xr(nq + b.v0 + 2)}, ve[3] = {xr(nq + b.v0 + 3), xr(nq + b.v0 + 4), xr(nq + b.v0 + 5)};
        mat_vec(f.R, om, f.ang);
        T rv[3], tx[3];
        mat_vec(f.R, ve, rv);
        cross3(f.t, f.ang, tx);
#pragma unroll
        for (int i = 0; i < 3; ++i) f.lin[i] = rv[i] + tx[i];
    }
}

// one thread per (environment, instruction): boundary arrays; one extra pass copies the bristle states
template <class T>
__global__ void __launch_bounds__(128) state_prologue_kernel(StateDev sd, long long n_env, long long n_real, int n_ins, int n_bristle,
                                                             const double* __restrict__ x, int seed0, double* __restrict__ X, double* __restrict__ twist,
                                                             double* __restrict__ s) {
    // n_env = n_chunk * n_real "environments", chunk-major: entry (chunk, env) reads the state of real environment env with the seeds
    // on x[seed0 + 6 chunk ..) -- the whole-Jacobian mode; n_real == n_env otherwise
    const long long n = n_env * n_ins;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x) {
        const long long env = id / n_ins;
        const int k = (int)(id - env * n_ins);
        const StateRead<T> xr{x + (env % n_real) * sd.n_x, seed0 + 6 * (int)(env / n_real)};
        Frame<T> f1, f2;
        body_frame(sd.bodies[sd.ins_body[2 * k]], xr, sd.nq, f1, true);
        body_frame(sd.bodies[sd.ins_body[2 * k + 1]], xr, sd.nq, f2, true);
        // x_r2_rw = inv(x_rw_r2);  x_r2_r1 = x_r2_rw * x_rw_r1   (non_friction.jl:109-113)
        T t_inv[3], t21[3];
        mat_t_vec(f2.R, f2.t, t_inv);
#pragma unroll
        for (int i = 0; i < 3; ++i) t_inv[i] = -t_inv[i];
        mat_t_vec(f2.R, f1.t, t21);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) store_scalar(X, 16 * id + 4 * j + i, f2.R[i] * f1.R[j] + f2.R[3 + i] * f1.R[3 + j] + f2.R[6 + i] * f1.R[6 + j]);
            store_scalar(X, 16 * id + 12 + i, t21[i] + t_inv[i]);
            store_scalar(X, 16 * id + 4 * i + 3, T(0.0));
        }
        store_scalar(X, 16 * id + 15, T(1.0));
        // twist_r2_r1 = -twist_w_r1 + twist_w_r2 in world, then transform(., x_r2_rw)   (:125-128)
        const T aw[3] = {f2.ang[0] - f1.ang[0], f2.ang[1] - f1.ang[1], f2.ang[2] - f1.ang[2]};
        const T lw[3] = {f2.lin[0] - f1.lin[0], f2.lin[1] - f1.lin[1], f2.lin[2] - f1.lin[2]};
        T ang[3], lin[3], tx[3];
        mat_t_vec(f2.R, aw, ang);
        mat_t_vec(f2.R, lw, lin);
        cross3(t_inv, ang, tx);
#pragma unroll
        for (int i = 0; i < 3; ++i) { store_scalar(twist, 6 * id + i, ang[i]); store_scalar(twist, 6 * id + 3 + i, lin[i] + tx[i]); }
    }
    const long long ns = n_env * 6 * n_bristle;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < ns; id += (long long)gridDim.x * blockDim.x) {
        const long long env = id / (6 * n_bristle);
        const StateRead<T> xr{x + (env % n_real) * sd.n_x, seed0 + 6 * (int)(env / n_real)};
        store_scalar(s, id, xr(sd.nq + sd.nv + (int)(id - env * 6 * n_bristle)));
    }
}

// The error bits of the per-(environment, instruction) flags, OR-ed into one device word: the host-pointer entry points read
// 4 bytes back instead of the whole flag array when the caller does not ask for it.
PFC_D void or_error_flags(const int* __restrict__ flags, long long n, int* __restrict__ status) {
    if (!status) return;
    int bad = 0;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x)
        bad |= flags[id] & (kFlagNonFinite | kFlagOverflow);
    if (bad) atomicOr(status, bad);
}

// J' w of every instruction that touches body b (addGeneralizedForcesThirdLaw!), summed in instruction order
template <class T>
PFC_D void body_generalized_force(const StateDev& sd, int b, const Frame<T>& fb, const StateRead<T>& xr, const double* __restrict__ wrench_env, T* fa, T* fl) {
#pragma unroll
    for (int i = 0; i < 3; ++i) { fa[i] = T(0.0); fl[i] = T(0.0); }
    for (int e = sd.body_ins_ptr[b]; e < sd.body_ins_ptr[b + 1]; ++e) {
        const int code = sd.body_ins[e];
        const int k = code >> 1;
        const double sign = (code & 1) ? 1.0 : -1.0;   // +J' w on body 2, -J' w on body 1
        Frame<T> f2;
        const int b2 = sd.ins_body[2 * k + 1];
        if (b2 == b) f2 = fb; else body_frame(sd.bodies[b2], xr, sd.nq, f2, false);
        T w[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) w[i] = load_scalar(wrench_env, 6 * k + i, (T*)nullptr);
        T lin_w[3], ang_w[3], tx[3];
        mat_vec(f2.R, w + 3, lin_w);
        mat_vec(f2.R, w, ang_w);
        cross3(f2.t, lin_w, tx);
#pragma unroll
        for (int i = 0; i < 3; ++i) ang_w[i] = ang_w[i] + tx[i];
        cross3(fb.t, lin_w, tx);
        const T m[3] = {ang_w[0] - tx[0], ang_w[1] - tx[1], ang_w[2] - tx[2]};
        T ja[3], jl[3];
        mat_t_vec(fb.R, m, ja);
        mat_t_vec(fb.R, lin_w, jl);
#pragma unroll
        for (int i = 0; i < 3; ++i) { fa[i] = fa[i] + ja[i] * sign; fl[i] = fl[i] + jl[i] * sign; }
    }
}

// one thread per (environment, body)
__global__ void __launch_bounds__(128) state_epilogue_kernel(StateDev sd, long long n_env, int n_ins, const double* __restrict__ x,
                                                             const double* __restrict__ wrench, double* __restrict__ f_gen,
                                                             const int* __restrict__ flags, int* __restrict__ status) {
    or_error_flags(flags, n_env * n_ins, status);
    const long long n = n_env * sd.n_body;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x) {
        const long long env = id / sd.n_body;
        const int b = (int)(id - env * sd.n_body);
        const BodyDev& body = sd.bodies[b];
        if (body.joint == 0) continue;   // jac == nothing: world-attached meshes take no generalized force
        const StateRead<double> xr{x + env * sd.n_x, 0};
        Frame<double> fb;
        body_frame(body, xr, sd.nq, fb, false);
        double fa[3], fl[3];
        body_generalized_force(sd, b, fb, xr, wrench + 6 * env * n_ins, fa, fl);
        double* fo = f_gen + env * sd.nv + body.v0;
#pragma unroll
        for (int i = 0; i < 3; ++i) { fo[i] = fa[i]; fo[3 + i] = fl[i]; }
    }
}

// calcXd! for floating bodies, one thread per (environment, body): J' w (as above), then
//   v_dot = H^-1 (f + tau_ext - v x* (H v)) + [0; R' g]     (mass_matrix!, dynamics_bias!, cholesky!/ldiv!: non_friction.jl:23-35;
//                                                            H is constant in the body frame, so its inverse is taken once, at pfc_set_dynamics)
//   q_dot = [B(p) w; R u],  B(p) = ((1 - p'p) I + 2 [p]x + 2 p p') / 4                  (configuration_derivative!, SPQuatFloating)
// and one extra pass copies s_dot behind [q_dot; v_dot] (copyto!, src/extensions.jl:40-50).
// wrench / sdot / xdot hold 1 (double) or 7 (Dual<6>: value, 6 partials) doubles per scalar.
// Where row `row` of x_dot goes.  Plain mode: xdot[env][row] (1 or 7 doubles).  Whole-Jacobian mode (jac != nullptr, Dual only): the
// partials are columns seed .. seed + 5 of jac[env][row][.] (row-major n_x x n_x per environment, the layout of calcJacobian!'s
// `jac`, /root/reference/src/radau/radau_functions.jl:2-26) and chunk 0 also writes the value to xdot[env][row] when asked to.
struct XdotOut { double* xdot; double* jac; int n_x; };
PFC_D void emit_row(const XdotOut& o, long long env_real, int row, int seed, bool first_chunk, double v) { o.xdot[env_real * o.n_x + row] = v; (void)seed; (void)first_chunk; }
PFC_D void emit_row(const XdotOut& o, long long env_real, int row, int seed, bool first_chunk, const D6& v) {
    if (!o.jac) { store_scalar(o.xdot, env_real * o.n_x + row, v); return; }
    double* j = o.jac + ((size_t)env_real * o.n_x + row) * o.n_x;
#pragma unroll
    for (int k = 0; k < 6; ++k) if (seed + k < o.n_x) j[seed + k] = v.p[k];
    if (first_chunk && o.xdot) o.xdot[env_real * o.n_x + row] = v.v;
}

// kTable: read H, H^-1 and gravity from the per-environment table of dd (pfc_set_body_params).  A separate instantiation, so the kernel
// without a table keeps its registers and stack frame (the run-time select cost the Dual<6> kernel 24 bytes of stack).
template <class T, bool kTable>
__global__ void __launch_bounds__(128) state_dynamics_kernel(StateDev sd, DynDev dd, long long n_env, long long n_real, int n_ins, int n_bristle,
                                                             const double* __restrict__ x, int seed0, const double* __restrict__ wrench,
                                                             const double* __restrict__ tau_ext, const double* __restrict__ sdot, XdotOut out,
                                                             const int* __restrict__ flags, int* __restrict__ status) {
    constexpr int W = sizeof(T) / sizeof(double);   // doubles per scalar
    or_error_flags(flags, n_real * n_ins, status);
    const long long n = n_env * sd.n_body;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x) {
        const long long env = id / sd.n_body;           // (chunk, real environment), chunk-major
        const int b = (int)(id - env * sd.n_body);
        const BodyDev& body = sd.bodies[b];
        if (body.joint == 0) continue;
        const long long er = env % n_real;
        const int seed = seed0 + 6 * (int)(env / n_real);
        const bool first = env < n_real;
        const StateRead<T> xr{x + er * sd.n_x, seed};
        T v[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) v[i] = xr(sd.nq + body.v0 + i);
        Frame<T> fb;
        body_frame(body, xr, sd.nq, fb, false);
        T f[6];
        body_generalized_force(sd, b, fb, xr, wrench + (size_t)W * 6 * env * n_ins, f, f + 3);
        if (tau_ext) {
#pragma unroll
            for (int i = 0; i < 6; ++i) f[i] = f[i] + tau_ext[er * sd.nv + body.v0 + i];
        }
        const double* H = dd.H + 36 * b;
        const double* Hi = dd.Hinv + 36 * b;
        double g[3] = {dd.gravity[0], dd.gravity[1], dd.gravity[2]};
        if (kTable) {   // the environment's row of the table
            const long long r = dd.row ? dd.row[er] : er;
            H = dd.H_env + 36 * (r * sd.n_body + b);
            Hi = dd.Hinv_env + 36 * (r * sd.n_body + b);
#pragma unroll
            for (int i = 0; i < 3; ++i) g[i] = dd.g_env[3 * r + i];
        }
        T h[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            T a = T(0.0);
#pragma unroll
            for (int j = 0; j < 6; ++j) a = a + v[j] * H[6 * i + j];
            h[i] = a;
        }
        T c1[3], c2[3], c3[3];
        cross3(v, h, c1);          // w x n
        cross3(v + 3, h + 3, c2);  // u x f
        cross3(v, h + 3, c3);      // w x f
        const T rhs[6] = {f[0] - (c1[0] + c2[0]), f[1] - (c1[1] + c2[1]), f[2] - (c1[2] + c2[2]), f[3] - c3[0], f[4] - c3[1], f[5] - c3[2]};
        T vd[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            T a = T(0.0);
#pragma unroll
            for (int j = 0; j < 6; ++j) a = a + rhs[j] * Hi[6 * i + j];
            vd[i] = a;
        }
        // the joint rotation (without the pose on the world) takes the body-frame velocity to q_dot; gravity uses the full rotation
        T p[3] = {xr(body.q0), xr(body.q0 + 1), xr(body.q0 + 2)};
        T Rj[9], g_b[3], qd_t[3];
        mrp_to_rot(p, Rj);
        mat_t_vec(fb.R, g, g_b);
        mat_vec(Rj, v + 3, qd_t);
        const T pp = p[0] * p[0] + p[1] * p[1] + p[2] * p[2], pw = p[0] * v[0] + p[1] * v[1] + p[2] * v[2];
        T pxw[3];
        cross3(p, v, pxw);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            emit_row(out, er, body.q0 + i, seed, first, ((1.0 - pp) * v[i] + 2.0 * pxw[i] + 2.0 * p[i] * pw) * 0.25);
            emit_row(out, er, body.q0 + 3 + i, seed, first, qd_t[i]);
            emit_row(out, er, sd.nq + body.v0 + i, seed, first, vd[i]);
            emit_row(out, er, sd.nq + body.v0 + 3 + i, seed, first, vd[3 + i] + g_b[i]);
        }
    }
    const long long ns = n_env * 6 * n_bristle;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < ns; id += (long long)gridDim.x * blockDim.x) {
        const long long env = id / (6 * n_bristle);
        emit_row(out, env % n_real, sd.nq + sd.nv + (int)(id - env * 6 * n_bristle), seed0 + 6 * (int)(env / n_real), env < n_real,
                 load_scalar(sdot, id, (T*)nullptr));
    }
}

unsigned state_blocks(long long n) { return (unsigned)((n + 127) / 128 < 148 * 16 ? (n + 127) / 128 : 148 * 16); }

// sum_m h[m] k[m] in the order m = 0 .. 5, as explicit FMAs: every mode of the feedback kernel rounds these sums alike
PFC_D double dot6(const double* h, const double* k) {
    double a = 0.0;
#pragma unroll
    for (int m = 0; m < 6; ++m) a = fma(h[m], k[m], a);
    return a;
}

// The feedback term of launch_state_feedback, one warp per (environment, body); see pfc_launch.h for the modes.  The term is subtracted
// as H^-1 K (x - x_ref): with K = 0 every sum is +0.0, so the outputs keep their bits (a signed zero included).  K is read coalesced,
// lanes over its columns; u = K (x - x_ref) is summed per lane in column order, then over the lanes by a butterfly that leaves the same
// bits in every lane, so the result does not depend on the batch or on the launch shape.
template <int kMode>
__global__ void __launch_bounds__(128) state_feedback_kernel(StateDev sd, DynDev dd, FeedbackDev fb, long long n_env, const double* __restrict__ x,
                                                             int seed0, double* __restrict__ xdot, double* __restrict__ jac) {
    const int lane = threadIdx.x & 31;
    const long long n = n_env * sd.n_body;
    for (long long id = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5; id < n; id += ((long long)gridDim.x * blockDim.x) >> 5) {
        const long long env = id / sd.n_body;
        const int b = (int)(id - env * sd.n_body);
        const BodyDev& body = sd.bodies[b];
        if (body.joint == 0) continue;   // the same for the whole warp
        const int nc = fb.ncol, nx = sd.n_x;
        const long long r = fb.row ? fb.row[env] : env;
        const double* Kb = fb.K + (r * sd.nv + body.v0) * nc;   // the body's six rows of K
        const double* xref = fb.x_ref + r * nc;
        const double* xe = x + env * nx;
        const double* Hi = dd.Hinv + 36 * b;
        if (dd.Hinv_env) Hi = dd.Hinv_env + 36 * ((dd.row ? dd.row[env] : env) * sd.n_body + b);
        double u[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int j = lane; j < nc; j += 32) {
            const double d = xe[j] - xref[j];
#pragma unroll
            for (int m = 0; m < 6; ++m) u[m] = fma(Kb[m * nc + j], d, u[m]);
        }
#pragma unroll
        for (int m = 0; m < 6; ++m)
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) u[m] = u[m] + __shfl_xor_sync(0xffffffffu, u[m], s);
        if (kMode == 2) {   // -(H^-1 K) into the [q; v] columns of the body's v_dot rows, once for all seed chunks
            double* jb = jac + ((size_t)env * nx + sd.nq + body.v0) * nx;
            for (int j = lane; j < nc; j += 32) {
                double kc[6];
#pragma unroll
                for (int m = 0; m < 6; ++m) kc[m] = Kb[m * nc + j];
#pragma unroll
                for (int i = 0; i < 6; ++i) jb[(size_t)i * nx + j] = jb[(size_t)i * nx + j] - dot6(Hi + 6 * i, kc);
            }
        }
        if (lane < 6) {   // lane i: v_dot row i of the body
            double h[6];
#pragma unroll
            for (int m = 0; m < 6; ++m) h[m] = Hi[6 * lane + m];
            const double a = dot6(h, u);
            const long long o = env * nx + sd.nq + body.v0 + lane;
            if (kMode == 0 || (kMode == 2 && xdot)) xdot[o] = xdot[o] - a;
            if (kMode == 1) {
                double* p = xdot + 7 * o;
                p[0] = p[0] - a;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const int col = seed0 + k;
                    if (col >= nc) break;   // bristle seeds: the feedback does not read s
                    double kc[6];
#pragma unroll
                    for (int m = 0; m < 6; ++m) kc[m] = Kb[m * nc + col];
                    p[1 + k] = p[1 + k] - dot6(h, kc);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) check_finite_kernel(const double* __restrict__ a, long long n, int* __restrict__ bad) {
    int b = 0;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x) b |= !isfinite(a[id]);
    if (__syncthreads_or(b) && threadIdx.x == 0) atomicOr(bad, 1);
}

}  // namespace

cudaError_t launch_state_prologue(const StateDev& sd, long long n_env, int n_ins, int n_bristle, const double* x, double* X, double* twist, double* s,
                                  cudaStream_t stream, int* n_launches) {
    const long long n = n_env * n_ins;
    if (n == 0) return cudaSuccess;
    state_prologue_kernel<double><<<state_blocks(n), 128, 0, stream>>>(sd, n_env, n_env, n_ins, n_bristle, x, 0, X, twist, s);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_state_prologue_dual6(const StateDev& sd, long long n_env, int n_ins, int n_bristle, const double* x, int seed0, double* X7, double* twist7,
                                        double* s7, cudaStream_t stream, int* n_launches, long long n_real) {
    const long long n = n_env * n_ins;
    if (n == 0) return cudaSuccess;
    state_prologue_kernel<D6><<<state_blocks(n), 128, 0, stream>>>(sd, n_env, n_real > 0 ? n_real : n_env, n_ins, n_bristle, x, seed0, X7, twist7, s7);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_state_epilogue(const StateDev& sd, long long n_env, int n_ins, const double* x, const double* wrench, double* f_gen, cudaStream_t stream,
                                  int* n_launches, const int* flags, int* status) {
    const long long n = n_env * sd.n_body;
    if (n == 0) return cudaSuccess;
    state_epilogue_kernel<<<state_blocks(n), 128, 0, stream>>>(sd, n_env, n_ins, x, wrench, f_gen, flags, status);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_state_dynamics(const StateDev& sd, const DynDev& dd, long long n_env, int n_ins, int n_bristle, const double* x, const double* wrench,
                                  const double* tau_ext, const double* sdot, double* xdot, cudaStream_t stream, int* n_launches, const int* flags, int* status) {
    const long long n = n_env * sd.n_body;
    if (n == 0) return cudaSuccess;
    (dd.H_env ? state_dynamics_kernel<double, true> : state_dynamics_kernel<double, false>)<<<state_blocks(n), 128, 0, stream>>>(
        sd, dd, n_env, n_env, n_ins, n_bristle, x, 0, wrench, tau_ext, sdot, XdotOut{xdot, nullptr, sd.n_x}, flags, status);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_state_dynamics_dual6(const StateDev& sd, const DynDev& dd, long long n_env, int n_ins, int n_bristle, const double* x, int seed0,
                                        const double* wrench7, const double* tau_ext, const double* sdot7, double* xdot7, cudaStream_t stream,
                                        int* n_launches, const int* flags, int* status, long long n_real, double* jac) {
    const long long n = n_env * sd.n_body;
    if (n == 0) return cudaSuccess;
    (dd.H_env ? state_dynamics_kernel<D6, true> : state_dynamics_kernel<D6, false>)<<<state_blocks(n), 128, 0, stream>>>(
        sd, dd, n_env, n_real > 0 ? n_real : n_env, n_ins, n_bristle, x, seed0, wrench7, tau_ext, sdot7, XdotOut{xdot7, jac, sd.n_x}, flags, status);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_state_feedback(const StateDev& sd, const DynDev& dd, const FeedbackDev& fb, long long n_env, const double* x, int mode, int seed0,
                                  double* xdot, double* jac, cudaStream_t stream, int* n_launches) {
    const long long n = n_env * sd.n_body;
    if (n == 0) return cudaSuccess;
    auto kern = mode == 0 ? state_feedback_kernel<0> : mode == 1 ? state_feedback_kernel<1> : state_feedback_kernel<2>;
    kern<<<state_blocks(32 * n), 128, 0, stream>>>(sd, dd, fb, n_env, x, seed0, xdot, jac);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t launch_check_finite(const double* a, long long n, int* bad, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const long long blocks = (n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8;
    check_finite_kernel<<<(unsigned)blocks, 256, 0, stream>>>(a, n, bad);
    return cudaGetLastError();
}

}  // namespace pfc
