// pfc_radau.cu -- the dense linear algebra of the reference's Radau step, batched over environments.
//
// updateInvC! (/root/reference/src/radau/radau_functions.jl:88-99) forms, for every stage i, the complex matrix
//     C_i = (h^-1 lambda_i) I - J      (the reference keeps -J in neg_J and adds the shift on the diagonal)
// and inverts it with LAPACK getrf! + getri!.  For a batch of environments this is thousands of independent NX x NX complex
// inversions (NX = 48 for test/boxes.jl), far too small for a library call per matrix and slow through batched cuSOLVER
// (17.6 ms for 4096 matrices measured on B200).  Here one CTA inverts one matrix in shared memory: in-place Gauss-Jordan with
// partial (row) pivoting, the pivot search by one warp, the rank-1 update by all threads; the column permutation is undone at
// the end.  Input is the REAL matrix -J shared by the stages of an environment plus the complex shift; output is interleaved
// (re, im) row-major, which is the memory layout of a torch.complex128 / Julia ComplexF64 array.
//
// The rest of the file is the adaptive step around those inverses (solveRadau, radau_solve.jl:1-34, for a batch): per round of attempts
// the plan kernel lists the pending environments' matrices and stage states; per Newton iteration the stage states of the still-active
// environments are packed (gather), evaluated by calcXd! on the host side of the launch sequence, and radau_newton_kernel (one CTA per
// active environment) does calcEw!, the mat-vecs with invC, updateStageX! and the convergence / divergence tests; radau_controller_kernel
// (one thread per environment) applies calc_and_update_h! / update_rule! at the end of each round.  A roll-out through knot times wraps that
// step: radau_select_kernel gathers the environments still under way into compact arrays the step runs on, radau_finish_kernel scatters them
// back and moves the environments that landed on their knot to the next one.
#include <cuda_runtime.h>

#include <algorithm>

#include <cub/block/block_scan.cuh>

#define PFC_RADAU_TABLE_STORAGE __constant__
#include "pfc_launch.h"
#include "pfc_radau_step.cuh"

namespace pfc {

namespace {

struct cplx { double re, im; };
__device__ __forceinline__ cplx cmul(const cplx& a, const cplx& b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ cplx cinv(const cplx& a) {   // Smith's algorithm (what LAPACK's zladiv guards against: overflow in |a|^2)
    if (fabs(a.re) >= fabs(a.im)) { const double r = a.im / a.re, d = a.re + a.im * r; return {1.0 / d, -r / d}; }
    const double r = a.re / a.im, d = a.re * r + a.im;
    return {r / d, -1.0 / d};
}

// grid: one CTA per matrix; dynamic shared memory: cplx A[n][n + 1] (odd-ish pitch) | int piv[n]
__global__ void __launch_bounds__(256) radau_inv_c_kernel(int n, const double* __restrict__ neg_J, const double* __restrict__ shift, const int* __restrict__ index,
                                                          double* __restrict__ inv_c, int* __restrict__ info) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int pitch = n + 1;
    cplx* A = reinterpret_cast<cplx*>(smem_raw);
    int* piv = reinterpret_cast<int*>(A + (size_t)n * pitch);
    __shared__ int s_p;
    __shared__ cplx s_pivinv;
    const long long mat = blockIdx.x;
    const long long src = index ? index[mat] : mat;             // environment whose -J this matrix is built from
    const double* J = neg_J + src * (long long)n * n;
    const cplx sh = {shift[2 * mat], shift[2 * mat + 1]};
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e - i * n;
        A[i * pitch + j] = {J[e] + (i == j ? sh.re : 0.0), (i == j ? sh.im : 0.0)};
    }
    __syncthreads();
    bool singular = false;
    for (int k = 0; k < n; ++k) {
        if (threadIdx.x < 32) {   // pivot: the row i >= k with the largest |re| + |im| in column k (izamax's measure)
            double best = -1.0; int bi = k;
            for (int i = k + (int)threadIdx.x; i < n; i += 32) {
                const double v = fabs(A[i * pitch + k].re) + fabs(A[i * pitch + k].im);
                if (v > best) { best = v; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
            }
            if (threadIdx.x == 0) { s_p = bi; piv[k] = bi; s_pivinv = (best > 0.0) ? cinv(A[bi * pitch + k]) : cplx{0.0, 0.0}; if (!(best > 0.0)) singular = true; }
        }
        __syncthreads();
        const int p = s_p;
        if (p != k) for (int j = threadIdx.x; j < n; j += blockDim.x) { const cplx t = A[k * pitch + j]; A[k * pitch + j] = A[p * pitch + j]; A[p * pitch + j] = t; }
        __syncthreads();
        // scale the pivot row (its pivot entry becomes the inverse of the pivot), then eliminate column k from every other row
        const cplx pinv = s_pivinv;
        for (int j = threadIdx.x; j < n; j += blockDim.x) A[k * pitch + j] = (j == k) ? pinv : cmul(A[k * pitch + j], pinv);
        __syncthreads();
        for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
            const int i = e / n, j = e - i * n;
            if (i == k || j == k) continue;
            const cplx f = A[i * pitch + k], r = A[k * pitch + j];
            A[i * pitch + j].re -= f.re * r.re - f.im * r.im;
            A[i * pitch + j].im -= f.re * r.im + f.im * r.re;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            if (i != k) { const cplx f = A[i * pitch + k]; const cplx t = cmul(f, pinv); A[i * pitch + k] = {-t.re, -t.im}; }
        __syncthreads();
    }
    for (int k = n - 1; k >= 0; --k) {   // undo the row interchanges as column interchanges, last first
        const int p = piv[k];
        if (p != k) for (int i = threadIdx.x; i < n; i += blockDim.x) { const cplx t = A[i * pitch + k]; A[i * pitch + k] = A[i * pitch + p]; A[i * pitch + p] = t; }
        __syncthreads();
    }
    double* out = inv_c + mat * 2ll * n * n;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n, j = e - i * n;
        out[2 * e] = A[i * pitch + j].re; out[2 * e + 1] = A[i * pitch + j].im;
    }
    if (threadIdx.x == 0 && singular && info) atomicOr(info, 1);
}

constexpr int kPlanThreads = 1024;

__global__ void __launch_bounds__(kPlanThreads) radau_plan_kernel(RadauBufs b, int mode) {
    using Scan = cub::BlockScan<int, kPlanThreads>;
    __shared__ typename Scan::TempStorage tmp;
    int base_s = 0, base_e = 0;
    for (long long c0 = 0; c0 < b.n_env; c0 += kPlanThreads) {
        const long long e = c0 + threadIdx.x;
        int flag = 0, s = 0;
        if (e < b.n_env) {
            RadauEnv& en = b.env[e];
            if (mode == 2) { en.pending = 1; en.n_rejected = 0; en.n_evals = 0; }
            flag = mode == 0 ? en.active : en.pending;
            s = flag ? 2 * en.rule - 1 : 0;
        }
        int ps, pe, agg_s, agg_e;
        Scan(tmp).ExclusiveSum(s, ps, agg_s);
        __syncthreads();
        Scan(tmp).ExclusiveSum(flag, pe, agg_e);
        __syncthreads();
        if (flag) {
            RadauEnv& en = b.env[e];
            const int pos = base_s + ps;
            b.env_list[base_e + pe] = (int)e;
            b.state_pos[e] = pos;
            for (int st = 0; st < s; ++st) b.state_list[pos + st] = (int)e * 8 + st;
            if (mode != 0) {   // a new attempt: its matrices (h^-1 lambda_i I - J)^-1 and simple_newton!'s initial state
                const RadauTableData& T = kRadauTables[en.rule - 1];
                const double h_inv = 1.0 / en.h;
                b.inv_base[e] = pos;
                for (int st = 0; st < s; ++st) {
                    b.index[pos + st] = (int)e;
                    b.shift[2 * (pos + st)] = h_inv * T.lam_re[st];
                    b.shift[2 * (pos + st) + 1] = h_inv * T.lam_im[st];
                }
                radau_attempt_begin(en);
            }
        }
        base_s += agg_s;
        base_e += agg_e;
    }
    if (threadIdx.x == 0) { b.counts[0] = base_s; b.counts[1] = base_e; }
}

__global__ void radau_prepare_kernel(RadauBufs b, const int* __restrict__ flags, int* __restrict__ status) {
    const long long n = b.n_env * (long long)b.nx * b.nx, nf = b.n_env * (long long)b.n_ins;
    int bad = 0;
    for (long long id = blockIdx.x * (long long)blockDim.x + threadIdx.x; id < n; id += (long long)gridDim.x * blockDim.x) {
        b.jac[id] = -b.jac[id];
        if (id < nf) bad |= flags[id] & (2 | 8);   // PFC_FLAG_NONFINITE | PFC_FLAG_OVERFLOW
    }
    if (bad) atomicOr(status, bad);
}

// one CTA per packed state: its stage vector (x0 at the first iteration of an attempt, which also initialises the stage), tau_ext, the
// environment's contact parameters and, with a body or a feedback table, the environment's row index (the rows themselves are not copied)
__global__ void __launch_bounds__(64) radau_gather_kernel(RadauBufs b) {
    const long long p = blockIdx.x;
    const int code = b.state_list[p], e = code >> 3, st = code & 7;
    const bool first = b.env[e].k_iter == 0;
    if (b.rowp && threadIdx.x == 0) b.rowp[p] = b.row ? b.row[e] : e;
    if (b.fb_rowp && threadIdx.x == 0) b.fb_rowp[p] = b.fb_row ? b.fb_row[e] : e;
    double* Xs = b.X + ((long long)e * b.s_max + st) * b.nx;
    const double* x0 = b.x + (long long)e * b.nx;
    for (int n = threadIdx.x; n < b.nx; n += blockDim.x) {
        const double v = first ? x0[n] : Xs[n];
        if (first) Xs[n] = v;
        b.Xp[p * b.nx + n] = v;
    }
    if (b.tau)
        for (int n = threadIdx.x; n < b.nv; n += blockDim.x) b.taup[p * b.nv + n] = b.tau[(long long)e * b.nv + n];
    if (b.params) {
        const double* src = reinterpret_cast<const double*>(b.params + (long long)e * b.n_ins);
        double* dst = reinterpret_cast<double*>(b.paramp + p * b.n_ins);
        for (int n = threadIdx.x; n < b.n_ins * (int)(sizeof(InsParam) / sizeof(double)); n += blockDim.x) dst[n] = src[n];
    }
}

// one Newton iteration of one environment (radau.py _simple_newton loop body); every element summed by one thread in a fixed order
constexpr int kNewtonThreads = 128;
__global__ void __launch_bounds__(kNewtonThreads) radau_newton_kernel(RadauBufs b) {
    extern __shared__ __align__(16) double sm[];
    __shared__ RadauEnv ctl;
    __shared__ double red[kRadauMaxStage];
    __shared__ unsigned div_mask;
    __shared__ int decision;
    const int e = b.env_list[blockIdx.x];
    const int nx = b.nx;
    if (threadIdx.x == 0) { ctl = b.env[e]; div_mask = 0u; }
    __syncthreads();
    const RadauTableData& T = kRadauTables[ctl.rule - 1];
    const int s = T.s, sn = s * nx;
    const double h = ctl.h, h_inv = 1.0 / h;
    double* x0 = sm;
    double* X = x0 + nx;
    double* F = X + sn;
    double* st = F + sn;
    double* ar = st + sn;
    double* ai = ar + sn;
    double* br = ai + sn;
    double* bi = br + sn;
    const double* x0g = b.x + (long long)e * nx;
    double* Xg = b.X + (long long)e * b.s_max * nx;
    const double* Fg = b.Fp + (long long)b.state_pos[e] * nx;
    const double* inv = b.invc + (long long)b.inv_base[e] * 2 * nx * nx;
    for (int id = threadIdx.x; id < sn; id += blockDim.x) { X[id] = Xg[id]; F[id] = Fg[id]; }
    for (int n = threadIdx.x; n < nx; n += blockDim.x) x0[n] = x0g[n];
    __syncthreads();
    for (int id = threadIdx.x; id < sn; id += blockDim.x) st[id] = radau_store(T, h, id / nx, id % nx, nx, x0, X, F);
    __syncthreads();
    if (threadIdx.x < s) {   // store_i . store_i
        double a = 0.0;
        for (int n = 0; n < nx; ++n) a = a + st[threadIdx.x * nx + n] * st[threadIdx.x * nx + n];
        red[threadIdx.x] = a;
    }
    for (int id = threadIdx.x; id < sn; id += blockDim.x) radau_ew(T, h_inv, id / nx, id % nx, nx, st, &ar[id], &ai[id]);
    __syncthreads();
    for (int id = threadIdx.x; id < sn; id += blockDim.x) {
        const int i = id / nx;
        radau_matvec_row(inv + (long long)i * 2 * nx * nx, nx, id % nx, ar + i * nx, ai + i * nx, &br[id], &bi[id]);
    }
    __syncthreads();
    unsigned mask = 0u;
    for (int id = threadIdx.x; id < sn; id += blockDim.x) {
        const double u = radau_update(T, id / nx, id % nx, nx, br, bi);
        st[id] = u;
        if (fabs(u) > 1.0e1) mask |= 1u << (id / nx);
    }
    if (mask) atomicOr(&div_mask, mask);
    __syncthreads();
    // updateStageX!: stages in order up to the first whose update exceeds 10
    const int first_div = div_mask ? __ffs(div_mask) - 1 : s;
    for (int id = threadIdx.x; id < first_div * nx; id += blockDim.x) { X[id] = X[id] - st[id]; Xg[id] = X[id]; }
    if (threadIdx.x == 0) {
        double residual = 0.0;
        for (int i = 0; i < s; ++i) residual += red[i];
        ctl.n_evals += s;
        decision = radau_newton_decide(ctl, ctl.k_iter + 1, residual, div_mask != 0u, b.tol_newton);
    }
    __syncthreads();
    if (decision == kRadauConverged) {   // update_x_err_norm! with this iteration's F, the updated last stage and invC of stage 0
        const double* xx0 = b.xx0 + (long long)e * nx;
        for (int n = threadIdx.x; n < nx; n += blockDim.x) ar[n] = radau_err_d(T, h, n, nx, xx0, F);
        __syncthreads();
        for (int r = threadIdx.x; r < nx; r += blockDim.x) ai[r] = radau_err_term(inv, nx, r, ar, X[(s - 1) * nx + r], x0[r]);
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0.0;
            for (int r = 0; r < nx; ++r) a = a + ai[r];
            ctl.err_norm = sqrt(a / nx);
        }
    }
    if (threadIdx.x == 0) {
        if (decision != kRadauIterate) ctl.active = 0;
        b.env[e] = ctl;
    }
}

// calc_and_update_h! / update_rule! of every environment whose attempt just ended; principal_value! on acceptance
__global__ void __launch_bounds__(128) radau_controller_kernel(RadauBufs b) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= b.n_env) return;
    RadauEnv ctl = b.env[e];
    if (!ctl.pending) return;
    const int s = 2 * ctl.rule - 1, k = ctl.k_iter;
    double h_taken = 0.0;
    const int rc = radau_control(ctl, b.max_rule, b.h_max, &h_taken);
    if (rc == kRadauAccepted) {
        double* x = b.x + e * b.nx;
        const double* Xl = b.X + (e * b.s_max + (s - 1)) * b.nx;
        for (int n = 0; n < b.nx; ++n) x[n] = Xl[n];
        for (int k2 = 0; k2 < b.n_body; ++k2) {
            if (b.bodies[k2].joint != 1) continue;
            double* p = x + b.bodies[k2].q0;
            const double n2 = p[0] * p[0] + p[1] * p[1] + p[2] * p[2];
            if (n2 > 1.0) { p[0] = -p[0] / n2; p[1] = -p[1] / n2; p[2] = -p[2] / n2; }
        }
        b.t[e] = b.t[e] + h_taken;
        b.h_taken[e] = h_taken;
        if (b.stats) { int* o = b.stats + 4 * e; o[0] = s; o[1] = k; o[2] = ctl.n_rejected; o[3] = ctl.n_evals; }
        ctl.pending = 0;
    } else if (rc == kRadauRetry) {
        ctl.n_rejected += 1;
    } else {
        atomicOr(b.counts + 2, rc == kRadauBadH ? 1 : 2);
        ctl.pending = 0;
    }
    b.env[e] = ctl;
}

// roll-out round: the environments with a knot ahead and steps left, in environment order, gathered into the compact slots
__global__ void __launch_bounds__(kPlanThreads) radau_select_kernel(RadauRolloutBufs b, int check) {
    using Scan = cub::BlockScan<int, kPlanThreads>;
    __shared__ typename Scan::TempStorage tmp;
    int bad = 0;
    if (check)
        for (long long e = threadIdx.x; e < b.n_env; e += kPlanThreads) bad |= !(b.knots[0] - b.t[e] >= kRadauHMin);
    if (__syncthreads_or(bad)) {
        if (threadIdx.x == 0) { b.count[0] = 0; b.count[1] = 1; }
        return;
    }
    int base = 0;
    for (long long c0 = 0; c0 < b.n_env; c0 += kPlanThreads) {
        const long long e = c0 + threadIdx.x;
        int flag = 0;
        if (e < b.n_env) flag = b.knot[e] < b.n_knot && b.steps[e] < b.max_steps;
        int pos, agg;
        Scan(tmp).ExclusiveSum(flag, pos, agg);
        __syncthreads();
        if (flag) {
            const long long p = base + pos;
            const int k = b.knot[e];
            RadauEnv en = b.env[e];
            const double t = b.t[e];
            b.h_save[p] = radau_knot_begin(en, t, b.knots[k]);
            b.list[p] = (int)e;
            b.env_c[p] = en;
            b.t_c[p] = t;
            for (int n = 0; n < b.nx; ++n) b.x_c[p * b.nx + n] = b.x[e * b.nx + n];
            if (b.tau) {
                const double* row = b.tau + ((long long)k * b.n_env + e) * b.nv;
                for (int n = 0; n < b.nv; ++n) b.tau_c[p * b.nv + n] = row[n];
            }
            if (b.params)
                for (int n = 0; n < b.n_ins; ++n) b.params_c[p * b.n_ins + n] = b.params[e * b.n_ins + n];
            if (b.fb_list) b.fb_list[p] = (int)((b.n_seg == 1 ? 0 : (long long)k) * b.n_env + e);
        }
        base += agg;
    }
    if (threadIdx.x == 0) { b.count[0] = base; b.count[1] = 0; }
}

// one thread per compact slot: the step's end relative to the knot, then everything back to the environment's own arrays
__global__ void __launch_bounds__(128) radau_finish_kernel(RadauRolloutBufs b, long long n_active) {
    const long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (p >= n_active) return;
    const long long e = b.list[p];
    const int k = b.knot[e];
    RadauEnv en = b.env_c[p];
    double t_new;
    const bool hit = radau_knot_end(en, b.t[e], b.knots[k], b.h_c[p], b.h_save[p], &t_new);
    b.t[e] = t_new;
    b.env[e] = en;
    b.steps[e] += 1;
    if (hit) b.knot[e] = k + 1;
    int* o = b.stats + 4 * e;
    const int* s = b.stats_c + 4 * p;
    o[0] += hit; o[1] += 1; o[2] += s[2]; o[3] += s[3];
    const double* xs = b.x_c + p * b.nx;
    double* xd = b.x + e * b.nx;
    double* row = hit && b.x_knot ? b.x_knot + ((long long)k * b.n_env + e) * b.nx : nullptr;
    for (int n = 0; n < b.nx; ++n) {
        xd[n] = xs[n];
        if (row) row[n] = xs[n];
    }
}

}  // namespace

cudaError_t launch_radau_select(const RadauRolloutBufs& b, int check, cudaStream_t stream) {
    radau_select_kernel<<<1, kPlanThreads, 0, stream>>>(b, check);
    return cudaGetLastError();
}

cudaError_t launch_radau_finish(const RadauRolloutBufs& b, long long n_active, cudaStream_t stream) {
    if (n_active == 0) return cudaSuccess;
    radau_finish_kernel<<<(unsigned)((n_active + 127) / 128), 128, 0, stream>>>(b, n_active);
    return cudaGetLastError();
}

cudaError_t launch_radau_plan(const RadauBufs& b, int mode, cudaStream_t stream) {
    radau_plan_kernel<<<1, kPlanThreads, 0, stream>>>(b, mode);
    return cudaGetLastError();
}

cudaError_t launch_radau_prepare(const RadauBufs& b, const int* flags, int* status, cudaStream_t stream) {
    const long long n = b.n_env * (long long)b.nx * b.nx;
    const long long blocks = std::min<long long>((n + 255) / 256, 148 * 16);
    radau_prepare_kernel<<<(unsigned)std::max<long long>(blocks, 1), 256, 0, stream>>>(b, flags, status);
    return cudaGetLastError();
}

cudaError_t launch_radau_gather(const RadauBufs& b, long long n_states, cudaStream_t stream) {
    if (n_states == 0) return cudaSuccess;
    radau_gather_kernel<<<(unsigned)n_states, 64, 0, stream>>>(b);
    return cudaGetLastError();
}

cudaError_t launch_radau_newton(const RadauBufs& b, long long n_active, cudaStream_t stream) {
    if (n_active == 0) return cudaSuccess;
    const size_t smem = sizeof(double) * ((size_t)b.nx + 7 * (size_t)b.s_max * b.nx);
    {
        struct Tag {};
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag>();
        if (smem > sl.smem) {
            cudaError_t e = cudaFuncSetAttribute(radau_newton_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            sl.smem = smem;
        }
    }
    radau_newton_kernel<<<(unsigned)n_active, kNewtonThreads, smem, stream>>>(b);
    return cudaGetLastError();
}

cudaError_t launch_radau_controller(const RadauBufs& b, cudaStream_t stream) {
    if (b.n_env == 0) return cudaSuccess;
    radau_controller_kernel<<<(unsigned)((b.n_env + 127) / 128), 128, 0, stream>>>(b);
    return cudaGetLastError();
}

cudaError_t launch_radau_inv_c(long long n_mat, int n, const double* neg_J, const double* shift, const int* index, double* inv_c, int* info, cudaStream_t stream) {
    if (n_mat == 0) return cudaSuccess;
    const size_t smem = sizeof(cplx) * (size_t)n * (n + 1) + sizeof(int) * n;
    {
        struct Tag {};
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag>();
        if (smem > sl.smem) {
            cudaError_t e = cudaFuncSetAttribute(radau_inv_c_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            sl.smem = smem;
        }
    }
    radau_inv_c_kernel<<<(unsigned)n_mat, 256, smem, stream>>>(n, neg_J, shift, index, inv_c, info);
    return cudaGetLastError();
}

}  // namespace pfc
