// pfc_sat.cuh -- oriented-box overlap test of the broad phase.
//
// Follows BB_BB_intersect (/root/reference/src/obb/bb_intersection.jl:2-74): compose
// inv(OBB_a) * X_a_b * OBB_b, add 1e-14 to |R|, then the 15 separating-axis tests of Ericson's
// table 4.1 with strict '<'.  The boolean must be bit-exact against the reference, so every
// product/sum below is an explicitly rounded, never-contracted operation in the reference's
// evaluation order (StaticArrays row-by-column sums, left to right).  Terms that multiply the
// constant 0/1 bottom row of a homogeneous matrix are dropped: adding +-0.0 cannot change a value
// that is later compared or passed through abs().
#pragma once
#include "pfc_math.cuh"
#include "pfc_types.cuh"

namespace pfc {

// M = inv(OBB_a) * X_a_b : the part of the composition that depends on node a only.
struct SatA { double R[9]; double t[3]; double e[3]; };

// Axis-aligned nodes (kind == kNodeInternalAabb: R == I exactly).  The reference multiplies by the identity all the same; with R = I every
// product is x * 1 or x * (+-0) and every sum is x + (+-0), so the composed entries are the operands themselves -- bit for bit for finite
// inputs, up to the sign of a zero, which neither fabs() nor '<' can see.  The identity products are therefore skipped (AABB = false keeps
// the general path: tests/test_device_sat_on_host.py checks that both give the same boolean everywhere).
template <bool AABB = true> PFC_D void sat_prepare_a(const NodeRec& a, const double* __restrict__ Rab, const double* __restrict__ tab, SatA& out) {
    if (AABB && a.kind == kNodeInternalAabb) {   // inv(OBB_a) = [I, -c]
#pragma unroll
        for (int k = 0; k < 9; ++k) out.R[k] = Rab[k];
#pragma unroll
        for (int i = 0; i < 3; ++i) out.t[i] = add_(tab[i], -a.c[i]);
        out.e[0] = a.e[0]; out.e[1] = a.e[1]; out.e[2] = a.e[2];
        return;
    }
    // i_dh_a = [a.R' , (-a.R') * a.c]
    double mt[3];
#pragma unroll
    for (int i = 0; i < 3; ++i)  // row i of a.R' is column i of a.R
        mt[i] = add_(add_(mul_(-a.R[0 + i], a.c[0]), mul_(-a.R[3 + i], a.c[1])), mul_(-a.R[6 + i], a.c[2]));
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double r0 = a.R[0 + i], r1 = a.R[3 + i], r2 = a.R[6 + i];
#pragma unroll
        for (int j = 0; j < 3; ++j) out.R[3 * i + j] = add_(add_(mul_(r0, Rab[0 + j]), mul_(r1, Rab[3 + j])), mul_(r2, Rab[6 + j]));
        out.t[i] = add_(add_(add_(mul_(r0, tab[0]), mul_(r1, tab[1])), mul_(r2, tab[2])), mt[i]);
    }
    out.e[0] = a.e[0]; out.e[1] = a.e[1]; out.e[2] = a.e[2];
}

// Rab/tab: row-major rotation and translation of x_r1_r2 (frame of tree 2 expressed in tree 1).
template <bool AABB = true> PFC_D bool sat_test(const SatA& A, const NodeRec& b) {
    double R[9], aR[9], t[3];
    const bool b_aabb = AABB && b.kind == kNodeInternalAabb;   // OBB_b = [I, c]: the rotation product is the left operand itself
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            R[3 * i + j] = b_aabb ? A.R[3 * i + j]
                                  : add_(add_(mul_(A.R[3 * i], b.R[0 + j]), mul_(A.R[3 * i + 1], b.R[3 + j])), mul_(A.R[3 * i + 2], b.R[6 + j]));
            aR[3 * i + j] = add_(fabs(R[3 * i + j]), 1.0e-14);
        }
        t[i] = add_(add_(add_(mul_(A.R[3 * i], b.c[0]), mul_(A.R[3 * i + 1], b.c[1])), mul_(A.R[3 * i + 2], b.c[2])), A.t[i]);
    }
    const double ea0 = A.e[0], ea1 = A.e[1], ea2 = A.e[2], eb0 = b.e[0], eb1 = b.e[1], eb2 = b.e[2];
    // All 15 axes are evaluated and OR-ed: the outcome equals the reference's early-exit chain, but
    // the 15 short dependency chains are independent, which is what hides the FP64 latency.
    bool sep = false;
    // face test 1/2: r_a = e_a, r_b = abs_R * e_b
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const double rb = add_(add_(mul_(aR[3 * i], eb0), mul_(aR[3 * i + 1], eb1)), mul_(aR[3 * i + 2], eb2));
        sep |= add_(A.e[i], rb) < fabs(t[i]);
    }
    // face test 2/2: T = |R' t|, r_a = abs_R' * e_a, r_b = e_b
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double T = fabs(add_(add_(mul_(R[j], t[0]), mul_(R[3 + j], t[1])), mul_(R[6 + j], t[2])));
        const double ra = add_(add_(mul_(aR[j], ea0), mul_(aR[3 + j], ea1)), mul_(aR[6 + j], ea2));
        sep |= add_(ra, b.e[j]) < T;
    }
    // edge-edge tests.  R0/R1/R2 are the rows of R; s100(v) = (v1, v0, v0), s221(v) = (v2, v2, v1).
    const double eb100[3] = {eb1, eb0, eb0}, eb221[3] = {eb2, eb2, eb1};
    const int i100[3] = {1, 0, 0}, i221[3] = {2, 2, 1};
    // cross 1/3: a0 x b_j
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double T = fabs(sub_(mul_(t[2], R[3 + j]), mul_(t[1], R[6 + j])));
        const double ra = add_(mul_(ea1, aR[6 + j]), mul_(ea2, aR[3 + j]));
        const double rb = add_(mul_(eb100[j], aR[i221[j]]), mul_(eb221[j], aR[i100[j]]));
        sep |= add_(ra, rb) < T;
    }
    // cross 2/3: a1 x b_j
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double T = fabs(sub_(mul_(t[0], R[6 + j]), mul_(t[2], R[j])));
        const double ra = add_(mul_(ea0, aR[6 + j]), mul_(ea2, aR[j]));
        const double rb = add_(mul_(eb100[j], aR[3 + i221[j]]), mul_(eb221[j], aR[3 + i100[j]]));
        sep |= add_(ra, rb) < T;
    }
    // cross 3/3: a2 x b_j
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const double T = fabs(sub_(mul_(t[1], R[j]), mul_(t[0], R[3 + j])));
        const double ra = add_(mul_(ea0, aR[3 + j]), mul_(ea1, aR[j]));
        const double rb = add_(mul_(eb100[j], aR[6 + i221[j]]), mul_(eb221[j], aR[6 + i100[j]]));
        sep |= add_(ra, rb) < T;
    }
    return !sep;
}

// ---- filtered test: the same boolean, decided in single precision wherever a certified error bound allows -------------------------
// The reference's FP64 arithmetic matters only for the boolean, and almost every test is far from its decision boundary.  sat_filter
// evaluates the 15 axes in float (contraction allowed) from records staged once in float, and returns kSatSeparated / kSatOverlap only
// when every axis it relies on is decided by more than an error bound B; otherwise kSatUndecided, and the caller runs the exact
// sat_prepare_a<false> + sat_test<false> on the FP64 records.
//
// Error bound.  Let m* be an axis margin |T| - (r_a + r_b) evaluated in exact arithmetic from the FP64 inputs, m_ref the reference's
// FP64 value (the comparison 'r_a + r_b < |T|' separates iff m_ref > 0) and m_f the filter's value.  If |m_f - m_ref| <= B, then
// m_f > B implies m_ref > 0 (separating axis) and m_f < -B implies m_ref < 0 (not separating); m_ref = 0 stays undecided.
//   Magnitudes.  Every rotation R (node records and the per-problem R_ab) passes ||R'R - I||_max <= 2^-20 (checked in FP64 when it is
//   staged; a record that fails is poisoned with a NaN and never decided), so ||R||_2 <= rho = sqrt(1 + 3 * 2^-20): every entry, row
//   and column norm of R, M = R_a' R_ab and R_tot = M R_b is at most rho^3, and powers of rho up to rho^6 < 1 + 2^-16 are absorbed by
//   the margin below.  With s = sum|c_a| + sum|c_b| + sum|t_ab| + sum|e_a| + sum|e_b| (all inputs, not the composed t: t can be the
//   small difference of large frame offsets) Cauchy-Schwarz gives ||t||_2 <= s, sum_i |t_i| <= sqrt(3) s, |aR_ij| <= 1 + 1e-14
//   (the reference's guard added to |R|), r_a + r_b <= s.
//   Per-operation bound: a sum of n products in any order, fused or not, is within gamma_n = n u (first order) of the exact sum,
//   relative to the sum of the absolute terms; u = 2^-53 for the reference, u = 2^-24 for float, whose inputs are rounded once more
//   (one extra u per input factor).  First-order errors of the composed quantities, in units of u (lengths in units of u s):
//                         M      t_A = R_a'(t_ab - c_a)   t      R_tot   aR = |R_tot| + 1e-14
//     reference (FP64)    3      7                        14     9       10
//     filter (float)      5      6                        16     13      14
//   Axes (propagated errors of the operands + the axis' own roundings, including r_a + r_b):
//     face a_i:   T = |t_i|                        reference 14 + 13 + 1 = 28      filter 16 + 18 + 2 = 36
//     face b_j:   T = |sum_i R_ij t_i|             reference 43 + 13 + 1 = 57      filter 53.2 + 18 + 2 = 73.2
//     a_i x b_j:  T = |t_k R_lj - t_l R_kj|        reference 34.5 + 13 = 47.5      filter 43 + 18 = 61
//   (face b_j's T: sum_i |dR_ij| |t_i| <= 9 u sqrt(3) s, sum_i |R_ij| |dt_i| <= 14 u s sqrt(3), rounding 3 u s for the reference; 13 and
//   16 in place of 9 and 14 for the filter.)  Hence |m_f - m_ref| <= 74 u_32 s + 57 u_64 s to first order.  B takes twice that, which
//   also covers the second-order terms, the rho powers, the rounding of the 1e-14 guard to float and the float rounding of s, B and the
//   final subtraction: B = (148 u_32 + 114 u_64) s + 2^-100.
//   The absolute 2^-100 term covers float underflow: an operand below 2^-126 loses relative precision, but each operation's absolute
//   error is then at most 2^-150, and no more than ~100 of them (scaled by at most rho^3 or by s, which the relative term covers)
//   reach a margin.  The build keeps IEEE denormals (no -ftz).
//   Non-finite inputs: a NaN anywhere makes s or the margins NaN; an infinity makes s infinite; s >= 2^100 (where float
//   intermediates could overflow) sets B = +inf.  Both comparisons below are false for NaN and for B = +inf, so such tests are
//   undecided, never decided wrongly.
enum { kSatSeparated = 0, kSatOverlap = 1, kSatUndecided = 2 };

// Node record of the filter, staged in shared memory: 80 B (five 16 B loads; five consecutive records cover all 32 banks once).
// s = sum|c| + sum|e| (this node's share of the scale), kind / right copied for the traversal's rebuild.
struct __align__(16) FiltNode {
    float c[3], e[3];
    float R[9];
    float s;
    int32_t kind, right;
    int32_t pad_[2];
};
static_assert(sizeof(FiltNode) == 80, "FiltNode is five 16 B words");

// Per-problem transform of the filter: R_ab, t_ab rounded to float, and st = sum|t_ab|.
struct FiltXf { float R[9]; float t[3]; float st; };

PFC_HD bool filt_rotation_ok(const double* R) {   // ||R'R - I||_max <= 2^-20 (false for NaN / inf entries)
    bool ok = true;
    for (int i = 0; i < 3; ++i)
        for (int j = i; j < 3; ++j) {
            const double d = R[i] * R[j] + R[3 + i] * R[3 + j] + R[6 + i] * R[6 + j] - (i == j ? 1.0 : 0.0);
            ok = ok && d >= -0x1p-20 && d <= 0x1p-20;
        }
    return ok;
}

PFC_HD void filt_node_from(const NodeRec& n, FiltNode& f) {
    float s = 0.0f;
    for (int k = 0; k < 3; ++k) { f.c[k] = (float)n.c[k]; f.e[k] = (float)n.e[k]; s += fabsf(f.c[k]) + fabsf(f.e[k]); }
    for (int k = 0; k < 9; ++k) f.R[k] = (float)n.R[k];
    f.s = filt_rotation_ok(n.R) ? s : NAN;   // NaN: every test of this node is undecided
    f.kind = n.kind; f.right = n.right; f.pad_[0] = f.pad_[1] = 0;
}

PFC_HD void filt_xf_from(const double* Rab, const double* tab, FiltXf& f) {
    float st = 0.0f;
    for (int k = 0; k < 9; ++k) f.R[k] = (float)Rab[k];
    for (int k = 0; k < 3; ++k) { f.t[k] = (float)tab[k]; st += fabsf(f.t[k]); }
    f.st = filt_rotation_ok(Rab) ? st : NAN;
}

PFC_HD int sat_filter(const FiltNode& a, const FiltNode& b, const FiltXf& X) {
    constexpr float kRel = (float)(148.0 * 0x1p-24 + 114.0 * 0x1p-53);
    const float s = a.s + b.s + X.st;
    const float B = s < 0x1p100f ? fmaf(kRel, s, 0x1p-100f) : INFINITY;
    // M = R_a' R_ab, t_A = R_a' (t_ab - c_a), R = M R_b, t = M c_b + t_A
    float M[9], R[9], aR[9], t[3];
    const float d0 = X.t[0] - a.c[0], d1 = X.t[1] - a.c[1], d2 = X.t[2] - a.c[2];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float r0 = a.R[i], r1 = a.R[3 + i], r2 = a.R[6 + i];
#pragma unroll
        for (int j = 0; j < 3; ++j) M[3 * i + j] = r0 * X.R[j] + r1 * X.R[3 + j] + r2 * X.R[6 + j];
        t[i] = r0 * d0 + r1 * d1 + r2 * d2;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            R[3 * i + j] = M[3 * i] * b.R[j] + M[3 * i + 1] * b.R[3 + j] + M[3 * i + 2] * b.R[6 + j];
            aR[3 * i + j] = fabsf(R[3 * i + j]) + 1.0e-14f;
        }
        t[i] += M[3 * i] * b.c[0] + M[3 * i + 1] * b.c[1] + M[3 * i + 2] * b.c[2];
    }
    // m = T - (r_a + r_b) per axis: some axis certainly separating -> separated; all certainly not -> overlapping
    bool sep = false, ovl = true;
    auto axis = [&](float T, float r) { const float m = T - r; sep |= m > B; ovl &= m < -B; };
#pragma unroll
    for (int i = 0; i < 3; ++i) axis(fabsf(t[i]), a.e[i] + (aR[3 * i] * b.e[0] + aR[3 * i + 1] * b.e[1] + aR[3 * i + 2] * b.e[2]));
#pragma unroll
    for (int j = 0; j < 3; ++j)
        axis(fabsf(R[j] * t[0] + R[3 + j] * t[1] + R[6 + j] * t[2]), (aR[j] * a.e[0] + aR[3 + j] * a.e[1] + aR[6 + j] * a.e[2]) + b.e[j]);
    const int i100[3] = {1, 0, 0}, i221[3] = {2, 2, 1};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const float eb100 = b.e[i100[j]], eb221 = b.e[i221[j]];
        axis(fabsf(t[2] * R[3 + j] - t[1] * R[6 + j]),
             (a.e[1] * aR[6 + j] + a.e[2] * aR[3 + j]) + (eb100 * aR[i221[j]] + eb221 * aR[i100[j]]));
        axis(fabsf(t[0] * R[6 + j] - t[2] * R[j]),
             (a.e[0] * aR[6 + j] + a.e[2] * aR[j]) + (eb100 * aR[3 + i221[j]] + eb221 * aR[3 + i100[j]]));
        axis(fabsf(t[1] * R[j] - t[0] * R[3 + j]),
             (a.e[0] * aR[3 + j] + a.e[1] * aR[j]) + (eb100 * aR[6 + i221[j]] + eb221 * aR[6 + i100[j]]));
    }
    return sep ? kSatSeparated : (ovl ? kSatOverlap : kSatUndecided);
}

}  // namespace pfc
