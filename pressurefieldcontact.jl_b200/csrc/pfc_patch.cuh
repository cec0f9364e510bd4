// pfc_patch.cuh -- per-pair narrow phase: clip -> polygon fan -> pressure quadrature -> traction.
//
// Reference (paths relative to /root/reference):
//   tri-tet pair ....... integrate_over!  src/contact_algorithms_non_friction.jl:196-215
//   tet-tet pair ....... integrate_over!  src/contact_algorithms_non_friction.jl:166-194
//   polygon fan ........ integrate_over_polygon_patch!  :217-234,  centroid  src/clip/poly_eight.jl:35-52
//   pressure law ....... fillTractionCacheInnerLoop!  :251-265
//   regularized law .... traction / yes_contact!  src/contact_algorithms_friction.jl:13-30, 50-72
//   (bristle friction: pfc_exact.cuh)
// The reference materialises a TractionCache list between the narrow phase and friction; here
// every quadrature point is consumed immediately by an accumulator (Accum::point) so nothing is
// written to memory.  The work is split in two stages so that a warp can keep its lanes busy:
//   stage A  clip_pair():        one candidate pair -> a PolyRec (clipped polygon in frame r2, its
//                                normal, centroid and the tet's pressure gradient), or nothing;
//   stage B  integrate_subtri(): one (polygon, edge) sub-triangle -> its 1 or 3 quadrature points.
// Most candidate pairs die in stage A; stage B is where the quadrature + friction FLOPs are, and
// its work items are dense.  integrate_pair() composes both for one-thread-per-pair callers.
#pragma once
#include "pfc_clip.cuh"
#include "pfc_math.cuh"
#include "pfc_types.cuh"

namespace pfc {

// XiaoGimbutas triangle rules 1 and 2 (src/clip/quadrature.jl:21-41)
#define PFC_Q1 0.33333333333333331483
#define PFC_QA 0.16666666666666674068
#define PFC_QB 0.66666666666666651864

enum AccMode { ACC_REGULARIZED = 0, ACC_DUMP = 4 };

// per (environment, instruction) data in mode T
template <class T> struct PatchCtx {
    Xform<T> x21;   // x_r2_r1: mesh-1 frame -> mesh-2 frame
    Xform<T> x12;   // its inverse (tet-tet only)
    Vec3<T> w_ang, w_lin;  // twist of r2 w.r.t. r1, expressed in r2
    double chi, Ebar1, Ebar2;
    int n_quad;
};

// A clipped contact polygon, ready for quadrature (stage A output / stage B input).
template <class T> struct PolyRec {
    Vec3<T> v[8];     // vertices in r2
    Vec3<T> nrm;      // unit normal, pointing into body 2
    Vec3<T> cen;      // area-weighted centroid
    double eps_r[4];  // pressure field of tet 2: gradient (0..2), offset (3)
    int n;
};

template <class T> PFC_D T clamped_piecewise(const T& x, double x1, double slope, double y1, double y2) {
    const T y = y1 + (x - x1) * slope;
    if (val(y) > y1) return T(y1);  // clamp(y, y2, y1): y2 <= y1
    if (val(y) < y2) return T(y2);
    return y;
}

template <class T> PFC_D Vec3<T> sub_proj(const Vec3<T>& v, const Vec3<T>& n) {  // vec_sub_vec_proj (muladd form)
    const T t = -dot(v, n);
    return mk<T>(fma_(t, n.x, v.x), fma_(t, n.y, v.y), fma_(t, n.z, v.z));
}

// Consumer of the quadrature points of the REGULARIZED friction model (and of the debug dump).  Bristle instructions do not come
// through here: pfc_exact.cuh evaluates them in the reference's operation order.
template <class T, int NA = 6> struct Accum {
    int mode;
    int n_points;
    T a[NA];            // wrench sums: torque (0..2), force (3..5)
    const double* fp;   // friction parameters (InsDev::p)
    Vec3<T> w_ang, w_lin;
    double* dump;       // ACC_DUMP: 8 doubles per point
    int dump_cap;

    PFC_D void reset(int m) {
        mode = m; n_points = 0;
#pragma unroll
        for (int k = 0; k < NA; ++k) a[k] = T(0.0);
    }

    PFC_D void point(const Vec3<T>& n, const Vec3<T>& r, const T& dA, const T& p) {
        const T p_dA = p * dA;
        if (mode == ACC_REGULARIZED) {
            // fp: mu_s, mu_d, v_c, v_mu_s, v_mu_d, slope, 1 / v_c
            const Vec3<T> vel = w_lin + cross(w_ang, r);
            const Vec3<T> vt = sub_proj(vel, n);
            const T mag2 = dot(vt, vt);
            const double mu_s = fp[0], v_c = fp[2];
            T coef;
            if (val(mag2) < v_c * v_c) {
                coef = T(-mu_s * fp[6]) * p_dA;
            } else {
                const T mag = sqrt_(mag2);
                coef = (clamped_piecewise(mag, fp[3], fp[5], mu_s, fp[1]) / mag) * (-p_dA);
            }
            const Vec3<T> tk = mk<T>(p_dA * n.x + vt.x * coef, p_dA * n.y + vt.y * coef, p_dA * n.z + vt.z * coef);
            const Vec3<T> m = cross(r, tk);
            a[0] += m.x; a[1] += m.y; a[2] += m.z; a[3] += tk.x; a[4] += tk.y; a[5] += tk.z;
        } else {  // ACC_DUMP (debug / parity): n(3) r(3) dA p, values only
            if (n_points < dump_cap) {
                double* o = dump + 8 * n_points;
                o[0] = val(n.x); o[1] = val(n.y); o[2] = val(n.z); o[3] = val(r.x); o[4] = val(r.y); o[5] = val(r.z);
                o[6] = val(dA); o[7] = val(p);
            }
        }
        ++n_points;
    }
};

// ---- stage B: one sub-triangle (v1, v2, centroid) of a contact polygon ------------------------------------
template <class T, int NA> PFC_D void quad_point(const Vec3<T>& v1, const Vec3<T>& v2, const Vec3<T>& cen, const Vec3<T>& nrm, double g0, double g1, double g2,
                                                 double g3, double za, double zb, double zc, const T& dA, const PatchCtx<T>& cx, Accum<T, NA>& acc) {
    const Vec3<T> r = mk<T>(v1.x * za + v2.x * zb + cen.x * zc, v1.y * za + v2.y * zb + cen.y * zc, v1.z * za + v2.z * zb + cen.z * zc);
    T eps = fma_(g0, r.x, g3);
    eps = fma_(g1, r.y, eps);
    eps = fma_(g2, r.z, eps);
    const Vec3<T> rd = cx.w_lin + cross(cx.w_ang, r);
    const T ee = -(g0 * rd.x + g1 * rd.y + g2 * rd.z);
    T damp = 1.0 + cx.chi * ee;
    if (val(damp) < 0.0) damp = T(0.0);
    const T p = eps * cx.Ebar2 * damp;
    if (0.0 < val(p)) acc.point(nrm, r, dA, p);
}
template <class T, int NA> PFC_D void integrate_subtri(const Vec3<T>& v1, const Vec3<T>& v2, const Vec3<T>& cen, const Vec3<T>& nrm, const double* eps_r,
                                                       const PatchCtx<T>& cx, Accum<T, NA>& acc) {
    const T area = dot(nrm, cross(v2 - v1, cen - v2) * 0.5);
    if (!(0.0 < val(area))) return;
    const double g0 = eps_r[0], g1 = eps_r[1], g2 = eps_r[2], g3 = eps_r[3];
    if (cx.n_quad == 1) { quad_point(v1, v2, cen, nrm, g0, g1, g2, g3, PFC_Q1, PFC_Q1, PFC_Q1, area * 1.0, cx, acc); return; }
    // rule 2: three points, written out so that their (independent) dependency chains can be interleaved by the scheduler
    const T dA = area * PFC_Q1;
    quad_point(v1, v2, cen, nrm, g0, g1, g2, g3, PFC_QA, PFC_QB, PFC_QA, dA, cx, acc);
    quad_point(v1, v2, cen, nrm, g0, g1, g2, g3, PFC_QB, PFC_QA, PFC_QA, dA, cx, acc);
    quad_point(v1, v2, cen, nrm, g0, g1, g2, g3, PFC_QA, PFC_QA, PFC_QB, dA, cx, acc);
}

// polygon in tetrahedral coordinates of tet 2 -> Cartesian vertices in r2 + area-weighted centroid
template <class T> PFC_D void finish_polygon(const Zeta<T>* z, int n, const TetRec& tet, PolyRec<T>& out) {
    out.n = n;
    for (int k = 0; k < n; ++k) {  // mul_then_un_pad(x_r2_zeta2, .)
        const T z0 = z[k].c[0], z1 = z[k].c[1], z2 = z[k].c[2], z3 = z[k].c[3];
        out.v[k] = mk<T>(tet.v[0] * z0 + tet.v[3] * z1 + tet.v[6] * z2 + tet.v[9] * z3, tet.v[1] * z0 + tet.v[4] * z1 + tet.v[7] * z2 + tet.v[10] * z3,
                         tet.v[2] * z0 + tet.v[5] * z1 + tet.v[8] * z2 + tet.v[11] * z3);
    }
    T cum_sum = T(0.0);
    Vec3<T> cum = mk<T>(T(0.0), T(0.0), T(0.0));
    for (int k = 2; k < n; ++k) {  // fan from vertex 0 (poly_eight.jl:35-52)
        const Vec3<T> a = out.v[0], b = out.v[k - 1], c = out.v[k];
        const T area = dot(out.nrm, cross(b - a, c - b) * 0.5);
        cum = cum + ((a + b + c) * (1.0 / 3.0)) * area;
        cum_sum += area;
    }
    out.cen = out.v[0];
    if (val(cum_sum) != 0.0) { const T inv = 1.0 / cum_sum; out.cen = mk<T>(cum.x * inv, cum.y * inv, cum.z * inv); }
#pragma unroll
    for (int k = 0; k < 4; ++k) out.eps_r[k] = tet.eps_r[k];
}

// ---- stage A -----------------------------------------------------------------------------------------------------
// triangle (mesh 1) against tetrahedron (mesh 2); returns false when the pair contributes nothing
template <class T> PFC_D bool clip_tri_tet(const TriRec& tri, const TetRec& tet, const PatchCtx<T>& cx, PolyRec<T>& out, int& flags) {
    Zeta<T> z[8];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const Vec3<T> p = apply_d(cx.x21, mk<double>(tri.v[3 * k], tri.v[3 * k + 1], tri.v[3 * k + 2]));
#pragma unroll
        for (int i = 0; i < 4; ++i) z[k].c[i] = tet.inv[4 * i] * p.x + tet.inv[4 * i + 1] * p.y + tet.inv[4 * i + 2] * p.z + tet.inv[4 * i + 3];
    }
    const int n = clip_tet(z, 3, flags);
    if (n < 3) return false;
    out.nrm = rot_d(cx.x21, mk<double>(tri.n[0], tri.n[1], tri.n[2]));
    finish_polygon(z, n, tet, out);
    return true;
}

// tetrahedron (mesh 1) against tetrahedron (mesh 2)
template <class T> PFC_D bool clip_tet_tet(const TetRec& t1, const TetRec& t2, const PatchCtx<T>& cx, PolyRec<T>& out, int& flags) {
    // plane of equal pressure in r2: E2 eps2 x_zeta2_r2 - E1 eps1 x_zeta1_r1 x_r1_r2
    T plane[4];
    {
        const double g0 = cx.Ebar1 * t1.eps_r[0], g1 = cx.Ebar1 * t1.eps_r[1], g2 = cx.Ebar1 * t1.eps_r[2], g3 = cx.Ebar1 * t1.eps_r[3];
        const Xform<T>& Y = cx.x12;
        const T p0 = g0 * Y.r[0] + g1 * Y.r[3] + g2 * Y.r[6];
        const T p1 = g0 * Y.r[1] + g1 * Y.r[4] + g2 * Y.r[7];
        const T p2 = g0 * Y.r[2] + g1 * Y.r[5] + g2 * Y.r[8];
        const T p3 = g0 * Y.t[0] + g1 * Y.t[1] + g2 * Y.t[2] + g3;
        plane[0] = cx.Ebar2 * t2.eps_r[0] - p0;
        plane[1] = cx.Ebar2 * t2.eps_r[1] - p1;
        plane[2] = cx.Ebar2 * t2.eps_r[2] - p2;
        plane[3] = cx.Ebar2 * t2.eps_r[3] - p3;
    }
    Vec3<T> v[4], poly[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) v[k] = apply_d(cx.x21, mk<double>(t1.v[3 * k], t1.v[3 * k + 1], t1.v[3 * k + 2]));
    const int n0 = plane_tet(plane, v, poly);
    if (n0 < 3) return false;
    Zeta<T> z[8];
    for (int k = 0; k < n0; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            z[k].c[i] = t2.inv[4 * i] * poly[k].x + t2.inv[4 * i + 1] * poly[k].y + t2.inv[4 * i + 2] * poly[k].z + t2.inv[4 * i + 3];
    zero_small(z, n0);
    const int n = clip_tet(z, n0, flags);
    if (n < 3) return false;
    const T inv_len = 1.0 / sqrt_(plane[0] * plane[0] + plane[1] * plane[1] + plane[2] * plane[2]);
    out.nrm = mk<T>(plane[0] * inv_len, plane[1] * inv_len, plane[2] * inv_len);
    finish_polygon(z, n, t2, out);
    return true;
}

// Cheap, exact rejection before the full clip (stage A1).  A triangle whose three vertices all have
// zeta_i <= 0 for one face i is clipped away whatever the other faces do: every vertex the clipper
// creates is c1 * z_pos - c2 * z_non with c1 >= 0 >= c2, so its zeta_i stays <= 0 and the
// reference returns the empty polygon at face i at the latest.  For tet-tet pairs the equal-pressure
// plane must have tet-1 vertices strictly on both sides (plane_tet_intersection.jl:27-29).
template <class T> PFC_D bool prefilter_pair(const SceneDev& sc, const InsDev& ins, int prim1, int prim2, const PatchCtx<T>& cx) {
    const TetRec& t2 = sc.tets[ins.prim_base2 + prim2];
    if (ins.kind1 == 0) {
        const TriRec& tri = sc.tris[ins.prim_base1 + prim1];
        unsigned all_non_pos = 0xfu;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const Vec3<T> p = apply_d(cx.x21, mk<double>(tri.v[3 * k], tri.v[3 * k + 1], tri.v[3 * k + 2]));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const T z = t2.inv[4 * i] * p.x + t2.inv[4 * i + 1] * p.y + t2.inv[4 * i + 2] * p.z + t2.inv[4 * i + 3];
                if (!(val(z) <= 0.0)) all_non_pos &= ~(1u << i);
            }
        }
        return all_non_pos == 0;
    }
    const TetRec& t1 = sc.tets[ins.prim_base1 + prim1];
    const double g0 = cx.Ebar1 * t1.eps_r[0], g1 = cx.Ebar1 * t1.eps_r[1], g2 = cx.Ebar1 * t1.eps_r[2], g3 = cx.Ebar1 * t1.eps_r[3];
    const Xform<T>& Y = cx.x12;
    const T pl0 = cx.Ebar2 * t2.eps_r[0] - (g0 * Y.r[0] + g1 * Y.r[3] + g2 * Y.r[6]);
    const T pl1 = cx.Ebar2 * t2.eps_r[1] - (g0 * Y.r[1] + g1 * Y.r[4] + g2 * Y.r[7]);
    const T pl2 = cx.Ebar2 * t2.eps_r[2] - (g0 * Y.r[2] + g1 * Y.r[5] + g2 * Y.r[8]);
    const T pl3 = cx.Ebar2 * t2.eps_r[3] - (g0 * Y.t[0] + g1 * Y.t[1] + g2 * Y.t[2] + g3);
    int n_pos = 0, n_neg = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const Vec3<T> v = apply_d(cx.x21, mk<double>(t1.v[3 * k], t1.v[3 * k + 1], t1.v[3 * k + 2]));
        const double pr = val(pl0 * v.x + pl1 * v.y + pl2 * v.z + pl3);
        n_pos += (0.0 < pr); n_neg += (pr < 0.0);
    }
    return n_pos != 0 && n_neg != 0;
}

// stage A dispatch on the kind of mesh 1
template <class T> PFC_D bool clip_pair(const SceneDev& sc, const InsDev& ins, int prim1, int prim2, const PatchCtx<T>& cx, PolyRec<T>& out, int& flags) {
    const TetRec& t2 = sc.tets[ins.prim_base2 + prim2];
    if (ins.kind1 == 0) return clip_tri_tet(sc.tris[ins.prim_base1 + prim1], t2, cx, out, flags);
    return clip_tet_tet(sc.tets[ins.prim_base1 + prim1], t2, cx, out, flags);
}

// ---- stage A, Float64, polygon kept in the caller's PolyRec slot (shared memory in the tile kernel) --------------------
// The slot's first 32 doubles hold the polygon in tetrahedral coordinates while it is clipped; the conversion to Cartesian
// vertices runs forward in place (vertex k lands in doubles [3k, 3k+3), which only overlaps coordinates already consumed).
PFC_D bool finish_polygon_slot(int n, const TetRec& tet_g, const Vec3<double>& nrm, PolyRec<double>& out) {
    double* z = reinterpret_cast<double*>(&out);
    struct { double v[12]; } tet;
    load_wide<12>(tet_g.v, tet.v);
    for (int k = 0; k < n; ++k) {  // mul_then_un_pad(x_r2_zeta2, .)
        const double z0 = z[4 * k], z1 = z[4 * k + 1], z2 = z[4 * k + 2], z3 = z[4 * k + 3];
        out.v[k] = mk<double>(tet.v[0] * z0 + tet.v[3] * z1 + tet.v[6] * z2 + tet.v[9] * z3, tet.v[1] * z0 + tet.v[4] * z1 + tet.v[7] * z2 + tet.v[10] * z3,
                              tet.v[2] * z0 + tet.v[5] * z1 + tet.v[8] * z2 + tet.v[11] * z3);
    }
    double cum_sum = 0.0;
    Vec3<double> cum = mk<double>(0.0, 0.0, 0.0);
    const Vec3<double> a = out.v[0];
    Vec3<double> b = out.v[1];
    for (int k = 2; k < n; ++k) {  // fan from vertex 0 (poly_eight.jl:35-52)
        const Vec3<double> c = out.v[k];
        const double area = dot(nrm, cross(b - a, c - b) * 0.5);
        cum = cum + ((a + b + c) * (1.0 / 3.0)) * area;
        cum_sum += area;
        b = c;
    }
    Vec3<double> cen = a;
    if (cum_sum != 0.0) { const double inv = 1.0 / cum_sum; cen = mk<double>(cum.x * inv, cum.y * inv, cum.z * inv); }
    out.nrm = nrm;
    out.cen = cen;
    load_wide<4>(tet_g.eps_r, out.eps_r);
    out.n = n;
    return true;
}

// ---- stage A split in two, for the tile kernel's compacted clip ---------------------------------------------------------
// start_polygon_zeta: everything before the first face cut -- the start polygon (the triangle, or the plane/tet section) in
// tetrahedral coordinates of tet 2, written to zr[4 * k + i] (the tile kernel passes a shared-memory staging area: 16 doubles
// held across its slot scan would cost it a local-memory frame); returns its vertex count, 0 when the pair is rejected (same
// tests, same arithmetic as clip_pair).  pair_normal: the polygon normal, recomputed from the records after the clip.
PFC_D int start_polygon_zeta(const SceneDev& sc, const InsDev& ins, int prim1, int prim2, const PatchCtx<double>& cx, double* zr) {
    const TetRec& t2 = sc.tets[ins.prim_base2 + prim2];
    if (ins.kind1 == 0) {
        struct { double v[9]; double n[3]; } tri;
        struct { double inv[16]; } t2r;
        load_wide<12>(sc.tris[ins.prim_base1 + prim1].v, tri.v);
        load_wide<16>(t2.inv, t2r.inv);
        unsigned all_non_pos = 0xfu;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const Vec3<double> p = apply_d(cx.x21, mk<double>(tri.v[3 * k], tri.v[3 * k + 1], tri.v[3 * k + 2]));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const double zz = t2r.inv[4 * i] * p.x + t2r.inv[4 * i + 1] * p.y + t2r.inv[4 * i + 2] * p.z + t2r.inv[4 * i + 3];
                zr[4 * k + i] = zz;
                if (!(zz <= 0.0)) all_non_pos &= ~(1u << i);
            }
        }
        return all_non_pos ? 0 : 3;
    }
    const TetRec& t1 = sc.tets[ins.prim_base1 + prim1];
    double plane[4];
    {
        const double g0 = cx.Ebar1 * t1.eps_r[0], g1 = cx.Ebar1 * t1.eps_r[1], g2 = cx.Ebar1 * t1.eps_r[2], g3 = cx.Ebar1 * t1.eps_r[3];
        const Xform<double>& Y = cx.x12;
        plane[0] = cx.Ebar2 * t2.eps_r[0] - (g0 * Y.r[0] + g1 * Y.r[3] + g2 * Y.r[6]);
        plane[1] = cx.Ebar2 * t2.eps_r[1] - (g0 * Y.r[1] + g1 * Y.r[4] + g2 * Y.r[7]);
        plane[2] = cx.Ebar2 * t2.eps_r[2] - (g0 * Y.r[2] + g1 * Y.r[5] + g2 * Y.r[8]);
        plane[3] = cx.Ebar2 * t2.eps_r[3] - (g0 * Y.t[0] + g1 * Y.t[1] + g2 * Y.t[2] + g3);
    }
    // tet 1's vertices in r2 are recomputed where they are needed, and each vertex of the section goes to tetrahedral coordinates
    // as soon as it exists: neither polygon is held in registers
    const auto vert = [&](int k) { return apply_d(cx.x21, mk<double>(t1.v[3 * k], t1.v[3 * k + 1], t1.v[3 * k + 2])); };
    const int n0 = plane_tet_inline(plane, vert, [&](int k, const Vec3<double>& p) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double zz = t2.inv[4 * i] * p.x + t2.inv[4 * i + 1] * p.y + t2.inv[4 * i + 2] * p.z + t2.inv[4 * i + 3];
            zr[4 * k + i] = zz * ((1.0e-14 < fabs(zz)) ? 1.0 : 0.0);   // zero_small_coordinates
        }
    });
    return n0 < 3 ? 0 : n0;
}

PFC_D Vec3<double> pair_normal(const SceneDev& sc, const InsDev& ins, int prim1, int prim2, const PatchCtx<double>& cx) {
    if (ins.kind1 == 0) {
        const TriRec& tri = sc.tris[ins.prim_base1 + prim1];
        return rot_d(cx.x21, mk<double>(tri.n[0], tri.n[1], tri.n[2]));
    }
    const TetRec& t1 = sc.tets[ins.prim_base1 + prim1];
    const TetRec& t2 = sc.tets[ins.prim_base2 + prim2];
    const double g0 = cx.Ebar1 * t1.eps_r[0], g1 = cx.Ebar1 * t1.eps_r[1], g2 = cx.Ebar1 * t1.eps_r[2];
    const Xform<double>& Y = cx.x12;
    const double p0 = cx.Ebar2 * t2.eps_r[0] - (g0 * Y.r[0] + g1 * Y.r[3] + g2 * Y.r[6]);
    const double p1 = cx.Ebar2 * t2.eps_r[1] - (g0 * Y.r[1] + g1 * Y.r[4] + g2 * Y.r[7]);
    const double p2 = cx.Ebar2 * t2.eps_r[2] - (g0 * Y.r[2] + g1 * Y.r[5] + g2 * Y.r[8]);
    const double inv_len = 1.0 / sqrt(p0 * p0 + p1 * p1 + p2 * p2);
    return mk<double>(p0 * inv_len, p1 * inv_len, p2 * inv_len);
}

// stages A + B for one pair on one thread, sub-triangles in the reference's order (previous vertex = last first)
template <class T, int NA> PFC_D void integrate_pair(const SceneDev& sc, const InsDev& ins, int prim1, int prim2, const PatchCtx<T>& cx, Accum<T, NA>& acc, int& flags) {
    PolyRec<T> pr;
    if (!clip_pair(sc, ins, prim1, prim2, cx, pr, flags)) return;
    Vec3<T> v2 = pr.v[pr.n - 1];
    for (int k = 0; k < pr.n; ++k) {
        const Vec3<T> v1 = v2;
        v2 = pr.v[k];
        integrate_subtri(v1, v2, pr.cen, pr.nrm, pr.eps_r, cx, acc);
    }
}

}  // namespace pfc
