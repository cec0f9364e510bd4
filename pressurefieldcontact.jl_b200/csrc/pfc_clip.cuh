// pfc_clip.cuh -- per-pair polygon clipping, one thread per candidate pair.
//
// Behaviour follows the reference's Clip module (/root/reference/src/clip):
//   * clip_tet      <- clip_in_tet_coordinates / clip / cut_clip / clip_node  static_clip.jl:7-201
//   * plane_tet     <- clip_plane_tet and its seven sign cases               plane_tet_intersection.jl:9-106
//   * zero_small    <- zero_small_coordinates                                 poly_eight.jl:106-126
// The reference unrolls the clip over the vertex count with one method per arity and recursion
// over the four faces; here it is a single loop over faces on a thread-private vertex array, with
// the reference's quirks kept: trailing non-positive vertices are dropped before the exit edge is
// cut, the "last vertex inside" comparison is strict for 3/4/5-gons and non-strict for 6/7-gons
// (static_clip.jl:140,152,164 vs :176,188), and a 7-gon that is cut returns immediately
// (static_clip.jl:185-195).
#pragma once
#include "pfc_math.cuh"
#include "pfc_types.cuh"

namespace pfc {

template <class T> struct Zeta { T c[4]; };

// weightPoly (src/math_kernel/utility.jl:21-26) on tetrahedral coordinates
template <class T> PFC_D Zeta<T> clip_node(const Zeta<T>& z_non, const Zeta<T>& z_pos, int i) {
    const T w1 = z_non.c[i], w2 = z_pos.c[i];
    const T inv = 1.0 / (w1 - w2);
    const T c1 = w1 * inv, c2 = w2 * inv;
    Zeta<T> r;
#pragma unroll
    for (int k = 0; k < 4; ++k) r.c[k] = c1 * z_pos.c[k] - c2 * z_non.c[k];
    return r;
}

// Clips the n-gon z (n = 3 or 4 on entry) against the four faces zeta_i >= 0.  Returns the vertex
// count (0 = clipped away); the result is left in z.  flags gets kFlagNonFinite on the
// reference's error("Non-finite vertex likely") path.
template <class T> __device__ __noinline__ int clip_tet(Zeta<T>* z, int n, int& flags) {
    for (int i = 0; i < 4; ++i) {
        bool all_non_pos = true, all_non_neg = true;
        unsigned non_pos = 0;
        for (int k = 0; k < n; ++k) {
            const double s = val(z[k].c[i]);
            const bool np = (s <= 0.0);
            non_pos |= (np ? 1u : 0u) << k;
            all_non_pos = all_non_pos && np;
            all_non_neg = all_non_neg && (0.0 <= s);
        }
        if (all_non_pos) return 0;
        if (all_non_neg) continue;
        int k0 = -1;
        for (int k = 0; k < n; ++k) {
            const int k1 = (k + 1 == n) ? 0 : k + 1;
            if (((non_pos >> k) & 1u) && !((non_pos >> k1) & 1u)) { k0 = k; break; }
        }
        if (k0 < 0) { flags |= kFlagNonFinite; return 0; }
        // rotate so that w[0] is non-positive and w[1] positive
        Zeta<T> w[8];
        for (int j = 0; j < n; ++j) { int k = k0 + j; if (k >= n) k -= n; w[j] = z[k]; }
        int m = n;
        while (m > 3 && val(w[m - 2].c[i]) <= 0.0) --m;  // cut_clip's arity-reducing recursion
        const Zeta<T> z_start = clip_node(w[0], w[1], i);
        const double last = val(w[m - 1].c[i]);
        const bool last_inside = (m <= 5) ? (0.0 < last) : (0.0 <= last);
        z[0] = z_start;
        if (last_inside) {
            for (int k = 1; k < m; ++k) z[k] = w[k];
            z[m] = clip_node(w[0], w[m - 1], i);
            n = m + 1;
        } else {
            for (int k = 1; k < m - 1; ++k) z[k] = w[k];
            z[m - 1] = clip_node(w[m - 1], w[m - 2], i);
            n = m;
        }
        if (m == 7) return n;  // the 7-vertex cut returns without visiting further faces
    }
    return n;
}

// The same clip, working IN PLACE on a polygon stored as z[4 * k + c] (Float64 mode; the tile kernel keeps it in the
// thread's shared-memory slot, so nothing goes through local memory).  Decisions are taken on three sign masks per face;
// the two cut edges are loaded before anything is overwritten; the kept vertices are rotated through registers only when
// the first kept vertex is not already in slot 1 (k0 != 0).  Same quirks as clip_tet above.
// Measured and rejected: arranging the loop by CUTS (each thread walks to its next face that cuts, then the threads of a warp run
// the cut body together, each on its own face) -- same results (bit for bit), but 172 us against 141 us for the tile kernel.  Not
// profiled: whether the threads really meet at the body is up to the compiler's reconvergence points.
PFC_D void clip_node_inplace(const double* zn, const double* zp, double w1, double w2, double* r) {   // w1, w2: coordinate i of zn, zp
    const double inv = 1.0 / (w1 - w2);
    const double c1 = w1 * inv, c2 = w2 * inv;
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] = c1 * zp[k] - c2 * zn[k];
}
PFC_D int clip_tet_inplace(double* z, int n, int& flags) {
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
        unsigned np = 0, nn = 0, ps = 0;   // bit k: s <= 0, 0 <= s, 0 < s  with s = zeta_i of vertex k
        for (int k = 0; k < n; ++k) {
            const double s = z[4 * k + i];
            np |= (s <= 0.0 ? 1u : 0u) << k;
            nn |= (0.0 <= s ? 1u : 0u) << k;
            ps |= (0.0 < s ? 1u : 0u) << k;
        }
        const unsigned full = (1u << n) - 1u;
        if (np == full) return 0;
        if (nn == full) continue;
        const unsigned trans = np & ~(((np >> 1) | (np << (n - 1))) & full);   // non-positive vertex followed by a positive one
        if (!trans) { flags |= kFlagNonFinite; return 0; }
        const int k0 = __ffs(trans) - 1;
        const unsigned rnp = ((np >> k0) | (np << (n - k0))) & full;            // masks in the rotated order w[j] = z[(k0 + j) mod n]
        const unsigned rnn = ((nn >> k0) | (nn << (n - k0))) & full;
        const unsigned rps = ((ps >> k0) | (ps << (n - k0))) & full;
        int m = n;
        while (m > 3 && ((rnp >> (m - 2)) & 1u)) --m;                           // cut_clip's arity-reducing recursion
        const bool last_inside = (((m <= 5) ? rps : rnn) >> (m - 1)) & 1u;
        const int keep_end = last_inside ? m - 1 : m - 2;                       // the output keeps w[1 .. keep_end]
        double w0[4], w1[4], wa[4], wb[4], zs[4], ze[4];
        {
            const int i1 = (k0 + 1 < n) ? k0 + 1 : k0 + 1 - n;
            const int ja = last_inside ? 0 : m - 1, jb = last_inside ? m - 1 : m - 2;   // z_end = clip_node(w[ja], w[jb])
            const int ia = (k0 + ja < n) ? k0 + ja : k0 + ja - n, ib = (k0 + jb < n) ? k0 + jb : k0 + jb - n;
#pragma unroll
            for (int c = 0; c < 4; ++c) { w0[c] = z[4 * k0 + c]; w1[c] = z[4 * i1 + c]; wa[c] = z[4 * ia + c]; wb[c] = z[4 * ib + c]; }
            // coordinate i again, by address: indexing the register copies with the loop variable would push them to local memory
            clip_node_inplace(w0, w1, z[4 * k0 + i], z[4 * i1 + i], zs);
            clip_node_inplace(wa, wb, z[4 * ia + i], z[4 * ib + i], ze);
        }
        if (k0 != 0) {   // one coordinate column at a time keeps the register footprint at 7 doubles
#pragma unroll 1
            for (int c = 0; c < 4; ++c) {
                double t[7];
#pragma unroll
                for (int j = 1; j <= 7; ++j)
                    if (j <= keep_end) { const int idx = (k0 + j < n) ? k0 + j : k0 + j - n; t[j - 1] = z[4 * idx + c]; }
#pragma unroll
                for (int j = 1; j <= 7; ++j)
                    if (j <= keep_end) z[4 * j + c] = t[j - 1];
            }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) { z[c] = zs[c]; z[4 * (keep_end + 1) + c] = ze[c]; }
        n = keep_end + 2;
        if (m == 7) return n;  // the 7-vertex cut returns without visiting further faces
    }
    return n;
}

// zero_small_coordinates: |x| <= 1e-14 -> 0 (decided on the value part)
template <class T> PFC_D void zero_small(Zeta<T>* z, int n) {
    for (int k = 0; k < n; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const bool keep = 1.0e-14 < fabs(val(z[k].c[i]));
            z[k].c[i] = z[k].c[i] * (keep ? 1.0 : 0.0);
        }
}

// weightPoly on Cartesian points
template <class T> PFC_D Vec3<T> weight_poly(const Vec3<T>& p1, const Vec3<T>& p2, const T& w1, const T& w2) {
    const T inv = 1.0 / (w1 - w2);
    const T c1 = w1 * inv, c2 = w2 * inv;
    return mk<T>(c1 * p2.x - c2 * p1.x, c1 * p2.y - c2 * p1.y, c1 * p2.z - c2 * p1.z);
}

// edge lists of plane_tet per case, 0-based (i1, i2) -> weightPoly(v[i1], v[i2], proj[i1], proj[i2])
// lone vertex k:   plane_tet_intersection.jl:52-79 ; two-two split: :81-106
constexpr signed char kPlaneTetTri[4][3][2] = {{{1, 0}, {3, 0}, {2, 0}}, {{0, 1}, {2, 1}, {3, 1}}, {{0, 2}, {3, 2}, {1, 2}}, {{0, 3}, {1, 3}, {2, 3}}};
constexpr signed char kPlaneTetQuad[3][4][2] = {{{1, 2}, {1, 3}, {0, 3}, {0, 2}}, {{0, 1}, {0, 3}, {2, 3}, {2, 1}}, {{0, 2}, {0, 1}, {3, 1}, {3, 2}}};
// The same lists as 4-bit fields i1 | i2 << 2 (case sel, edge k at bit 4 * (n_edges * sel + k)): a shift of a constant instead of a
// table in local memory.
constexpr unsigned long long plane_tet_edge_bits(bool quad) {
    unsigned long long b = 0;
    for (int s = 0; s < (quad ? 3 : 4); ++s)
        for (int k = 0; k < (quad ? 4 : 3); ++k) {
            const signed char* e = quad ? kPlaneTetQuad[s][k] : kPlaneTetTri[s][k];
            b |= (unsigned long long)(e[0] | e[1] << 2) << (4 * ((quad ? 4 : 3) * s + k));
        }
    return b;
}
constexpr unsigned long long kPlaneTetTriBits = plane_tet_edge_bits(false), kPlaneTetQuadBits = plane_tet_edge_bits(true);
template <class T> PFC_D T pick4(int i, const T& a, const T& b, const T& c, const T& d) { return i == 0 ? a : i == 1 ? b : i == 2 ? c : d; }

// Plane (4 coefficients) against a tetrahedron whose vertex k is vert(k): hands the vertices of a 3- or 4-gon with the plane's
// orientation to emit(j, vertex), j = 0, 1, ..., and returns its size (0 when all vertices are on one side).  Every array index is
// a constant once the loops are unrolled, and vert is asked again for the two ends of each cut edge instead of holding all four
// vertices: a caller that inlines this keeps what it needs in registers, and few of them.
template <class T, class Vert, class Emit> PFC_D int plane_tet_inline(const T* plane, Vert&& vert, Emit&& emit) {
    T proj[4];
    int n_neg = 0, n_pos = 0;
    unsigned pos = 0, neg = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const Vec3<T> v = vert(k);
        proj[k] = plane[0] * v.x + plane[1] * v.y + plane[2] * v.z + plane[3];
        const double p = val(proj[k]);
        if (p < 0.0) { ++n_neg; neg |= 1u << k; }
        if (0.0 < p) { ++n_pos; pos |= 1u << k; }
    }
    if (n_pos == 0 || n_neg == 0) return 0;
    int cnt, sel;
    bool forward;
    if (n_pos == 1) { sel = __ffs(pos) - 1; cnt = 3; forward = true; }
    else if (n_neg == 1) { sel = __ffs(neg) - 1; cnt = 3; forward = false; }
    else {
        const unsigned p0 = pos & 1u;
        if (((pos >> 1) & 1u) == p0) sel = 0;
        else if (((pos >> 2) & 1u) == p0) sel = 1;
        else if (((pos >> 3) & 1u) == p0) sel = 2;
        else return 0;  // a vertex exactly on the plane in a 2-2 split: the reference falls through (returns nothing)
        cnt = 4;
        forward = (0.0 < val(proj[0]));
    }
    const unsigned long long edges = (cnt == 3) ? kPlaneTetTriBits : kPlaneTetQuadBits;
#pragma unroll
    for (int j = 0; j < 4; ++j)   // output vertex j is edge k of the case's list
        if (j < cnt) {
            const int k = forward ? j : cnt - 1 - j;
            const unsigned e = unsigned(edges >> (4 * (cnt * sel + k))) & 15u;
            const int i1 = e & 3u, i2 = e >> 2;
            emit(j, weight_poly(vert(i1), vert(i2), pick4(i1, proj[0], proj[1], proj[2], proj[3]), pick4(i2, proj[0], proj[1], proj[2], proj[3])));
        }
    return cnt;
}
// The same for callers that do not inline it: tet vertices v[0 .. 4), the polygon written to out[0 .. size).
template <class T> __device__ __noinline__ int plane_tet(const T* plane, const Vec3<T>* v, Vec3<T>* out) {
    return plane_tet_inline(plane, [&](int k) { return v[k]; }, [&](int j, const Vec3<T>& p) { out[j] = p; });
}

}  // namespace pfc
