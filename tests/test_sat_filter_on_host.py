"""CPU-only: the broad phase's filtered box-overlap test (csrc/pfc_sat.cuh: sat_filter, float with a certified error bound, and the
exact FP64 sat_prepare_a<false> + sat_test<false> for what it leaves undecided) compiled for the host with g++ and compared with the
oracle's BB_BB_intersect (oracle/pfc_oracle.hpp).

  * test_filtered_sat_equals_oracle_everywhere: random box pairs, each also bisected down to neighbouring doubles where the oracle's
    answer flips, plus adversarial inputs -- frames far from the origin with adjacent nodes (cancellation in t), flat and zero-extent
    boxes, +-0, subnormal centres, boxes at subnormal and near-overflow scales, non-rotation matrices, NaN and infinite inputs.  Filter +
    fallback must equal the oracle on every evaluation, and every answer the filter gives alone must equal the oracle's.  The
    non-finite and non-rotation inputs must all be left undecided, so they get exactly the answer of the FP64 test (which drops the
    products with the homogeneous 0/1 row, so with an infinite input it need not agree with the oracle: 0 * inf is NaN there).
  * test_filtered_traversal_replays_oracle_pair_lists: the dual-tree recursion of tree_tree_intersect replayed with the filtered test on
    settled-stack states of test/boxes.jl (the benchmark's workload, tests/helpers.py::boxes_env_states): the pair lists must equal
    the oracle's, in order, and the share of tests the filter leaves undecided must stay below 1 % (a bound that sends everything to
    the fallback would be correct and slow)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HARNESS = r"""
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>
#include "pfc_oracle.hpp"
#define __host__
#define __device__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __shfl_xor_sync(unsigned, double v, int, int = 32) { return v; }
#define PFC_HOST_CHECK 1
#include "pfc_sat.cuh"

static bool exact_says(const pfc::NodeRec& a, const pfc::NodeRec& b, const double* Rab, const double* tab) {
    pfc::SatA A;
    pfc::sat_prepare_a<false>(a, Rab, tab, A);
    return pfc::sat_test<false>(A, b);
}
static int filter_says(const pfc::NodeRec& a, const pfc::NodeRec& b, const double* Rab, const double* tab) {
    pfc::FiltNode fa, fb;
    pfc::FiltXf fx;
    pfc::filt_node_from(a, fa); pfc::filt_node_from(b, fb); pfc::filt_xf_from(Rab, tab, fx);
    return pfc::sat_filter(fa, fb, fx);
}

// ---------------------------------------------------------------------------------------------------------------------------------
static std::mt19937_64 g(2718);
static std::uniform_real_distribution<double> u(-1.0, 1.0), u01(0.0, 1.0);
static void random_rotation(double* R) {   // row-major
    double q[4] = {u(g), u(g), u(g), u(g)};
    const double qn = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (double& x : q) x /= qn;
    const double M[9] = {1 - 2 * (q[2] * q[2] + q[3] * q[3]), 2 * (q[1] * q[2] - q[0] * q[3]), 2 * (q[1] * q[3] + q[0] * q[2]),
                         2 * (q[1] * q[2] + q[0] * q[3]), 1 - 2 * (q[1] * q[1] + q[3] * q[3]), 2 * (q[2] * q[3] - q[0] * q[1]),
                         2 * (q[1] * q[3] - q[0] * q[2]), 2 * (q[2] * q[3] + q[0] * q[1]), 1 - 2 * (q[1] * q[1] + q[2] * q[2])};
    std::memcpy(R, M, sizeof M);
}
struct Case { pfc::NodeRec a, b; double Rab[9], base[3], dir[3]; };
static bool oracle_says(const Case& c, const double* tab) {
    orc::OBB A, B;
    orc::M3<double> R;
    orc::V3<double> t;
    for (int i = 0; i < 3; ++i) {
        A.c[i] = c.a.c[i]; A.e[i] = c.a.e[i]; B.c[i] = c.b.c[i]; B.e[i] = c.b.e[i]; t[i] = tab[i];
        for (int j = 0; j < 3; ++j) { A.R(i, j) = c.a.R[3 * i + j]; B.R(i, j) = c.b.R[3 * i + j]; R(i, j) = c.Rab[3 * i + j]; }
    }
    return orc::BB_BB_intersect<double>(R, t, A, B);
}

static long n_eval = 0, n_decided = 0, n_away = 0, n_away_decided = 0, n_boundary = 0, bad = 0, bad_filter = 0, n_must_undecide = 0, bad_undecided = 0;
static bool check(const Case& c, double s, bool must_undecide, long k, bool away = false) {
    double tab[3];
    for (int i = 0; i < 3; ++i) tab[i] = c.base[i] + s * c.dir[i];
    const bool o = oracle_says(c, tab);
    const int f = filter_says(c.a, c.b, c.Rab, tab);
    const bool got = f == pfc::kSatUndecided ? exact_says(c.a, c.b, c.Rab, tab) : f == pfc::kSatOverlap;
    ++n_eval;
    n_away += away; n_away_decided += away && f != pfc::kSatUndecided;
    if (f != pfc::kSatUndecided) {
        ++n_decided;
        if ((f == pfc::kSatOverlap) != o && bad_filter++ < 5) std::printf("case %ld at s = %.17g: oracle %d, filter decided %d\n", k, s, (int)o, f);
    }
    if (got != o && !must_undecide && bad++ < 5) std::printf("case %ld at s = %.17g: oracle %d, filter + fallback %d\n", k, s, (int)o, (int)got);
    if (must_undecide) {
        ++n_must_undecide;
        if (f != pfc::kSatUndecided && bad_undecided++ < 5) std::printf("case %ld: non-finite / non-rotation input decided (%d)\n", k, f);
    }
    return o;
}
static void run_case(const Case& c, long k, bool must_undecide) {
    for (int r = 0; r < 4; ++r) check(c, 4.0 * u01(g), must_undecide, k, !must_undecide);
    if (must_undecide) return;
    double lo = 0.0, hi = 16.0;   // bisect the flip along dir, then evaluate 4 ulps to either side of it
    double t0[3], t1[3];
    for (int i = 0; i < 3; ++i) { t0[i] = c.base[i]; t1[i] = c.base[i] + hi * c.dir[i]; }
    if (!oracle_says(c, t0) || oracle_says(c, t1)) return;
    for (int it = 0; it < 200 && std::nextafter(lo, hi) < hi; ++it) {
        const double mid = 0.5 * (lo + hi);
        double tm[3];
        for (int i = 0; i < 3; ++i) tm[i] = c.base[i] + mid * c.dir[i];
        (oracle_says(c, tm) ? lo : hi) = mid;
    }
    ++n_boundary;
    double s = lo;
    for (int r = 0; r < 4; ++r) s = std::nextafter(s, 0.0);
    for (int r = 0; r < 9; ++r) { check(c, s, false, k); s = std::nextafter(s, 32.0); }
}

static void random_case(Case& c, long k) {
    std::memset(&c, 0, sizeof c);
    random_rotation(c.a.R); random_rotation(c.b.R); random_rotation(c.Rab);
    const double I9[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (k % 5 == 0) { std::memcpy(c.b.R, I9, sizeof I9); std::memcpy(c.Rab, I9, sizeof I9); std::memcpy(c.a.R, I9, sizeof I9); }   // parallel edges
    for (int i = 0; i < 3; ++i) { c.a.c[i] = 0.2 * u(g); c.b.c[i] = 0.2 * u(g); c.a.e[i] = 0.05 + u01(g); c.b.e[i] = 0.05 + u01(g); c.dir[i] = u(g); }
    c.a.kind = c.b.kind = pfc::kNodeInternal;
    if (k % 3 == 1) std::memcpy(c.a.R, I9, sizeof I9);
    if (k % 3 == 2) std::memcpy(c.b.R, I9, sizeof I9);
}

int main(int argc, char** argv) {
    const long n_case = argc > 1 ? atol(argv[1]) : 20000;
    long k = 0;
    for (; k < n_case; ++k) { Case c; random_case(c, k); run_case(c, k, false); }
    // ---- adversarial inputs
    const double big[4] = {1.0e2, 1.0e4, 1.0e6, 1.0e9};
    for (long r = 0; r < n_case / 4; ++r, ++k) {
        Case c; random_case(c, k);
        switch (r % 10) {
        case 0: case 1: {   // both frames far from the origin, nodes adjacent: t_ab and c_a nearly cancel
            const double L = big[(r / 10) % 4];
            for (int i = 0; i < 3; ++i) { c.a.c[i] += L * (i + 1); c.base[i] = c.a.c[i] - c.b.c[i]; }
            break;
        }
        case 2: c.b.e[r % 3] = 0.0; c.b.e[(r + 1) % 3] = 0.0; c.a.e[(r + 2) % 3] = 0.0; break;   // zero-extent: a segment against a flat box
        case 3:   // +-0 in the records and the transform
            c.a.c[r % 3] = -0.0; c.b.c[(r + 1) % 3] = 0.0; c.b.e[r % 3] = -0.0; c.base[(r + 2) % 3] = -0.0; c.dir[r % 3] = -0.0;
            for (int j = 0; j < 9; ++j) { if (c.Rab[j] == 0.0) c.Rab[j] = -0.0; if (c.a.R[j] == 0.0 && (r & 1)) c.a.R[j] = -0.0; }
            break;
        case 4: c.a.c[r % 3] = 4.9e-324; c.b.c[(r + 1) % 3] = -2.2e-308; c.base[(r + 2) % 3] = 1.0e-310; break;   // subnormal centres
        case 5: {   // the whole configuration scaled into float's subnormal range, below it, and up to float's overflow
            const double sc[5] = {1.0e-20, 1.0e-40, 1.0e-300, 1.0e29, 1.0e36};
            const double f = sc[(r / 10) % 5];
            for (int i = 0; i < 3; ++i) { c.a.c[i] *= f; c.b.c[i] *= f; c.a.e[i] *= f; c.b.e[i] *= f; c.dir[i] *= f; }
            break;
        }
        default: break;
        }
        if (r % 10 <= 5) { run_case(c, k, false); continue; }
        // non-finite and non-rotation inputs: never decided by the filter
        const double bad_v[3] = {NAN, INFINITY, -INFINITY};
        const double v = bad_v[r % 3];
        switch ((r / 10) % 7) {
        case 0: c.a.c[r % 3] = v; break;
        case 1: c.b.e[r % 3] = v; break;
        case 2: c.a.R[r % 9] = v; break;
        case 3: c.b.R[r % 9] = v; break;
        case 4: c.Rab[r % 9] = v; break;
        case 5: c.base[r % 3] = v; break;
        default: for (int j = 0; j < 9; ++j) ((r & 1) ? c.b.R : c.Rab)[j] *= 1.001; break;   // not a rotation
        }
        run_case(c, k, true);
    }
    std::printf("evaluations %ld decided %ld away %ld away_decided %ld boundaries %ld bad %ld bad_filter %ld must_undecide %ld bad_undecided %ld\n", n_eval, n_decided,
                n_away, n_away_decided, n_boundary, bad, bad_filter, n_must_undecide, bad_undecided);
    return bad != 0 || bad_filter != 0 || bad_undecided != 0;
}
"""

REPLAY = r"""
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>
#define __host__
#define __device__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __shfl_xor_sync(unsigned, double v, int, int = 32) { return v; }
#define PFC_HOST_CHECK 1
#include "pfc_sat.cuh"

// input (float64 / int32 little-endian, written by the test): n_tree, per tree n_node then c, e, R (row-major) as doubles and left, right,
// leaf_id as int32; n_ins, (tree_1, tree_2) per instruction; n_env; X_r2_r1 [env][ins][16] column-major.
// output: per (env, ins) the pair count and the (leaf_1, leaf_2) pairs; last line the test counts.
struct Tree { std::vector<pfc::NodeRec> rec; std::vector<pfc::FiltNode> f; std::vector<int32_t> left, right, leaf; };
static long n_test = 0, n_undecided = 0;

static bool overlap(const Tree& t1, int n1, const Tree& t2, int n2, const double* Rab, const double* tab, const pfc::FiltXf& fx) {
    ++n_test;
    const int f = pfc::sat_filter(t1.f[n1], t2.f[n2], fx);
    if (f != pfc::kSatUndecided) return f == pfc::kSatOverlap;
    ++n_undecided;
    pfc::SatA A;
    pfc::sat_prepare_a<false>(t1.rec[n1], Rab, tab, A);
    return pfc::sat_test<false>(A, t2.rec[n2]);
}
static void recurse(std::vector<int32_t>& out, const Tree& t1, int n1, const Tree& t2, int n2, const double* Rab, const double* tab,
                    const pfc::FiltXf& fx) {   // tree_tree_intersect's visiting order
    if (!overlap(t1, n1, t2, n2, Rab, tab, fx)) return;
    const bool l1 = t1.leaf[n1] >= 0, l2 = t2.leaf[n2] >= 0;
    if (l1 && l2) { out.push_back(t1.leaf[n1]); out.push_back(t2.leaf[n2]); }
    else if (l1) { recurse(out, t1, n1, t2, t2.left[n2], Rab, tab, fx); recurse(out, t1, n1, t2, t2.right[n2], Rab, tab, fx); }
    else if (l2) { recurse(out, t1, t1.left[n1], t2, n2, Rab, tab, fx); recurse(out, t1, t1.right[n1], t2, n2, Rab, tab, fx); }
    else {
        recurse(out, t1, t1.left[n1], t2, t2.left[n2], Rab, tab, fx); recurse(out, t1, t1.right[n1], t2, t2.left[n2], Rab, tab, fx);
        recurse(out, t1, t1.left[n1], t2, t2.right[n2], Rab, tab, fx); recurse(out, t1, t1.right[n1], t2, t2.right[n2], Rab, tab, fx);
    }
}
template <class V> static void rd(FILE* fp, V* p, size_t n) { if (fread(p, sizeof(V), n, fp) != n) { std::printf("short input\n"); exit(2); } }

int main(int argc, char** argv) {
    FILE* fp = std::fopen(argv[1], "rb");
    FILE* fo = std::fopen(argv[2], "wb");
    int32_t n_tree; rd(fp, &n_tree, 1);
    std::vector<Tree> trees(n_tree);
    for (Tree& t : trees) {
        int32_t n; rd(fp, &n, 1);
        std::vector<double> c(3 * n), e(3 * n), R(9 * n);
        rd(fp, c.data(), c.size()); rd(fp, e.data(), e.size()); rd(fp, R.data(), R.size());
        t.left.resize(n); t.right.resize(n); t.leaf.resize(n); t.rec.resize(n); t.f.resize(n);
        rd(fp, t.left.data(), n); rd(fp, t.right.data(), n); rd(fp, t.leaf.data(), n);
        for (int k = 0; k < n; ++k) {
            pfc::NodeRec& r = t.rec[k];
            std::memset(&r, 0, sizeof r);
            for (int i = 0; i < 3; ++i) { r.c[i] = c[3 * k + i]; r.e[i] = e[3 * k + i]; }
            for (int i = 0; i < 9; ++i) r.R[i] = R[9 * k + i];
            r.kind = t.leaf[k] >= 0 ? pfc::kNodeLeaf : pfc::kNodeInternal;
            pfc::filt_node_from(r, t.f[k]);
        }
    }
    int32_t n_ins; rd(fp, &n_ins, 1);
    std::vector<int32_t> ins(2 * n_ins); rd(fp, ins.data(), ins.size());
    int32_t n_env; rd(fp, &n_env, 1);
    std::vector<double> X(16 * (size_t)n_env * n_ins); rd(fp, X.data(), X.size());
    std::vector<int32_t> out;
    for (int env = 0; env < n_env; ++env)
        for (int k = 0; k < n_ins; ++k) {
            const double* x = X.data() + 16 * ((size_t)env * n_ins + k);
            double Rab[9], tab[3];   // x_r1_r2 with the reference's rounding, as the broad kernel forms it
            for (int l = 0; l < 9; ++l) Rab[l] = x[4 * (l / 3) + l % 3];
            for (int i = 0; i < 3; ++i) tab[i] = -((x[4 * i] * x[12] + x[4 * i + 1] * x[13]) + x[4 * i + 2] * x[14]);
            pfc::FiltXf fx;
            pfc::filt_xf_from(Rab, tab, fx);
            out.clear();
            recurse(out, trees[ins[2 * k]], 0, trees[ins[2 * k + 1]], 0, Rab, tab, fx);
            const int32_t n = (int32_t)out.size() / 2;
            std::fwrite(&n, 4, 1, fo);
            std::fwrite(out.data(), 4, out.size(), fo);
        }
    std::fclose(fo);
    std::printf("tests %ld undecided %ld\n", n_test, n_undecided);
    return 0;
}
"""

INC = ["-I", os.path.join(ROOT, "oracle"), "-I", os.path.join(ROOT, "pressurefieldcontact.jl_b200", "csrc"), "-I", "/usr/local/cuda/include"]


def _build(tmp_path, name, src):
    cpp = tmp_path / f"{name}.cpp"
    cpp.write_text(src)
    exe = tmp_path / name
    # -ffp-contract=off for the exact test's host stand-ins of __dmul_rn / __dadd_rn; the filter's bound holds with or without contraction
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-w", *INC, "-o", str(exe), str(cpp)])
    return exe


def test_filtered_sat_equals_oracle_everywhere(tmp_path):
    exe = _build(tmp_path, "sat_filter_host", HARNESS)
    out = subprocess.run([str(exe), "20000"], capture_output=True, text=True)
    sys.stdout.write(out.stdout)
    assert out.returncode == 0, out.stdout[-2000:]
    f = out.stdout.split()
    st = {f[i]: int(f[i + 1]) for i in range(len(f) - 1) if f[i] in ("evaluations", "away", "away_decided", "boundaries", "must_undecide")}
    assert st["boundaries"] > 10000 and st["evaluations"] > 150000 and st["must_undecide"] > 5000
    # away from the bisected boundaries the filter decides most tests alone (what it leaves: mostly the axis-aligned cases, whose exactly
    # parallel edges put cross-product axes at a margin of ~1e-14)
    assert st["away_decided"] >= 0.8 * st["away"]


def test_filtered_traversal_replays_oracle_pair_lists(tmp_path):
    from helpers import boxes_env_states, scene_boxes
    from oracle import orc
    from pfc_b200 import scenario as S

    n_env = 256
    m, _ = scene_boxes(orc.OracleContext())
    X, tw, _ = S.boundary_arrays(m, boxes_env_states(m, n_env))
    m.backend.eval_f64(X, tw, None, keep=True)
    mesh_ids = sorted({i for ci in m.ContactInstructions for i in (ci.id_1, ci.id_2)})
    slot = {mid: k for k, mid in enumerate(mesh_ids)}
    inp = tmp_path / "replay.bin"
    with open(inp, "wb") as fp:
        fp.write(np.int32(len(mesh_ids)).tobytes())
        for mid in mesh_ids:
            t = m.MeshCache[mid].tree
            R_rowmajor = np.asarray(t.R, np.float64).reshape(-1, 3, 3).transpose(0, 2, 1)   # FlatTree.R is column-major
            fp.write(np.int32(t.n_node).tobytes())
            for a in (t.c, t.e, R_rowmajor):
                fp.write(np.ascontiguousarray(a, np.float64).tobytes())
            for a in (t.left, t.right, t.leaf_id):
                fp.write(np.ascontiguousarray(a, np.int32).tobytes())
        fp.write(np.int32(len(m.ContactInstructions)).tobytes())
        fp.write(np.array([(slot[ci.id_1], slot[ci.id_2]) for ci in m.ContactInstructions], np.int32).tobytes())
        fp.write(np.int32(n_env).tobytes())
        fp.write(np.ascontiguousarray(X, np.float64).tobytes())
    exe = _build(tmp_path, "sat_filter_replay", REPLAY)
    outp = tmp_path / "pairs.bin"
    out = subprocess.run([str(exe), str(inp), str(outp)], capture_output=True, text=True)
    sys.stdout.write(out.stdout)
    assert out.returncode == 0, out.stdout[-2000:]
    got = np.fromfile(outp, np.int32)
    at, n_pairs = 0, 0
    for env in range(n_env):
        for k in range(len(m.ContactInstructions)):
            n = int(got[at])
            pairs = got[at + 1:at + 1 + 2 * n].reshape(n, 2)
            at += 1 + 2 * n
            ref = m.backend.get_pairs(env, k)
            assert np.array_equal(pairs, ref), (env, k)
            n_pairs += n
    assert at == got.size and n_pairs > 0
    f = out.stdout.split()
    n_test, n_und = int(f[f.index("tests") + 1]), int(f[f.index("undecided") + 1])
    print(f"{n_env} environments: {n_pairs} candidate pairs, {n_test} box tests, {n_und} undecided ({100.0 * n_und / n_test:.3f} %)")
    assert n_und <= 0.01 * n_test
