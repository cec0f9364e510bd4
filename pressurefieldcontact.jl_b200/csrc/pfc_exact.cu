// pfc_exact.cu -- bristle-friction instructions, evaluated in the reference's operation order (pfc_exact.cuh says why).
// COMPILED WITH -fmad=false: every product and sum below is a separately rounded IEEE operation unless the source says fma().
//
// Reference: integrate_over! + yes_contact!(::Bristle) / no_contact!
// (/root/reference/src/contact_algorithms_non_friction.jl:136-265, src/contact_algorithms_friction.jl:76-201,
//  src/contact_algorithms_normal.jl:17-34).  The reference materialises a TractionCache list per instruction and makes three
// sequential passes over it; so does this file, for Float64 and for the Jacobian mode (T = XD<6>):
//   exact_points_kernel   a CTA takes a unit of 256 consecutive candidate pairs of one (environment, bristle instruction), one pair
//                         per thread: clip + quadrature in the reference's arithmetic -> its traction points; a block scan packs the
//                         unit's points, in pair order, into the TractionCache buffer (one atomicAdd per unit reserves the space;
//                         like the reference's VectorCache the buffer grows and the evaluation is repeated when it was too small);
//   exact_bristle_kernel  one warp per (environment, bristle instruction) walks its units in order.  Per pass, 32 (8 in Jacobian
//                         mode) points at a time: lane l computes the terms of point l into shared memory, then lane e adds term
//                         e of the points ONE AFTER THE OTHER onto its running sum -- the association of the reference's loop.
//                         Between the passes one lane runs the patch-level steps (centre of pressure, decompose_K!, Delta^2,
//                         s-dot).
// Work per point is small and bristle instructions are few; what matters here is the bit pattern, not the FLOP rate.
#include <algorithm>
#include <cstdio>

#include "pfc_exact.cuh"
#include "pfc_exact.h"

namespace pfc {

namespace {

using namespace ex;
typedef XD<6> X6;

#define ECU(call)                         \
    do {                                  \
        cudaError_t e_ = (call);          \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

constexpr int kUnit = 256;   // pairs per unit == kChunk of the large path (its unit_start table is reused)

template <class T> struct NC;   // doubles per scalar
template <> struct NC<double> { static constexpr int n = 1; };
template <> struct NC<X6> { static constexpr int n = 7; };
template <class T> __device__ inline T ldT(const double* p, long long idx);
template <> __device__ inline double ldT<double>(const double* p, long long idx) { return p[idx]; }
template <> __device__ inline X6 ldT<X6>(const double* p, long long idx) { X6 r; r.v = p[7 * idx]; for (int i = 0; i < 6; ++i) r.p[i] = p[7 * idx + 1 + i]; return r; }
template <class T> __device__ inline void stT(double* p, long long idx, const T& x);
template <> __device__ inline void stT<double>(double* p, long long idx, const double& x) { p[idx] = x; }
template <> __device__ inline void stT<X6>(double* p, long long idx, const X6& x) { p[7 * idx] = x.v; for (int i = 0; i < 6; ++i) p[7 * idx + 1 + i] = x.p[i]; }

// one TractionCache entry (src/mechanism_scenario.jl:51-58): n(3) r(3) dA p
template <class T> struct ExRec { T n[3]; T r[3]; T dA; T p; };

// the unit a CTA / the units a warp works on
struct UnitWork { long long ei; long long env; int k; int first; int count; int large_p; };

// unit index space: [0, W_small) = U_s slots per (environment, bristle instruction); [W_small, W_small + n_units) = the large path's units
__device__ inline bool resolve_small_unit(const SceneDev& sc, const ExactScene& es, const long long* n_pairs, long long w, int U_s, UnitWork& uw) {
    const long long pb = w / U_s;
    const int chunk = int(w - pb * U_s);
    const long long env = pb / es.n_bris;
    const int k = es.bris_ins[pb - env * es.n_bris];
    if (!sc.ins[k].small) return false;
    uw.env = env; uw.k = k; uw.ei = env * sc.n_ins + k;
    const int n = (int)n_pairs[uw.ei];
    uw.first = chunk * kUnit;
    uw.count = n - uw.first < kUnit ? n - uw.first : kUnit;
    uw.large_p = -1;
    return uw.count > 0;
}

template <class T> __device__ inline void load_ctx(const SceneDev& sc, const ExactIO& io, const UnitWork& uw, ExCtx<T>& cx) {
    const InsDev& ins = sc.ins[uw.k];
    for (int j = 0; j < 16; ++j) cx.X21[j] = ldT<T>(io.X, 16 * uw.ei + j);
    for (int j = 0; j < 6; ++j) cx.twist[j] = ldT<T>(io.twist, 6 * uw.ei + j);
    make_x12(cx);
    const InsParam* cp = io.params ? io.params + uw.ei : nullptr;
    if (cp) { cx.chi = cp->chi; cx.Ebar1 = cp->Ebar1; cx.Ebar2 = cp->Ebar2; }
    else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
    cx.n_quad = ins.n_quad;
}

template <class T>
__global__ void __launch_bounds__(kUnit) exact_points_kernel(SceneDev sc, ExactScene es, ExactIO io, ExactPairs ps, ExRec<T>* recs, unsigned cap_points, unsigned* ctr,
                                                           unsigned* unit_off, unsigned* unit_cnt, int U_s) {
    __shared__ int warp_tot[kUnit / 32];
    __shared__ unsigned s_base;
    __shared__ int s_prob;
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    const long long W_small = io.n_env * es.n_bris * U_s;
    const long long n_large_units = ps.n_units ? (long long)*ps.n_units : 0;
    for (long long w = blockIdx.x; w < W_small + n_large_units; w += gridDim.x) {
        UnitWork uw;
        bool work;
        if (w < W_small) work = resolve_small_unit(sc, es, io.n_pairs, w, U_s, uw);
        else {
            const unsigned u = (unsigned)(w - W_small);
            __syncthreads();
            if (tid == 0) {   // unit -> problem of the large list by binary search in unit_start
                unsigned lo = 0, hi = (unsigned)(io.n_env * ps.n_large);
                while (hi - lo > 1) { const unsigned mid = (lo + hi) >> 1; if (ps.unit_start[mid] <= u) lo = mid; else hi = mid; }
                s_prob = (int)lo;
            }
            __syncthreads();
            const int p = s_prob;
            uw.env = p / ps.n_large;
            uw.k = ps.large_ins[p - uw.env * ps.n_large];
            uw.ei = uw.env * sc.n_ins + uw.k;
            uw.large_p = p;
            uw.first = (int)(ps.seg_start[p] + (u - ps.unit_start[p]) * kUnit);
            const int left = (int)ps.seg_end[p] - uw.first;
            uw.count = left < kUnit ? left : kUnit;
            work = sc.ins[uw.k].model == PFC_MODEL_BRISTLE && uw.count > 0;
        }
        if (!work) { if (tid == 0) { unit_off[w] = 0; unit_cnt[w] = 0; } continue; }   // (block-uniform)
        const InsDev& ins = sc.ins[uw.k];
        ExPoint<T> pts[kExMaxPoints];
        X3<T> n2;
        int np = 0, fl = 0;
        if (tid < uw.count) {
            ExCtx<T> cx;
            load_ctx(sc, io, uw, cx);
            int a, b;
            if (uw.large_p < 0) { const unsigned e = ps.small_pairs[(size_t)ps.small_cap * uw.ei + uw.first + tid]; a = int((e >> 15) & 0x7fffu); b = int(e & 0x7fffu); }
            else { const int3 e = ps.sorted[uw.first + tid]; a = e.y; b = e.z; }
            const TetRec& t2 = sc.tets[ins.prim_base2 + b];
            if (ins.kind1 == 0) np = pair_points_tri_tet(sc.tris[ins.prim_base1 + a], t2, cx, n2, pts, fl);
            else np = pair_points_tet_tet(sc.tets[ins.prim_base1 + a], es.tet_eps + 4 * (size_t)(ins.prim_base1 + a), t2, es.tet_eps + 4 * (size_t)(ins.prim_base2 + b), cx, n2, pts, fl);
        }
        // block scan of the point counts: the unit's points are packed in pair order
        int incl = np;
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        __syncthreads();   // warp_tot / s_base of the previous unit have been read
        if (lane == 31) warp_tot[wib] = incl;
        __syncthreads();
        int before = 0, total = 0;
        for (int q = 0; q < kUnit / 32; ++q) { const int t = warp_tot[q]; if (q < wib) before += t; total += t; }
        if (tid == 0) s_base = total > 0 ? atomicAdd(ctr, (unsigned)total) : 0u;
        __syncthreads();
        const unsigned base = s_base;
        const bool fits = (unsigned long long)base + (unsigned)total <= cap_points;
        if (fits) {
            ExRec<T>* out = recs + base + before + incl - np;
            for (int j = 0; j < np; ++j) {
                ExRec<T>& o = out[j];
                o.n[0] = n2[0]; o.n[1] = n2[1]; o.n[2] = n2[2];
                o.r[0] = pts[j].r[0]; o.r[1] = pts[j].r[1]; o.r[2] = pts[j].r[2];
                o.dA = pts[j].dA; o.p = pts[j].p;
            }
        }
        if (tid == 0) {
            unit_off[w] = base; unit_cnt[w] = fits ? (unsigned)total : 0u;
            if (!fits) atomicOr(ctr + 1, 1u);
        }
        if (fl) atomicOr(&io.flags[uw.ei], fl);
    }
}

// shared memory of one warp of exact_bristle_kernel
template <class T, int PTS> struct BristleSmem {
    T terms[PTS][27];
    T acc[27];
    T s10[10];
    T cop[3];
    T Sinv[6];
    T Kh[6][6];
    T D2[6];
    T s[6];
    T twist[6];
    PatchScratch<T> scr;
};

template <class T, int PTS, int WPB>
__global__ void __launch_bounds__(32 * WPB) exact_bristle_kernel(SceneDev sc, ExactScene es, ExactIO io, ExactPairs ps, const ExRec<T>* __restrict__ recs,
                                                                 const unsigned* __restrict__ unit_off, const unsigned* __restrict__ unit_cnt, int U_s) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int nc = NC<T>::n;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    BristleSmem<T, PTS>& sm = reinterpret_cast<BristleSmem<T, PTS>*>(smem_raw)[wib];
    const long long W_small = io.n_env * es.n_bris * U_s;
    const long long n_prob = io.n_env * es.n_bris;
    for (long long pb = (long long)blockIdx.x * WPB + wib; pb < n_prob; pb += (long long)gridDim.x * WPB) {
        const long long env = pb / es.n_bris;
        const int k = es.bris_ins[pb - env * es.n_bris];
        const InsDev& ins = sc.ins[k];
        if (!ins.small && es.skip_large) continue;
        const long long ei = env * sc.n_ins + k;
        long long u0, u1;   // this problem's units
        if (ins.small) { u0 = pb * U_s; u1 = u0 + U_s; }
        else { const long long p = env * ps.n_large + es.large_index[k]; u0 = W_small + ps.unit_start[p]; u1 = W_small + ps.unit_start[p + 1]; }
        const double* fp = io.params ? io.params[ei].p : ins.p;
        const BristleP bf = {fp[0], fp[1], fp[2], fp[3], fp[4], fp[5], fp[6]};
        const long long sb = 6 * ((long long)sc.n_bristle * env + ins.bristle_id);
        if (lane < 6) { sm.s[lane] = ldT<T>(io.s, sb + lane); sm.twist[lane] = ldT<T>(io.twist, 6 * ei + lane); }
        long long n_points = 0;
        for (long long u = u0; u < u1; ++u) n_points += unit_cnt[u];
        __syncwarp();
        if (n_points > 0) {
            for (int pass = 0; pass < 3; ++pass) {
                const int nt = pass == 0 ? 10 : (pass == 1 ? 27 : 6);
                double* accd = reinterpret_cast<double*>(sm.acc);
                for (int e = lane; e < nt * nc; e += 32) accd[e] = 0.0;
                __syncwarp();
                for (long long u = u0; u < u1; ++u) {
                    const unsigned off = unit_off[u], cnt = unit_cnt[u];
                    for (unsigned base = 0; base < cnt; base += PTS) {
                        const int m = (int)(cnt - base < (unsigned)PTS ? cnt - base : (unsigned)PTS);
                        if (lane < m) {
                            const ExRec<T>& rc = recs[off + base + lane];
                            const X3<T> n = x3<T>(rc.n[0], rc.n[1], rc.n[2]), r = x3<T>(rc.r[0], rc.r[1], rc.r[2]);
                            if (pass == 0) terms_cop(n, r, rc.dA, rc.p, sm.terms[lane]);
                            else if (pass == 1) terms_stiffness(n, r, rc.dA, rc.p, x3<T>(sm.cop[0], sm.cop[1], sm.cop[2]), sm.terms[lane]);
                            else terms_friction(bf, n, r, rc.dA, rc.p, x3<T>(sm.cop[0], sm.cop[1], sm.cop[2]), sm.D2, sm.twist, sm.terms[lane]);
                        }
                        __syncwarp();
                        // lane e owns scalar e of the running sums and adds the points one after the other (the reference's association)
                        for (int e = lane; e < nt * nc; e += 32) {
                            double a = accd[e];
                            const bool subtract = pass == 1 && e >= 18 * nc;   // K11 -= ...
                            for (int q = 0; q < m; ++q) {
                                const double t = reinterpret_cast<const double*>(sm.terms[q])[e];
                                a = subtract ? a - t : a + t;
                            }
                            accd[e] = a;
                        }
                        __syncwarp();
                    }
                }
                if (pass == 1) bristle_after_stiffness(sm.acc, bf, sm.s, sm.Sinv, sm.Kh, sm.D2, sm.scr, Coop{lane});   // every lane: the eigen-decomposition is dealt to the warp
                else if (lane == 0) {
                    if (pass == 0) {
                        for (int j = 0; j < 10; ++j) sm.s10[j] = sm.acc[j];
                        const X3<T> cop = xdivide(x3<T>(sm.acc[7], sm.acc[8], sm.acc[9]), sm.acc[6]);
                        sm.cop[0] = cop[0]; sm.cop[1] = cop[1]; sm.cop[2] = cop[2];
                    } else {
                        T w[6], sd[6];
                        bristle_finish(sm.s10, sm.acc, x3<T>(sm.cop[0], sm.cop[1], sm.cop[2]), bf, sm.s, sm.Sinv, sm.Kh, w, sd);
                        for (int j = 0; j < 6; ++j) { stT<T>(io.wrench, 6 * ei + j, w[j]); stT<T>(io.sdot, sb + j, sd[j]); }
                    }
                }
                __syncwarp();
            }
        } else if (lane == 0) {   // no_contact!(::Bristle) (friction.jl:76-81)
            const double ti = -(1 / bf.tau);
            for (int j = 0; j < 6; ++j) { stT<T>(io.wrench, 6 * ei + j, T(0.0)); stT<T>(io.sdot, sb + j, ti * sm.s[j]); }
        }
        if (lane == 0) io.flags[ei] = (io.flags[ei] & ~kFlagContact) | (n_points > 0 ? kFlagContact : 0);
        __syncwarp();
    }
}

template <class T> cudaError_t ensure_buf(T*& p, size_t& cap, size_t need) {
    if (need <= cap) return cudaSuccess;
    alloc_generation()++;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, need * sizeof(T));
    if (e == cudaSuccess) cap = need;
    return e;
}

}  // namespace

struct ExactBuffers {
    unsigned* ctr = nullptr;          // [0] points reserved so far, [1] overflow
    unsigned* h_ctr = nullptr;        // pinned copy, read by exact_check() after the caller's synchronisation
    bool check_pending = false;
    double* recs = nullptr; size_t cap_rec_doubles = 0;
    unsigned* unit_off = nullptr; size_t cap_off = 0;
    unsigned* unit_cnt = nullptr; size_t cap_cnt = 0;
    size_t want_points = 1u << 16;
    size_t cap_points = 0;
    unsigned last_points = 0;
};
ExactBuffers* exact_buffers_create() { return new ExactBuffers(); }
void exact_buffers_destroy(ExactBuffers* b) {
    if (!b) return;
    cudaFree(b->ctr); cudaFree(b->recs); cudaFree(b->unit_off); cudaFree(b->unit_cnt);
    if (b->h_ctr) cudaFreeHost(b->h_ctr);
    delete b;
}
unsigned exact_last_points(const ExactBuffers* b) { return b->last_points; }

// Queues the two kernels; nothing is read back here.  The TractionCache buffer grows like the reference's VectorCache
// (src/obb/vector_cache.jl:11-15), after the fact: the caller synchronises once at the end of the evaluation it queued and asks
// exact_check(), which raises the capacity to what the counter says was needed and tells the caller to queue the evaluation again.
template <class T> static cudaError_t exact_eval_t(const SceneDev& sc, const ExactScene& es, const ExactIO& io, const ExactPairs& ps, ExactBuffers* b,
                                                   cudaStream_t stream, int* n_launches) {
    const long long n_prob = io.n_env * es.n_bris;
    if (n_prob <= 0) return cudaSuccess;
    constexpr int nc = NC<T>::n;
    const int U_s = (ps.small_cap + kUnit - 1) / kUnit > 0 ? (ps.small_cap + kUnit - 1) / kUnit : 1;
    const size_t n_unit_slots = (size_t)n_prob * U_s + ps.max_large_units;
    if (n_unit_slots >= (1ull << 31)) return cudaErrorMemoryAllocation;
    int n_sm = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    if (!b->ctr) ECU(cudaMalloc(&b->ctr, 2 * sizeof(unsigned)));
    if (!b->h_ctr) ECU(cudaHostAlloc(reinterpret_cast<void**>(&b->h_ctr), 2 * sizeof(unsigned), cudaHostAllocDefault));
    ECU(ensure_buf(b->unit_off, b->cap_off, n_unit_slots));
    ECU(ensure_buf(b->unit_cnt, b->cap_cnt, n_unit_slots));
    constexpr int PTS = nc == 1 ? 32 : 8;
    constexpr int WPB = nc == 1 ? 4 : 2;
    const size_t smem = sizeof(BristleSmem<T, PTS>) * WPB;
    {
        struct Tag {};
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag, 2>(nc == 1 ? 0 : 1);
        if (sl.smem < smem) { ECU(cudaFuncSetAttribute(exact_bristle_kernel<T, PTS, WPB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); sl.smem = smem; }
    }
    b->cap_points = std::min<size_t>(std::max(b->want_points, b->cap_points), 0xfffffff0u);
    ECU(ensure_buf(b->recs, b->cap_rec_doubles, b->cap_points * 8 * 7));   // sized for the Jacobian mode: both modes share the buffer
    ECU(cudaMemsetAsync(b->ctr, 0, 2 * sizeof(unsigned), stream));
    const unsigned grid_p = (unsigned)std::min<size_t>(n_unit_slots, (size_t)n_sm * 8);
    exact_points_kernel<T><<<grid_p, kUnit, 0, stream>>>(sc, es, io, ps, reinterpret_cast<ExRec<T>*>(b->recs), (unsigned)b->cap_points, b->ctr, b->unit_off, b->unit_cnt, U_s);
    const unsigned grid_b = (unsigned)std::min<long long>((n_prob + WPB - 1) / WPB, (long long)n_sm * 8);
    exact_bristle_kernel<T, PTS, WPB><<<grid_b, 32 * WPB, smem, stream>>>(sc, es, io, ps, reinterpret_cast<const ExRec<T>*>(b->recs), b->unit_off, b->unit_cnt, U_s);
    if (n_launches) *n_launches += 2;
    ECU(cudaGetLastError());
    ECU(cudaMemcpyAsync(b->h_ctr, b->ctr, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    b->check_pending = true;
    return cudaSuccess;
}

cudaError_t exact_bristle_eval(const SceneDev& sc, const ExactScene& es, const ExactIO& io, const ExactPairs& ps, int dual, ExactBuffers* b, cudaStream_t stream,
                               int* n_launches) {
    return dual ? exact_eval_t<X6>(sc, es, io, ps, b, stream, n_launches) : exact_eval_t<double>(sc, es, io, ps, b, stream, n_launches);
}

// After the caller synchronised the stream: 0 = the TractionCache buffer sufficed, 1 = it did not (capacity raised: queue the evaluation
// again), -1 = it cannot be made large enough.
void exact_mark_clear(ExactBuffers* b) { if (b) b->check_pending = false; }
void exact_mark_pending(ExactBuffers* b) { if (b && b->h_ctr) b->check_pending = true; }
int exact_check(ExactBuffers* b) {
    if (!b || !b->check_pending) return 0;
    b->check_pending = false;
    b->last_points = b->h_ctr[0];
    if (!b->h_ctr[1]) return 0;
    if (b->cap_points >= 0xfffffff0u) return -1;
    b->want_points = (size_t)b->h_ctr[0] + (size_t)b->h_ctr[0] / 4 + 1024;   // the counter kept counting: the need is known exactly
    return 1;
}

}  // namespace pfc
