// pfc_dual_chunked.cu -- Jacobian mode of the regularized-friction instructions: the 6 partials travel in three chunks of 2.
//
// Radau obtains the Jacobian of the ODE right-hand side by forward-mode AD in chunks of 6
// (/root/reference/src/radau/radau_functions.jl:2-26, N_chunk = 6 at src/mechanism_scenario.jl:181):
// forceAllElasticIntersections! then runs on ForwardDiff.Dual{Nothing,Float64,6}, i.e. every scalar that depends on the state carries
// its value and 6 partials, while the candidate-pair lists come from the Float64 state (calcTriTetIntersections! always uses m.float,
// non_friction.jl:94-101).  The device code is the templated source of the Float64 path (pfc_clip.cuh, pfc_patch.cuh) on Dual<2>.
// Bristle instructions are skipped here: pfc_exact.cu evaluates them on Dual<6> in the reference's operation order.
#include <algorithm>
#include <mutex>

#include "pfc_dual.cuh"
#include "pfc_launch.h"

namespace pfc {

namespace {

// ---- the 6 partials in three chunks of 2, work pooled over a tile of problems -------------------------------------------------------
// One sub-triangle on Dual<6> keeps ~240 doubles alive (its polygon, the twist, the accumulators, temporaries): twice the register
// file per thread.  A Dual<2> needs 3 doubles per scalar instead of 7, and carrying the 6 partials as 3 independent (pair, chunk) items
// triples the parallelism.  The value part is recomputed by every chunk (9 instead of 7 units of work per pair); the three chunks of a
// pair produce bit-identical value parts, chunk 0's is the one stored.
//
// A CTA of 128 threads owns a TILE of kDP consecutive problems ((chunk, environment, instruction) in whole-Jacobian mode) and every
// phase is flattened over the tile, like narrow_tile_kernel:
//   1. problem contexts: Dual<2> transforms / twists of the three chunks, the Float64 value context, "is any input seeded?";
//   2. the tile's candidate pairs are dealt one per thread for the Float64 clip (two thirds clip to nothing; decisions are value-only)
//      -- or come already filtered from dual_prefilter_kernel, once per evaluation for all seed chunks; a block scan packs the
//      survivors in candidate order;
//   3. survivors of problems whose TRANSFORM depends on the seeds become 3 work items (one per chunk of partials), the whole pair on
//      Dual<2>; survivors of problems whose twist alone does (velocity seeds) ONE item: Float64 polygon, the twist-dependent part on
//      Dual<2> three times (pfc_twist.cuh); problems none of whose inputs depends on the seeds (the seeds sit on another body: 18 of 32
//      (instruction, chunk) pairs of boxes.jl) copy the Float64 wrench of the same evaluation when the caller has it (one Float64 item
//      per survivor otherwise); items are dealt one per thread, their 42 output scalars + point count go to shared memory;
//   4. one thread per (problem, output scalar) adds its items in candidate order (sequential, fixed order: reproducible, no atomics).
// The warp-per-problem kernel this replaces left 19 of 32 lanes idle and 3 of 8 resident warps without work (ncu, round 1).
typedef Dual<2> D2;
constexpr int kDP = 16;           // problems per tile (boxes.jl: four environments' instructions of one seed chunk, ~240 items on 128 threads;
                                  // measured 8 / 16 / 20 problems: 5.08 / 4.54 / 4.82 ms for the whole Jacobian of 4096 environments)
constexpr int kDT = 128;          // threads per CTA
constexpr int kResStride = 43;    // per item: the 42 output scalars [7 comp + (0 = value, 1 + d = partial d)] + point count, odd stride
constexpr int kTotStride = 43;    // 42 output scalars + point count

struct DualTileSmem {
    PatchCtx<D2> cx[kDP][3];
    PatchCtx<double> cxv[kDP];
    double res[kDT * kResStride];
    double tot[kDP][kTotStride + 1];
    long long ei[kDP], er[kDP];   // problem index among the (chunk, env, ins) entries / among the real (env, ins) ones; ei = -1: nothing to do
    const unsigned* pl_s[kDP];
    const int3* pl_l[kDP];
    const double* fp[kDP];        // friction parameters of problem q (InsDev::p, or its environment's row of the parameter table)
    int ins[kDP], seeded[kDP], pflags[kDP], prefiltered[kDP], copied[kDP];
    int pre[kDP + 1];             // candidates before problem q
    int surv_a[kDT], surv_b[kDT];
    int item_off[kDT + 1];
    int q_lo[kDP], q_hi[kDP];     // item range of problem q in the current survivor round
    unsigned char surv_q[kDT];
    int warp_tot[kDT / 32];
    long long next_tile;
};

// exclusive block scan of one int per thread (kDT threads); returns the total through `total`
PFC_D int block_scan_excl(int v, int* warp_tot, int& total) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    __syncthreads();   // warp_tot of the previous scan has been read
    if (lane == 31) warp_tot[wib] = incl;
    __syncthreads();
    int before = 0;
    total = 0;
#pragma unroll
    for (int w = 0; w < kDT / 32; ++w) { const int t = warp_tot[w]; if (w < wib) before += t; total += t; }
    return before + incl - v;
}

// Float64 clip of every candidate pair of the small regularized instructions, once per REAL (environment, instruction): the survivors,
// packed in candidate order, are what every seed chunk of the Jacobian works on (two thirds of the candidates clip to nothing).  One warp
// per problem, 32 candidates per pass.
__global__ void __launch_bounds__(128) dual_prefilter_kernel(SceneDev sc, long long n_env, const double* __restrict__ X, const long long* __restrict__ n_pairs,
                                                             const unsigned* __restrict__ pairs, int cap, unsigned* __restrict__ surv, int* __restrict__ surv_n,
                                                             const InsParam* __restrict__ params) {
    const int lane = threadIdx.x & 31;
    const long long n_prob = n_env * sc.n_ins;
    for (long long ei = (long long)blockIdx.x * 4 + (threadIdx.x >> 5); ei < n_prob; ei += (long long)gridDim.x * 4) {
        const int k = int(ei % sc.n_ins);
        const InsDev& ins = sc.ins[k];
        if (!ins.small || ins.model != PFC_MODEL_REGULARIZED) { if (lane == 0) surv_n[ei] = 0; continue; }
        const int n = (int)n_pairs[ei];
        PatchCtx<double> cx;
        {
            const double* Xe = X + 16 * ei;   // col-major 4x4 -> row-major rotation + translation
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
                for (int j = 0; j < 3; ++j) cx.x21.r[3 * i + j] = Xe[4 * j + i];
                cx.x21.t[i] = Xe[12 + i];
            }
        }
        cx.x12 = inverse(cx.x21);
        cx.w_ang = mk<double>(0.0, 0.0, 0.0); cx.w_lin = cx.w_ang;
        if (params) { cx.chi = params[ei].chi; cx.Ebar1 = params[ei].Ebar1; cx.Ebar2 = params[ei].Ebar2; }
        else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
        cx.n_quad = ins.n_quad;
        const unsigned* in = pairs + (size_t)cap * ei;
        unsigned* out = surv + (size_t)cap * ei;
        int kept = 0;
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            unsigned e = 0;
            bool keep = false;
            if (i < n) { e = in[i]; keep = survives_f64(sc, ins, int((e >> 15) & 0x7fffu), int(e & 0x7fffu), cx); }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) out[kept + __popc(m & ((1u << lane) - 1u))] = e;
            kept += __popc(m);
        }
        if (lane == 0) surv_n[ei] = kept;
    }
}

__global__ void __launch_bounds__(kDT) eval_dual6_tile_kernel(SceneDev sc, DualIO io, PairSource ps, unsigned* __restrict__ ticket) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DualTileSmem& sm = *reinterpret_cast<DualTileSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    const long long n_prob = io.n_env * sc.n_ins;
    const long long n_tile = (n_prob + kDP - 1) / kDP;
    for (long long tile = blockIdx.x; tile < n_tile;) {
        // ---- 1. contexts: warp w fills problems w, w + 4, ...
        for (int q = wib; q < kDP; q += kDT / 32) {
            const long long ei = tile * kDP + q;
            bool active = false;
            if (ei < n_prob) {
                const long long env_v = ei / sc.n_ins;
                const int k = int(ei - env_v * sc.n_ins);
                const long long env = env_v % io.n_real, er = env * sc.n_ins + k;   // the real environment whose pair list this problem reads
                const InsDev& ins = sc.ins[k];
                if (ins.model == PFC_MODEL_REGULARIZED) {   // bristle: pfc_exact.cu
                    active = true;
                    const InsParam* cp = io.params ? io.params + er : nullptr;   // the real environment's contact parameters, if it has its own
                    const double* Xp = io.X7 + 112 * ei;
                    const double* tw = io.twist7 + 42 * ei;
                    bool mine_x = false, mine_t = false;   // does the transform / the twist depend on the seeds?  (lanes share the 18 x 6 partials)
                    for (int e = lane; e < 18 * 6; e += 32) {
                        const int sc_i = e / 6, d = e - sc_i * 6;
                        const double* base = sc_i < 12 ? Xp + 7 * (sc_i < 9 ? (4 * (sc_i % 3) + sc_i / 3) : (12 + sc_i - 9)) : tw + 7 * (sc_i - 12);
                        const bool nz = base[1 + d] != 0.0;
                        if (sc_i < 12) mine_x |= nz; else mine_t |= nz;
                    }
                    const int seeded = __any_sync(0xffffffffu, mine_x) ? 2 : (__any_sync(0xffffffffu, mine_t) ? 1 : 0);
                    const bool copy_only = seeded == 0 && ps.w_f64;   // nothing to differentiate and the values exist: no contexts needed
                    if (lane < 3 && !copy_only) {   // chunk `lane`'s context: partials 2 lane and 2 lane + 1
                        PatchCtx<D2>& cx = sm.cx[q][lane];
                        auto ld = [&](const double* p7) { D2 r; r.v = p7[0]; r.p[0] = p7[1 + 2 * lane]; r.p[1] = p7[2 + 2 * lane]; return r; };
#pragma unroll
                        for (int i = 0; i < 3; ++i) {
#pragma unroll
                            for (int j = 0; j < 3; ++j) cx.x21.r[3 * i + j] = ld(Xp + 7 * (4 * j + i));
                            cx.x21.t[i] = ld(Xp + 7 * (12 + i));
                        }
                        cx.x12 = inverse(cx.x21);
                        cx.w_ang = mk<D2>(ld(tw), ld(tw + 7), ld(tw + 14));
                        cx.w_lin = mk<D2>(ld(tw + 21), ld(tw + 28), ld(tw + 35));
                        if (cp) { cx.chi = cp->chi; cx.Ebar1 = cp->Ebar1; cx.Ebar2 = cp->Ebar2; }
                        else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
                        cx.n_quad = ins.n_quad;
                    }
                    __syncwarp();
                    if (lane == 0) {
                        if (!copy_only) {
                            const PatchCtx<D2>& c0 = sm.cx[q][0];
                            PatchCtx<double>& cxv = sm.cxv[q];
#pragma unroll
                            for (int i = 0; i < 9; ++i) { cxv.x21.r[i] = c0.x21.r[i].v; cxv.x12.r[i] = c0.x12.r[i].v; }
#pragma unroll
                            for (int i = 0; i < 3; ++i) { cxv.x21.t[i] = c0.x21.t[i].v; cxv.x12.t[i] = c0.x12.t[i].v; }
                            cxv.w_ang = mk<double>(c0.w_ang.x.v, c0.w_ang.y.v, c0.w_ang.z.v);
                            cxv.w_lin = mk<double>(c0.w_lin.x.v, c0.w_lin.y.v, c0.w_lin.z.v);
                            cxv.chi = c0.chi; cxv.Ebar1 = c0.Ebar1; cxv.Ebar2 = c0.Ebar2; cxv.n_quad = c0.n_quad;
                        }
                        sm.ei[q] = ei; sm.er[q] = er; sm.ins[q] = k; sm.seeded[q] = seeded; sm.pflags[q] = 0; sm.fp[q] = cp ? cp->p : ins.p;
                        const bool pf = ins.small && ps.surv_pairs;       // survivors of the Float64 clip are listed already
                        const bool cp = seeded == 0 && ps.w_f64;          // nothing to differentiate and the values exist: copy them
                        sm.prefiltered[q] = pf ? 1 : 0; sm.copied[q] = cp ? 1 : 0;
                        sm.pre[q + 1] = cp ? 0 : (pf ? ps.surv_n[er] : (int)io.n_pairs[er]);   // turned into a prefix below
                        sm.pl_s[q] = ins.small ? (pf ? ps.surv_pairs : ps.small_pairs) + (size_t)ps.small_cap * er : nullptr;
                        sm.pl_l[q] = ins.small ? nullptr : ps.large_sorted + ps.seg_start[env * ps.n_large + ps.large_index[k]];
                    }
                }
            }
            if (!active && lane == 0) { sm.fp[q] = nullptr; sm.ei[q] = -1; sm.er[q] = 0; sm.ins[q] = 0; sm.seeded[q] = 0; sm.pflags[q] = 0; sm.pre[q + 1] = 0; sm.pl_s[q] = nullptr; sm.pl_l[q] = nullptr; sm.prefiltered[q] = 0; sm.copied[q] = 0; }
            for (int j = lane; j <= kTotStride; j += 32) sm.tot[q][j] = 0.0;
        }
        __syncthreads();
        if (tid == 0) {
            sm.pre[0] = 0;
            for (int q = 0; q < kDP; ++q) sm.pre[q + 1] += sm.pre[q];
            sm.next_tile = (long long)gridDim.x + atomicAdd(ticket, 1u);
        }
        __syncthreads();
        const int n_cand = sm.pre[kDP];
        for (int c0 = 0; c0 < n_cand; c0 += kDT) {
            // ---- 2. Float64 clip of one candidate per thread; survivors packed in candidate order
            const int c = c0 + tid;
            int a = 0, b = 0, q = 0;
            bool keep = false;
            if (c < n_cand) {
#pragma unroll
                for (int r = 1; r < kDP; ++r) q += (c >= sm.pre[r]);
                const int i = c - sm.pre[q];
                if (sm.pl_s[q]) { const unsigned e = sm.pl_s[q][i]; a = int((e >> 15) & 0x7fffu); b = int(e & 0x7fffu); }
                else { const int3 e = sm.pl_l[q][i]; a = e.y; b = e.z; }
                keep = sm.prefiltered[q] ? true : survives_f64(sc, sc.ins[sm.ins[q]], a, b, sm.cxv[q]);
            }
            int n_surv;
            const int slot = block_scan_excl(keep ? 1 : 0, sm.warp_tot, n_surv);
            if (keep) { sm.surv_a[slot] = a; sm.surv_b[slot] = b; sm.surv_q[slot] = (unsigned char)q; }
            if (tid < kDP) { sm.q_lo[tid] = 0; sm.q_hi[tid] = 0; }
            __syncthreads();
            if (n_surv == 0) continue;   // block-uniform
            // ---- 3a. items: 3 per survivor of a seeded problem, 1 otherwise
            int n_items;
            const int mine_n = tid < n_surv ? (sm.seeded[sm.surv_q[tid]] == 2 ? 3 : 1) : 0;
            const int off = block_scan_excl(mine_n, sm.warp_tot, n_items);
            if (tid < n_surv) {
                sm.item_off[tid] = off;
                const int sq = sm.surv_q[tid];
                if (tid == 0 || (int)sm.surv_q[tid - 1] != sq) sm.q_lo[sq] = off;
                if (tid == n_surv - 1 || (int)sm.surv_q[tid + 1] != sq) sm.q_hi[sq] = off + mine_n;
            }
            if (tid == 0) sm.item_off[n_surv] = n_items;
            __syncthreads();
            for (int i0 = 0; i0 < n_items; i0 += kDT) {
                const int i1 = min(n_items, i0 + kDT);
                // ---- 3b. one item per thread
                const int it = i0 + tid;
                if (it < i1) {
                    int lo = 0, hi = n_surv - 1;   // the survivor s with item_off[s] <= it < item_off[s + 1]
                    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (sm.item_off[mid] <= it) lo = mid; else hi = mid - 1; }
                    const int sq = sm.surv_q[lo], chunk = it - sm.item_off[lo];
                    const InsDev& ins = sc.ins[sm.ins[sq]];
                    double* res = sm.res + tid * kResStride;
                    int flags = 0, pts;
                    if (sm.seeded[sq] == 2) {          // the transform carries partials: the whole pair on Dual<2>, this item's 2 partials
                        const PatchCtx<D2>& cx = sm.cx[sq][chunk];
                        Accum<D2, 6> acc;
                        acc.fp = sm.fp[sq]; acc.w_ang = cx.w_ang; acc.w_lin = cx.w_lin; acc.dump = nullptr; acc.dump_cap = 0;
                        acc.reset(ACC_REGULARIZED);
                        integrate_pair(sc, ins, sm.surv_a[lo], sm.surv_b[lo], cx, acc, flags);
#pragma unroll
                        for (int j = 0; j < 6; ++j) { res[7 * j] = acc.a[j].v; res[7 * j + 1 + 2 * chunk] = acc.a[j].p[0]; res[7 * j + 2 + 2 * chunk] = acc.a[j].p[1]; }
                        pts = acc.n_points;
                    } else if (sm.seeded[sq] == 1) {   // only the twist does: Float64 polygon, the three chunks of partials one after another
                        const PatchCtx<double>& cxv = sm.cxv[sq];
                        PolyRec<double> pr;
                        pts = 0;
                        const bool hit = clip_pair(sc, ins, sm.surv_a[lo], sm.surv_b[lo], cxv, pr, flags);
#pragma unroll 1
                        for (int c3 = 0; c3 < 3; ++c3) {
                            const PatchCtx<D2>& cx = sm.cx[sq][c3];
                            TwistAcc<2> acc;
                            acc.fp = sm.fp[sq]; acc.w_ang = cx.w_ang; acc.w_lin = cx.w_lin; acc.n_points = 0;
#pragma unroll
                            for (int j = 0; j < 6; ++j) acc.a[j] = D2(0.0);
                            if (hit) {
                                Vec3<double> v2 = pr.v[pr.n - 1];
                                for (int k = 0; k < pr.n; ++k) {
                                    const Vec3<double> v1 = v2;
                                    v2 = pr.v[k];
                                    integrate_subtri_tw(v1, v2, pr.cen, pr.nrm, pr.eps_r, cxv.chi, cxv.Ebar2, cxv.n_quad, acc);
                                }
                            }
#pragma unroll
                            for (int j = 0; j < 6; ++j) { res[7 * j] = acc.a[j].v; res[7 * j + 1 + 2 * c3] = acc.a[j].p[0]; res[7 * j + 2 + 2 * c3] = acc.a[j].p[1]; }
                            pts = acc.n_points;
                        }
                    } else {                            // nothing does: the Float64 evaluation
                        const PatchCtx<double>& cx = sm.cxv[sq];
                        Accum<double, 6> acc;
                        acc.fp = sm.fp[sq]; acc.w_ang = cx.w_ang; acc.w_lin = cx.w_lin; acc.dump = nullptr; acc.dump_cap = 0;
                        acc.reset(ACC_REGULARIZED);
                        integrate_pair(sc, ins, sm.surv_a[lo], sm.surv_b[lo], cx, acc, flags);
#pragma unroll
                        for (int j = 0; j < 6; ++j) res[7 * j] = acc.a[j];
                        pts = acc.n_points;
                    }
                    res[42] = (double)pts;
                    if (flags) atomicOr(&sm.pflags[sq], flags);
                }
                __syncthreads();
                // ---- 4. fixed-order sums: thread (problem, scalar) adds this round's items of its problem in candidate order
                for (int o = tid; o < kDP * kTotStride; o += kDT) {
                    const int oq = o / kTotStride, j = o - oq * kTotStride;
                    const int lo = sm.q_lo[oq], a_ = max(lo, i0), b_ = min(sm.q_hi[oq], i1);
                    if (a_ >= b_) continue;
                    double sum = sm.tot[oq][j];
                    const int which = j == 42 ? 0 : j % 7;
                    if (sm.seeded[oq] == 2) {
                        // item (survivor k, chunk c) sits at lo + 3 k + c; the value and the point count come from chunk 0, partial d from chunk d / 2
                        const int c_ = which == 0 ? 0 : (which - 1) >> 1;
                        const int first = a_ + ((c_ - (a_ - lo)) % 3 + 3) % 3;
                        for (int it2 = first; it2 < b_; it2 += 3) sum += sm.res[(it2 - i0) * kResStride + j];
                    } else {
                        if (sm.seeded[oq] == 0 && which != 0) continue;   // partials of an instruction that does not depend on the seeds: 0
                        for (int it2 = a_; it2 < b_; ++it2) sum += sm.res[(it2 - i0) * kResStride + j];
                    }
                    sm.tot[oq][j] = sum;
                }
                __syncthreads();
            }
        }
        // ---- results: wrench (zero without contact), flags
        for (int o = tid; o < kDP * 42; o += kDT) {
            const int q = o / 42, j = o - 42 * q;
            if (sm.ei[q] < 0) continue;
            if (sm.copied[q]) io.wrench7[42 * sm.ei[q] + j] = (j % 7 == 0) ? ps.w_f64[6 * sm.er[q] + j / 7] : 0.0;   // (zero without contact already)
            else io.wrench7[42 * sm.ei[q] + j] = sm.tot[q][42] > 0.0 ? sm.tot[q][j] : 0.0;
        }
        if (tid < kDP && sm.ei[tid] >= 0 && !sm.copied[tid]) {   // (a copied problem's contact flag was set by the Float64 evaluation)
            const int fl = sm.pflags[tid] | (sm.tot[tid][42] > 0.0 ? kFlagContact : 0);
            int* f = &io.flags[sm.er[tid]];
            if (io.n_real == io.n_env) *f = (*f & ~kFlagContact) | fl;
            else if (fl) atomicOr(f, fl);   // several chunks share the word
        }
        __syncthreads();
        tile = sm.next_tile;
    }
}

}  // namespace

const unsigned* large_seg_start_ptr(const LargeBuffers* b);
const int3* large_sorted_ptr(const LargeBuffers* b);

cudaError_t launch_eval_dual6(const SceneDev& sc, long long n_env, const double* X7, const double* twist7, const double* s7, double* wrench7, double* sdot7,
                              const long long* n_pairs, int* flags, const unsigned* small_pairs, int small_cap, const LargeBuffers* lb,
                              const int32_t* large_index, int n_large, const InsParam* params, cudaStream_t stream, unsigned* ticket, long long n_real,
                              const DualShared* shared) {
    DualIO io{n_env, X7, twist7, s7, wrench7, sdot7, n_pairs, flags, n_real > 0 ? n_real : n_env, params};
    PairSource ps{small_pairs, small_cap, lb ? large_sorted_ptr(lb) : nullptr, lb ? large_seg_start_ptr(lb) : nullptr, large_index, n_large,
                  shared ? shared->surv_pairs : nullptr, shared ? shared->surv_n : nullptr, shared ? shared->w_f64 : nullptr};
    const long long n_prob = n_env * sc.n_ins;
    if (n_prob == 0) return cudaSuccess;
    struct DualTileTag {};
    cudaError_t err = cudaSuccess;
    int resident;
    {
        std::lock_guard<std::mutex> lock(launch_mutex());
        LaunchSlot& slot = launch_slot<DualTileTag>();
        if (!slot.blocks) {
            slot.blocks = persistent_blocks((const void*)eval_dual6_tile_kernel, kDT, sizeof(DualTileSmem), &err);
            if (err != cudaSuccess) return err;
        }
        resident = slot.blocks;
    }
    const long long n_tile = (n_prob + kDP - 1) / kDP;
    const unsigned blocks = (unsigned)std::min<long long>(n_tile, resident);
    err = cudaMemsetAsync(ticket, 0, sizeof(unsigned), stream);   // the tile ticket of this launch (owned by the calling context)
    if (err != cudaSuccess) return err;
    eval_dual6_tile_kernel<<<blocks, kDT, sizeof(DualTileSmem), stream>>>(sc, io, ps, ticket);
    return cudaGetLastError();
}


cudaError_t launch_dual_prefilter(const SceneDev& sc, long long n_env, const double* X, const long long* n_pairs, const unsigned* small_pairs, int small_cap,
                                  unsigned* surv_pairs, int* surv_n, const InsParam* params, cudaStream_t stream) {
    const long long n_prob = n_env * sc.n_ins;
    if (n_prob == 0) return cudaSuccess;
    int n_sm = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    const unsigned blocks = (unsigned)std::min<long long>((n_prob + 3) / 4, (long long)n_sm * 8);
    dual_prefilter_kernel<<<blocks, 128, 0, stream>>>(sc, n_env, X, n_pairs, small_pairs, small_cap, surv_pairs, surv_n, params);
    return cudaGetLastError();
}

}  // namespace pfc
