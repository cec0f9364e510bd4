// pfc_small.cu -- contact-wrench evaluation for SMALL instructions (n_leaf1 * n_leaf2 <= 512), batched over environments:
// everything on chip, two launches per batch.
//
// This is the batched-environments path (config C3: thousands of copies of test/boxes.jl).  What the reference does per
// instruction in force_single_elastic_intersection! (/root/reference/src/contact_algorithms_non_friction.jl:70-84) --
//   calcTriTetIntersections! (dual-tree traversal, src/obb/tree_types.jl:88-111)
//   integrate_over!          (loop over candidate pairs, :136-143)
//   yes_contact!/no_contact! (src/contact_algorithms_friction.jl:50-81, 119-143)
// -- is done by two persistent-grid kernels (split so that each runs at the occupancy its register needs allow):
//   1. broad_tile_kernel    one warp per tile of 4 problems over a node table staged in shared memory: level-synchronous expansion
//                           of a flattened frontier (SAT on the open pairs, lanes dense; ordered rebuild) that ends in exactly the
//                           reference's recursion (DFS) order -- no atomics, no sort, deterministic, bit-exact pair lists;
//   2. narrow_tile_kernel   one CTA per tile of 4 problems, every phase flattened over them: clip in place in shared-memory polygon
//                           slots, (polygon, edge) sub-triangles dealt one per thread for quadrature + friction, per-problem sums in
//                           item order (bitwise reproducible; no floating-point atomics);
//   Bristle instructions on this path keep their pair lists from kernel 1 and are evaluated in the reference's operation order by
//   pfc_exact.cu (TractionCache materialised, three sequential passes).
// HBM traffic per instruction is the boundary data only: 22 doubles in, 6 doubles + 2 words out.
#include <cstdlib>

#include "pfc_launch.h"
#include "pfc_patch.cuh"
#include "pfc_sat.cuh"

namespace pfc {

namespace {

constexpr unsigned kDone = 0x80000000u;
PFC_D unsigned enc(int a, int b) { return (unsigned(a) << 15) | unsigned(b); }
PFC_D int dec_a(unsigned e) { return int((e >> 15) & 0x7fffu); }
PFC_D int dec_b(unsigned e) { return int(e & 0x7fffu); }

PFC_D int warp_sum_int(int x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}
PFC_D int warp_incl_scan(int x, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += v; }
    return x;
}

// Loads x_r2_r1 (col-major 4x4) into a row-major rotation + translation.
PFC_D void load_xform(const double* __restrict__ X, Xform<double>& x) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) x.r[3 * i + j] = X[4 * j + i];
        x.t[i] = X[12 + i];
    }
}

// x_r1_r2 for the broad phase with the reference's rounding: R' and -(R' * t), products summed left to right.
PFC_D void broad_phase_xform(const Xform<double>& x21, double* Rab, double* tab) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) Rab[3 * i + j] = x21.r[3 * j + i];
        tab[i] = -add_(add_(mul_(x21.r[i], x21.t[0]), mul_(x21.r[3 + i], x21.t[1])), mul_(x21.r[6 + i], x21.t[2]));
    }
}

// ---- kernel 1: broad phase, one WARP per tile of P problems, node table in shared memory ----------------------------
// What limited the first version of this kernel (one group of 16 lanes per problem, node records read from global memory) was
// not the FP64 pipe but the L1 data pipe: every lane gathered its two 128 B node records with its own vector loads, so one warp-wide load instruction touched 32 different lines and cost 32 wavefronts
// for 16 useful bytes each (ncu: l1tex__data_pipe_lsu_wavefronts ~ 66 % of peak, profiles/r1_v7_*).  Here
//   * the persistent CTA stages the node records of all small instructions ONCE in shared memory, as the float records of the
//     filtered SAT (FiltNode, 80 B: five 16 B loads per record);
//   * each warp owns a tile of P consecutive problems whose frontiers form ONE flattened array (problem-major, DFS order
//     inside a problem), and every level runs in two phases:
//       A. the OPEN node pairs (a compact work list of frontier slots) are tested one per lane, lanes dense: the filtered 15-axis
//          SAT in float (pfc_sat.cuh: sat_filter, a certified error bound) -> a result code per slot; the few slots it cannot
//          decide are compacted and tested again, one per lane, with the reference's FP64 arithmetic, operation by operation, on
//          the global node records;
//       B. an ordered rebuild over the whole frontier (integer work only): finished pairs are copied, hits are replaced by
//          their children in the reference's visiting order, a warp scan gives the positions; the open children form the
//          next work list.
//     When no pair is open the frontier is exactly the reference's recursion order: no atomics, no sort, bit-exact lists.
// Warps never synchronise with each other after the staging barrier.
constexpr int kNodeTabMax = 320;       // nodes staged at most (25 KB of FiltNode); larger scenes test every pair exactly from global memory
template <int P> struct BroadTileLayout {
    // per warp: double xf[P][12] | long long ei[P] | FiltXf fxf[P] | unsigned front[2][P * cap] | int pre[2][P + 1] | int ins[P] |
    // u16 olist[2][P * cap] | u8 res[P * cap]
    __host__ __device__ static size_t warp_bytes(int cap) {
        const size_t b = sizeof(double) * P * 12 + sizeof(long long) * P + sizeof(FiltXf) * P + sizeof(unsigned) * 2 * P * cap +
                         sizeof(int) * (2 * (P + 1) + P) + sizeof(unsigned short) * 2 * P * cap + (size_t)P * cap;
        return (b + 15) / 16 * 16;
    }
    __host__ __device__ static size_t bytes(int cap, int n_warps, int n_stage) { return sizeof(FiltNode) * n_stage + warp_bytes(cap) * n_warps; }
};

template <int P, int NW, int MINB>
__global__ void __launch_bounds__(32 * NW, MINB) broad_tile_kernel(SceneDev sc, EvalIO io, int cap, int n_stage, unsigned* __restrict__ pairs_out) {
    constexpr int T = 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) pairs_out[(size_t)cap * io.n_env * sc.n_ins] = 0u;   // the narrow tile kernel's tile ticket
    // ---- node table of the filtered SAT (float records, kind / right for the rebuild): staged once per (persistent) CTA
    FiltNode* ftab_s = reinterpret_cast<FiltNode*>(smem_raw);
    for (int j = threadIdx.x; j < n_stage; j += 32 * NW) filt_node_from(sc.nodes[sc.small_node_lo + j], ftab_s[j]);
    __syncthreads();
    const FiltNode* ftab = ftab_s - sc.small_node_lo;
    const bool staged = n_stage > 0;   // otherwise every pair takes the exact test and the rebuild reads the FP64 records
    auto right_of = [&](int node) { return staged ? ftab[node].right : sc.nodes[node].right; };

    unsigned char* wbase = smem_raw + sizeof(FiltNode) * n_stage + BroadTileLayout<P>::warp_bytes(cap) * wib;
    double* xf = reinterpret_cast<double*>(wbase);
    long long* s_ei = reinterpret_cast<long long*>(xf + P * 12);
    FiltXf* fxf = reinterpret_cast<FiltXf*>(s_ei + P);
    unsigned* front = reinterpret_cast<unsigned*>(fxf + P);
    int* pre = reinterpret_cast<int*>(front + 2 * (size_t)P * cap);   // pre[b][q + 1]: end of problem q's segment in frontier b
    int* s_ins = pre + 2 * (P + 1);
    unsigned short* olist = reinterpret_cast<unsigned short*>(s_ins + P);
    unsigned char* res = reinterpret_cast<unsigned char*>(olist + 2 * (size_t)P * cap);
    const int fcap = P * cap;
    const long long n_prob = io.n_env * sc.n_small;
    const long long n_tile = (n_prob + P - 1) / P;
    for (long long tile = (long long)blockIdx.x * NW + wib; tile < n_tile; tile += (long long)gridDim.x * NW) {
        // ---- 0. per-problem transform of the broad phase (x_r1_r2 = inverse of x_r2_r1, the reference's rounding): 16 lanes per problem
        for (int j = lane; j < 16 * P; j += T) {
            const int q = j >> 4, l = j & 15;
            const long long prob = tile * P + q;
            if (prob < n_prob) {
                const long long jj = prob / io.n_env;   // scheduling order: instruction-major, heaviest instruction first
                const long long env = prob - jj * io.n_env;
                const int k = sc.small_heavy_first[jj];
                const long long ei = env * sc.n_ins + k;
                const double* X = io.X + 16 * ei;
                if (l < 9) xf[12 * q + l] = X[4 * (l / 3) + l % 3];
                else if (l < 12) { const int i = l - 9; xf[12 * q + l] = -add_(add_(mul_(X[4 * i], X[12]), mul_(X[4 * i + 1], X[13])), mul_(X[4 * i + 2], X[14])); }
                else if (l == 12) { s_ei[q] = ei; s_ins[q] = k; front[q] = enc(0, 0); olist[q] = (unsigned short)q; }
            } else if (l == 12) { s_ei[q] = -1; s_ins[q] = 0; }
        }
        const int n_valid = (int)((n_prob - tile * P) < P ? (n_prob - tile * P) : P);
        for (int j = lane; j <= P; j += T) pre[j] = j < n_valid ? j : n_valid;
        __syncwarp();
        if (lane < n_valid) filt_xf_from(xf + 12 * lane, xf + 12 * lane + 9, fxf[lane]);
        __syncwarp();
        int cur = 0, n_open = n_valid;
        int flags = 0;
        bool tile_overflow = false;   // warp-uniform
        unsigned dead = 0;   // problems whose frontier is empty (nobody writes their segment end any more); identical in every lane
#pragma unroll
        for (int q = 0; q < P; ++q) dead |= (q >= n_valid ? 1u : 0u) << q;
        int pc[P + 1];
        for (;;) {
            const int* pcs = pre + cur * (P + 1);
            int* pn = pre + (cur ^ 1) * (P + 1);
            const unsigned* fc = front + (size_t)cur * fcap;
            unsigned* fn = front + (size_t)(cur ^ 1) * fcap;
            const unsigned short* olc = olist + (size_t)cur * fcap;
            unsigned short* oln = olist + (size_t)(cur ^ 1) * fcap;
            pc[0] = 0;
#pragma unroll
            for (int q = 0; q < P; ++q) {
                pc[q + 1] = ((dead >> q) & 1u) ? pc[q] : pcs[q + 1];
                if (pc[q + 1] == pc[q]) dead |= 1u << q;
            }
            const int total = pc[P];
            if (n_open == 0) break;
            // ---- A1. filtered SAT on the open node pairs, one per lane (pfc_sat.cuh: float, certified bound); the slots it cannot decide
            // are listed in oln, which is free until the rebuild
            int n_und = 0;   // warp-uniform
            for (int j0 = 0; j0 < n_open; j0 += T) {
                const int j = j0 + lane;
                int c = 0;
                bool und = false;
                if (j < n_open) {
                    c = olc[j];
                    und = true;
                    if (staged) {
                        int q = 0;
#pragma unroll
                        for (int r = 1; r < P; ++r) q += (c >= pc[r]);
                        const unsigned e = fc[c];
                        const InsDev& ins = sc.ins[s_ins[q]];
                        const FiltNode a = ftab[ins.node_base1 + dec_a(e)], b = ftab[ins.node_base2 + dec_b(e)];
                        const int f = sat_filter(a, b, fxf[q]);
                        und = f == kSatUndecided;
                        if (!und) res[c] = (unsigned char)(f == kSatSeparated ? 0 : ((a.kind < 0) ? ((b.kind < 0) ? 1 : 2) : ((b.kind < 0) ? 3 : 4)));
                    }
                }
                const unsigned m = __ballot_sync(0xffffffffu, und);
                if (und) oln[n_und + __popc(m & ((1u << lane) - 1u))] = (unsigned short)c;
                n_und += __popc(m);
            }
            __syncwarp();
            // ---- A2. the reference's FP64 test on the undecided slots, from the global node records
            for (int k = lane; k < n_und; k += T) {
                const int c = oln[k];
                int q = 0;
#pragma unroll
                for (int r = 1; r < P; ++r) q += (c >= pc[r]);
                const unsigned e = fc[c];
                const InsDev& ins = sc.ins[s_ins[q]];
                const NodeRec& a = sc.nodes[ins.node_base1 + dec_a(e)];
                const NodeRec& b = sc.nodes[ins.node_base2 + dec_b(e)];
                // (the general path for every node: skipping the identity products of axis-aligned nodes, as the large path's traversal does,
                // makes the lanes of a work list diverge by node kind here -- measured 88 us against 84 us on 4096 environments)
                SatA A;
                sat_prepare_a<false>(a, xf + 12 * q, xf + 12 * q + 9, A);
                int code = 0;
                if (sat_test<false>(A, b)) code = (a.kind < 0) ? ((b.kind < 0) ? 1 : 2) : ((b.kind < 0) ? 3 : 4);
                res[c] = (unsigned char)code;
            }
            __syncwarp();
            // ---- B. ordered rebuild: children replace their parent in place (reference order), open children form the next work list
            int carry = 0;
            for (int c0 = 0; c0 < total; c0 += T) {
                const int c = c0 + lane;
                int cnt = 0, ocnt = 0, q = 0;
                unsigned ch0 = 0, ch1 = 0, ch2 = 0, ch3 = 0;
                if (c < total) {
#pragma unroll
                    for (int r = 1; r < P; ++r) q += (c >= pc[r]);
                    const unsigned e = fc[c];
                    if (e & kDone) { cnt = 1; ch0 = e; }
                    else {
                        const int code = res[c];
                        if (code) {
                            const int ia = dec_a(e), ib = dec_b(e);
                            const InsDev& ins = sc.ins[s_ins[q]];
                            const int al = ia + 1, ar = right_of(ins.node_base1 + ia), bl = ib + 1, br = right_of(ins.node_base2 + ib);   // pre-order: child 1 is the next record
                            if (code == 1) { cnt = 1; ch0 = kDone | enc(ar, br); }
                            else if (code == 2) { cnt = ocnt = 2; ch0 = enc(ia, bl); ch1 = enc(ia, br); }
                            else if (code == 3) { cnt = ocnt = 2; ch0 = enc(al, ib); ch1 = enc(ar, ib); }
                            else { cnt = ocnt = 4; ch0 = enc(al, bl); ch1 = enc(ar, bl); ch2 = enc(al, br); ch3 = enc(ar, br); }
                        }
                    }
                }
                const int mine = cnt | (ocnt << 16);
                int incl = mine;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
                const int chunk_total = __shfl_sync(0xffffffffu, incl, 31);
                const int excl = carry + incl - mine;
                const int at = excl & 0xffff, oat = excl >> 16;
                if (at + cnt <= fcap) {
                    if (cnt > 0) fn[at] = ch0;
                    if (cnt > 1) fn[at + 1] = ch1;
                    if (cnt > 2) { fn[at + 2] = ch2; fn[at + 3] = ch3; }
                    for (int k = 0; k < ocnt; ++k) oln[oat + k] = (unsigned short)(at + k);
                }
                // only instructions whose slot is smaller than n_leaf1 * n_leaf2 (mid-size trees) can overflow it: the tile is given up --
                // the host moves the instruction to the large path and repeats the evaluation
                tile_overflow |= __any_sync(0xffffffffu, cnt > 0 && at + cnt > fcap);
                if (c < total) {   // the last slot of problem q closes its segment.  pc[] is read with compile-time indices only: end_q is the
                    // first segment end above c (an 'r == q + 1' select chain is folded back into pc[q + 1], which puts pc[] in local memory)
                    int end_q = pc[P];
#pragma unroll
                    for (int r = P - 1; r >= 1; --r) end_q = c < pc[r] ? pc[r] : end_q;
                    if (c + 1 == end_q) pn[q + 1] = min(at + cnt, fcap);
                }
                carry += chunk_total;
            }
            n_open = carry >> 16;
            __syncwarp();
            cur ^= 1;
            if (tile_overflow) break;
        }
        if (tile_overflow) {
#pragma unroll
            for (int q = 0; q < P; ++q)
                if (lane == q && s_ei[q] >= 0) {
                    io.n_pairs[s_ei[q]] = 0;
                    io.flags[s_ei[q]] = kFlagOverflow;
                    if (sc.ins_overflow) sc.ins_overflow[s_ins[q]] = 1;
                }
            __syncwarp();
            continue;
        }
        // ---- results: pair lists (DFS order), counts, flags (pc[] holds the final segments)
        {
            const unsigned* fc = front + (size_t)cur * fcap;
            const int total = pc[P];
            for (int c = lane; c < total; c += T) {
                int q = 0;
#pragma unroll
                for (int r = 1; r < P; ++r) q += (c >= pc[r]);
                int beg_q = 0;   // the last segment start at or below c (compile-time indices, as above)
#pragma unroll
                for (int r = 1; r < P; ++r) beg_q = c >= pc[r] ? pc[r] : beg_q;
                const int i = c - beg_q;
                const unsigned e = fc[c];
                if (i < cap) pairs_out[(size_t)cap * s_ei[q] + i] = e;
                if (io.dbg_pairs && i < io.dbg_cap) {
                    int* out = io.dbg_pairs + 2 * ((long long)io.dbg_cap * s_ei[q] + i);
                    out[0] = dec_a(e); out[1] = dec_b(e);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) flags |= __shfl_xor_sync(0xffffffffu, flags, o);
#pragma unroll
            for (int q = 0; q < P; ++q)
                if (lane == q && s_ei[q] >= 0) {
                    const int n = pc[q + 1] - pc[q];
                    io.n_pairs[s_ei[q]] = n < cap ? n : cap;
                    if (n > cap && sc.ins_overflow) { sc.ins_overflow[s_ins[q]] = 1; flags |= kFlagOverflow; }
                    io.flags[s_ei[q]] = flags;
                }
        }
        __syncwarp();
    }
}

// ---- kernel 2: narrow phase of the regularized small instructions: one CTA per TILE of P problems ----
// A warp-per-problem kernel leaves lanes idle (about 29 candidates, 21 clip jobs and 49 sub-triangles per boxes.jl
// instruction on a 32-lane warp) and a warp runs its phases strictly one after another.  Here a CTA of 128 threads owns P
// consecutive (environment, instruction) problems and every phase is flattened over all of them:
//   1. 32 threads per problem fill the problem's shared context (transform, inverse, twist, constants), one element each;
//   2. the tile's candidate pairs (about 118 for P = 4 boxes.jl instructions) are dealt one per thread and taken up to their
//      start polygon, staged in the free upper half of the thread's own slot (start_polygon_zeta: about 3 of 10 pairs are
//      rejected there); a block scan packs the survivors, in candidate order, into the shared-memory PolyRec slots (stride 35
//      doubles: conflict-free); slot d is clipped IN PLACE by thread d, centroid -> a finished PolyRec.  The kernel has no
//      local-memory frame and no spills at 128 registers (tests/test_small_kernel_resources.py).  The clip -- the most divergent part
//      of the step -- so starts with all lanes of the leading warps busy, and a tile with more than 128 candidates (19 % of
//      the settled boxes.jl stacks) needs one clip / quadrature / summation round instead of two because its survivors fit
//      the 128 slots (164 -> 144 us on 4096 environments).  When the survivors of a round do not fit, the round after the
//      clip starts again at the first candidate left out (rare);
//   3. a block scan over the vertex counts turns the polygons into a dense (slot, edge) work list, dealt one sub-triangle
//      per thread for quadrature + friction; every item leaves its 6 sums (+ point count) in shared memory;
//   4. the items are ordered by problem, so a warp's 32 items belong to one to three problems: per problem a masked xor-butterfly
//      over the warp into the warp's running sums, added in warp order at the end of the tile: a fixed item -> lane assignment and
//      a fixed tree, bitwise reproducible, no atomics, no per-item results in shared memory, no barrier between the rounds.
// Measured and rejected: one WARP per tile (32 slots per warp, __syncwarp only, per-lane register accumulators flushed by a
// butterfly per problem) -- no barrier waits, but the sub-triangles of a 32-slot round split into per-problem segments that
// fill 6 of 10 lanes: 196 us against 146 us for this kernel.  Fetching the next tile's boundary data (x_r2_r1, twist, pair count)
// into registers one tile ahead: no change (145 us) -- the other three CTAs of the SM already cover that DRAM round trip.  Tiles of
// 8 problems on 256 threads (2 CTAs per SM): 152 us against 141 us -- a barrier then waits for the slowest of 256 clips.
// 3 CTAs per SM at 168 registers (no spills, 12 warps instead of 16): 151 us.  5 CTAs per SM (96 registers, 360 B of spills; possible
// since the per-item results left shared memory: 41 KB per CTA): 152 us against 135 us -- the kernel wants its 128 registers more than
// a fifth CTA.
constexpr int kPolyStride = 35;    // doubles per PolyRec slot
static_assert(sizeof(PolyRec<double>) == kPolyStride * sizeof(double), "PolyRec<double> is 35 doubles");

template <int P> struct TileSmem {   // P problems, P warps
    static constexpr int kThreads = 32 * P;
    double poly[kThreads * kPolyStride];   // PolyRec per thread
    PatchCtx<double> cx[P];
    long long ei[P];
    const double* fp[P];
    int ins[P];
    int n_cand[P];
    double wtot[P][P][8];   // [warp][problem]: running sums of the warp's items of the problem (6 sums + point count)
    int warp_tot[P];
    int pflags[P];
    unsigned short items[kThreads * 8];
    unsigned char poly_prob[kThreads];
    // pair code and start-polygon size per occupied slot, friction parameters per problem
    unsigned slot_pair[kThreads];
    unsigned char slot_n[kThreads];
    int resume_c;
    long long next_tile;    // drawn from the ticket counter by thread 0
    double fpv[P][8];
};
// 4 CTAs per SM (the launch's grid and the register budget assume it): 228 KB of shared memory per SM, 1 KB reserved per CTA
static_assert(sizeof(TileSmem<4>) <= 56 * 1024, "4 CTAs per SM need <= 56 KB each");

#define PFC_TILE_KERNEL narrow_tile_kernel
#define PFC_TILE_PARAMS false
#include "pfc_narrow_tile.cuh"
#undef PFC_TILE_KERNEL
#undef PFC_TILE_PARAMS
#define PFC_TILE_KERNEL narrow_tile_params_kernel
#define PFC_TILE_PARAMS true
#include "pfc_narrow_tile.cuh"
#undef PFC_TILE_KERNEL
#undef PFC_TILE_PARAMS

// One thread walks a given pair list in order and records every traction point (TractionCache).
__global__ void dump_traction_kernel(SceneDev sc, EvalIO io, long long env, int k, const int* pairs, long long n_pairs, double* out, int cap, int* n_points) {
    const InsDev& ins = sc.ins[k];
    const long long ei = env * sc.n_ins + k;
    PatchCtx<double> cx;
    load_xform(io.X + 16 * ei, cx.x21);
    cx.x12 = inverse(cx.x21);
    const double* tw = io.twist + 6 * ei;
    cx.w_ang = mk<double>(tw[0], tw[1], tw[2]);
    cx.w_lin = mk<double>(tw[3], tw[4], tw[5]);
    const InsParam* cp = io.params ? io.params + ei : nullptr;
    if (cp) { cx.chi = cp->chi; cx.Ebar1 = cp->Ebar1; cx.Ebar2 = cp->Ebar2; }
    else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
    cx.n_quad = ins.n_quad;
    Accum<double> acc;
    acc.fp = cp ? cp->p : ins.p; acc.w_ang = cx.w_ang; acc.w_lin = cx.w_lin; acc.dump = out; acc.dump_cap = cap;
    acc.reset(ACC_DUMP);
    int flags = 0;
    for (long long i = 0; i < n_pairs; ++i) integrate_pair(sc, ins, pairs[2 * i], pairs[2 * i + 1], cx, acc, flags);
    *n_points = acc.n_points;
}

}  // namespace

int persistent_blocks(const void* kern, int threads, size_t smem, cudaError_t* err) {
    int per_sm = 0, dev = 0, n_sm = 0;
    *err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (*err != cudaSuccess) return 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    *err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
    return n_sm * (per_sm > 0 ? per_sm : 1);
}

namespace {

template <int P, int NW, int MINB>
cudaError_t launch_broad_tile(const SceneDev& sc, const EvalIO& io, int cap, unsigned* pairs, cudaStream_t stream) {
    struct Tag {};
    auto kern = broad_tile_kernel<P, NW, MINB>;
    const int n_stage = sc.small_node_n <= kNodeTabMax ? sc.small_node_n : 0;
    const size_t smem = BroadTileLayout<P>::bytes(cap, NW, n_stage);
    int cached_blocks;
    {
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag>();
        if (sl.key0 != cap || sl.key1 != n_stage) {
            cudaError_t e;
            sl.blocks = persistent_blocks((const void*)kern, 32 * NW, smem, &e);
            if (e != cudaSuccess) return e;
            sl.key0 = cap; sl.key1 = n_stage;
        }
        cached_blocks = sl.blocks;
    }
    const long long n_tile = (io.n_env * sc.n_small + P - 1) / P;
    long long blocks = (n_tile + NW - 1) / NW;
    if (blocks > cached_blocks) blocks = cached_blocks;
    kern<<<(unsigned)blocks, 32 * NW, smem, stream>>>(sc, io, cap, n_stage, pairs);
    return cudaGetLastError();
}

// 4 problems per tile whatever the batch size: a tile of 4 is one environment's instructions, whose light (box on plane) and heavy
// (box on box) pair lists balance each other over the CTA's 128 threads.  Measured: 4096 environments 137 / 170 / 200 us for
// 4 / 2 / 1 problems per tile; 512 environments 30 / 48 / 52 us.
cudaError_t launch_narrow_tile(const SceneDev& sc, const EvalIO& io, int cap, const unsigned* pairs, cudaStream_t stream) {
    constexpr int P = 4;
    struct Tag {};
    const bool per_env = io.params != nullptr;
    auto kern = per_env ? narrow_tile_params_kernel<P, 4> : narrow_tile_kernel<P, 4>;   // 4 CTAs per SM
    const size_t smem = sizeof(TileSmem<P>);
    int cached_blocks;
    {
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag, 2>(per_env ? 1 : 0);
        if (sl.blocks == 0) {
            cudaError_t e;
            sl.blocks = persistent_blocks((const void*)kern, 32 * P, smem, &e);
            if (e != cudaSuccess) return e;
        }
        cached_blocks = sl.blocks;
    }
    long long blocks = (io.n_env * sc.n_small + P - 1) / P;
    if (blocks > cached_blocks) blocks = cached_blocks;
    kern<<<(unsigned)blocks, 32 * P, smem, stream>>>(sc, io, cap, pairs, const_cast<unsigned*>(pairs) + (size_t)cap * io.n_env * sc.n_ins);
    return cudaGetLastError();
}

// Broad phase of the small path.  Measured on B200 (4096 boxes.jl environments): 4 problems per warp, 8 warps per CTA, 2 CTAs per SM
// (124 registers) is the fastest; squeezing the SAT into 80-92 registers for more warps per SM costs more than the occupancy returns.
cudaError_t launch_broad(const SceneDev& sc, const EvalIO& io, int cap, unsigned* pairs, cudaStream_t stream) {
    // (4096 tiles on 2368 resident warps are 1.7 waves; finer tiles even the waves out but thin the lanes: 3 problems per warp 90 us,
    // 2 problems 102 us, 4 problems 85 us.)  Small batches: a warp's tile of 4 problems takes ~42 us whatever the load (level after level of
    // dependent phases), so when the problems do not fill the resident warps 4 at a time, smaller tiles shorten the critical path:
    // 512 environments 27.6 / 29.7 / 42.0 us for 1 / 2 / 4 problems per warp, 1024 environments 46.0 / 37.9 / 42.1 us.
    const long long n_prob = io.n_env * sc.n_small;
    int n_sm = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    int p = n_prob <= 16LL * n_sm ? 1 : (n_prob <= 32LL * n_sm ? 2 : 4);
    if (cap > 256) p = 1;   // slots of kMidCap entries (mid-size trees): the frontiers of one problem per warp are what fits in shared memory
    if (p == 1) return launch_broad_tile<1, 8, 2>(sc, io, cap, pairs, stream);
    if (p == 2) return launch_broad_tile<2, 8, 2>(sc, io, cap, pairs, stream);
    return launch_broad_tile<4, 8, 2>(sc, io, cap, pairs, stream);
}

}  // namespace

// max_pairs: the largest n_leaf1 * n_leaf2 over the small instructions (frontier capacity needed);
// pairs: scratch of n_env * n_ins * small_cap(max_pairs) words.
int small_cap(int max_pairs) { return ((max_pairs > 1 ? max_pairs : 1) + 31) / 32 * 32; }

cudaError_t launch_eval_small_f64(const SceneDev& sc, const EvalIO& io, int max_pairs, unsigned* pairs, cudaStream_t stream, int* n_launches,
                                  cudaEvent_t* ev, cudaEvent_t after_broad) {
    if (io.n_env * sc.n_small == 0) return cudaSuccess;
    const int cap = small_cap(max_pairs);
    if (ev) cudaEventRecord(ev[0], stream);
    cudaError_t e = launch_broad(sc, io, cap, pairs, stream);
    if (e != cudaSuccess) return e;
    if (ev) cudaEventRecord(ev[1], stream);
    if (after_broad) cudaEventRecord(after_broad, stream);   // the pair lists exist: what only needs them may start on another stream
    // regularized instructions: the tile kernel (4 problems per CTA, 4 CTAs per SM).  Bristle instructions are skipped here: they are
    // evaluated in the reference's operation order by pfc_exact.cu from the pair lists the broad kernel left
    e = launch_narrow_tile(sc, io, cap, pairs, stream);
    if (ev) cudaEventRecord(ev[2], stream);
    if (n_launches) *n_launches += 2;
    return e;
}

cudaError_t launch_broad_small_only(const SceneDev& sc, const EvalIO& io, int max_pairs, unsigned* pairs, cudaStream_t stream, int* n_launches) {
    if (io.n_env * sc.n_small == 0) return cudaSuccess;
    if (n_launches) *n_launches += 1;
    return launch_broad(sc, io, small_cap(max_pairs), pairs, stream);
}

cudaError_t launch_dump_traction(const SceneDev& sc, const EvalIO& io, long long env, int ins, const int* pairs, long long n_pairs, double* out,
                                 int cap_points, int* n_points, cudaStream_t stream) {
    dump_traction_kernel<<<1, 1, 0, stream>>>(sc, io, env, ins, pairs, n_pairs, out, cap_points, n_points);
    return cudaGetLastError();
}

}  // namespace pfc
