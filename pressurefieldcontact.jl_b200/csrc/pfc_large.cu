// pfc_large.cu -- contact-wrench evaluation for LARGE instructions (big trees, 1e5..1e6+ candidate
// pairs per evaluation; configs C4/C5).  Multi-kernel pipeline over global work lists:
//
//   K1a broad_bfs_kernel   a few level-synchronous expansions of the node-pair frontier until there
//                          are enough independent sub-problems (seeds) for the whole GPU
//   K1b broad_dfs_kernel   persistent warps pull seeds from a global queue and run a warp-cooperative,
//                          stack-based dual-tree traversal: the stack lives in shared memory, every
//                          lane tests one node pair per iteration (bit-exact 15-axis SAT), children are
//                          pushed with a warp prefix sum, leaf pairs are appended to the global pair
//                          list with ONE atomicAdd per warp per iteration (warp-aggregated atomics).
//                          Contact patches are small compared with the meshes, so a few seeds own nearly
//                          all of the work: a warp whose stack is deep while the queue runs dry DONATES
//                          the oldest half of its stack (the sub-trees nearest the root) back to the
//                          queue; idle warps keep polling until no seed is outstanding.
//   K1c key + radix sort   the pair list arrives in nondeterministic order; each pair gets the key of
//                          its position in the reference's recursion (src/obb/tree_types.jl:88-111):
//                          the root-to-leaf turns of both leaves interleaved, tree 2's turn first
//                          (children are visited (1.1,2.1),(1.2,2.1),(1.1,2.2),(1.2,2.2)).  A stable
//                          LSD radix sort on (problem, key) restores exactly the reference's order, so
//                          the pair lists are bit-exact and every later sum has a fixed order.
//   K2  narrow_large_kernel one thread per sorted pair of a regularized instruction (clip + quadrature +
//                          friction), fixed-order block reduction per 256-pair chunk of a problem's segment
//   K3  finish_large_kernel one warp per problem sums its chunk partials in order
//   Bristle instructions keep their sorted lists; pfc_exact.cu evaluates them in the reference's operation order.
//
// Reference: calcTriTetIntersections! + integrate_over! + yes_contact!/no_contact!
// (/root/reference/src/contact_algorithms_non_friction.jl:70-143, src/contact_algorithms_friction.jl:50-143).
#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include <cuda_pipeline_primitives.h>

#include "pfc_exact.h"
#include "pfc_large.h"
#include "pfc_patch.cuh"
#include "pfc_sat.cuh"

namespace pfc {

namespace {

#define LCU(call)                         \
    do {                                  \
        cudaError_t e_ = (call);          \
        if (e_ != cudaSuccess) return e_; \
    } while (0)

constexpr int kStackCap = 1024;   // node pairs per warp stack (8 KB)
constexpr int kDfsWarps = 4;
constexpr int kChunk = 256;       // pairs per reduction chunk (= narrow kernel block size)
constexpr int kNA = 6;            // accumulator slots per chunk partial (regularized wrench)
static_assert(kLargePartStride == kNA + 2, "partial record = kNA sums + point count + pair count");

constexpr int kMaxLevels = 132;   // breadth-first levels at most: two trees of depth <= 62 plus the roots (pfc_add_mesh rejects deeper trees)
struct Counters {                 // device-resident
    unsigned int frontier_max;    // largest frontier any breadth-first level asked for (sizes the buffers of a repeated evaluation)
    unsigned int epoch;           // evaluation counter (kept across evaluations): tags the seeds donated during one traversal
    unsigned int seed_head;       // next seed to hand out
    unsigned int n_pairs;         // leaf pairs appended
    unsigned int overflow;        // bit0 frontier, bit1 pairs, bit2 stack
    unsigned int n_units;         // narrow-phase work units
    unsigned int pad0[26];        // the polled queue words below get their own 128 B line (pollers must not slow the pair-list atomics)
    unsigned int q_head;          // seed queue: next seed to hand out
    unsigned int q_tail;          //             slots reserved (initial seeds + donations); a donated slot is readable once its tag is set
    unsigned int n_seed0;         //             seeds the breadth-first levels left (readable without a tag)
    int outstanding;              //             seeds queued or being traversed; 0 = traversal finished
    unsigned long long n_tests;   // node pairs tested (statistics)
    unsigned long long n_donated; // seeds donated (statistics)
    unsigned int level_n[kMaxLevels + 2];   // frontier size of every breadth-first level (level 0 = the root pairs)
};

// prob = index into the large-problem list; a, b mesh-local node ids; tag = traversal epoch for donated seeds (0 otherwise).
// Two 8-byte words: a donor stores (a, b), fences, then stores (prob, tag); a waiter polls (prob, tag).
struct __align__(16) Seed { int prob; unsigned tag; int a; int b; };
static_assert(offsetof(Counters, q_head) == 128, "queue words start a new 128 B line");

PFC_D void load_xform_l(const double* __restrict__ X, Xform<double>& x) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) x.r[3 * i + j] = X[4 * j + i];
        x.t[i] = X[12 + i];
    }
}
PFC_D void broad_xform_l(const double* __restrict__ X, double* Rab, double* tab) {
    Xform<double> x21;
    load_xform_l(X, x21);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) Rab[3 * i + j] = x21.r[3 * j + i];
        tab[i] = -add_(add_(mul_(x21.r[i], x21.t[0]), mul_(x21.r[3 + i], x21.t[1])), mul_(x21.r[6 + i], x21.t[2]));
    }
}

// problem p of the large list -> (env, instruction)
PFC_D void prob_to_ei(const SceneDev& sc, const LargeScene& ls, int p, long long& env, int& k) {
    env = p / ls.n_large;
    k = ls.large_ins[p - env * ls.n_large];
}

// Tests one node pair and classifies the outcome: returns the number of children (0, 2, 4) written to
// ch[], or -1 for a leaf pair (prims in ch[0]); 0 also when the boxes are disjoint.
// A 128 B node record as four 256-bit loads (sm_100: ld.global.v4.b64).  Every lane gathers its own two records, so each load
// instruction touches 32 different lines; fewer, wider requests are what the L1 data pipe is short of here.
// Axis-aligned internal nodes (most of what a traversal of big trees visits) need only the first 64 B: centre, extents, links, kind.
PFC_D void load_node(const NodeRec* __restrict__ p, NodeRec& out) {
    unsigned long long* o = reinterpret_cast<unsigned long long*>(&out);
#pragma unroll
    for (int j = 0; j < 2; ++j)
        asm volatile("ld.global.nc.v4.b64 {%0, %1, %2, %3}, [%4];"
                     : "=l"(o[4 * j]), "=l"(o[4 * j + 1]), "=l"(o[4 * j + 2]), "=l"(o[4 * j + 3])
                     : "l"(reinterpret_cast<const char*>(p) + 32 * j));
    if (out.kind != kNodeInternalAabb) {
#pragma unroll
        for (int j = 2; j < 4; ++j)
            asm volatile("ld.global.nc.v4.b64 {%0, %1, %2, %3}, [%4];"
                         : "=l"(o[4 * j]), "=l"(o[4 * j + 1]), "=l"(o[4 * j + 2]), "=l"(o[4 * j + 3])
                         : "l"(reinterpret_cast<const char*>(p) + 32 * j));
    }
}

// What a traversal thread needs to know about its problem, one 128 B record per (environment, large instruction), written once per
// evaluation by init_frontier_kernel: the transform of frame a into frame b as the SAT wants it, the two trees' offsets in the node
// array, whether the multi-GPU split applies.  A seed names its nodes by their GLOBAL index in the node array, so a thread can fetch
// both node records straight after its seed -- side by side with the problem record instead of behind three dependent look-ups
// (problem -> instruction -> node base / transform -> node).
struct __align__(16) ProbRec { double Rab[9]; double tab[3]; int base1, base2, split, pad_; double pad2_; };
static_assert(sizeof(ProbRec) == 128, "ProbRec is one 128 B line");

// ga, gb: global node indices; children / leaf primitives in ch[] (children as global indices, primitives as mesh-local ids)
PFC_D int expand_nodes(const NodeRec& a, const NodeRec& b, int base1, int base2, const double* Rab, const double* tab, int ga, int gb, int2* ch);
PFC_D int expand_pair(const NodeRec* __restrict__ nodes, int base1, int base2, const double* Rab, const double* tab, int ga, int gb, int2* ch) {
    NodeRec a, b;
    load_node(nodes + ga, a);
    load_node(nodes + gb, b);
    return expand_nodes(a, b, base1, base2, Rab, tab, ga, gb, ch);
}
PFC_D int expand_nodes(const NodeRec& a, const NodeRec& b, int base1, int base2, const double* Rab, const double* tab, int ga, int gb, int2* ch) {
    SatA A;
    sat_prepare_a(a, Rab, tab, A);
    if (!sat_test(A, b)) return 0;
    if (a.kind < 0) {
        if (b.kind < 0) { ch[0] = make_int2(a.right, b.right); return -1; }   // (a leaf's `right` is its primitive)
        ch[0] = make_int2(ga, gb + 1); ch[1] = make_int2(ga, base2 + b.right); return 2;
    }
    const int al = ga + 1, ar = base1 + a.right;   // pre-order: child 1 is the next record
    if (b.kind < 0) { ch[0] = make_int2(al, gb); ch[1] = make_int2(ar, gb); return 2; }
    const int bl = gb + 1, br = base2 + b.right;
    ch[0] = make_int2(al, bl); ch[1] = make_int2(ar, bl); ch[2] = make_int2(al, br); ch[3] = make_int2(ar, br);
    return 4;
}

__global__ void init_frontier_kernel(SceneDev sc, LargeScene ls, long long n_env, const double* __restrict__ X, Seed* frontier, ProbRec* ptab, Counters* cnt) {
    const long long n = n_env * ls.n_large;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        long long env; int k;
        prob_to_ei(sc, ls, (int)p, env, k);
        const InsDev& ins = sc.ins[k];
        ProbRec r;
        broad_xform_l(X + 16 * (env * sc.n_ins + k), r.Rab, r.tab);
        r.base1 = ins.node_base1; r.base2 = ins.node_base2; r.split = ins.model != PFC_MODEL_BRISTLE ? 1 : 0; r.pad_ = 0; r.pad2_ = 0.0;
        ptab[p] = r;
        frontier[p] = Seed{(int)p, 0u, ins.node_base1, ins.node_base2};   // the two roots
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        cnt->epoch += 1;   // (on the device, so that a captured CUDA graph of the evaluation can be replayed)
        cnt->frontier_max = (unsigned)n; cnt->seed_head = 0; cnt->n_pairs = 0; cnt->overflow = 0; cnt->n_units = 0;
        cnt->level_n[0] = (unsigned)n;
        for (int l = 1; l < kMaxLevels + 2; ++l) cnt->level_n[l] = 0;
        cnt->n_tests = 0; cnt->n_donated = 0; cnt->q_head = 0; cnt->q_tail = 0; cnt->n_seed0 = 0; cnt->outstanding = 0;
    }
}

// K1a: one level of breadth-first expansion (order is irrelevant here: the sort restores it)
// Multi-GPU split of one large scene: every rank runs the (cheap) breadth-first levels, then owns the seeds -- and the leaf pairs the
// breadth-first levels emit directly -- whose hash falls on it.  A sub-tree is traversed by exactly one rank, so the pair lists of the
// ranks are disjoint and their union is the full list; nothing is exchanged before the per-instruction partial sums.
// Bristle instructions are not split: their sums must run sequentially over the WHOLE TractionCache list (pfc_exact.cuh), so every rank
// lists and evaluates them completely (identical bits on every rank, nothing exchanged).
PFC_D bool prob_is_split(const SceneDev& sc, const LargeScene& ls, int prob) {
    return sc.ins[ls.large_ins[prob % ls.n_large]].model != PFC_MODEL_BRISTLE;
}
PFC_D unsigned item_hash(int prob, int a, int b) {
    unsigned h = (unsigned)prob * 0x9E3779B1u ^ (unsigned)a * 0x85EBCA77u ^ (unsigned)b * 0xC2B2AE3Du;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12;
    return h;
}

__global__ void __launch_bounds__(256, 2) broad_bfs_kernel(SceneDev sc, const ProbRec* __restrict__ ptab, const Seed* __restrict__ in, Seed* out,
                                                        int level, int split_level, unsigned cap_frontier, int3* pairs, unsigned cap_pairs, Counters* cnt,
                                                        unsigned hrank, unsigned hworld, unsigned per_warp_from) {
    const unsigned n_raw = cnt->level_n[level];
    const unsigned n = n_raw < cap_frontier ? n_raw : cap_frontier;   // (an overflowing level is cut short; the host repeats the evaluation)
    if (n == 0) return;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    // Multi-GPU split: up to split_level every rank expands the same frontier; AT split_level a rank keeps only the children (sub-trees)
    // whose hash falls on it; below, everything in its frontier is its own.  Leaf pairs found on the shared levels go to the rank their
    // own hash names.
    const bool shared = hworld > 1u && level <= split_level;
    // Space in the next frontier and in the pair list is reserved with ONE atomic per counter and reservation (the high-water mark the
    // first version also kept with an atomicMax is read off the level counters by the host): same-address atomics retire at ~2 ns each,
    // and a level's duration was three of them per warp.  Levels below per_warp_from entries reserve once per CTA and iteration (block
    // scan, two barriers: C4's levels of <= 1 M node pairs, 0.397 -> 0.384 ms); bigger levels once per warp without a barrier (C5's two
    // levels of 5 M node pairs: 373 / 364 -> ~300 us each; C5 1.45 -> 1.28 ms).  Measured thresholds 0 / 1 M / 3 M / never: C5 1.297 /
    // 1.277 / 1.289 / 1.453 ms, C4 0.397 / 0.384 / 0.385 / 0.385 ms.
    __shared__ unsigned warp_child[8], warp_leaf[8], base_child, base_leaf;
    unsigned long long tests = 0;
    const unsigned stride = gridDim.x * blockDim.x;
    const bool per_warp = n >= per_warp_from;
    for (unsigned base = blockIdx.x * blockDim.x; base < n; base += stride) {   // CTA-uniform trip count
        const unsigned i = base + threadIdx.x;
        int r = 0;
        int2 ch[4];
        Seed s{};
        bool split = false;
        if (i < n) {
            s = in[i];
            const ProbRec& pr = ptab[s.prob];
            r = expand_pair(sc.nodes, pr.base1, pr.base2, pr.Rab, pr.tab, s.a, s.b, ch);
            ++tests;
            split = shared && pr.split;
        }
        int n_child = r > 0 ? r : 0;
        if (split && level == split_level) {   // keep this rank's sub-trees only
            int kept = 0;
            for (int c = 0; c < n_child; ++c)
                if (item_hash(s.prob, ch[c].x, ch[c].y) % hworld == hrank) ch[kept++] = ch[c];
            n_child = kept;
        }
        const bool emit = r < 0 && (!split || item_hash(s.prob, ch[0].x, ch[0].y) % hworld == hrank);
        // scan of (children, leaf pairs): children in the low 16 bits of one word, leaves in the high 16
        unsigned incl = (unsigned)n_child | (emit ? 0x10000u : 0u);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        unsigned at, pat;
        if (per_warp) {   // (grid-uniform) one reservation per warp, no barrier
            const unsigned tot = __shfl_sync(0xffffffffu, incl, 31);
            unsigned bc = 0, bl = 0;
            if (lane == 31) {
                if (tot & 0xffffu) bc = atomicAdd(&cnt->level_n[level + 1], tot & 0xffffu);
                if (tot >> 16) bl = atomicAdd(&cnt->n_pairs, tot >> 16);
            }
            bc = __shfl_sync(0xffffffffu, bc, 31); bl = __shfl_sync(0xffffffffu, bl, 31);
            at = bc + (incl & 0xffffu) - (unsigned)n_child;
            pat = bl + (incl >> 16) - 1u;
        } else {
            if (lane == 31) { warp_child[wib] = incl & 0xffffu; warp_leaf[wib] = incl >> 16; }
            __syncthreads();
            unsigned before_c = 0, before_l = 0, tot_c = 0, tot_l = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) { const unsigned c = warp_child[w], l = warp_leaf[w]; if (w < wib) { before_c += c; before_l += l; } tot_c += c; tot_l += l; }
            if (threadIdx.x == 0) {
                base_child = tot_c ? atomicAdd(&cnt->level_n[level + 1], tot_c) : 0u;
                base_leaf = tot_l ? atomicAdd(&cnt->n_pairs, tot_l) : 0u;
            }
            __syncthreads();
            at = base_child + before_c + (incl & 0xffffu) - (unsigned)n_child;
            pat = base_leaf + before_l + (incl >> 16) - 1u;
        }
        if (at + n_child <= cap_frontier) { for (int c = 0; c < n_child; ++c) out[at + c] = Seed{s.prob, 0u, ch[c].x, ch[c].y}; }
        else if (n_child > 0) atomicOr(&cnt->overflow, 1u);
        if (emit) {
            if (pat < cap_pairs) pairs[pat] = make_int3(s.prob, ch[0].x, ch[0].y); else atomicOr(&cnt->overflow, 2u);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tests += __shfl_xor_sync(0xffffffffu, tests, o);
    if (lane == 0 && tests) atomicAdd(&cnt->n_tests, tests);
}

// the seeds the breadth-first levels left in frontier[src] become the initial content of the queue
__global__ void dfs_queue_init_kernel(Counters* cnt, int level, unsigned cap_frontier) {
    const unsigned n_raw = cnt->level_n[level];
    const unsigned n = n_raw < cap_frontier ? n_raw : cap_frontier;
    cnt->q_head = 0; cnt->q_tail = n; cnt->n_seed0 = n; cnt->outstanding = (int)n;
}

PFC_D unsigned ld_volatile_u32(const unsigned* p) { return *reinterpret_cast<const volatile unsigned*>(p); }

// K1b: warp-cooperative stack-based traversal of the seeds, with work donation
template <int MINB>
__global__ void __launch_bounds__(kDfsWarps * 32, MINB) broad_dfs_kernel(SceneDev sc, const ProbRec* __restrict__ ptab, Seed* seeds, unsigned cap_seeds,
                                                                   int3* pairs, unsigned cap_pairs, Counters* cnt, unsigned hrank,
                                                                   unsigned hworld) {
    __shared__ int2 stack_mem[kDfsWarps][kStackCap];   // per-warp circular stack: entry i lives at (base + i) & (kStackCap - 1)
    const unsigned epoch = cnt->epoch;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int2* stack = stack_mem[wib];
    const unsigned n_seed0 = cnt->n_seed0;
    unsigned long long tests = 0;
    unsigned donated = 0;
    for (;;) {
        // ---- acquire a seed: take a ticket; tickets below n_seed0 are the seeds of the breadth-first levels, later ones are
        // donated slots that become readable when their tag equals this traversal's epoch.  A waiter gives up when no seed is
        // outstanding: every reserved slot has then been traversed, so an abandoned ticket can never receive work.
        Seed seed;
        seed.prob = -1;
        if (lane == 0) {
            const unsigned ticket = atomicAdd(&cnt->q_head, 1u);
            if (ticket < n_seed0) {
                seed = seeds[ticket];
                if (hworld > 1u && ptab[seed.prob].split && item_hash(seed.prob, seed.a, seed.b) % hworld != hrank) {   // another rank's sub-tree
                    atomicSub(&cnt->outstanding, 1);
                    seed.prob = -2;
                }
            } else {
                unsigned backoff = 64, spins = 0;
                for (;;) {
                    if (ticket < cap_seeds) {
                        const unsigned long long w0 = *reinterpret_cast<const volatile unsigned long long*>(&seeds[ticket]);   // (prob, tag)
                        if ((unsigned)(w0 >> 32) == epoch) {
                            __threadfence();   // acquire: (a, b) were stored before the tag
                            const unsigned long long w1 = *(reinterpret_cast<const volatile unsigned long long*>(&seeds[ticket]) + 1);
                            seed.prob = (int)(unsigned)(w0 & 0xffffffffull); seed.a = (int)(unsigned)(w1 & 0xffffffffull); seed.b = (int)(unsigned)(w1 >> 32);
                            break;
                        }
                    }
                    if ((spins++ & 3u) == 0 && *reinterpret_cast<const volatile int*>(&cnt->outstanding) <= 0) break;
                    __nanosleep(backoff);
                    if (backoff < 2000) backoff *= 2;
                }
            }
        }
        seed.prob = __shfl_sync(0xffffffffu, seed.prob, 0);
        seed.a = __shfl_sync(0xffffffffu, seed.a, 0);
        seed.b = __shfl_sync(0xffffffffu, seed.b, 0);
        if (seed.prob == -2) continue;
        if (seed.prob < 0) break;
        double Rab[9], tab[3];
        int base1, base2;
        {
            const ProbRec& pr = ptab[seed.prob];
#pragma unroll
            for (int i = 0; i < 9; ++i) Rab[i] = pr.Rab[i];
#pragma unroll
            for (int i = 0; i < 3; ++i) tab[i] = pr.tab[i];
            base1 = pr.base1; base2 = pr.base2;
        }
        int n = 1;
        unsigned base = 0;
        if (lane == 0) stack[0] = make_int2(seed.a, seed.b);
        __syncwarp();
        while (n > 0) {
            // idle warps = tickets issued beyond the reserved slots; loaded early, consumed after the tests (the latency hides behind the SAT)
            unsigned qh = 0, qt = 0;
            const bool may_donate = n >= 32;
            if (may_donate && lane == 0) { qh = ld_volatile_u32(&cnt->q_head); qt = ld_volatile_u32(&cnt->q_tail); }
            // pop as many entries as the stack can absorb children for (each pops 1, pushes <= 4)
            int take = n < 32 ? n : 32;
            const int room = (kStackCap - n) / 3;
            if (take > room) take = room > 0 ? room : 1;
            int r = 0;
            int2 ch[4];
            if (lane < take) {
                const int2 e = stack[(base + n - 1 - lane) & (kStackCap - 1)];
                r = expand_pair(sc.nodes, base1, base2, Rab, tab, e.x, e.y, ch);
                ++tests;
            }
            __syncwarp();
            n -= take;
            const int n_child = r > 0 ? r : 0;
            int incl = n_child;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            const int tot = __shfl_sync(0xffffffffu, incl, 31);
            const int at = n + incl - n_child;
            if (n + tot <= kStackCap) { for (int c = 0; c < n_child; ++c) stack[(base + at + c) & (kStackCap - 1)] = ch[c]; }
            else if (lane == 0) atomicOr(&cnt->overflow, 4u);  // cannot happen: take was limited by room
            n = (n + tot <= kStackCap) ? n + tot : n;
            const unsigned leaf_mask = __ballot_sync(0xffffffffu, r < 0);
            if (leaf_mask) {
                unsigned pat = 0;
                if (lane == 0) pat = atomicAdd(&cnt->n_pairs, (unsigned)__popc(leaf_mask));
                pat = __shfl_sync(0xffffffffu, pat, 0) + __popc(leaf_mask & ((1u << lane) - 1u));
                if (r < 0) { if (pat < cap_pairs) pairs[pat] = make_int3(seed.prob, ch[0].x, ch[0].y); else atomicOr(&cnt->overflow, 2u); }
            }
            __syncwarp();
            // ---- donation: warps are waiting for work and this stack is deep -> hand over its oldest entries (the sub-trees
            // nearest the root), at most half of the stack and about two per waiting warp
            int give = 0;
            if (may_donate && lane == 0 && n >= 32) {
                const int waiting = (int)(qh - qt);
                if (waiting > 0) { give = n / 2; if (give > 2 * waiting) give = 2 * waiting; if (give > 256) give = 256; }
            }
            give = __shfl_sync(0xffffffffu, give, 0);
            if (give > 0) {
                unsigned q0 = 0;
                if (lane == 0) { atomicAdd(&cnt->outstanding, give); q0 = atomicAdd(&cnt->q_tail, (unsigned)give); }
                q0 = __shfl_sync(0xffffffffu, q0, 0);
                const bool fits = q0 + (unsigned)give <= cap_seeds;
                if (fits) {
                    for (int j = lane; j < give; j += 32) {
                        const int2 e = stack[(base + j) & (kStackCap - 1)];
                        *reinterpret_cast<int2*>(&seeds[q0 + j].a) = e;
                    }
                    __threadfence();
                    for (int j = lane; j < give; j += 32)
                        *reinterpret_cast<volatile unsigned long long*>(&seeds[q0 + j]) = ((unsigned long long)epoch << 32) | (unsigned)seed.prob;
                } else if (lane == 0) {
                    atomicOr(&cnt->overflow, 1u);            // the host grows the queue and re-runs the traversal;
                    atomicSub(&cnt->outstanding, give);      // these seeds are dropped so that this run still terminates
                }
                base = (base + give) & (kStackCap - 1);
                n -= give;
                donated += give;
                __syncwarp();
            }
        }
        if (lane == 0) { __threadfence(); atomicSub(&cnt->outstanding, 1); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tests += __shfl_xor_sync(0xffffffffu, tests, o);
    if (lane == 0 && tests) atomicAdd(&cnt->n_tests, tests);
    if (lane == 0 && donated) atomicAdd(&cnt->n_donated, (unsigned long long)donated);
}

// K1c: DFS-order key of every pair.  key = (prob << key_bits) | interleaved path bits (left-aligned in key_bits)
// the number of pairs the traversal left (never more than the buffers hold: an overflowing evaluation is repeated by the host)
PFC_D unsigned listed_pairs(const Counters* cnt, unsigned cap_pairs) { const unsigned n = cnt->n_pairs; return n < cap_pairs ? n : cap_pairs; }

__global__ void build_keys_kernel(SceneDev sc, LargeScene ls, const int3* __restrict__ pairs, const Counters* cnt, unsigned cap_pairs, unsigned long long* keys,
                                  unsigned* vals) {
    const unsigned n = listed_pairs(cnt, cap_pairs);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int3 p = pairs[i];
        long long env; int k;
        prob_to_ei(sc, ls, p.x, env, k);
        const InsDev& ins = sc.ins[k];
        const unsigned long long pa = ls.leaf_path[ins.path_base1 + p.y], pb = ls.leaf_path[ins.path_base2 + p.z];
        const int da = ls.leaf_depth[ins.path_base1 + p.y], db = ls.leaf_depth[ins.path_base2 + p.z];
        unsigned long long key = 0;
        int nb = 0;
        const int dm = da > db ? da : db;
        for (int l = 0; l < dm; ++l) {
            if (l < db) { key = (key << 1) | ((pb >> (db - 1 - l)) & 1ull); ++nb; }
            if (l < da) { key = (key << 1) | ((pa >> (da - 1 - l)) & 1ull); ++nb; }
        }
        key <<= (ls.key_bits - nb);  // left-align: keys of different lengths compare like the recursion order
        keys[i] = (ls.key_bits < 64 ? ((unsigned long long)(unsigned)p.x << ls.key_bits) : 0ull) | key;   // (64 key bits leave room for one problem only)
        vals[i] = i;
    }
}

// ---- stable LSD radix sort, 8 bits per pass, one warp per 512-element tile ---------------------------------------
// Per pass: (1) per-tile digit histograms, digit-major; (2) one block per digit scans its row of tile counts (exclusive) and
// leaves the digit total; (3) every tile turns the 256 digit totals into digit bases with a warp scan, adds its row offsets and
// scatters its keys in order (ranks inside a 32-key chunk from __match_any_sync), so the sort is stable.
constexpr int kTile = 512;
// (n comes from the device counter, so the whole evaluation is queued without a host round trip: grids are sized for the buffers'
// capacity -- cap_tiles tiles -- and the tiles beyond the list return at once; lists of at most kSmallSort pairs go to small_sort_kernel)
constexpr unsigned kSmallSort = 2048;   // beyond a few thousand keys the radix passes win (measured: 6 695 keys, 421 vs 363 us per evaluation)
__global__ void __launch_bounds__(128) radix_hist_kernel(const unsigned long long* __restrict__ keys, const Counters* cnt, unsigned cap_pairs, int shift, unsigned* hist,
                                                         unsigned cap_tiles) {
    __shared__ unsigned h[4][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned n = listed_pairs(cnt, cap_pairs);
    if (n <= kSmallSort) return;
    const unsigned n_tiles = (n + kTile - 1) / kTile;
    const unsigned tile = blockIdx.x * 4 + wib;
    for (int d = lane; d < 256; d += 32) h[wib][d] = 0;
    __syncwarp();
    if (tile < n_tiles) {
        const unsigned beg = tile * kTile, end = min(beg + kTile, n);
        unsigned long long k[kTile / 32];
#pragma unroll
        for (int j = 0; j < kTile / 32; ++j) { const unsigned i = beg + 32 * j + lane; k[j] = i < end ? keys[i] : 0ull; }   // all loads in flight at once
#pragma unroll
        for (int j = 0; j < kTile / 32; ++j) if (beg + 32 * j + lane < end) atomicAdd(&h[wib][(k[j] >> shift) & 255u], 1u);
        __syncwarp();
        for (int d = lane; d < 256; d += 32) hist[(size_t)d * cap_tiles + tile] = h[wib][d];  // digit-major for the row scans
    }
}
// block d: exclusive scan of row d (n_tiles counts) in place, row total -> tot[d]
__global__ void __launch_bounds__(256) radix_rowscan_kernel(unsigned* hist, const Counters* cnt, unsigned cap_pairs, unsigned cap_tiles, unsigned* tot) {
    __shared__ unsigned warp_sums[8];
    const unsigned n = listed_pairs(cnt, cap_pairs);
    if (n <= kSmallSort) return;
    const unsigned n_tiles = (n + kTile - 1) / kTile;
    unsigned* row = hist + (size_t)blockIdx.x * cap_tiles;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned carry = 0;
    constexpr int IT = 8;   // consecutive counts per thread
    for (unsigned base = 0; base < n_tiles; base += 256 * IT) {
        unsigned v[IT], s = 0;
#pragma unroll
        for (int j = 0; j < IT; ++j) { const unsigned i = base + threadIdx.x * IT + j; v[j] = i < n_tiles ? row[i] : 0u; s += v[j]; }
        unsigned incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) warp_sums[w] = incl;
        __syncthreads();
        unsigned before = carry + incl - s, total = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const unsigned t = warp_sums[k]; if (k < w) before += t; total += t; }
#pragma unroll
        for (int j = 0; j < IT; ++j) { const unsigned i = base + threadIdx.x * IT + j; if (i < n_tiles) row[i] = before; before += v[j]; }
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) tot[blockIdx.x] = carry;
}
__global__ void __launch_bounds__(128) radix_scatter_kernel(const unsigned long long* __restrict__ keys_in, const unsigned* __restrict__ vals_in, const Counters* cnt,
                                                            unsigned cap_pairs, int shift, const unsigned* __restrict__ hist, const unsigned* __restrict__ tot,
                                                            unsigned cap_tiles, unsigned long long* keys_out, unsigned* vals_out) {
    __shared__ unsigned base[4][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned n = listed_pairs(cnt, cap_pairs);
    if (n <= kSmallSort) return;
    const unsigned n_tiles = (n + kTile - 1) / kTile;
    const unsigned tile = blockIdx.x * 4 + wib;
    if (tile >= n_tiles) return;
    {   // digit bases: exclusive prefix of the 256 digit totals (lane l owns digits 8 l .. 8 l + 7) + this tile's row offsets
        unsigned t[8], s = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { t[j] = tot[8 * lane + j]; s += t[j]; }
        unsigned incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        unsigned run = incl - s;
#pragma unroll
        for (int j = 0; j < 8; ++j) { base[wib][8 * lane + j] = run + hist[(size_t)(8 * lane + j) * cap_tiles + tile]; run += t[j]; }
    }
    __syncwarp();
    const unsigned beg = tile * kTile, end = min(beg + kTile, n);
    constexpr int B = 8;   // chunks whose keys are loaded together (the global-load latency is paid once per batch)
    for (unsigned c0 = beg; c0 < end; c0 += 32 * B) {
        unsigned long long kk[B]; unsigned vv[B];
#pragma unroll
        for (int j = 0; j < B; ++j) { const unsigned i = c0 + 32 * j + lane; const bool ok = i < end; kk[j] = ok ? keys_in[i] : 0ull; vv[j] = ok ? vals_in[i] : 0u; }
#pragma unroll
        for (int j = 0; j < B; ++j) {   // chunks in order, lanes in order => stable
            const unsigned i = c0 + 32 * j + lane;
            const bool valid = i < end;
            const unsigned d = valid ? (unsigned)((kk[j] >> shift) & 255u) : 256u + lane;  // invalid lanes get unique digits
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            const unsigned rank = __popc(peers & ((1u << lane) - 1u));
            unsigned pos = 0;
            if (valid) pos = base[wib][d] + rank;
            __syncwarp();
            if (valid && rank == (unsigned)__popc(peers) - 1) base[wib][d] = pos + 1;  // the last peer advances the digit's cursor
            __syncwarp();
            if (valid) { keys_out[pos] = kk[j]; vals_out[pos] = vv[j]; }
        }
    }
}

// Short lists (a single small scene): one CTA sorts (key, value) in shared memory with a bitonic network instead of 5 x 3 launches of
// the radix passes.  Keys are distinct (a key encodes both root-to-leaf paths), so stability is not needed.
// (may run in place: everything is read into shared memory before anything is written)
// radix_queued = 0: the host left the radix passes out (the previous evaluation's list was short); a list that turns out longer raises
// overflow bit 8 and the host repeats the evaluation with the passes queued.
__global__ void __launch_bounds__(1024) small_sort_kernel(const unsigned long long* keys_in, const unsigned* vals_in, Counters* cnt, unsigned cap_pairs,
                                                          unsigned long long* keys_out, unsigned* vals_out, int radix_queued) {
    extern __shared__ __align__(16) unsigned char sort_smem[];
    const unsigned n = listed_pairs(cnt, cap_pairs);
    if (n > kSmallSort && !radix_queued && threadIdx.x == 0) atomicOr(&cnt->overflow, 8u);
    if (n == 0 || n > kSmallSort) return;
    unsigned m = 1;
    while (m < n) m <<= 1;
    unsigned long long* k = reinterpret_cast<unsigned long long*>(sort_smem);
    unsigned* v = reinterpret_cast<unsigned*>(k + m);
    for (unsigned i = threadIdx.x; i < m; i += blockDim.x) { k[i] = i < n ? keys_in[i] : ~0ull; v[i] = i < n ? vals_in[i] : 0u; }
    __syncthreads();
    for (unsigned size = 2; size <= m; size <<= 1)
        for (unsigned stride = size >> 1; stride > 0; stride >>= 1) {
            for (unsigned t = threadIdx.x; t < m / 2; t += blockDim.x) {
                const unsigned lo = 2 * t - (t & (stride - 1)), hi = lo + stride;   // the t-th compare-exchange of this step
                const bool up = (lo & size) == 0;
                const unsigned long long a = k[lo], b = k[hi];
                if ((a > b) == up) { k[lo] = b; k[hi] = a; const unsigned tv = v[lo]; v[lo] = v[hi]; v[hi] = tv; }
            }
            __syncthreads();
        }
    for (unsigned i = threadIdx.x; i < n; i += blockDim.x) { keys_out[i] = k[i]; vals_out[i] = v[i]; }
}

// sorted order -> (prob, a, b) arrays + per-problem segments
__global__ void gather_sorted_kernel(const int3* __restrict__ pairs, const unsigned* __restrict__ vals, const Counters* cnt, unsigned cap_pairs, int3* sorted,
                                     unsigned* seg_start, unsigned* seg_end) {
    const unsigned n = listed_pairs(cnt, cap_pairs);
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int3 p = pairs[vals[i]];
        sorted[i] = p;
        const int prev = i > 0 ? pairs[vals[i - 1]].x : -1;
        if (p.x != prev) { seg_start[p.x] = i; if (prev >= 0) seg_end[prev] = i; }
        if (i == n - 1) seg_end[p.x] = n;
    }
}
// unit_start[p] = sum_{q < p} ceil(len_q / kChunk); one block (problem counts on the large path are modest)
__global__ void __launch_bounds__(1024) units_scan_kernel(const unsigned* __restrict__ seg_start, const unsigned* __restrict__ seg_end, unsigned n_prob, unsigned* unit_start,
                                                          Counters* cnt, unsigned shard_rank, unsigned shard_world) {
    __shared__ unsigned warp_sums[32];
    __shared__ unsigned carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (unsigned base = 0; base < n_prob; base += 1024) {
        const unsigned i = base + threadIdx.x;
        const unsigned v = i < n_prob ? (seg_end[i] - seg_start[i] + kChunk - 1) / kChunk : 0;
        unsigned incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) warp_sums[w] = incl;
        __syncthreads();
        if (w == 0) {
            unsigned s = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += t; }
            warp_sums[lane] = s;
        }
        __syncthreads();
        const unsigned before = carry + (w > 0 ? warp_sums[w - 1] : 0) + incl - v;
        if (i < n_prob) unit_start[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) { unit_start[n_prob] = carry; cnt->n_units = carry; }
    (void)shard_rank; (void)shard_world;
}

// K2: narrow phase of the REGULARIZED instructions, one CTA per unit of 256 sorted pairs of one problem, in the phases of the small path's
// tile kernel (pfc_small.cu) so that the divergent clip and the dense quadrature each get full warps:
//   1. one candidate pair per thread up to its start polygon in registers (exact rejection);
//   2. block scan: the survivors are packed, in pair order, into shared-memory polygon slots; slot d is clipped in place by thread d;
//   3. block scan of the vertex counts -> dense (slot, edge) list, one sub-triangle per thread (quadrature, pressure law, friction);
//   4. the unit's 6 sums + point count in item order by one warp (lane-strided partials + xor-butterfly: bitwise reproducible).
// (Bristle instructions keep their sorted pair lists and are evaluated by the reference-order pipeline, pfc_exact.cu.)
// The first version ran one thread per pair through clip + all sub-triangles: 12.7 of 32 lanes busy, 389 us for the 0.9 M pairs of C5.
constexpr int kLPolyStride = 35;
static_assert(sizeof(PolyRec<double>) == kLPolyStride * sizeof(double), "PolyRec<double> is 35 doubles");
struct NarrowLargeSmem {
    double poly[kChunk * kLPolyStride];
    double item_res[kChunk * 7];
    PatchCtx<double> cx;
    double fpv[8];
    double tot[8];
    unsigned short items[kChunk * 8];
    int2 slot_pair[kChunk];
    unsigned char slot_n[kChunk];
    int warp_tot[kChunk / 32];
    int s_prob;
    int pflags;
};

__global__ void __launch_bounds__(kChunk, 2) narrow_large_kernel(SceneDev sc, LargeScene ls, EvalIO io, const int3* __restrict__ sorted, const unsigned* __restrict__ seg_start,
                                                                 const unsigned* __restrict__ seg_end, const unsigned* __restrict__ unit_start, unsigned n_prob,
                                                                 const Counters* cnt, double* chunk_out, int* chunk_points, int* prob_flags) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    NarrowLargeSmem& sm = *reinterpret_cast<NarrowLargeSmem*>(smem_raw);
    const unsigned n_units = cnt->n_units;
    const int tid = threadIdx.x, lane = tid & 31, wib = tid >> 5;
    constexpr int NW = kChunk / 32;
    for (unsigned u = blockIdx.x; u < n_units; u += gridDim.x) {
        if (tid == 0) {  // unit -> problem by binary search in unit_start
            unsigned lo = 0, hi = n_prob;
            while (hi - lo > 1) { const unsigned mid = (lo + hi) >> 1; if (unit_start[mid] <= u) lo = mid; else hi = mid; }
            sm.s_prob = (int)lo;
            sm.pflags = 0;
        }
        __syncthreads();
        const int p = sm.s_prob;
        long long env; int k;
        prob_to_ei(sc, ls, p, env, k);
        const InsDev& ins = sc.ins[k];
        if (ins.model != PFC_MODEL_REGULARIZED) { __syncthreads(); continue; }   // (block-uniform)
        const long long ei = env * sc.n_ins + k;
        // ---- context: one element per lane of warp 0
        if (wib == 0) {
            const double* X = io.X + 16 * ei;
            const double* twist = io.twist + 6 * ei;
            PatchCtx<double>& cx = sm.cx;
            const InsParam* cp = io.params ? io.params + ei : nullptr;   // this environment's contact parameters, if it has its own
            if (lane < 8) sm.fpv[lane] = cp ? cp->p[lane] : ins.p[lane];
            if (lane < 9) { const int i = lane / 3, j = lane % 3; cx.x21.r[lane] = X[4 * j + i]; }
            else if (lane < 12) cx.x21.t[lane - 9] = X[12 + lane - 9];
            else if (lane < 21) { const int e = lane - 12, i = e / 3, j = e % 3; cx.x12.r[e] = X[4 * i + j]; }
            else if (lane < 24) { const int i = lane - 21; cx.x12.t[i] = -(X[4 * i] * X[12] + X[4 * i + 1] * X[13] + X[4 * i + 2] * X[14]); }
            else if (lane < 27) (&cx.w_ang.x)[lane - 24] = twist[lane - 24];
            else if (lane < 30) (&cx.w_lin.x)[lane - 27] = twist[lane - 24];
            else if (lane == 30) {
                if (cp) { cx.chi = cp->chi; cx.Ebar1 = cp->Ebar1; cx.Ebar2 = cp->Ebar2; }
                else { cx.chi = ins.chi; cx.Ebar1 = ins.Ebar1; cx.Ebar2 = ins.Ebar2; }
                cx.n_quad = ins.n_quad;
            }
            if (lane < 8) sm.tot[lane] = 0.0;
        }
        __syncthreads();
        // ---- 1. start polygons, staged in doubles [16, 32) of slot tid (the compaction below writes doubles [0, 16) of a slot only)
        const unsigned i = seg_start[p] + (u - unit_start[p]) * kChunk + tid;
        double* zr = sm.poly + tid * kLPolyStride + 16;
        int n0 = 0;
        int3 pr = make_int3(0, 0, 0);
        if (i < seg_end[p]) {
            pr = sorted[i];
            n0 = start_polygon_zeta(sc, ins, pr.y, pr.z, sm.cx, zr);
        }
        // ---- 2. survivors -> slots in pair order; clip in place
        const unsigned alive = __ballot_sync(0xffffffffu, n0 > 0);
        if (lane == 0) sm.warp_tot[wib] = __popc(alive);
        __syncthreads();
        int before = 0, n_slot = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { const int t = sm.warp_tot[w]; if (w < wib) before += t; n_slot += t; }
        if (n0 > 0) {
            const int slot = before + __popc(alive & ((1u << lane) - 1u));
            double* z = sm.poly + slot * kLPolyStride;
#pragma unroll
            for (int j = 0; j < 16; ++j)
                if (j < 4 * n0) z[j] = zr[j];
            sm.slot_pair[slot] = make_int2(pr.y, pr.z); sm.slot_n[slot] = (unsigned char)n0;
        }
        __syncthreads();
        int nv = 0;
        if (tid < n_slot) {
            const int2 e = sm.slot_pair[tid];
            PolyRec<double>& out = *reinterpret_cast<PolyRec<double>*>(sm.poly + tid * kLPolyStride);
            int flags = 0;
            const int n = clip_tet_inplace(reinterpret_cast<double*>(&out), (int)sm.slot_n[tid], flags);
            if (n >= 3) {
                finish_polygon_slot(n, sc.tets[ins.prim_base2 + e.y], pair_normal(sc, ins, e.x, e.y, sm.cx), out);
                nv = n;
            }
            if (flags) atomicOr(&sm.pflags, flags);
        }
        // ---- 3. (slot, edge) items
        int incl = nv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        __syncthreads();   // warp_tot of step 2 has been read
        if (lane == 31) sm.warp_tot[wib] = incl;
        __syncthreads();
        int ibefore = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { const int t = sm.warp_tot[w]; if (w < wib) ibefore += t; total += t; }
        const int at = ibefore + incl - nv;
        for (int q = 0; q < nv; ++q) sm.items[at + q] = (unsigned short)((tid << 3) | q);
        __syncthreads();
        for (int i0 = 0; i0 < total; i0 += kChunk) {
            const int i1 = min(total, i0 + kChunk);
            const int it = i0 + tid;
            if (it < i1) {
                const int code = sm.items[it];
                const int slot = code >> 3, q = code & 7;
                const PolyRec<double>& prc = *reinterpret_cast<const PolyRec<double>*>(sm.poly + slot * kLPolyStride);
                Accum<double, 6> tmp;
                tmp.fp = sm.fpv; tmp.w_ang = sm.cx.w_ang; tmp.w_lin = sm.cx.w_lin; tmp.dump = nullptr; tmp.dump_cap = 0;
                tmp.reset(ACC_REGULARIZED);
                const int qp = (q == 0) ? prc.n - 1 : q - 1;
                integrate_subtri(prc.v[qp], prc.v[q], prc.cen, prc.nrm, prc.eps_r, sm.cx, tmp);
                double* res = sm.item_res + tid * 7;
#pragma unroll
                for (int j = 0; j < 6; ++j) res[j] = tmp.a[j];
                reinterpret_cast<int*>(res + 6)[0] = tmp.n_points;
            }
            __syncthreads();
            // ---- 4. the round's items in order: lane l adds items l, l + 32, ..., then a xor-butterfly
            if (wib == 0) {
                double part[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
                int part_n = 0;
                for (int j = lane; j < i1 - i0; j += 32) {
                    const double* res = sm.item_res + j * 7;
#pragma unroll
                    for (int c = 0; c < 6; ++c) part[c] += res[c];
                    part_n += reinterpret_cast<const int*>(res + 6)[0];
                }
                int pn = part_n;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) pn += __shfl_xor_sync(0xffffffffu, pn, o);
                double mine = (double)pn;
#pragma unroll
                for (int c = 0; c < 6; ++c) { const double t = warp_sum(part[c]); mine = (lane == c) ? t : mine; }
                if (lane < 7) sm.tot[lane] += mine;
            }
            __syncthreads();
        }
        if (tid < kNA) chunk_out[(size_t)u * kNA + tid] = sm.tot[tid];
        if (tid == 0) { chunk_points[u] = (int)sm.tot[6]; if (sm.pflags) atomicOr(&prob_flags[p], sm.pflags); }
        __syncthreads();
    }
}

// K3: one warp per problem: ordered sum of its chunk partials -> wrench, pair count, flags.
// In sharded (multi-GPU) mode the chunk sums of the other ranks are missing: `part_out` makes the kernel write the raw per-problem
// partial sums (6 sums, point count, pair count) for the caller's reduction over the ranks instead; `apply_parts` finishes from the
// reduced buffer.  Bristle instructions only get their pair count published here (exact_bristle: pfc_exact.cu evaluates them).
__global__ void __launch_bounds__(128) finish_large_kernel(SceneDev sc, LargeScene ls, EvalIO io, const unsigned* __restrict__ seg_start, const unsigned* __restrict__ seg_end,
                                                           const unsigned* __restrict__ unit_start, unsigned n_prob, const double* __restrict__ chunk_out,
                                                           const int* __restrict__ chunk_points, const int* __restrict__ prob_flags, double* part_out, int apply_parts) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    for (unsigned p = blockIdx.x * 4 + wib; p < n_prob; p += gridDim.x * 4) {
        long long env; int k;
        prob_to_ei(sc, ls, (int)p, env, k);
        const InsDev& ins = sc.ins[k];
        const long long ei = env * sc.n_ins + k;
        if (ins.model == PFC_MODEL_BRISTLE) {   // never split over ranks: the list is complete here
            if (lane == 0 && !apply_parts) { io.n_pairs[ei] = (long long)seg_end[p] - (long long)seg_start[p]; io.flags[ei] = prob_flags[p]; }
            if (lane == 0 && part_out && !apply_parts) for (int j = 0; j < kLargePartStride; ++j) part_out[(size_t)p * kLargePartStride + j] = 0.0;
            continue;
        }
        double sum[kNA];
        int pts = 0;
        if (apply_parts) {  // sums were reduced across ranks by the caller
            for (int j = 0; j < kNA; ++j) sum[j] = part_out[(size_t)p * kLargePartStride + j];
            pts = (int)part_out[(size_t)p * kLargePartStride + kNA];
        } else {
            // lane l sums chunks l, l+32, ... of this problem in order; then a fixed butterfly
            const unsigned c0 = unit_start[p], c1 = unit_start[p + 1];
            for (int j = 0; j < kNA; ++j) sum[j] = 0.0;
            for (unsigned c = c0 + lane; c < c1; c += 32) {
                for (int j = 0; j < kNA; ++j) sum[j] += chunk_out[(size_t)c * kNA + j];
                pts += chunk_points[c];
            }
            for (int j = 0; j < kNA; ++j) sum[j] = warp_sum(sum[j]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) pts += __shfl_xor_sync(0xffffffffu, pts, o);
            if (part_out) {  // sharded: hand the partial sums to the caller and stop here
                if (lane == 0) {
                    for (int j = 0; j < kNA; ++j) part_out[(size_t)p * kLargePartStride + j] = sum[j];
                    part_out[(size_t)p * kLargePartStride + kNA] = (double)pts;
                    part_out[(size_t)p * kLargePartStride + kNA + 1] = (double)(seg_end[p] - seg_start[p]);
                }
                continue;
            }
        }
        // sharded: the ranks hold disjoint parts of the pair list; the count travels with the partial sums
        const long long n_pairs = apply_parts ? (long long)part_out[(size_t)p * kLargePartStride + kNA + 1] : (long long)seg_end[p] - (long long)seg_start[p];
        if (lane == 0) {
            const bool contact = pts > 0;
            double* wo = io.wrench + 6 * ei;
            for (int j = 0; j < 6; ++j) wo[j] = contact ? sum[j] : 0.0;
            io.n_pairs[ei] = n_pairs;
            io.flags[ei] = prob_flags[p] | (contact ? kFlagContact : 0);
        }
    }
}

__global__ void zero_int_kernel(int* p, unsigned n) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = 0;
}
__global__ void init_segments_kernel(unsigned* seg_start, unsigned* seg_end, unsigned n) {
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { seg_start[i] = 0; seg_end[i] = 0; }
}

template <class T> cudaError_t ensure(T*& p, size_t& cap, size_t need) {
    if (need <= cap) return cudaSuccess;
    alloc_generation()++;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, need * sizeof(T));
    if (e != cudaSuccess) return e;
    cap = need;
    return cudaMemset(p, 0, need * sizeof(T));   // seed tags of a fresh queue must not match any epoch
}

}  // namespace

struct LargeBuffers {
    Counters* cnt = nullptr;
    Seed* frontier[2] = {nullptr, nullptr}; size_t cap_frontier = 0;
    int3* pairs = nullptr; int3* sorted = nullptr; size_t cap_pairs = 0;
    unsigned long long* keys[2] = {nullptr, nullptr}; unsigned* vals[2] = {nullptr, nullptr}; size_t cap_keys = 0, cap_keys2 = 0, cap_vals = 0, cap_vals2 = 0, cap_sorted = 0;
    unsigned* hist = nullptr; size_t cap_hist = 0;
    unsigned* seg_start = nullptr; unsigned* seg_end = nullptr; unsigned* unit_start = nullptr; size_t cap_seg = 0, cap_seg2 = 0, cap_unit = 0;
    int* prob_flags = nullptr; size_t cap_pf = 0;
    ProbRec* ptab = nullptr; size_t cap_ptab = 0;
    double* chunk_out = nullptr; size_t cap_chunk = 0;
    int* chunk_points = nullptr; size_t cap_cp = 0;
    double* part = nullptr; size_t cap_part = 0;
    size_t cf2 = 0;
    Counters* h_cnt = nullptr;          // pinned copy of the counters of the last traversal
    bool check_pending = false;         // a traversal has been queued whose counters have not been looked at yet
    size_t want_frontier = 0, want_pairs = 0;
    bool force_radix = false, radix_wanted = true;
    unsigned last_n_pairs = 0;
    unsigned long long last_n_tests = 0;
};

LargeBuffers* large_buffers_create() { return new LargeBuffers(); }
void large_buffers_destroy(LargeBuffers* b) {
    if (!b) return;
    cudaFree(b->cnt); cudaFree(b->frontier[0]); cudaFree(b->frontier[1]); cudaFree(b->pairs); cudaFree(b->sorted);
    cudaFree(b->keys[0]); cudaFree(b->keys[1]); cudaFree(b->vals[0]); cudaFree(b->vals[1]); cudaFree(b->hist);
    cudaFree(b->seg_start); cudaFree(b->seg_end); cudaFree(b->unit_start); cudaFree(b->prob_flags); cudaFree(b->ptab);
    cudaFree(b->chunk_out); cudaFree(b->chunk_points); cudaFree(b->part);
    if (b->h_cnt) cudaFreeHost(b->h_cnt);
    delete b;
}

unsigned large_last_pairs(const LargeBuffers* b) { return b->last_n_pairs; }
unsigned long long large_last_tests(const LargeBuffers* b) { return b->last_n_tests; }
double* large_part_buffer(LargeBuffers* b) { return b->part; }

// Copies the sorted pair list of problem `prob` (device -> host).
cudaError_t large_get_pairs(LargeBuffers* b, int prob, int* out, long long cap, long long* n_out, cudaStream_t stream) {
    unsigned se[2] = {0, 0};
    LCU(cudaMemcpyAsync(&se[0], b->seg_start + prob, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    LCU(cudaMemcpyAsync(&se[1], b->seg_end + prob, sizeof(unsigned), cudaMemcpyDeviceToHost, stream));
    LCU(cudaStreamSynchronize(stream));
    const long long n = (long long)se[1] - se[0];
    if (n_out) *n_out = n;
    const long long m = std::min(n, cap);
    if (out && m > 0) {
        std::vector<int3> tmp(m);
        LCU(cudaMemcpy(tmp.data(), b->sorted + se[0], sizeof(int3) * m, cudaMemcpyDeviceToHost));
        for (long long i = 0; i < m; ++i) { out[2 * i] = tmp[i].y; out[2 * i + 1] = tmp[i].z; }
    }
    return cudaSuccess;
}
const int3* large_sorted_ptr(const LargeBuffers* b) { return b->sorted; }
// what the reference-order bristle pipeline needs of the last broad phase
void large_exact_view(const LargeBuffers* b, const LargeScene& ls, long long n_env, ExactPairs& ps) {
    ps.sorted = b->sorted; ps.seg_start = b->seg_start; ps.seg_end = b->seg_end; ps.unit_start = b->unit_start;
    ps.n_units = b->cnt ? &b->cnt->n_units : nullptr;
    ps.large_ins = ls.large_ins; ps.n_large = ls.n_large;
    ps.max_large_units = (size_t)(b->cap_pairs / kChunk) + (size_t)(n_env * ls.n_large) + 1;
}
const unsigned* large_seg_start_ptr(const LargeBuffers* b) { return b->seg_start; }

namespace {
__global__ void write_counts_kernel(SceneDev sc, LargeScene ls, EvalIO io, const unsigned* seg_start, const unsigned* seg_end, unsigned n_prob) {
    for (unsigned p = blockIdx.x * blockDim.x + threadIdx.x; p < n_prob; p += gridDim.x * blockDim.x) {
        long long env; int k;
        prob_to_ei(sc, ls, (int)p, env, k);
        io.n_pairs[env * sc.n_ins + k] = (long long)seg_end[p] - (long long)seg_start[p];
        io.flags[env * sc.n_ins + k] = 0;
    }
}
}  // namespace

// Broad phase only (Jacobian mode): publish the pair counts of the large instructions.
cudaError_t large_write_counts(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, cudaStream_t stream) {
    const unsigned n_prob = (unsigned)(io.n_env * ls.n_large);
    if (n_prob == 0) return cudaSuccess;
    write_counts_kernel<<<std::min<unsigned>((n_prob + 255) / 256, 1024), 256, 0, stream>>>(sc, ls, io, b->seg_start, b->seg_end, n_prob);
    return cudaGetLastError();
}

// Broad phase + sort + segments, queued on the stream WITHOUT a host round trip: the pair count stays on the device (every later kernel
// reads it from the counters), grids are sized for the buffers' capacity.  The capacities grow like the reference's VectorCache
// (src/obb/vector_cache.jl:11-15), but after the fact: the counters are copied to pinned memory behind the traversal, the caller
// synchronises once at the END of the evaluation it queued and asks large_check(), which doubles what overflowed and tells the caller
// to queue the evaluation again.
cudaError_t large_broad_phase(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, cudaStream_t stream, int* n_launches,
                              int hash_rank, int hash_world) {
    const long long n_prob_ll = io.n_env * ls.n_large;
    if (n_prob_ll <= 0) return cudaSuccess;
    if (n_prob_ll > (1LL << 30)) return cudaErrorInvalidValue;
    const unsigned n_prob = (unsigned)n_prob_ll;
    int prob_bits = 0;
    while ((1ull << prob_bits) < (unsigned long long)n_prob) ++prob_bits;
    if (ls.key_bits + prob_bits > 64) return cudaErrorMemoryAllocation;   // (problem, DFS key) must fit one 64-bit sort key -> PFC_E_CAPACITY
    if (!b->cnt) { LCU(cudaMalloc(&b->cnt, sizeof(Counters))); LCU(cudaMemset(b->cnt, 0, sizeof(Counters))); }
    if (!b->h_cnt) LCU(cudaHostAlloc(reinterpret_cast<void**>(&b->h_cnt), sizeof(Counters), cudaHostAllocDefault));
    b->want_frontier = std::max<size_t>(b->want_frontier, std::max<size_t>(std::max<size_t>(b->cap_frontier, 1u << 18), (size_t)n_prob * 4));
    b->want_pairs = std::max<size_t>(b->want_pairs, std::max<size_t>(b->cap_pairs, 1u << 20));
    int n_sm = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    // the traversal kernel is persistent: every block must be resident, because idle warps wait for donated work
    static const int dfs_minb = getenv("PFC_DFS_MINB") ? atoi(getenv("PFC_DFS_MINB")) : 1;   // (experiment switch)
    int dfs_blocks_per_sm = 0;
    {
        struct Tag {};
        std::lock_guard<std::mutex> g(launch_mutex());
        LaunchSlot& sl = launch_slot<Tag>();
        if (sl.blocks == 0) {
            LCU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sl.blocks, dfs_minb == 4 ? broad_dfs_kernel<4> : (dfs_minb == 3 ? broad_dfs_kernel<3> : broad_dfs_kernel<1>), kDfsWarps * 32, 0));
            if (sl.blocks < 1) sl.blocks = 1;
        }
        dfs_blocks_per_sm = sl.blocks;
        struct TagSort {};
        LaunchSlot& ss = launch_slot<TagSort>();
        if (ss.key0 != 1) {
            LCU(cudaFuncSetAttribute(small_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kSmallSort * 12)));
            ss.key0 = 1;
        }
    }
    const int dfs_blocks = n_sm * dfs_blocks_per_sm;
    // How the dual-tree recursion is walked.  Big scenes: LEVEL BY LEVEL to the leaves -- one launch per level of the recursion, one thread
    // per node pair of the level's frontier, children appended to the next frontier with warp-aggregated atomics.  Every lane of the
    // machine works on a node pair whatever the shape of the contact (a few instructions out of thousands carry all of the work in a
    // pile; a contact patch is a small corner of two big trees), which the per-warp stacks of the depth-first kernel cannot offer: measured
    // on the 64-body pile 1.78 ms (stack traversal from the root pairs, work donated between warps) against the level-by-level walk.
    // The order the pairs are found in does not matter: the sort below restores the reference's order.
    // Small scenes (one gripper pad against another): a few levels to get one seed per resident warp, then the stack traversal in
    // ONE launch -- a launch per level would cost more than the work.
    const bool by_level = ls.max_leaves >= 16384 || n_prob >= 64;
    int levels = 0;
    { double f = (double)n_prob; const double target = 1.0 * dfs_blocks * kDfsWarps; while (f < target && levels < 12) { f *= 4.0; ++levels; } }
    // split over several GPUs: a contact patch is small against the meshes, so a few sub-trees carry nearly all of the work; three more
    // breadth-first levels make the hash-partitioned pieces ~64x finer, which is what balances the ranks
    static const int split_extra = getenv("PFC_SPLIT_EXTRA") ? atoi(getenv("PFC_SPLIT_EXTRA")) : 3;   // (experiment switch)
    if (hash_world > 1) levels = std::min(levels + split_extra, 16);
    const int split_level = levels - 1;             // the level whose children are dealt to the ranks by hash
    // (a level descends both trees until one of them is at a leaf, then the other alone: a leaf pair at depths (d1, d2) is reached at
    // level max(d1, d2), so max_depth + 1 levels test every pair of the recursion)
    if (by_level) levels = std::max(levels, std::min(ls.max_depth + 1, kMaxLevels));
    LCU(ensure(b->frontier[0], b->cap_frontier, b->want_frontier));
    LCU(ensure(b->frontier[1], b->cf2, b->want_frontier));
    LCU(ensure(b->pairs, b->cap_pairs, b->want_pairs));
    const size_t cap = b->cap_pairs;
    LCU(ensure(b->keys[0], b->cap_keys, cap)); LCU(ensure(b->keys[1], b->cap_keys2, cap));
    LCU(ensure(b->vals[0], b->cap_vals, cap)); LCU(ensure(b->vals[1], b->cap_vals2, cap));
    LCU(ensure(b->sorted, b->cap_sorted, cap));
    const unsigned cap_tiles = (unsigned)((cap + kTile - 1) / kTile);
    LCU(ensure(b->hist, b->cap_hist, (size_t)256 * cap_tiles + 256));   // + the 256 digit totals
    LCU(ensure(b->seg_start, b->cap_seg, (size_t)n_prob + 1));
    LCU(ensure(b->seg_end, b->cap_seg2, (size_t)n_prob + 1));
    LCU(ensure(b->unit_start, b->cap_unit, (size_t)n_prob + 2));
    LCU(ensure(b->prob_flags, b->cap_pf, (size_t)n_prob));
    LCU(ensure(b->ptab, b->cap_ptab, (size_t)n_prob));
    // ---- traversal
    init_frontier_kernel<<<std::min<unsigned>((n_prob + 255) / 256, 1024), 256, 0, stream>>>(sc, ls, io.n_env, io.X, b->frontier[0], b->ptab, b->cnt);
    int src = 0;
    static const unsigned per_warp_from = getenv("PFC_BFS_PER_WARP_FROM") ? (unsigned)atoll(getenv("PFC_BFS_PER_WARP_FROM")) : (1u << 20);   // (experiment switch)
    for (int l = 0; l < levels; ++l) {
        broad_bfs_kernel<<<n_sm * 8, 256, 0, stream>>>(sc, b->ptab, b->frontier[src], b->frontier[src ^ 1], l, split_level, (unsigned)b->cap_frontier, b->pairs,
                                                     (unsigned)b->cap_pairs, b->cnt, (unsigned)hash_rank, (unsigned)hash_world, per_warp_from);
        src ^= 1;
    }
    // what the levels left (nothing, when they ran to the leaves) is traversed with per-warp stacks; the split has been made by then
    dfs_queue_init_kernel<<<1, 1, 0, stream>>>(b->cnt, levels, (unsigned)b->cap_frontier);
    if (dfs_minb == 4)
        broad_dfs_kernel<4><<<dfs_blocks, kDfsWarps * 32, 0, stream>>>(sc, b->ptab, b->frontier[src], (unsigned)b->cap_frontier, b->pairs, (unsigned)b->cap_pairs,
                                                                     b->cnt, 0u, 1u);
    else if (dfs_minb == 3)
        broad_dfs_kernel<3><<<dfs_blocks, kDfsWarps * 32, 0, stream>>>(sc, b->ptab, b->frontier[src], (unsigned)b->cap_frontier, b->pairs, (unsigned)b->cap_pairs,
                                                                     b->cnt, 0u, 1u);
    else
        broad_dfs_kernel<1><<<dfs_blocks, kDfsWarps * 32, 0, stream>>>(sc, b->ptab, b->frontier[src], (unsigned)b->cap_frontier, b->pairs, (unsigned)b->cap_pairs,
                                                                     b->cnt, 0u, 1u);
    LCU(cudaMemcpyAsync(b->h_cnt, b->cnt, sizeof(Counters), cudaMemcpyDeviceToHost, stream));   // read by large_check() after the caller's synchronisation
    b->check_pending = true;
    if (n_launches) *n_launches += 3 + levels;
    // ---- segments + keys + sort (n on the device)
    init_segments_kernel<<<std::min<unsigned>((n_prob + 255) / 256, 1024), 256, 0, stream>>>(b->seg_start, b->seg_end, n_prob);
    zero_int_kernel<<<std::min<unsigned>((n_prob + 255) / 256, 1024), 256, 0, stream>>>(b->prob_flags, n_prob);
    unsigned* tot = b->hist + (size_t)256 * cap_tiles;
    const unsigned g = std::min<unsigned>((unsigned)((cap + 255) / 256), (unsigned)n_sm * 16);
    build_keys_kernel<<<g, 256, 0, stream>>>(sc, ls, b->pairs, b->cnt, (unsigned)cap, b->keys[0], b->vals[0]);
    const int total_bits = ls.key_bits + prob_bits;
    const int n_pass = (total_bits + 7) / 8;
    const int fin = n_pass & 1;   // where the radix passes leave the sorted keys; short lists are sorted into the same buffer by one CTA
    // single small scenes: when the previous evaluation listed few pairs the 3 x n_pass radix launches (which would all return at once) are
    // left out; small_sort_kernel raises a flag if the list is long after all
    const bool radix_queued = b->radix_wanted;   // (decided by large_check after the previous evaluation)
    int cur = 0;
    for (int pass = 0; pass < n_pass && radix_queued; ++pass) {
        radix_hist_kernel<<<(cap_tiles + 3) / 4, 128, 0, stream>>>(b->keys[cur], b->cnt, (unsigned)cap, 8 * pass, b->hist, cap_tiles);
        radix_rowscan_kernel<<<256, 256, 0, stream>>>(b->hist, b->cnt, (unsigned)cap, cap_tiles, tot);
        radix_scatter_kernel<<<(cap_tiles + 3) / 4, 128, 0, stream>>>(b->keys[cur], b->vals[cur], b->cnt, (unsigned)cap, 8 * pass, b->hist, tot, cap_tiles, b->keys[cur ^ 1],
                                                                    b->vals[cur ^ 1]);
        cur ^= 1;
    }
    small_sort_kernel<<<1, 1024, kSmallSort * 12, stream>>>(b->keys[0], b->vals[0], b->cnt, (unsigned)cap, b->keys[fin], b->vals[fin], radix_queued ? 1 : 0);
    gather_sorted_kernel<<<g, 256, 0, stream>>>(b->pairs, b->vals[fin], b->cnt, (unsigned)cap, b->sorted, b->seg_start, b->seg_end);
    units_scan_kernel<<<1, 1024, 0, stream>>>(b->seg_start, b->seg_end, n_prob, b->unit_start, b->cnt, 0, 1);
    if (n_launches) *n_launches += 6 + (radix_queued ? 3 * n_pass : 0);
    return cudaGetLastError();
}

// After the caller synchronised the stream: did the traversal queued by the last large_broad_phase fit its buffers?
// 0 = yes; 1 = no, the capacities have been raised and the evaluation must be queued again; -1 = it cannot fit.
// a replayed CUDA graph of an evaluation contains the traversal and the copy of its counters: they must be looked at again
void large_mark_clear(LargeBuffers* b) { if (b) b->check_pending = false; }
void large_mark_pending(LargeBuffers* b) { if (b && b->h_cnt) b->check_pending = true; }
int large_check(LargeBuffers* b) {
    if (!b || !b->check_pending) return 0;
    b->check_pending = false;
    const Counters& h = *b->h_cnt;
    if (h.overflow & 4u) return -1;
    bool again = false;
    if (h.overflow & 8u) { b->force_radix = true; b->radix_wanted = true; alloc_generation()++; again = true; }   // the list outgrew the one-CTA sort
    if (h.overflow & 1u) {
        unsigned level_max = h.frontier_max;   // the level counters kept counting past the capacity: the need of the levels that ran is known
        for (int l = 0; l < kMaxLevels + 2; ++l) level_max = std::max(level_max, h.level_n[l]);
        const size_t need = (size_t)std::max(level_max, h.q_tail) + 1024;   // (levels below an overflowing one were cut short: leave room)
        b->want_frontier = std::max<size_t>(b->cap_frontier * 2, need * 2);
        again = true;
    }
    if (h.overflow & 2u) {
        b->want_pairs = std::max<size_t>(b->cap_pairs * 2, (size_t)h.n_pairs + 1024);   // the counter kept counting: the need is known
        again = true;
    }
    if (again) return (b->want_pairs > (1ull << 31) || b->want_frontier > (1ull << 31)) ? -1 : 1;
    b->last_n_pairs = h.n_pairs;
    b->last_n_tests = h.n_tests;
    const bool want = b->force_radix || h.n_pairs > kSmallSort / 2;
    if (want != b->radix_wanted) { b->radix_wanted = want; alloc_generation()++; }   // the launch sequence changes: a captured graph of it is stale
    return 0;
}

// Narrow phase + friction + reduction of the regularized instructions over the pair lists produced by large_broad_phase.
// partial_only (sharded contexts): leave the per-problem partial sums (kLargePartStride doubles each) in large_part_buffer(); the caller
// reduces them over the ranks and calls again with apply_parts = 1.
cudaError_t large_narrow_stage(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, int partial_only, int apply_parts,
                               cudaStream_t stream, int* n_launches) {
    const unsigned n_prob = (unsigned)(io.n_env * ls.n_large);
    if (n_prob == 0) return cudaSuccess;
    const size_t max_units = (size_t)(b->cap_pairs / kChunk) + n_prob + 1;   // (the pair count itself stays on the device)
    int n_sm = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    LCU(ensure(b->chunk_out, b->cap_chunk, max_units * kNA));
    LCU(ensure(b->chunk_points, b->cap_cp, max_units));
    if (partial_only) LCU(ensure(b->part, b->cap_part, (size_t)n_prob * kLargePartStride));
    if (!apply_parts) {
        {
            struct Tag {};
            std::lock_guard<std::mutex> g(launch_mutex());
            LaunchSlot& sl = launch_slot<Tag>();
            if (sl.key0 != 1) { LCU(cudaFuncSetAttribute(narrow_large_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NarrowLargeSmem))); sl.key0 = 1; }
        }
        const unsigned grid = (unsigned)std::min<size_t>(max_units, (size_t)n_sm * 2);   // persistent: 2 CTAs per SM (93 KB of shared memory each)
        narrow_large_kernel<<<grid, kChunk, sizeof(NarrowLargeSmem), stream>>>(sc, ls, io, b->sorted, b->seg_start, b->seg_end, b->unit_start, n_prob, b->cnt, b->chunk_out,
                                                                               b->chunk_points, b->prob_flags);
        if (n_launches) *n_launches += 1;
    }
    finish_large_kernel<<<std::min<unsigned>((n_prob + 3) / 4, (unsigned)n_sm * 8), 128, 0, stream>>>(
        sc, ls, io, b->seg_start, b->seg_end, b->unit_start, n_prob, b->chunk_out, b->chunk_points, b->prob_flags, partial_only ? b->part : nullptr, apply_parts);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

}  // namespace pfc
