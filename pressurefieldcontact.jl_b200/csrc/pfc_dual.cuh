// pfc_dual.cuh -- declarations of the Jacobian mode of the regularized-friction instructions (pfc_dual_chunked.cu).
#pragma once
#include "pfc_large.h"
#include "pfc_patch.cuh"
#include "pfc_twist.cuh"

namespace pfc {

struct DualIO {
    long long n_env;
    const double* X7;       // [env][ins][16][7]
    const double* twist7;   // [env][ins][6][7]
    const double* s7;       // [env][bristle][6][7]
    double* wrench7;        // [env][ins][6][7]
    double* sdot7;          // [env][bristle][6][7]
    const long long* n_pairs;  // [env][ins] (from the Float64 broad phase)
    int* flags;             // [env][ins]
    long long n_real;       // whole-Jacobian mode: the n_env "environments" are n_env / n_real seed chunks of n_real real ones
                            // (chunk-major); pair lists, counts and flags exist once per REAL environment.  Otherwise = n_env.
    const InsParam* params; // [real env][ins] contact parameters, or nullptr for the scene's own
};

// pair list access for both paths
struct PairSource {
    const unsigned* small_pairs; int small_cap;           // [env][ins][cap] packed (a << 15 | b)
    const int3* large_sorted; const unsigned* seg_start;  // sorted (prob, a, b) + per-problem segment starts
    const int32_t* large_index;                           // instruction -> index in the large list or -1
    int n_large;
    // optional, small instructions only: the pairs that survive the Float64 clip, packed in candidate order by dual_prefilter_kernel
    // ([env][ins][cap] + counts [env][ins]); without them the Dual kernel clips every candidate in Float64 itself
    const unsigned* surv_pairs; const int* surv_n;
    // optional: Float64 wrenches [env][ins][6] of the same evaluation; problems none of whose inputs depends on the seeds copy their values
    const double* w_f64;
};

// value part of the Dual context: what the Float64 pass of the same evaluation works with

// Two thirds of the candidate pairs clip to nothing.  Whether a pair survives is decided by value parts only (the clipper compares
// values; the value part of every Dual operation used on the way is the Float64 operation), so the Float64 clip runs first and the
// 7x more expensive Dual pipeline only sees the pairs that leave a polygon.
PFC_D bool survives_f64(const SceneDev& sc, const InsDev& ins, int a, int b, const PatchCtx<double>& cxv) {
    if (!prefilter_pair(sc, ins, a, b, cxv)) return false;
    PolyRec<double> tmp;
    int fl = 0;
    const bool keep = clip_pair(sc, ins, a, b, cxv, tmp, fl);
    return keep || fl != 0;   // error paths (non-finite vertex) are left to the Dual pass, which records the flag
}

}  // namespace pfc
