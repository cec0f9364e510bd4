// pfc_exact.h -- host-side interface of the reference-order bristle pipeline (pfc_exact.cu).
#pragma once
#include <cuda_runtime.h>

#include "pfc_launch.h"
#include "pfc_types.cuh"

namespace pfc {

// static tables (uploaded by pfc_finalize)
struct ExactScene {
    const double* tet_eps;        // [n_tet][4]: the pressure-field value at each vertex of every tetrahedron
    const int32_t* bris_ins;      // the bristle instructions, in instruction order
    const int32_t* large_index;   // instruction -> index in the large list, or -1
    int32_t n_bris;
    int32_t skip_large;           // 1: large bristle instructions are not evaluated here (sharded contexts)
};
// boundary arrays of one evaluation; in Jacobian mode every scalar is 7 doubles (value, 6 partials)
struct ExactIO {
    long long n_env;
    const double* X;       // [env][ins][16]
    const double* twist;   // [env][ins][6]
    const double* s;       // [env][bristle][6]
    double* wrench;        // [env][ins][6]
    double* sdot;          // [env][bristle][6]
    const long long* n_pairs;   // [env][ins] (small instructions)
    int* flags;            // [env][ins]
    const InsParam* params;     // [env][ins] contact parameters, or nullptr for the scene's own
};
// candidate-pair lists of the Float64 broad phase
struct ExactPairs {
    const unsigned* small_pairs; int small_cap;   // [env][ins][cap], (a << 15) | b
    const int3* sorted;                           // large path: (problem, a, b) in the reference's order
    const unsigned* seg_start; const unsigned* seg_end; const unsigned* unit_start; const unsigned* n_units;
    const int32_t* large_ins; int n_large;
    size_t max_large_units;                       // host-side upper bound of *n_units
};
struct ExactBuffers;
ExactBuffers* exact_buffers_create();
void exact_buffers_destroy(ExactBuffers* b);
unsigned exact_last_points(const ExactBuffers* b);
// Queues the evaluation of every bristle instruction of the scene (wrench, s-dot, contact flag) on the stream.  The TractionCache buffer
// grows like the reference's VectorCache (src/obb/vector_cache.jl:11-15): after the caller synchronised the stream, exact_check() says
// whether it sufficed (0), or was raised so that the evaluation must be queued again (1), or cannot be made large enough (-1).
int exact_check(ExactBuffers* b);
void exact_mark_pending(ExactBuffers* b);
void exact_mark_clear(ExactBuffers* b);   // after replaying a captured evaluation
cudaError_t exact_bristle_eval(const SceneDev& sc, const ExactScene& es, const ExactIO& io, const ExactPairs& ps, int dual, ExactBuffers* b, cudaStream_t stream,
                               int* n_launches);

}  // namespace pfc
