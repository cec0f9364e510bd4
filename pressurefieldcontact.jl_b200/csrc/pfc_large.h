// pfc_large.h -- host-side interface of the large-instruction pipeline (pfc_large.cu).
#pragma once
#include <cuda_runtime.h>

#include "pfc_launch.h"
#include "pfc_types.cuh"

namespace pfc {

// device-resident tables of the large path
struct LargeScene {
    const int32_t* large_ins;             // instruction indices handled by the large path
    const unsigned long long* leaf_path;  // per primitive (all meshes concatenated): root-to-leaf turns, MSB first in the low `depth` bits
    const unsigned char* leaf_depth;      // per primitive: depth of its leaf
    int32_t n_large;
    int32_t key_bits;                     // max over large instructions of depth(tree 1) + depth(tree 2)
    int32_t max_leaves;                   // max over large instructions of max(n_leaf 1, n_leaf 2)
    int32_t max_depth;                    // max over large instructions of max(depth(tree 1), depth(tree 2))
};

struct LargeBuffers;
LargeBuffers* large_buffers_create();
void large_buffers_destroy(LargeBuffers* b);

// hash_rank / hash_world: multi-GPU split of one large scene -- this context traverses (and lists) only the sub-trees whose hash falls on it
cudaError_t large_broad_phase(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, cudaStream_t stream, int* n_launches,
                              int hash_rank = 0, int hash_world = 1);
// regularized instructions over the lists of large_broad_phase (bristle instructions: pfc_exact.cu).
// partial_only: leave the per-problem partial sums (+ point and pair counts) in large_part_buffer() for the caller's reduction over the ranks;
// apply_parts: the buffer holds the sums over all ranks -- finish from it
cudaError_t large_narrow_stage(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, int partial_only, int apply_parts,
                               cudaStream_t stream, int* n_launches);
struct ExactPairs;
void large_exact_view(const LargeBuffers* b, const LargeScene& ls, long long n_env, ExactPairs& ps);
// after the caller's stream synchronisation: 0 = the last traversal fit its buffers, 1 = it did not (capacities raised: queue the evaluation
// again), -1 = it cannot fit
int large_check(LargeBuffers* b);
void large_mark_pending(LargeBuffers* b);
void large_mark_clear(LargeBuffers* b);   // after replaying a captured evaluation
cudaError_t large_write_counts(const SceneDev& sc, const LargeScene& ls, const EvalIO& io, LargeBuffers* b, cudaStream_t stream);
unsigned large_last_pairs(const LargeBuffers* b);
unsigned long long large_last_tests(const LargeBuffers* b);
double* large_part_buffer(LargeBuffers* b);     // [n_problem][8]: 6 partial sums, point count, pair count (sharded mode)
constexpr int kLargePartStride = 8;
cudaError_t large_get_pairs(LargeBuffers* b, int prob, int* out, long long cap, long long* n_out, cudaStream_t stream);

// Jacobian mode of the regularized instructions (pfc_dual_chunked.cu): narrow phase + friction + reduction on Duals over existing pair lists.
// What the seed chunks of one Jacobian share (all optional): survivors of the Float64 clip of the small instructions' candidates
// (launch_dual_prefilter) and the Float64 wrenches of the same evaluation.
struct DualShared { const unsigned* surv_pairs; const int* surv_n; const double* w_f64; };
// params: [real env][ins] contact parameters, or nullptr for the scene's own
cudaError_t launch_dual_prefilter(const SceneDev& sc, long long n_env, const double* X, const long long* n_pairs, const unsigned* small_pairs, int small_cap,
                                  unsigned* surv_pairs, int* surv_n, const InsParam* params, cudaStream_t stream);
cudaError_t launch_eval_dual6(const SceneDev& sc, long long n_env, const double* X7, const double* twist7, const double* s7, double* wrench7, double* sdot7,
                              const long long* n_pairs, int* flags, const unsigned* small_pairs, int small_cap, const LargeBuffers* lb,
                              const int32_t* large_index, int n_large, const InsParam* params, cudaStream_t stream, unsigned* ticket,
                              long long n_real = 0, const DualShared* shared = nullptr);

}  // namespace pfc
