// pfc_launch.h -- host-side launchers of the kernels (implemented in the .cu files).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <mutex>

#include "pfc_types.cuh"

namespace pfc {

// Launch-configuration cache.  cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device and the persistent grid sizes depend on
// the device's SM count, so what a launcher caches is keyed by (kernel family tag, variant, current device) -- several contexts on
// different devices may live in one process (single-process multi-device, pfc_group) -- and guarded by one mutex.
// Counts device (re)allocations of the growable buffers: a captured CUDA graph of an evaluation holds raw pointers, so it is only replayed
// while this number is what it was at capture time.
inline std::atomic<unsigned long long>& alloc_generation() { static std::atomic<unsigned long long> g{0}; return g; }

struct LaunchSlot { int key0 = -1, key1 = -1, blocks = 0; size_t smem = 0; };
constexpr int kMaxLaunchDevices = 64;
inline std::mutex& launch_mutex() { static std::mutex m; return m; }
template <class Tag, int Variants = 1> inline LaunchSlot& launch_slot(int variant = 0) {   // call with launch_mutex() held
    static LaunchSlot slots[kMaxLaunchDevices][Variants];
    int dev = 0;
    cudaGetDevice(&dev);
    return slots[dev % kMaxLaunchDevices][variant];
}

struct EvalIO {
    long long n_env;
    const double* X;      // [env][ins][16] col-major x_r2_r1
    const double* twist;  // [env][ins][6]  angular, linear
    const double* s;      // [env][bristle][6] or nullptr
    double* wrench;       // [env][ins][6]
    double* sdot;         // [env][bristle][6] or nullptr
    long long* n_pairs;   // [env][ins]
    int* flags;           // [env][ins]
    int* dbg_pairs;       // optional [env*n_ins][dbg_cap][2] (prim ids, DFS order) or nullptr
    int dbg_cap;
    const InsParam* params;   // [env][ins] contact parameters, or nullptr for the scene's own
};

constexpr int kSmallCap = 512;      // frontier / pair capacity of the fused small path

int small_cap(int max_pairs);
int persistent_blocks(const void* kern, int threads, size_t smem, cudaError_t* err);   // resident CTAs of a persistent kernel on the current device (pfc_small.cu)
constexpr int kSmallPairsSlack = 32;   // words after the pair lists: [0] is the narrow tile kernel's tile ticket (zeroed by the broad kernel)
// ev: optional array of 3 events recorded before the broad kernel, between the two kernels and after the narrow kernel
cudaError_t launch_eval_small_f64(const SceneDev& sc, const EvalIO& io, int max_pairs, unsigned* pairs, cudaStream_t stream, int* n_launches,
                                  cudaEvent_t* ev = nullptr, cudaEvent_t after_broad = nullptr);

// broad phase of the small path only (Jacobian mode re-traverses with the Float64 state, then evaluates on Duals)
cudaError_t launch_broad_small_only(const SceneDev& sc, const EvalIO& io, int max_pairs, unsigned* pairs, cudaStream_t stream, int* n_launches);

// single-thread debug kernel: re-runs the narrow phase of one (env, ins) over a given pair list in
// order and writes the traction points (8 doubles each) -- the reference's TractionCache.
cudaError_t launch_dump_traction(const SceneDev& sc, const EvalIO& io, long long env, int ins, const int* pairs, long long n_pairs, double* out,
                                 int cap_points, int* n_points, cudaStream_t stream);

// FP64 DFMA throughput of the current device in TFLOP/s (best of a few bursts).
cudaError_t measure_fp64_peak(cudaStream_t stream, double* tflops);


// ---- device-side prologue / epilogue for floating-joint scenes (pfc_state.cu) ----
struct BodyDev {
    int joint;      // 0 = world-attached (no joint), 1 = SPQuatFloating
    int q0, v0;     // offsets of the joint's coordinates in q and v
    int pad;
    double pose_R[9];   // joint pose on the world (row-major), pose_t
    double pose_t[3];
};
struct StateDev {
    const BodyDev* bodies;
    const int* ins_body;       // [n_ins][2]: body of mesh_1, body of mesh_2
    const int* body_ins_ptr;   // CSR over bodies: the instructions that touch a body, in instruction order ...
    const int* body_ins;       // ... as (instruction << 1) | (1 if the body carries mesh_2)
    int n_body, nq, nv, n_x;   // n_x = nq + nv + 6 n_bristle: stride of one environment's state
};
// rigid-body data for the device-side calcXd! (pfc_set_dynamics): per body the 6x6 spatial inertia about the body origin in the
// body frame ([angular; linear], row-major) and its inverse; gravity in the world frame
struct DynDev {
    const double* H;      // [n_body][36]
    const double* Hinv;   // [n_body][36]
    double gravity[3];
};
cudaError_t launch_state_dynamics(const StateDev& sd, const DynDev& dd, long long n_env, int n_ins, int n_bristle, const double* x, const double* wrench,
                                  const double* tau_ext, const double* sdot, double* xdot, cudaStream_t stream, int* n_launches,
                                  const int* flags = nullptr, int* status = nullptr);
cudaError_t launch_state_prologue(const StateDev& sd, long long n_env, int n_ins, int n_bristle, const double* x, double* X, double* twist, double* s,
                                  cudaStream_t stream, int* n_launches);
// Jacobian mode of the same kernels (Dual<6>, seeds on x[seed0 .. seed0 + 6)): every output scalar is 7 doubles (value, 6 partials)
cudaError_t launch_state_prologue_dual6(const StateDev& sd, long long n_env, int n_ins, int n_bristle, const double* x, int seed0, double* X7, double* twist7,
                                        double* s7, cudaStream_t stream, int* n_launches, long long n_real = 0);
cudaError_t launch_state_dynamics_dual6(const StateDev& sd, const DynDev& dd, long long n_env, int n_ins, int n_bristle, const double* x, int seed0,
                                        const double* wrench7, const double* tau_ext, const double* sdot7, double* xdot7, cudaStream_t stream,
                                        int* n_launches, const int* flags = nullptr, int* status = nullptr, long long n_real = 0, double* jac = nullptr);
// (n_real > 0: whole-Jacobian mode -- the n_env entries are n_env / n_real seed chunks of n_real real environments, chunk-major, chunk g
//  seeded on x[seed0 + 6 g ..); with jac the partials go to jac[env][row][seed + k] (row-major n_x x n_x) and chunk 0's values to xdot7[env][row])
// flags / status (optional): OR the error bits of flags[n_env * n_ins] into *status (see or_error_flags)
cudaError_t launch_state_epilogue(const StateDev& sd, long long n_env, int n_ins, const double* x, const double* wrench, double* f_gen, cudaStream_t stream,
                                  int* n_launches, const int* flags = nullptr, int* status = nullptr);

// Refit of one mesh after its vertices moved (pfc_refit.cu): primitive records, leaf boxes, internal boxes bottom-up.  idx / eps / xyz /
// level_nodes are device arrays of the mesh; nodes / tris / tets point at the mesh's slices; level_ptr is a HOST array of n_level + 1
// offsets into level_nodes (internal nodes grouped by depth); aabb is scratch of 6 n_node doubles; *err gets bit 0 for a bad tetrahedron.
cudaError_t launch_refit(int kind, long long n_prim, long long n_node, const int* idx, const double* eps, const double* xyz, TriRec* tris, TetRec* tets,
                         NodeRec* nodes, double* aabb, const int* level_nodes, const int* level_ptr, int n_level, int* err, cudaStream_t stream,
                         int* n_launches);

// Batched updateInvC! of the Radau step (pfc_radau.cu): inv_c[m] = inverse((shift[m]) I + neg_J[index ? index[m] : m]), n x n complex, interleaved
cudaError_t launch_radau_inv_c(long long n_mat, int n, const double* neg_J, const double* shift, const int* index, double* inv_c, int* info, cudaStream_t stream);

// The adaptive Radau IIA step of a batch (pfc_radau.cu; per-environment arithmetic in pfc_radau_step.cuh).  A "state" is one (environment,
// stage) pair of the current attempt; the packed arrays hold the states of the still-active environments in environment order.
struct RadauEnv;
struct RadauBufs {
    long long n_env;
    int nx, nv, n_ins, s_max, max_rule;
    double h_max, tol_newton;
    RadauEnv* env;              // [env] controller state
    double* x;                  // [env][nx] the step's start state, overwritten by the accepted state
    const double* tau;          // [env][nv] or nullptr
    double* t;                  // [env]
    double* h_taken;            // [env]
    int* stats;                 // [env][4] or nullptr
    double* X;                  // [env][s_max][nx] stage states
    double* Xp; double* Fp;     // [state][nx] packed stage states / their derivatives
    double* taup;               // [state][nv] (with tau)
    const InsParam* params;     // [env][n_ins] contact parameters, or nullptr for the scene's own
    InsParam* paramp;           // [state][n_ins] (with params): the environment's rows, gathered next to taup
    const double* xx0;          // [env][nx] calcXd!(x)
    double* jac;                // [env][nx][nx] d xdot / d x, negated in place into -J
    double* invc;               // [matrix][nx][nx] complex: (h^-1 lambda_i I - J)^-1, matrices in the order of the round's plan
    double* shift;              // [matrix][2]
    int* index;                 // [matrix] environment
    int* state_list;            // [state] env * 8 + stage
    int* env_list;              // [active env]
    int* state_pos;             // [env] first packed state of the environment in this iteration
    int* inv_base;              // [env] first matrix of the environment in this round
    int* counts;                // [4]: states, environments of the last plan / compaction; step-size error bits; spare
    const BodyDev* bodies; int n_body;   // principal_value! of the floating bodies' MRPs
};
// mode 2: first round of a step (every environment pending), 1: a new attempt round of the pending environments (matrix list, attempt
// reset), 0: compaction of the active environments between Newton iterations.  One CTA; writes counts[0..1].
cudaError_t launch_radau_plan(const RadauBufs& b, int mode, cudaStream_t stream);
// -J from the Jacobian in place, and the error bits of the Jacobian's flags [env][ins] into *status
cudaError_t launch_radau_prepare(const RadauBufs& b, const int* flags, int* status, cudaStream_t stream);
cudaError_t launch_radau_gather(const RadauBufs& b, long long n_states, cudaStream_t stream);
cudaError_t launch_radau_newton(const RadauBufs& b, long long n_active, cudaStream_t stream);
cudaError_t launch_radau_controller(const RadauBufs& b, cudaStream_t stream);

// A roll-out through shared knot times (pfc_radau_rollout): per round of steps, the environments that still have a knot ahead and steps
// left are gathered into compact arrays, take one step as a sub-batch (the RadauBufs sequence above on the compact arrays), and are
// scattered back.
struct RadauRolloutBufs {
    long long n_env, max_steps;
    int nx, nv, n_knot;
    const double* knots;        // [knot] absolute times
    RadauEnv* env;              // [env] controller state
    double* x;                  // [env][nx]
    const double* tau;          // [knot][env][nv] or nullptr
    double* t;                  // [env]
    const InsParam* params;     // [env][n_ins] contact parameters, or nullptr for the scene's own
    double* x_knot;             // [knot][env][nx] or nullptr
    int* knot;                  // [env] next knot
    int* steps;                 // [env] accepted steps of this roll-out
    int* stats;                 // [env][4] knots reached, accepted steps, rejected attempts, stage evaluations
    int* list;                  // [slot] environment of the compact slot
    RadauEnv* env_c; double* x_c; double* tau_c; double* t_c; double* h_c; double* h_save; int* stats_c;   // [slot] compact step arrays
    InsParam* params_c;         // [slot][n_ins] (with params)
    int n_ins;
    int* count;                 // [2]: compact slots of the last selection; 1 if some environment starts within h_min of knot 0
};
// One CTA: lists the environments with knot < n_knot and steps < max_steps (environment order), gathers them (with their parameter rows)
// and prepares the knot step (radau_knot_begin).  check: also test t_knot[0] - t >= h_min for every environment (count[1]; nothing is gathered when it fails).
cudaError_t launch_radau_select(const RadauRolloutBufs& b, int check, cudaStream_t stream);
// After the compact step: radau_knot_end, the x_knot rows, the statistics and the write-back of the n_active slots.
cudaError_t launch_radau_finish(const RadauRolloutBufs& b, long long n_active, cudaStream_t stream);

}  // namespace pfc
