/* pfc.h -- C ABI of libpfc_b200.so: B200-native contact-wrench evaluation for pressure-field
 * contact (drop-in for the hot path of ryanelandt/PressureFieldContact.jl).
 *
 * The boundary replaces the reference's forceAllElasticIntersections!(m, tm)
 * (src/contact_algorithms_non_friction.jl:60-68) as called from calcXd! (:18-38), which is the
 * function MechanismScenario.de holds (src/mechanism_scenario.jl:175,181,196) and Radau calls with
 * Vector{Float64} (src/radau/radau_functions.jl:67) and Vector{Dual{Nothing,Float64,6}} (:9).
 * Rigid-body kinematics before it (refreshBodyBodyTransform!/refreshBodyBodyCache!, :103-134) and
 * the J' * wrench epilogue after it (addGeneralizedForcesThirdLaw!, :267-286) stay with the
 * caller (RigidBodyDynamics on the Julia side); INTEGRATION.md shows the ccall shim.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative PFC_E_* code;
 *     pfc_last_error() returns a thread-local message for the last failure on this thread.
 *   - the caller owns every host buffer; the library copies on entry and never keeps a caller
 *     pointer after the call returns.  Device memory and the CUDA stream belong to the context.
 *   - a context is not thread-safe: one context per host thread / per GPU.
 *   - indices are 0-based int32 (the reference uses 1-based Int64).
 *   - matrices: 4x4 transforms are column-major (Julia SMatrix layout); twists and wrenches are
 *     [angular(3); linear(3)] (as_static_vector, src/utility.jl:13-14).
 *   - the wrench returned for an instruction is about the origin of mesh_2's frame r2, expressed
 *     in r2, applied TO body 2; the normal points into body 2; the relative velocity is v2 - v1
 *     (src/contact_algorithms_non_friction.jl:10-17).
 */
#ifndef PFC_H
#define PFC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pfc_ctx pfc_ctx;
typedef struct pfc_group pfc_group;   /* several contexts (one per GPU) sharing one scene and one library-owned NCCL communicator */

enum {
    PFC_OK = 0,
    PFC_E_ARG = -1,       /* bad argument / call order */
    PFC_E_CUDA = -2,      /* CUDA runtime error (message has the CUDA string) */
    PFC_E_CAPACITY = -3,  /* a fixed capacity was exceeded and could not be grown */
    PFC_E_NONFINITE = -4, /* the reference's error("Non-finite vertex likely"), src/clip/static_clip.jl:52 */
    PFC_E_MESH = -5,      /* invalid mesh (inverted tetrahedron, src/obb/obb_construction.jl:30; bad tree) */
    PFC_E_STEP = -6       /* error("time step is too small, something is wrong") / unacceptable h (src/radau/radau_solve.jl, adaptive.jl:52-57) */
};

/* per-(environment, instruction) flag bits */
enum { PFC_FLAG_CONTACT = 1, PFC_FLAG_NONFINITE = 2, PFC_FLAG_BAD_ARITY = 4, PFC_FLAG_OVERFLOW = 8 };

/* MechanismScenario() -- src/mechanism_scenario.jl:181-198.  Creates an empty scene on CUDA device `device`. */
int pfc_create(int device, pfc_ctx** out);
int pfc_destroy(pfc_ctx* ctx);

/* add_contact! / MeshCache -- src/mechanism_scenario.jl:298-314, src/structs.jl:33-54.
 * kind: 0 = triangle mesh (eps == NULL, Ebar ignored), 1 = tetrahedral mesh (eps per point, Ebar =
 * ContactProperties.E).  idx: n_prim x 3 or n_prim x 4.  The bounding-volume tree is the host-built
 * bin_BB_Tree (src/obb/tree_types.jl:1-16) flattened into arrays: node 0 is the root; node_R is
 * column-major 3x3 per node; node_left/right are node indices (-1 for a leaf); node_leaf_id is
 * the 0-based primitive index for leaves and -1 for internal nodes (the reference's id == -9999). */
int pfc_add_mesh(pfc_ctx* ctx, int kind, int64_t n_point, const double* xyz, int64_t n_prim, const int32_t* idx, const double* eps, double Ebar,
                 int64_t n_node, const double* node_c, const double* node_e, const double* node_R, const int32_t* node_left,
                 const int32_t* node_right, const int32_t* node_leaf_id, int* mesh_id_out);

/* ContactInstructions + add_friction_regularize! / add_friction_bristle! -- src/mechanism_scenario.jl:36-49, 365-416.
 * mesh_2 must be a tetrahedral mesh (the caller applies the Tri/Tet ordering rule, :399-416).
 * model 0 = Regularized, params = {mu_s, mu_d, v_c}; model 1 = Bristle, params = {tau, k_bar, mu_s, mu_d, magic};
 * bristle ids are assigned in call order.  n_quad_rule in {1, 2} (:45). */
int pfc_add_instruction(pfc_ctx* ctx, int mesh_1, int mesh_2, double chi, int model, const double* params, int n_quad_rule, int* ins_id_out);

/* finalize! -- src/mechanism_scenario.jl:206-231: uploads the static scene and sizes the per-batch buffers for max_env environments. */
int pfc_finalize(pfc_ctx* ctx, int64_t max_env);

/* Per-environment contact parameters, after pfc_finalize (domain randomization, system identification, parameter sweeps as one batch).
 * params[env][ins][8] = {chi, Ebar_1, Ebar_2, q0, q1, q2, q3, q4}: q = {mu_s, mu_d, v_c, -, -} for a regularized instruction,
 * {tau, k_bar, mu_s, mu_d, magic} for a bristle one (pfc_add_instruction's order); Ebar_1 / Ebar_2 take the place of the Ebar that
 * pfc_add_mesh gave mesh_1 / mesh_2 (Ebar_1 is ignored when mesh_1 is a triangle mesh); entries marked - are ignored.  Host pointer,
 * copied.  While a table is set, environment e of every evaluation (pfc_eval_f64[_device], pfc_eval_dual6, pfc_eval_state_f64[_device],
 * pfc_calcxd_*, pfc_radau_step[_device], pfc_radau_rollout[_device], pfc_get_traction) gives the bits of a context whose scene was built
 * with row e's values, evaluated on the same batch.  (In a scene whose number of small instructions is not a multiple of 4, a narrow
 * tile holds problems of neighbouring environments and a wrench's last bits depend on their contact patches, with or without a table:
 * bit-for-bit equality then needs the environments that share e's tiles to carry row e too; otherwise e agrees to rounding.)  Those
 * entry points (and pfc_radau_init) require n_env to equal the table's.  The candidate-pair lists do not
 * depend on these values.  n_env = 0 clears the table.  PFC_E_ARG, with the table in force unchanged, before pfc_finalize, for n_env
 * outside 0..max_env, a NULL params with n_env > 0, or a non-finite entry that the instruction's model uses.  The sharded and group
 * evaluations (pfc_eval_sharded_*, pfc_group_eval_f64) return PFC_E_ARG while a table is set. */
int pfc_set_contact_params(pfc_ctx* ctx, int64_t n_env, const double* params);

/* forceAllElasticIntersections!, Float64 mode -- src/contact_algorithms_non_friction.jl:60-84, for n_env independent states of the scene.
 *   X_r2_r1 [env][ins][16]  b.x_r2_r1.mat (:112)          twist_r2 [env][ins][6]  b.twist_r2_r1_r2 (:128)
 *   s       [env][bristle][6] bristle state (tm.s)         sdot     [env][bristle][6] tm.s-dot   (both may be NULL without bristles)
 *   wrench_r2 [env][ins][6]  the wrench yes_contact! returns (zero when no contact)
 *   n_pairs [env][ins] length(m.TT_Cache) (:74)            flags    [env][ins] PFC_FLAG_* bits         (either may be NULL)
 * Host pointers; copies in and out are part of the call; synchronous at return. */
int pfc_eval_f64(pfc_ctx* ctx, int64_t n_env, const double* X_r2_r1, const double* twist_r2, const double* s, double* wrench_r2, double* sdot,
                 int64_t* n_pairs, int32_t* flags);

/* Same evaluation on buffers already resident in device memory (all pointers are device pointers,
 * none may be NULL except s/sdot without bristles); enqueued on the context's stream.  Asynchronous for scenes whose instructions all
 * take the small path (n_leaf_1 * n_leaf_2 <= 512, e.g. test/boxes.jl) and use regularized friction; scenes with large instructions
 * synchronise the stream once inside the call (the candidate-pair count is read back to size the sort and to grow the pair buffers like
 * the reference's VectorCache), and so do scenes with bristle instructions (the TractionCache buffer grows the same way). */
int pfc_eval_f64_device(pfc_ctx* ctx, int64_t n_env, const double* X_r2_r1, const double* twist_r2, const double* s, double* wrench_r2,
                        double* sdot, int64_t* n_pairs, int32_t* flags);

/* forceAllElasticIntersections!, Dual{Nothing,Float64,6} mode (the Jacobian chunks of src/radau/radau_functions.jl:2-26).
 * Every Dual scalar is 7 doubles: value, then 6 partials.  X_bp is the Float64 transform the broad phase uses: the reference always
 * traverses with m.float's state (src/contact_algorithms_non_friction.jl:94-101); pass NULL to reuse the pair lists of the previous
 * pfc_eval_f64 call on this context. */
int pfc_eval_dual6(pfc_ctx* ctx, int64_t n_env, const double* X_bp, const double* X7_r2_r1, const double* twist7_r2, const double* s7,
                   double* wrench7_r2, double* sdot7, int64_t* n_pairs, int32_t* flags);

/* Device-side prologue / epilogue for scenes whose bodies are world-attached or float on SPQuatFloating joints (the batched MPC
 * roll-out case).  pfc_set_bodies (after pfc_finalize) describes the mechanism: joint_type[b] 0 = world-attached, 1 = SPQuatFloating
 * (q = [MRP(3); trans(3)], v = [omega(3); vel(3)] in the body frame, src/mechanism_scenario.jl:247-256); q0/v0 = offsets of the joint's
 * coordinates; pose = joint pose on the world, 12 doubles per body (R row-major, then t) or NULL for identity; mesh_body[mesh] = body. */
int pfc_set_bodies(pfc_ctx* ctx, int n_body, const int32_t* joint_type, const int32_t* q0, const int32_t* v0, const double* pose,
                   const int32_t* mesh_body, int nq, int nv);
/* forceAllElasticIntersections! including refreshBodyBodyTransform!/refreshBodyBodyCache! (src/contact_algorithms_non_friction.jl:103-134)
 * and addGeneralizedForcesThirdLaw! (:267-286), for n_env states x = [q; v; s] (stride nq + nv + 6 n_bristle, src/extensions.jl:21-50):
 *   f_generalized [env][nv]   sdot [env][bristle][6]   n_pairs / flags [env][ins] (may be NULL in the host version).  Host pointers. */
int pfc_eval_state_f64(pfc_ctx* ctx, int64_t n_env, const double* x, double* f_generalized, double* sdot, int64_t* n_pairs, int32_t* flags);
/* Same on device buffers, asynchronous on the context's stream (f_generalized must be zero-initialised for world-attached dofs). */
int pfc_eval_state_f64_device(pfc_ctx* ctx, int64_t n_env, const double* x, double* f_generalized, double* sdot, int64_t* n_pairs, int32_t* flags);
/* calcXd! (src/contact_algorithms_non_friction.jl:18-38) on the device for the same class of scenes: mass_matrix!, dynamics_bias!,
 * configuration_derivative!, forceAllElasticIntersections!, sum_all_forces! (:40-52) and the Cholesky solve.  pfc_set_dynamics (after
 * pfc_set_bodies): spatial_inertia[body][36] = the body's 6x6 spatial inertia about its origin in the body frame, row-major,
 * [angular; linear] ordering (newBodyFromInertia, src/body_inertia.jl:2-9; ignored for world-attached bodies); gravity[3] in the world frame
 * (src/mechanism_scenario.jl:184).  The mass matrix of such a scene is block diagonal and constant, so it is factored once, here. */
int pfc_set_dynamics(pfc_ctx* ctx, int n_body, const double* spatial_inertia, const double* gravity);
/* x[env][n_x] -> xdot[env][n_x] = [q_dot; v_dot; s_dot] (copyto!, src/extensions.jl:40-50).  tau_ext[env][nv] = external generalized
 * forces (the controller's tau_ext, :46-47) or NULL.  Host pointers; n_pairs / flags [env][ins] may be NULL. */
int pfc_calcxd_f64(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, double* xdot, int64_t* n_pairs, int32_t* flags);
/* Same on device buffers, asynchronous on the context's stream (xdot must be zero-initialised for world-attached coordinates). */
int pfc_calcxd_f64_device(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, double* xdot, int64_t* n_pairs, int32_t* flags);
/* calcXd! in Jacobian mode (Vector{Dual{Nothing,Float64,6}}: calcJacobian!, src/radau/radau_functions.jl:2-26) for the same scenes.
 * x[env][n_x] are Float64 states; the 6 Dual seeds sit on x[seed_start .. seed_start + 6) (seed_indices!, :16-26).  xdot7[env][n_x][7] =
 * value followed by the partials d xdot / d x[seed_start + k], k = 0..5 (write_indices!, :28-42, takes its columns of -J from them).
 * The candidate pairs come from the Float64 state, like the reference (:94-101).  Host pointers; tau_ext / n_pairs / flags may be NULL. */
int pfc_calcxd_dual6(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, int seed_start, double* xdot7, int64_t* n_pairs,
                     int32_t* flags);
/* Same on device buffers (none may be NULL except tau_ext), asynchronous on the context's stream; xdot7 must be zero-initialised for
 * world-attached coordinates. */
int pfc_calcxd_dual6_device(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, int seed_start, double* xdot7, int64_t* n_pairs,
                            int32_t* flags);
/* The whole Jacobian of calcXd! in one call (calcJacobian!, src/radau/radau_functions.jl:2-26: ceil(n_x / 6) Dual-6 passes of calcXd!).
 * jac[env][n_x][n_x], row-major: jac[env][i][j] = d xdot_i / d x_j (calcJacobian! stores its negative: J = -jac).  xdot[env][n_x] (may be
 * NULL) receives calcXd!(x) itself, the value part of the first pass.  The Float64 kinematics and the broad phase run once (the reference
 * repeats the traversal in every pass, on the same Float64 state: non_friction.jl:94-101) and the seed chunks run side by side as a grid
 * axis of the Dual kernels, so the result equals ceil(n_x / 6) calls of pfc_calcxd_dual6 bit for bit.  Host pointers; tau_ext / xdot /
 * n_pairs / flags may be NULL. */
int pfc_calcxd_jacobian(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, double* jac, double* xdot, int64_t* n_pairs,
                        int32_t* flags);
/* Same on device buffers (tau_ext and xdot may be NULL), asynchronous on the context's stream.  Every entry of jac / xdot is written. */
int pfc_calcxd_jacobian_device(pfc_ctx* ctx, int64_t n_env, const double* x, const double* tau_ext, double* jac, double* xdot, int64_t* n_pairs,
                               int32_t* flags);
/* Refit of one mesh after its vertices moved (same connectivity, same tree topology), on the device: rebuilds the mesh's primitive records
 * (triangle normals; inv([V; 1]) and the pressure gradient of every tetrahedron, src/contact_algorithms_non_friction.jl:145-164) and refits
 * every box of its tree with the construction rules of eMesh_to_tree (leaves: fit_tri_obb / fit_tet_obb, src/obb/obb_construction.jl; internal
 * nodes: OBB(a, b) of the children's axis-aligned boxes, src/obb/box_types.jl:11-15, bottom-up).  xyz[n_point][3] is a host pointer.
 * Returns PFC_E_MESH for a non-finite vertex or an inverted tetrahedron (src/obb/obb_construction.jl:30). */
int pfc_refit_mesh(pfc_ctx* ctx, int mesh_id, int64_t n_point, const double* xyz);

/* updateInvC! (src/radau/radau_functions.jl:88-99) for a batch: inv_c[m] = inverse(shift[m] I + neg_J[index ? index[m] : m]) for m < n_mat, where
 * neg_J[e] is the real n x n matrix -J of environment e (row-major), shift[m] = h^-1 lambda_stage as (re, im), and inv_c[m] is n x n complex,
 * row-major, interleaved (re, im) -- the layout of Julia's Matrix{ComplexF64} transposed / of a torch.complex128 tensor.  One CTA per matrix,
 * Gauss-Jordan with partial pivoting in shared memory.  *info (optional) gets bit 0 if a pivot vanished.  Device pointers; asynchronous. */
int pfc_radau_inv_c_device(pfc_ctx* ctx, int64_t n_mat, int n, const double* neg_J, const double* shift, const int32_t* index, double* inv_c,
                           int32_t* info);
/* Adaptive Radau IIA (src/radau) for n_env environments of a pfc_set_dynamics scene, every array on the device.
 * pfc_radau_init resets the per-environment controller to the reference's initial state (RadauStep / RadauRule, radau_struct.jl:64-95:
 * h = h0, rule 1, cooldown 10, Psi 9999) and sizes the buffers.  max_rule in 1..3 (NR; stages 2 rule - 1); n_x <= 96; tol_newton >= 0.
 * tol_a = tol_r = 1e-4, h_min = 1e-8, k_iter_max = 15 are the reference's constants.  The context owns the work space; the largest part is
 * the inverses (h^-1 lambda_i I - J)^-1: n_env (2 max_rule - 1) n_x^2 complex doubles -- 453 MB for 4096 environments of n_x = 48 at
 * max_rule = 2 -- besides the Jacobians (n_env n_x^2 doubles) and the stage states. */
int pfc_radau_init(pfc_ctx* ctx, int64_t n_env, int max_rule, double h0, double h_max, double tol_newton);
/* solveRadau (radau_solve.jl:1-34) for every environment: ONE accepted step each.  x[env][n_x] in/out (principal_value! applied to the
 * MRPs of SPQuatFloating bodies after the step), t[env] in/out, h_taken[env] out, tau_ext[env][nv] (held constant over the step) or NULL,
 * stats[env][4] (or NULL) = {stages of the accepted attempt, its Newton iterations, rejected attempts, stage evaluations over all attempts}.
 * An environment whose attempt fails retries with its own smaller h and rule while the others wait; the Jacobian is not recomputed for a
 * retry (radau_solve.jl:23-28).  Every environment takes the decisions the single-scene integrator would take for it alone, and its
 * result does not depend on the batch it is in.  Device pointers; the call synchronises the stream once per Newton iteration to read how
 * many (environment, stage) states are still active, and once per round of attempts; outputs are ready in stream order when it returns.
 * Returns PFC_E_STEP when an environment's step size falls below h_min (or becomes unacceptable), PFC_E_NONFINITE / PFC_E_CAPACITY as
 * pfc_calcxd_f64 does for the evaluations of the step; the outputs are then undefined. */
int pfc_radau_step_device(pfc_ctx* ctx, int64_t n_env, double* x, const double* tau_ext, double* t, double* h_taken, int32_t* stats);
/* Same on host pointers (copies in and out are part of the call). */
int pfc_radau_step(pfc_ctx* ctx, int64_t n_env, double* x, const double* tau_ext, double* t, double* h_taken, int32_t* stats);
/* A roll-out with a piecewise-constant tau_ext: every environment is advanced through the knot times t_knot[0..n_knot) (a HOST array,
 * shared by the batch, strictly increasing with gaps of at least h_min = 1e-8; t_knot[0] - t[env] >= h_min), tau_ext[k][env][nv] (or NULL)
 * acting on (t_knot[k-1], t_knot[k]].  Steps are pfc_radau_step's, from the controller state the context keeps, with one rule at the knots:
 * when h >= (t_knot[k] - t) - h_min the step is a knot step of exactly t_knot[k] - t (a rejected one retries with a smaller, ordinary h);
 * once accepted, t = t_knot[k] exactly, x (after principal_value!) is written to x_knot[k][env] (or nowhere if x_knot is NULL), and a
 * controller proposal of at least the knot step's h is raised back to the h the knot step replaced.  So no ordinary step leaves less than
 * h_min to a knot, and a roll-out through K knots equals K roll-outs through one knot each, bit for bit.  Environments go through their
 * knots independently; a round of steps takes the Jacobian of the environments still under way only.  max_steps >= 1 bounds each
 * environment's accepted steps: one that exhausts it stops where it is, its unreached x_knot rows are NaN, and the call returns PFC_OK.
 * x[env][n_x] and t[env] in/out; stats[env][4] (or NULL) = {knots reached, accepted steps, rejected attempts, stage evaluations} of the call.
 * PFC_E_ARG (nothing modified) for a bad knot array, max_steps < 1, an n_env other than pfc_radau_init's, or an environment that starts
 * less than h_min before t_knot[0] (checked on the device before the first step); otherwise the errors of pfc_radau_step.  Device pointers
 * except t_knot; one more host synchronisation per round of steps. */
int pfc_radau_rollout_device(pfc_ctx* ctx, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps, double* x, const double* tau_ext,
                             double* t, double* x_knot, int32_t* stats);
/* Same on host pointers. */
int pfc_radau_rollout(pfc_ctx* ctx, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps, double* x, const double* tau_ext, double* t,
                      double* x_knot, int32_t* stats);
/* Of the last pfc_radau_step[_device] or pfc_radau_rollout[_device] call (sums over a roll-out's steps): counts[0] = rounds of attempts,
 * counts[1] = host synchronisations; ms[0..3] = device time of the Jacobian, the stage evaluations, the inverses, and the Newton +
 * controller kernels (CUDA events; zeros unless pfc_set_timing is on).  Either pointer may be NULL. */
int pfc_radau_step_info(pfc_ctx* ctx, double* ms, int64_t* counts);
/* Debug / parity: the boundary arrays (X_r2_r1, twist_r2) the prologue computed and the per-instruction wrenches of the last
 * host-pointer evaluation; any pointer may be NULL. */
int pfc_get_boundary(pfc_ctx* ctx, int64_t n_env, double* X_r2_r1, double* twist_r2, double* wrench_r2);

/* Debug / parity: keep the candidate-pair lists (TT_Cache, src/obb/tree_types.jl:32-50) of subsequent evaluations. */
int pfc_set_debug(pfc_ctx* ctx, int keep_pairs);
/* Pair list of (env, ins) from the last evaluation, in the reference's traversal order: pairs[2k] = primitive of mesh_1, pairs[2k+1] = of mesh_2. */
int pfc_get_pairs(pfc_ctx* ctx, int64_t env, int ins, int32_t* pairs, int64_t cap, int64_t* n_out);
/* TractionCache (src/mechanism_scenario.jl:51-58) of (env, ins) from the last evaluation: 8 doubles per point: n(3), r_cart(3), dA, p. */
int pfc_get_traction(pfc_ctx* ctx, int64_t env, int ins, double* out, int64_t cap_points, int64_t* n_out);

/* Multi-GPU for one very large scene: this context traverses, lists and evaluates only the sub-trees of every large REGULARIZED
 * instruction's dual-tree recursion whose hash falls on `rank` of `world` (disjoint pair lists, no exchange before the sums); the partial
 * sums are then reduced over the ranks.  Bristle instructions are never split: their sums run sequentially over the whole TractionCache
 * list (the reference's order, src/contact_algorithms_friction.jl:147-201), so every rank lists and evaluates them completely and ends with
 * identical bits.  pfc_get_pairs returns this rank's part of a split list. */
int pfc_set_shard(pfc_ctx* ctx, int rank, int world);
/* Sharded evaluation protocol (device pointers; see INTEGRATION.md):
 *   begin:    breadth-first levels (every rank), this rank's share of the traversal, sort, narrow phase over its own pairs;
 *   partials: the buffer the caller must sum over all ranks in place: count doubles (8 per (env, large instruction): 6 wrench sums,
 *             traction-point count, pair count);
 *   step:     applies the summed buffer (wrench, counts, flags); *more is always 0 (one exchange per evaluation). */
int pfc_eval_sharded_begin(pfc_ctx* ctx, int64_t n_env, const double* X_r2_r1, const double* twist_r2, const double* s, double* wrench_r2,
                           double* sdot, int64_t* n_pairs, int32_t* flags);
int pfc_eval_sharded_partials(pfc_ctx* ctx, double** dev_ptr, int64_t* count);
int pfc_eval_sharded_step(pfc_ctx* ctx, int* more);

/* The same evaluation with the exchange done by the library (SURVEY.md section 8b "pfc_group"): a Julia caller cannot issue NCCL calls, so
 * the library owns the communicator.  The ranks' partial sums are ALL-GATHERED over NCCL (NVLink / NVSwitch) and added in rank order on
 * every rank, so all ranks -- and repeated runs -- end with the same bits (an all-reduce leaves the association to the collective).
 * NCCL is resolved at run time (dlopen of libnccl.so.2: the copy the host program already loaded, else the system's).
 *
 * One process per GPU (MPI / torchrun-style launchers): rank 0 calls pfc_comm_unique_id and hands the 128 bytes to the other ranks by any
 * means; every rank then calls pfc_comm_init_rank (which also makes the context rank `rank` of `world`, like pfc_set_shard) and evaluates
 * with pfc_eval_sharded_f64_device (device pointers, as pfc_eval_sharded_begin; queued on the context's stream after one
 * synchronisation for the buffer check; every rank ends with the full wrenches, counts and flags). */
int pfc_comm_unique_id(void* id128);
int pfc_comm_init_rank(pfc_ctx* ctx, const void* id128, int rank, int world);
int pfc_eval_sharded_f64_device(pfc_ctx* ctx, int64_t n_env, const double* X_r2_r1, const double* twist_r2, const double* s, double* wrench_r2,
                                double* sdot, int64_t* n_pairs, int32_t* flags);
/* One process, several GPUs (what a single Julia process drives): pfc_group_create makes one context per listed device and one
 * communicator over them (ncclCommInitAll).  The scene is described once -- pfc_group_add_mesh / _add_instruction / _finalize forward to
 * every context -- and pfc_group_eval_f64 is forceAllElasticIntersections! with the large instructions' candidate-pair lists split over
 * the devices (host pointers in and out, exactly like pfc_eval_f64; synchronous at return).  pfc_group_ctx(g, r) is device r's context
 * (e.g. for pfc_get_pairs, which returns that rank's part of a split list). */
int pfc_group_create(int n_dev, const int* devices, pfc_group** out);
int pfc_group_destroy(pfc_group* g);
int pfc_group_size(pfc_group* g);
pfc_ctx* pfc_group_ctx(pfc_group* g, int rank);
int pfc_group_add_mesh(pfc_group* g, int kind, int64_t n_point, const double* xyz, int64_t n_prim, const int32_t* idx, const double* eps, double Ebar,
                       int64_t n_node, const double* node_c, const double* node_e, const double* node_R, const int32_t* node_left,
                       const int32_t* node_right, const int32_t* node_leaf_id, int* mesh_id_out);
int pfc_group_add_instruction(pfc_group* g, int mesh_1, int mesh_2, double chi, int model, const double* params, int n_quad_rule, int* ins_id_out);
int pfc_group_finalize(pfc_group* g, int64_t max_env);
int pfc_group_eval_f64(pfc_group* g, int64_t n_env, const double* X_r2_r1, const double* twist_r2, const double* s, double* wrench_r2, double* sdot,
                       int64_t* n_pairs, int32_t* flags);

/* Plumbing */
int pfc_sync(pfc_ctx* ctx);
void* pfc_stream(pfc_ctx* ctx);            /* the cudaStream_t kernels are launched on (for CUDA-event timing) */
int64_t pfc_launch_count(pfc_ctx* ctx);   /* kernels launched by this context so far */
/* Per-kernel device timing (CUDA events on the context's stream): enable, evaluate, then read the durations in
 * milliseconds of the last evaluation: ms[0] = broad-phase kernel, ms[1] = narrow-phase/friction/reduction kernel. */
int pfc_set_timing(pfc_ctx* ctx, int on);
int pfc_kernel_times(pfc_ctx* ctx, double* ms, int n);
/* FP64 (DFMA) throughput of the context's device in TFLOP/s: the roofline denominator of the clip/quadrature kernels. */
int pfc_measure_fp64_peak(pfc_ctx* ctx, double* tflops);
int pfc_counters(pfc_ctx* ctx, int64_t* n_node_pairs_tested, int64_t* n_candidate_pairs);
const char* pfc_last_error(void);
const char* pfc_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PFC_H */
