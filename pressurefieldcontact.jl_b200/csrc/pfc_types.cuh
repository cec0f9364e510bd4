// pfc_types.cuh -- device-resident scene layout (uploaded once by pfc_finalize).
//
// What the reference keeps in MeshCache / bin_BB_Tree / ContactInstructions
// (/root/reference/src/structs.jl:33-54, src/obb/tree_types.jl:1-16,
// src/mechanism_scenario.jl:36-49) is flattened into three record arrays shared by all meshes:
//   NodeRec  128 B per tree node   (box + child links; one 128 B line per node visit)
//   TetRec   256 B per tetrahedron (vertices, inverse of [V;1], pressure gradient)
//   TriRec    96 B per triangle    (vertices, unit normal)
// The per-tet 4x4 inverse and eps gradient are per-primitive constants that the reference
// recomputes for every candidate pair (src/contact_algorithms_non_friction.jl:150-162); here they
// are computed once at upload.
#pragma once
#include <cstdint>

namespace pfc {

// Trees are stored PRE-ORDER (pfc_add_mesh re-flattens them), so child 1 of an internal node is the next record and needs no link.
// Internal nodes are axis-aligned boxes merged from their children (R = I, src/obb/box_types.jl:11-15); only leaves carry a fitted
// rotation.  The first 64 B of a record hold everything an axis-aligned node needs: the traversal loads the second half (the rest of
// R) only for nodes whose kind says the rotation is not the identity.
enum { kNodeLeaf = -1, kNodeInternal = 0, kNodeInternalAabb = 1 };
struct NodeRec {
    double c[3];
    double e[3];
    int32_t kind;  // kNodeLeaf, or kNodeInternal / kNodeInternalAabb (R == I exactly); child 1 of an internal node is this node + 1
    int32_t right; // mesh-local node index of child 2, or the 0-based primitive id for a leaf
    double R[9];   // row-major: R[3*i+j]
};
static_assert(sizeof(NodeRec) == 128, "NodeRec must be one 128 B line");

struct TetRec {
    double v[12];     // v[3*k + c]: vertex k (columns of x_r_zeta)
    double inv[16];   // row-major x_zeta_r: zeta_i = inv[4i+0] x + inv[4i+1] y + inv[4i+2] z + inv[4i+3]
    double eps_r[4];  // eps * x_zeta_r: pressure-field gradient (0..2) and offset (3)
};
static_assert(sizeof(TetRec) == 256, "TetRec must be 256 B");

struct TriRec {
    double v[9];  // v[3*k + c]
    double n[3];  // triangleNormal in the mesh frame
};

enum { PFC_MODEL_REGULARIZED = 0, PFC_MODEL_BRISTLE = 1 };

struct InsDev {
    int32_t kind1;       // 0 = Tri, 1 = Tet (mesh_2 is always Tet)
    int32_t model;
    int32_t n_quad;      // 1 or 3 quadrature points per sub-triangle
    int32_t bristle_id;  // -1 for regularized
    int32_t node_base1, node_base2; // first node of each mesh in the node array (the root: trees are stored pre-order)
    int32_t prim_base1, prim_base2; // offsets into the tri / tet record arrays
    int32_t path_base1, path_base2; // offsets into the per-primitive leaf path / depth tables (large path)
    int32_t n_leaf1, n_leaf2;
    int32_t small;       // 1: handled by the fused warp-per-instruction kernel
    int32_t key_bits;    // max DFS-key length (depth1 + depth2) for the large path's sort
    double chi, Ebar1, Ebar2;
    // regularized: mu_s, mu_d, v_c, v_mu_s, v_mu_d, slope = (mu_d - mu_s) / (v_mu_d - v_mu_s), 1 / v_c
    // bristle:     tau, k_bar, mu_s, mu_d, Ts_mu_s, Ts_mu_d, magic, slope = (mu_d - mu_s) / (Ts_mu_d - Ts_mu_s)
    double p[8];
};

// The contact parameters of one instruction in one environment (pfc_set_contact_params): the fields InsDev ends with, derived by the same
// host code.  A table of rows [env][ins], passed to the kernels as an optional pointer (nullptr: every environment uses the InsDev values).
struct InsParam {
    double chi, Ebar1, Ebar2;
    double p[8];
};

// flags written per (env, instruction)
enum { kFlagContact = 1, kFlagNonFinite = 2, kFlagBadArity = 4, kFlagOverflow = 8 };  // == PFC_FLAG_* of include/pfc.h

// everything a kernel needs to find the static scene
struct SceneDev {
    const NodeRec* nodes;
    const TetRec* tets;
    const TriRec* tris;
    const InsDev* ins;
    const int32_t* small_ins;  // indices of the instructions on the fused small path
    const int32_t* small_heavy_first;  // the same instructions ordered by n_leaf1 * n_leaf2, largest first (broad-phase scheduling order)
    int32_t n_ins, n_small, n_bristle;
    int32_t n_small_bristle;   // bristle instructions among the small ones (selects the narrow-phase kernel)
    int32_t* ins_overflow;     // per instruction: set when a small-path pair-list / frontier slot was too small (nullptr when none can be)
    int32_t small_node_lo, small_node_n;  // range of the node array that holds the trees of the small instructions (staged in shared memory when it fits)
};

}  // namespace pfc
