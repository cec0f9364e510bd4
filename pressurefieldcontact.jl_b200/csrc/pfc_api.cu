// pfc_api.cu -- the C ABI of include/pfc.h: scene container, one-time upload, evaluation entry points.
#include <dlfcn.h>
#include <nccl.h>   // declarations only: the library is loaded at run time (nccl_api), so libpfc_b200.so has no link-time dependency on it

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "../../include/pfc.h"
#include "pfc_exact.h"
#include "pfc_large.h"
#include "pfc_launch.h"
#include "pfc_radau_step.cuh"

using namespace pfc;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) return fail(e_ == cudaErrorMemoryAllocation ? PFC_E_CAPACITY : PFC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

struct HostMesh {
    int kind;
    int64_t n_point, n_prim;
    std::vector<double> xyz, eps;
    std::vector<int32_t> idx;
    double Ebar;
    std::vector<NodeRec> nodes;  // pre-order, mesh-local links
    std::vector<int32_t> leaf_depth;     // per primitive: depth of its leaf node
    std::vector<uint64_t> leaf_path;     // per primitive: root-to-leaf turns, MSB-first in the low `depth` bits
    int depth;                           // max leaf depth
    int node_base, prim_base, path_base;
};

struct HostIns {
    int mesh_1, mesh_2, model, n_quad_rule, bristle_id;
    double chi, params[5];
};

// ---- NCCL, resolved at run time ------------------------------------------------------------------------------------------------
// dlopen("libnccl.so.2") picks up the copy a host program has already loaded (PyTorch ships its own under the same soname), else
// the system's.  Only what the per-instruction partial sums of a split scene need: communicator set-up and all-gather.
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string error;
    bool ok() const { return handle && error.empty(); }
};
NcclApi& nccl_api() {
    static NcclApi a = [] {
        NcclApi n;
        n.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!n.handle) n.handle = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!n.handle) { n.error = std::string("NCCL is not available: ") + dlerror(); return n; }
        auto sym = [&](const char* name) { void* p = dlsym(n.handle, name); if (!p && n.error.empty()) n.error = std::string("NCCL symbol missing: ") + name; return p; };
        n.GetUniqueId = reinterpret_cast<decltype(n.GetUniqueId)>(sym("ncclGetUniqueId"));
        n.CommInitRank = reinterpret_cast<decltype(n.CommInitRank)>(sym("ncclCommInitRank"));
        n.CommInitAll = reinterpret_cast<decltype(n.CommInitAll)>(sym("ncclCommInitAll"));
        n.CommDestroy = reinterpret_cast<decltype(n.CommDestroy)>(sym("ncclCommDestroy"));
        n.AllGather = reinterpret_cast<decltype(n.AllGather)>(sym("ncclAllGather"));
        n.GroupStart = reinterpret_cast<decltype(n.GroupStart)>(sym("ncclGroupStart"));
        n.GroupEnd = reinterpret_cast<decltype(n.GroupEnd)>(sym("ncclGroupEnd"));
        n.GetErrorString = reinterpret_cast<decltype(n.GetErrorString)>(sym("ncclGetErrorString"));
        return n;
    }();
    return a;
}
#define NC(call)                                                                                                               \
    do {                                                                                                                       \
        ncclResult_t r_ = (call);                                                                                              \
        if (r_ != ncclSuccess) return fail(PFC_E_CUDA, std::string(#call) + ": " + nccl_api().GetErrorString(r_));            \
    } while (0)

// out[i] = ((g[0][i] + g[1][i]) + g[2][i]) + ... : the ranks' partial sums added in RANK ORDER on every rank, so all ranks end with the
// same bits whatever order the network delivered them in (an all-reduce leaves the association to the collective's algorithm)
__global__ void sum_ranks_kernel(const double* __restrict__ gathered, int world, long long count, double* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        double a = gathered[i];
        for (int r = 1; r < world; ++r) a += gathered[(long long)r * count + i];
        out[i] = a;
    }
}

template <class T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
    ~DevBuf() { release(); }   // every buffer a context owns goes with it (pfc_destroy deletes the context on its device)
    cudaError_t ensure(size_t count) {
        if (count <= n) return cudaSuccess;
        alloc_generation()++;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

}  // namespace

struct pfc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;                 // bristle pipeline beside the regularized narrow phase (eval_device_once)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool finalized = false;
    std::vector<HostMesh> mesh;
    std::vector<HostIns> ins;
    int n_bristle = 0;
    int64_t max_env = 0;
    // static scene on the device
    DevBuf<NodeRec> d_nodes;
    DevBuf<TetRec> d_tets;
    DevBuf<TriRec> d_tris;
    DevBuf<InsDev> d_ins;
    DevBuf<int32_t> d_small;
    DevBuf<int32_t> d_small_heavy;
    std::vector<InsDev> h_ins;
    SceneDev scene{};
    // per-batch staging (host-pointer entry points)
    DevBuf<double> d_X, d_tw, d_s, d_w, d_sd;
    DevBuf<long long> d_np;
    DevBuf<int> d_fl;
    // debug
    bool keep_pairs = false;
    DevBuf<int> d_dbg_pairs;
    int dbg_cap = 0;
    int64_t dbg_n_env = 0;
    DevBuf<long long> d_last_np;   // n_pairs of the last evaluation (device copy kept for get_pairs)
    const double* last_X = nullptr; const double* last_tw = nullptr;  // device pointers of the last evaluation
    int64_t launches = 0;
    int shard_rank = 0, shard_world = 1;
    int small_max_pairs = 1;
    int n_mid = 0;                       // instructions on the small path whose pair-list slot can overflow (see build_tables)
    std::vector<char> force_large;       // instructions moved to the large path after such an overflow
    DevBuf<int> d_ins_overflow;
    int* h_ins_overflow = nullptr;       // pinned
    bool mid_check_pending = false;
    DevBuf<unsigned> d_small_pairs;  // broad -> narrow pair lists of the small path: [env][ins][cap]
    // large path
    DevBuf<int32_t> d_large;
    DevBuf<unsigned long long> d_leaf_path;
    DevBuf<unsigned char> d_leaf_depth;
    LargeScene large_scene{};
    LargeBuffers* large_buf = nullptr;
    std::vector<int32_t> large_ins_host;
    // reference-order pipeline of the bristle instructions (pfc_exact.cu)
    DevBuf<double> d_tet_eps;
    DevBuf<int32_t> d_bris_ins;
    ExactScene exact_scene{};
    ExactBuffers* exact_buf = nullptr;
    bool has_large_bristle = false;
    // CUDA graph of the last evaluation's launch sequence (scenes with large / bristle instructions queue dozens of short kernels)
    struct GraphCache {
        cudaGraphExec_t exec = nullptr;
        unsigned long long key = 0, gen = ~0ull;   // what was evaluated (entry point, batch size, buffers) and the allocation generation then
        bool seen = false;                          // the same evaluation ran eagerly once: everything it needs is allocated
        int launches = 0;
        bool disabled = false;
    } graph, graph_host, graph_pack;   // graph: one device-level evaluation of a many-kernel scene; graph_host: a whole host-pointer call of a small-path scene
    ncclComm_t comm = nullptr;   // library-owned communicator of a split scene (pfc_comm_init_rank / pfc_group_create)
    DevBuf<double> d_gather;     // [world][count]: the ranks' partial sums after the all-gather
    int sharded_stage = -1;   // >= 0 while a sharded evaluation is in flight
    EvalIO sharded_io{};
    // Jacobian mode staging + the pair lists it may reuse
    DevBuf<double> d_X7, d_tw7, d_s7, d_w7, d_sd7, d_jac;
    DevBuf<unsigned> d_dual_ticket;   // tile ticket of the Dual kernel
    DevBuf<unsigned> d_surv;          // Jacobian mode: pairs that survive the Float64 clip [env][ins][cap]
    DevBuf<int> d_surv_n;
    DevBuf<int32_t> d_large_index;
    int64_t lists_n_env = -1;   // n_env of the evaluation whose pair lists (d_small_pairs / large_buf, lists_np, lists_fl) are current
    long long* lists_np = nullptr;   // where that evaluation left its pair counts / flags (d_np / d_fl, or the packed block of a small call)
    int* lists_fl = nullptr;
    DevBuf<unsigned char> d_pack_in, d_pack_out;   // small host-pointer calls: all inputs / all outputs in one block each (one copy each way)
    // device-side kinematics (pfc_set_bodies / pfc_eval_state_f64)
    bool has_bodies = false;
    std::vector<BodyDev> h_bodies;
    std::vector<int> h_mesh_body;
    DevBuf<BodyDev> d_bodies;
    DevBuf<int> d_ins_body, d_body_ins_ptr, d_body_ins;
    StateDev state{};
    DevBuf<double> d_x, d_fgen;
    // device-side calcXd! (pfc_set_dynamics / pfc_calcxd_f64)
    bool has_dynamics = false;
    DevBuf<double> d_H, d_Hinv, d_xdot, d_tau;
    DevBuf<int> d_status;       // OR of the error flag bits of a state-level evaluation
    // device-side refit (pfc_refit_mesh): per mesh, built on first use
    struct RefitDev { DevBuf<int> idx; DevBuf<double> eps; DevBuf<int> level_nodes; std::vector<int> level_ptr; bool ready = false; };
    std::vector<RefitDev> refit;
    DevBuf<double> d_refit_xyz, d_refit_aabb;
    // pinned staging arena for small host-pointer calls (a single scene moves a few hundred bytes per array: copying through pinned
    // memory keeps every cudaMemcpyAsync truly asynchronous instead of the driver's staged, synchronising path for pageable memory)
    unsigned char* h_arena = nullptr;
    size_t arena_cap = 0, arena_used = 0;
    struct PendingOut { void* dst; const void* src; size_t bytes; };
    std::vector<PendingOut> arena_out;
    bool large_index_dirty = true;
    int* h_status = nullptr;    // pinned
    DynDev dyn{};
    // batched Radau step (pfc_radau_init / pfc_radau_step): controller state and work space for radau_n_env environments
    struct RadauState {
        int64_t n_env = -1;
        int max_rule = 0, s_max = 0;
        double h_max = 0.0, tol_newton = 0.0;
        DevBuf<RadauEnv> env;
        DevBuf<double> X, Xp, Fp, taup, xx0, jac, invc, shift, x, tau, t, h;
        DevBuf<InsParam> paramp, params_c;   // contact-parameter rows gathered per stage state / per compact roll-out slot: grown on first use
        DevBuf<int> index, state_list, env_list, state_pos, inv_base, counts, stats, flags, flags_stage, info;
        DevBuf<long long> np, np_stage;
        // roll-outs (pfc_radau_rollout): grown on first use
        DevBuf<RadauEnv> env_c;
        DevBuf<double> knots, x_c, tau_c, t_c, h_c, h_save, x_knot;
        DevBuf<int> knot, steps, ro_stats, list, stats_c, ro_count;
        int* h_counts = nullptr;   // pinned: counts[0..3] + the status word; [5..6] a roll-out's ro_count
        int64_t rounds = 0, syncs = 0;   // of the last step or roll-out
        double ms[4] = {0, 0, 0, 0};     // of the last step or roll-out with pfc_set_timing on: Jacobian, stage evaluations, inverses, Newton + controller
        std::vector<cudaEvent_t> ev_pool;
    } radau;
    bool timing = false;
    cudaEvent_t ev[8] = {};
    bool ev_valid = false;
    // per-environment contact parameters (pfc_set_contact_params): rows [env][ins]; params_n_env = 0 while no table is set
    DevBuf<InsParam> d_params;
    int64_t params_n_env = 0;
    const InsParam* last_params = nullptr;   // the table the last evaluation read (pfc_get_traction re-runs its narrow phase)
};

namespace {

// inverse of A = [v0 v1 v2 v3; 1 1 1 1] (columns are the homogeneous vertices): the explicit adjugate / determinant formula for a 4x4
// (what StaticArrays' inv(::SMatrix{4,4}) amounts to; the reference inverts per candidate pair, src/contact_algorithms_non_friction.jl:158-162).
// The expression order is fixed -- every cofactor as a left-to-right sum of triple products of the column-major entries m[], then one
// division and 16 scalings -- because the reference-order bristle path (pfc_exact.cuh) reproduces the reference's K matrix bit for bit
// from these per-tetrahedron constants.  Row-major output.
bool invert_tet_matrix(const double v[12], double out[16]) {
    double m[16];  // column-major: m[4*c + r]
    for (int c = 0; c < 4; ++c) { m[4 * c] = v[3 * c]; m[4 * c + 1] = v[3 * c + 1]; m[4 * c + 2] = v[3 * c + 2]; m[4 * c + 3] = 1.0; }
    double inv[16];
    inv[0] = m[5] * m[10] * m[15] - m[5] * m[11] * m[14] - m[9] * m[6] * m[15] + m[9] * m[7] * m[14] + m[13] * m[6] * m[11] - m[13] * m[7] * m[10];
    inv[4] = -m[4] * m[10] * m[15] + m[4] * m[11] * m[14] + m[8] * m[6] * m[15] - m[8] * m[7] * m[14] - m[12] * m[6] * m[11] + m[12] * m[7] * m[10];
    inv[8] = m[4] * m[9] * m[15] - m[4] * m[11] * m[13] - m[8] * m[5] * m[15] + m[8] * m[7] * m[13] + m[12] * m[5] * m[11] - m[12] * m[7] * m[9];
    inv[12] = -m[4] * m[9] * m[14] + m[4] * m[10] * m[13] + m[8] * m[5] * m[14] - m[8] * m[6] * m[13] - m[12] * m[5] * m[10] + m[12] * m[6] * m[9];
    inv[1] = -m[1] * m[10] * m[15] + m[1] * m[11] * m[14] + m[9] * m[2] * m[15] - m[9] * m[3] * m[14] - m[13] * m[2] * m[11] + m[13] * m[3] * m[10];
    inv[5] = m[0] * m[10] * m[15] - m[0] * m[11] * m[14] - m[8] * m[2] * m[15] + m[8] * m[3] * m[14] + m[12] * m[2] * m[11] - m[12] * m[3] * m[10];
    inv[9] = -m[0] * m[9] * m[15] + m[0] * m[11] * m[13] + m[8] * m[1] * m[15] - m[8] * m[3] * m[13] - m[12] * m[1] * m[11] + m[12] * m[3] * m[9];
    inv[13] = m[0] * m[9] * m[14] - m[0] * m[10] * m[13] - m[8] * m[1] * m[14] + m[8] * m[2] * m[13] + m[12] * m[1] * m[10] - m[12] * m[2] * m[9];
    inv[2] = m[1] * m[6] * m[15] - m[1] * m[7] * m[14] - m[5] * m[2] * m[15] + m[5] * m[3] * m[14] + m[13] * m[2] * m[7] - m[13] * m[3] * m[6];
    inv[6] = -m[0] * m[6] * m[15] + m[0] * m[7] * m[14] + m[4] * m[2] * m[15] - m[4] * m[3] * m[14] - m[12] * m[2] * m[7] + m[12] * m[3] * m[6];
    inv[10] = m[0] * m[5] * m[15] - m[0] * m[7] * m[13] - m[4] * m[1] * m[15] + m[4] * m[3] * m[13] + m[12] * m[1] * m[7] - m[12] * m[3] * m[5];
    inv[14] = -m[0] * m[5] * m[14] + m[0] * m[6] * m[13] + m[4] * m[1] * m[14] - m[4] * m[2] * m[13] - m[12] * m[1] * m[6] + m[12] * m[2] * m[5];
    inv[3] = -m[1] * m[6] * m[11] + m[1] * m[7] * m[10] + m[5] * m[2] * m[11] - m[5] * m[3] * m[10] - m[9] * m[2] * m[7] + m[9] * m[3] * m[6];
    inv[7] = m[0] * m[6] * m[11] - m[0] * m[7] * m[10] - m[4] * m[2] * m[11] + m[4] * m[3] * m[10] + m[8] * m[2] * m[7] - m[8] * m[3] * m[6];
    inv[11] = -m[0] * m[5] * m[11] + m[0] * m[7] * m[9] + m[4] * m[1] * m[11] - m[4] * m[3] * m[9] - m[8] * m[1] * m[7] + m[8] * m[3] * m[5];
    inv[15] = m[0] * m[5] * m[10] - m[0] * m[6] * m[9] - m[4] * m[1] * m[10] + m[4] * m[2] * m[9] + m[8] * m[1] * m[6] - m[8] * m[2] * m[5];
    const double det = m[0] * inv[0] + m[1] * inv[4] + m[2] * inv[8] + m[3] * inv[12];
    if (!(det != 0.0) || !std::isfinite(det)) return false;
    const double idet = 1.0 / det;
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) out[4 * r + c] = inv[4 * c + r] * idet;   // column-major adjugate -> row-major inverse
    return true;
}

double tet_volume6(const double v[12]) {  // 6 * signed volume, positive for the reference's orientation
    const double* a = v; const double* b = v + 3; const double* c = v + 6; const double* d = v + 9;
    double V = (b[0] - a[0]) * (c[1] * d[2] - c[2] * d[1]);
    V += (b[1] - a[1]) * (c[2] * d[0] - c[0] * d[2]);
    V += (b[2] - a[2]) * (c[0] * d[1] - c[1] * d[0]);
    V += (c[0] - d[0]) * (a[2] * b[1] - a[1] * b[2]);
    V += (c[1] - d[1]) * (a[0] * b[2] - a[2] * b[0]);
    V += (c[2] - d[2]) * (a[1] * b[0] - a[0] * b[1]);
    return V;
}

}  // namespace

extern "C" {

const char* pfc_last_error(void) { return g_err.c_str(); }
const char* pfc_version(void) { return "pfc-b200 0.1 (sm_100a)"; }

int pfc_create(int device, pfc_ctx** out) {
    if (!out) return fail(PFC_E_ARG, "pfc_create: out is NULL");
    int n_dev = 0;
    CU(cudaGetDeviceCount(&n_dev));
    if (device < 0 || device >= n_dev) return fail(PFC_E_ARG, "pfc_create: no such CUDA device");
    CU(cudaSetDevice(device));
    pfc_ctx* c = new pfc_ctx();
    c->device = device;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { delete c; return fail(PFC_E_CUDA, cudaGetErrorString(e)); }
    *out = c;
    return PFC_OK;
}

int pfc_destroy(pfc_ctx* c) {
    if (!c) return PFC_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->graph.exec) { cudaGraphExecDestroy(c->graph.exec); c->graph.exec = nullptr; }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->stream2) cudaStreamDestroy(c->stream2);
    if (c->graph_host.exec) { cudaGraphExecDestroy(c->graph_host.exec); c->graph_host.exec = nullptr; }
    if (c->graph_pack.exec) { cudaGraphExecDestroy(c->graph_pack.exec); c->graph_pack.exec = nullptr; }
    if (c->comm && nccl_api().ok()) { nccl_api().CommDestroy(c->comm); c->comm = nullptr; }
    if (c->stream) cudaStreamDestroy(c->stream);
    c->d_nodes.release(); c->d_tets.release(); c->d_tris.release(); c->d_ins.release(); c->d_small.release(); c->d_small_heavy.release();
    c->d_X.release(); c->d_tw.release(); c->d_s.release(); c->d_w.release(); c->d_sd.release(); c->d_np.release(); c->d_fl.release();
    c->d_dbg_pairs.release(); c->d_last_np.release(); c->d_small_pairs.release();
    c->d_H.release(); c->d_Hinv.release(); c->d_xdot.release(); c->d_tau.release(); c->d_status.release(); c->d_refit_xyz.release(); c->d_refit_aabb.release();
    for (auto& r : c->refit) { r.idx.release(); r.eps.release(); r.level_nodes.release(); }
    if (c->h_status) { cudaFreeHost(c->h_status); c->h_status = nullptr; }
    if (c->radau.h_counts) { cudaFreeHost(c->radau.h_counts); c->radau.h_counts = nullptr; }
    for (cudaEvent_t ev : c->radau.ev_pool) cudaEventDestroy(ev);
    if (c->h_ins_overflow) { cudaFreeHost(c->h_ins_overflow); c->h_ins_overflow = nullptr; }
    if (c->h_arena) { cudaFreeHost(c->h_arena); c->h_arena = nullptr; }
    for (int k = 0; k < 8; ++k) if (c->ev[k]) cudaEventDestroy(c->ev[k]);
    c->d_large.release(); c->d_leaf_path.release(); c->d_leaf_depth.release();
    c->d_X7.release(); c->d_tw7.release(); c->d_s7.release(); c->d_w7.release(); c->d_sd7.release(); c->d_large_index.release();
    large_buffers_destroy(c->large_buf);
    exact_buffers_destroy(c->exact_buf);
    delete c;
    return PFC_OK;
}

int pfc_add_mesh(pfc_ctx* c, int kind, int64_t n_point, const double* xyz, int64_t n_prim, const int32_t* idx, const double* eps, double Ebar,
                 int64_t n_node, const double* node_c, const double* node_e, const double* node_R, const int32_t* node_left,
                 const int32_t* node_right, const int32_t* node_leaf_id, int* mesh_id_out) {
    if (!c || c->finalized) return fail(PFC_E_ARG, "pfc_add_mesh: context missing or already finalized");
    if (kind != 0 && kind != 1) return fail(PFC_E_ARG, "pfc_add_mesh: kind must be 0 (tri) or 1 (tet)");
    if (!xyz || !idx || n_point <= 0 || n_prim <= 0) return fail(PFC_E_ARG, "pfc_add_mesh: empty mesh");
    if (kind == 1 && !eps) return fail(PFC_E_ARG, "pfc_add_mesh: tet mesh needs eps");
    if (n_node != 2 * n_prim - 1) return fail(PFC_E_MESH, "pfc_add_mesh: a binary tree over n_prim leaves has 2 n_prim - 1 nodes");
    const int w = kind == 0 ? 3 : 4;
    HostMesh m;
    m.kind = kind; m.n_point = n_point; m.n_prim = n_prim; m.Ebar = Ebar;
    m.xyz.assign(xyz, xyz + 3 * n_point);
    m.idx.assign(idx, idx + w * n_prim);
    if (kind == 1) m.eps.assign(eps, eps + n_point);
    for (int64_t k = 0; k < w * n_prim; ++k)
        if (idx[k] < 0 || idx[k] >= n_point) return fail(PFC_E_MESH, "pfc_add_mesh: vertex index out of range");
    // re-flatten the tree in pre-order from node 0, recording each leaf's root-to-leaf path
    m.nodes.resize(n_node);
    m.leaf_depth.assign(n_prim, -1);
    m.leaf_path.assign(n_prim, 0);
    m.depth = 0;
    struct Item { int32_t src; int32_t parent_dst; int side; int depth; uint64_t path; };
    std::vector<Item> stack;
    stack.push_back({0, -1, 0, 0, 0});
    int32_t next = 0;
    std::vector<char> seen(n_node, 0);
    while (!stack.empty()) {
        Item it = stack.back();
        stack.pop_back();
        if (it.src < 0 || it.src >= n_node || seen[it.src]) return fail(PFC_E_MESH, "pfc_add_mesh: tree links are not a tree");
        seen[it.src] = 1;
        const int32_t dst = next++;
        NodeRec& nd = m.nodes[dst];
        for (int i = 0; i < 3; ++i) {
            nd.c[i] = node_c[3 * it.src + i];
            nd.e[i] = node_e[3 * it.src + i];
            for (int j = 0; j < 3; ++j) nd.R[3 * i + j] = node_R[9 * it.src + 3 * j + i];  // column-major in, row-major stored
        }
        if (it.parent_dst >= 0) {   // pre-order: child 1 is the record after its parent (no link stored), child 2 is linked
            if (it.side == 0) { if (dst != it.parent_dst + 1) return fail(PFC_E_MESH, "pfc_add_mesh: internal error (pre-order)"); }
            else m.nodes[it.parent_dst].right = dst;
        }
        const int32_t leaf = node_leaf_id[it.src];
        if (leaf >= 0) {
            if (leaf >= n_prim || m.leaf_depth[leaf] >= 0) return fail(PFC_E_MESH, "pfc_add_mesh: leaf ids are not a permutation of the primitives");
            nd.kind = kNodeLeaf; nd.right = leaf;
            m.leaf_depth[leaf] = it.depth;
            m.leaf_path[leaf] = it.path;
            if (it.depth > m.depth) m.depth = it.depth;
        } else {
            if (it.depth >= 62) return fail(PFC_E_MESH, "pfc_add_mesh: tree deeper than 62 levels");
            bool identity = true;   // internal boxes are merged axis-aligned boxes (src/obb/box_types.jl:11-15): the SAT skips the identity products
            for (int i = 0; i < 9; ++i) identity = identity && (nd.R[i] == ((i % 4 == 0) ? 1.0 : 0.0));
            nd.kind = identity ? kNodeInternalAabb : kNodeInternal;
            nd.right = -1;
            stack.push_back({node_right[it.src], dst, 1, it.depth + 1, (it.path << 1) | 1u});
            stack.push_back({node_left[it.src], dst, 0, it.depth + 1, (it.path << 1)});
        }
    }
    if (next != n_node) return fail(PFC_E_MESH, "pfc_add_mesh: unreachable tree nodes");
    if (kind == 1) {
        for (int64_t k = 0; k < n_prim; ++k) {
            double v[12];
            for (int j = 0; j < 4; ++j) for (int i = 0; i < 3; ++i) v[3 * j + i] = xyz[3 * idx[4 * k + j] + i];
            if (!(0.0 < tet_volume6(v))) return fail(PFC_E_MESH, "pfc_add_mesh: inverted tetrahedron");
        }
    }
    c->mesh.push_back(std::move(m));
    if (mesh_id_out) *mesh_id_out = int(c->mesh.size()) - 1;
    return PFC_OK;
}

int pfc_add_instruction(pfc_ctx* c, int mesh_1, int mesh_2, double chi, int model, const double* params, int n_quad_rule, int* ins_id_out) {
    if (!c || c->finalized) return fail(PFC_E_ARG, "pfc_add_instruction: context missing or already finalized");
    const int nm = int(c->mesh.size());
    if (mesh_1 < 0 || mesh_1 >= nm || mesh_2 < 0 || mesh_2 >= nm) return fail(PFC_E_ARG, "pfc_add_instruction: no such mesh");
    if (c->mesh[mesh_2].kind != 1) return fail(PFC_E_ARG, "pfc_add_instruction: mesh_2 must be a tetrahedral mesh (add_friction! ordering rule)");
    if (model != 0 && model != 1) return fail(PFC_E_ARG, "pfc_add_instruction: model must be 0 (regularized) or 1 (bristle)");
    if (n_quad_rule < 1 || n_quad_rule > 2) return fail(PFC_E_ARG, "only quadrature rules 1 (first order) and 2 (second? order) are currently implemented");
    if (!params) return fail(PFC_E_ARG, "pfc_add_instruction: params is NULL");
    HostIns h{};
    h.mesh_1 = mesh_1; h.mesh_2 = mesh_2; h.model = model; h.n_quad_rule = n_quad_rule; h.chi = chi;
    const int np = model == 0 ? 3 : 5;
    for (int k = 0; k < np; ++k) h.params[k] = params[k];
    h.bristle_id = model == 1 ? c->n_bristle++ : -1;
    c->ins.push_back(h);
    if (ins_id_out) *ins_id_out = int(c->ins.size()) - 1;
    return PFC_OK;
}

// The contact parameters of an instruction as the kernels use them, from the values a scene is built with (pfc_add_mesh's Ebar,
// pfc_add_instruction's chi and params): for pfc_finalize's scene table and for every row of a per-environment table alike, so equal
// values give equal bits.  Ebar1 is 0 for a triangle mesh_1.
static InsParam derive_contact_params(int model, double chi, double Ebar1, double Ebar2, const double* q) {
    InsParam d{};
    d.chi = chi; d.Ebar1 = Ebar1; d.Ebar2 = Ebar2;
    if (model == 0) { d.p[0] = q[0]; d.p[1] = q[1]; d.p[2] = q[2]; d.p[3] = 2 * q[2]; d.p[4] = 3 * q[2];
        d.p[5] = (d.p[1] - d.p[0]) / (d.p[4] - d.p[3]); d.p[6] = 1.0 / d.p[2]; }
    else { d.p[0] = q[0]; d.p[1] = q[1]; d.p[2] = q[2]; d.p[3] = q[3]; d.p[4] = 2 * q[2]; d.p[5] = 3 * q[2]; d.p[6] = q[4];
        d.p[7] = (d.p[3] - d.p[2]) / (d.p[5] - d.p[4]); }
    return d;
}

// Which path every instruction takes, and the device tables that follow from it.
//   small  n_leaf1 * n_leaf2 <= 512: broad and narrow phase on chip, two launches per batch; the pair list cannot outgrow its slot.
//   mid    both trees <= kMidLeaves leaves (gripper pads, coarse spheres): the same two kernels with a frontier / pair-list slot of
//          kMidCap entries -- contact patches touch a small corner of such trees.  A frontier that outgrows the slot raises a per-instruction
//          flag; the host then moves the instruction to the large path for good (force_large) and repeats the evaluation.
//   large  everything else: the multi-kernel pipeline of pfc_large.cu.
constexpr int kMidLeaves = 1024;
constexpr int kMidCap = 1024;
static int build_tables(pfc_ctx* c) {
    const long long mid_leaves = getenv("PFC_MID_LEAVES") ? atoll(getenv("PFC_MID_LEAVES")) : kMidLeaves;   // (0: tests that want the large path on small trees)
    c->h_ins.clear();
    std::vector<int32_t> small, large;
    int large_key_bits = 0;
    c->small_max_pairs = 1;
    c->n_mid = 0;
    for (size_t k = 0; k < c->ins.size(); ++k) {
        const HostIns& h = c->ins[k];
        const HostMesh& m1 = c->mesh[h.mesh_1];
        const HostMesh& m2 = c->mesh[h.mesh_2];
        InsDev d{};
        d.kind1 = m1.kind; d.model = h.model; d.n_quad = h.n_quad_rule == 1 ? 1 : 3; d.bristle_id = h.bristle_id;
        d.node_base1 = m1.node_base; d.node_base2 = m2.node_base; d.prim_base1 = m1.prim_base; d.prim_base2 = m2.prim_base;
        d.n_leaf1 = int(m1.n_prim); d.n_leaf2 = int(m2.n_prim);
        d.key_bits = m1.depth + m2.depth;
        if (d.key_bits > 64) return fail(PFC_E_MESH, "pfc_finalize: tree depths sum to more than 64 levels");
        const bool fits_slot = m1.n_prim * m2.n_prim <= kSmallCap;
        const bool mid = !fits_slot && m1.n_prim <= mid_leaves && m2.n_prim <= mid_leaves && !c->force_large[k];
        d.small = (fits_slot || mid) ? 1 : 0;
        {
            const InsParam cp = derive_contact_params(h.model, h.chi, m1.kind == 1 ? m1.Ebar : 0.0, m2.Ebar, h.params);
            d.chi = cp.chi; d.Ebar1 = cp.Ebar1; d.Ebar2 = cp.Ebar2;
            for (int j = 0; j < 8; ++j) d.p[j] = cp.p[j];
        }
        d.path_base1 = m1.path_base; d.path_base2 = m2.path_base;
        if (d.small) {
            small.push_back(int32_t(k));
            c->small_max_pairs = std::max(c->small_max_pairs, mid ? kMidCap : int(m1.n_prim * m2.n_prim));
            c->n_mid += mid;
        } else { large.push_back(int32_t(k)); large_key_bits = std::max(large_key_bits, d.key_bits); }
        c->h_ins.push_back(d);
    }
    c->large_ins_host = large;
    c->large_scene = LargeScene{};
    if (!large.empty()) {
        CU(c->d_large.ensure(large.size()));
        CU(cudaMemcpy(c->d_large.p, large.data(), large.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        c->large_scene.large_ins = c->d_large.p;
        c->large_scene.leaf_path = c->d_leaf_path.p;
        c->large_scene.leaf_depth = c->d_leaf_depth.p;
        c->large_scene.n_large = int(large.size());
        c->large_scene.key_bits = large_key_bits;
        for (int32_t k : large) {
            c->large_scene.max_leaves = std::max(c->large_scene.max_leaves, std::max(c->h_ins[k].n_leaf1, c->h_ins[k].n_leaf2));
            c->large_scene.max_depth = std::max(c->large_scene.max_depth, std::max(c->mesh[c->ins[k].mesh_1].depth, c->mesh[c->ins[k].mesh_2].depth));
        }
        if (!c->large_buf) c->large_buf = large_buffers_create();
    }
    CU(c->d_ins.ensure(c->h_ins.size()));
    CU(c->d_small.ensure(std::max<size_t>(small.size(), 1)));
    CU(cudaMemcpy(c->d_ins.p, c->h_ins.data(), c->h_ins.size() * sizeof(InsDev), cudaMemcpyHostToDevice));
    if (!small.empty()) CU(cudaMemcpy(c->d_small.p, small.data(), small.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    {   // broad-phase scheduling order: instruction-major, the instructions with the largest trees first
        std::vector<int32_t> heavy(small);
        std::stable_sort(heavy.begin(), heavy.end(), [&](int32_t a, int32_t b) {
            return (long long)c->h_ins[a].n_leaf1 * c->h_ins[a].n_leaf2 > (long long)c->h_ins[b].n_leaf1 * c->h_ins[b].n_leaf2; });
        CU(c->d_small_heavy.ensure(std::max<size_t>(heavy.size(), 1)));
        if (!heavy.empty()) CU(cudaMemcpy(c->d_small_heavy.p, heavy.data(), heavy.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        c->scene.small_heavy_first = c->d_small_heavy.p;
        int lo = INT32_MAX, hi = 0;
        for (int32_t k : small) {
            const InsDev& in = c->h_ins[k];
            lo = std::min(lo, std::min(in.node_base1, in.node_base2));
            hi = std::max(hi, std::max(in.node_base1 + 2 * in.n_leaf1 - 1, in.node_base2 + 2 * in.n_leaf2 - 1));
        }
        c->scene.small_node_lo = small.empty() ? 0 : lo;
        c->scene.small_node_n = small.empty() ? 0 : hi - lo;
    }
    if (c->n_mid > 0) {   // per-instruction overflow marks of the mid instructions
        CU(c->d_ins_overflow.ensure(c->h_ins.size()));
        CU(cudaMemset(c->d_ins_overflow.p, 0, sizeof(int) * c->h_ins.size()));
        if (!c->h_ins_overflow) CU(cudaHostAlloc(reinterpret_cast<void**>(&c->h_ins_overflow), sizeof(int) * std::max<size_t>(c->h_ins.size(), 1), cudaHostAllocDefault));
    }
    c->scene.nodes = c->d_nodes.p; c->scene.tets = c->d_tets.p; c->scene.tris = c->d_tris.p; c->scene.ins = c->d_ins.p;
    c->scene.small_ins = c->d_small.p;
    c->scene.ins_overflow = c->n_mid > 0 ? c->d_ins_overflow.p : nullptr;
    c->scene.n_ins = int(c->h_ins.size()); c->scene.n_small = int(small.size()); c->scene.n_bristle = c->n_bristle;
    c->scene.n_small_bristle = 0;
    for (int32_t k : small) c->scene.n_small_bristle += (c->h_ins[k].model == PFC_MODEL_BRISTLE);
    {   // bristle instructions: tables of the reference-order pipeline
        std::vector<int32_t> bris, large_index(c->h_ins.size(), -1);
        for (size_t k = 0; k < c->h_ins.size(); ++k) if (c->h_ins[k].model == PFC_MODEL_BRISTLE) bris.push_back(int32_t(k));
        for (size_t k = 0; k < large.size(); ++k) large_index[large[k]] = int32_t(k);
        CU(c->d_large_index.ensure(large_index.size()));
        CU(cudaMemcpy(c->d_large_index.p, large_index.data(), sizeof(int32_t) * large_index.size(), cudaMemcpyHostToDevice));
        c->large_index_dirty = false;
        c->has_large_bristle = false;
        for (int32_t k : large) c->has_large_bristle |= (c->h_ins[k].model == PFC_MODEL_BRISTLE);
        if (!bris.empty()) {
            CU(c->d_bris_ins.ensure(bris.size()));
            CU(cudaMemcpy(c->d_bris_ins.p, bris.data(), sizeof(int32_t) * bris.size(), cudaMemcpyHostToDevice));
            if (!c->exact_buf) c->exact_buf = exact_buffers_create();
        }
        c->exact_scene.tet_eps = c->d_tet_eps.p; c->exact_scene.bris_ins = c->d_bris_ins.p; c->exact_scene.large_index = c->d_large_index.p;
        c->exact_scene.n_bris = int32_t(bris.size()); c->exact_scene.skip_large = 0;
    }
    alloc_generation()++;   // (a captured evaluation graph holds the old tables' launch sequence)
    return PFC_OK;
}

int pfc_finalize(pfc_ctx* c, int64_t max_env) {
    if (!c || c->finalized) return fail(PFC_E_ARG, "pfc_finalize: context missing or already finalized");
    if (c->ins.empty()) return fail(PFC_E_ARG, "pfc_finalize: no contact instructions");
    if (max_env < 1) max_env = 1;
    CU(cudaSetDevice(c->device));
    std::vector<NodeRec> nodes;
    std::vector<TetRec> tets;
    std::vector<TriRec> tris;
    std::vector<double> tet_eps;   // per tetrahedron: the pressure-field value at its 4 vertices
    for (auto& m : c->mesh) {
        m.node_base = int(nodes.size());
        nodes.insert(nodes.end(), m.nodes.begin(), m.nodes.end());
        if (m.kind == 1) {
            m.prim_base = int(tets.size());
            for (int64_t k = 0; k < m.n_prim; ++k) {
                TetRec t;
                double e4[4];
                for (int j = 0; j < 4; ++j) {
                    const int32_t vi = m.idx[4 * k + j];
                    for (int i = 0; i < 3; ++i) t.v[3 * j + i] = m.xyz[3 * vi + i];
                    e4[j] = m.eps[vi];
                }
                if (!invert_tet_matrix(t.v, t.inv)) return fail(PFC_E_MESH, "pfc_finalize: degenerate tetrahedron");
                for (int j = 0; j < 4; ++j) t.eps_r[j] = e4[0] * t.inv[j] + e4[1] * t.inv[4 + j] + e4[2] * t.inv[8 + j] + e4[3] * t.inv[12 + j];
                tets.push_back(t);
                tet_eps.insert(tet_eps.end(), e4, e4 + 4);
            }
        } else {
            m.prim_base = int(tris.size());
            for (int64_t k = 0; k < m.n_prim; ++k) {
                TriRec t;
                for (int j = 0; j < 3; ++j) for (int i = 0; i < 3; ++i) t.v[3 * j + i] = m.xyz[3 * m.idx[3 * k + j] + i];
                // triangleNormal = normalize(cross(v2 - v1, v3 - v2) * 0.5)
                const double ax = t.v[3] - t.v[0], ay = t.v[4] - t.v[1], az = t.v[5] - t.v[2];
                const double bx = t.v[6] - t.v[3], by = t.v[7] - t.v[4], bz = t.v[8] - t.v[5];
                const double nx = (ay * bz - az * by) * 0.5, ny = (az * bx - ax * bz) * 0.5, nz = (ax * by - ay * bx) * 0.5;
                const double len = std::sqrt(nx * nx + ny * ny + nz * nz);
                t.n[0] = nx / len; t.n[1] = ny / len; t.n[2] = nz / len;
                tris.push_back(t);
            }
        }
    }
    {   // per-primitive leaf paths (the DFS keys of the large path) for every mesh: uploaded whether or not an instruction needs them yet
        std::vector<unsigned long long> leaf_path;
        std::vector<unsigned char> leaf_depth;
        for (auto& m : c->mesh) {
            m.path_base = int(leaf_path.size());
            for (int64_t k = 0; k < m.n_prim; ++k) { leaf_path.push_back(m.leaf_path[k]); leaf_depth.push_back((unsigned char)m.leaf_depth[k]); }
        }
        CU(c->d_leaf_path.ensure(std::max<size_t>(leaf_path.size(), 1)));
        CU(c->d_leaf_depth.ensure(std::max<size_t>(leaf_depth.size(), 1)));
        CU(cudaMemcpy(c->d_leaf_path.p, leaf_path.data(), leaf_path.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(c->d_leaf_depth.p, leaf_depth.data(), leaf_depth.size(), cudaMemcpyHostToDevice));
    }
    CU(c->d_nodes.ensure(nodes.size()));
    CU(c->d_tets.ensure(std::max<size_t>(tets.size(), 1)));
    CU(c->d_tris.ensure(std::max<size_t>(tris.size(), 1)));
    CU(cudaMemcpy(c->d_nodes.p, nodes.data(), nodes.size() * sizeof(NodeRec), cudaMemcpyHostToDevice));
    if (!tets.empty()) CU(cudaMemcpy(c->d_tets.p, tets.data(), tets.size() * sizeof(TetRec), cudaMemcpyHostToDevice));
    if (!tris.empty()) CU(cudaMemcpy(c->d_tris.p, tris.data(), tris.size() * sizeof(TriRec), cudaMemcpyHostToDevice));
    CU(c->d_tet_eps.ensure(std::max<size_t>(tet_eps.size(), 4)));
    if (!tet_eps.empty()) CU(cudaMemcpy(c->d_tet_eps.p, tet_eps.data(), sizeof(double) * tet_eps.size(), cudaMemcpyHostToDevice));
    c->force_large.assign(c->ins.size(), 0);
    {
        const int rc = build_tables(c);
        if (rc != PFC_OK) return rc;
    }
    c->max_env = max_env;
    c->finalized = true;
    return PFC_OK;
}

// The bristle instructions of an evaluation, in the reference's operation order (pfc_exact.cu), from the pair lists the Float64 broad
// phase left.  dual: Jacobian mode (every scalar of X / twist / s / wrench / sdot is 7 doubles).  skip_large: a sharded context keeps its
// large bristle instructions on the partial-sum protocol.  Synchronises the stream once (see exact_bristle_eval).
static int eval_bristle_exact(pfc_ctx* c, long long n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot,
                              const long long* n_pairs, int* flags, const InsParam* params, int dual, bool skip_large, int* nl, cudaStream_t stream = nullptr) {
    if (c->exact_scene.n_bris == 0) return PFC_OK;
    ExactIO xio{n_env, X, twist, s, wrench, sdot, n_pairs, flags, params};
    ExactPairs ps{};
    ps.small_pairs = c->d_small_pairs.p; ps.small_cap = small_cap(c->small_max_pairs);
    if (c->large_scene.n_large > 0 && c->has_large_bristle && !skip_large) large_exact_view(c->large_buf, c->large_scene, n_env, ps);
    ExactScene es = c->exact_scene;
    es.skip_large = skip_large ? 1 : 0;
    CU(exact_bristle_eval(c->scene, es, xio, ps, dual, c->exact_buf, stream ? stream : c->stream, nl));
    return PFC_OK;
}

// The large path and the bristle pipeline queue their work without a host round trip and size their buffers from earlier evaluations.
// After an evaluation has been queued: one synchronisation, then the device-side counters say whether everything fit.  Returns 0 (it
// did, or nothing growable was involved: no synchronisation then), 1 (capacities raised: queue the same evaluation again) or a
// negative PFC_E_* code.
static int build_tables(pfc_ctx* c);
static int evaluation_fits(pfc_ctx* c) {
    const bool lg = c->large_buf != nullptr, ex = c->exact_buf != nullptr, mid = c->n_mid > 0;
    if (!lg && !ex && !mid) return 0;
    cudaError_t e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return fail(PFC_E_CUDA, std::string("cudaStreamSynchronize: ") + cudaGetErrorString(e));
    int m = 0;
    if (mid && c->mid_check_pending) {   // a mid-size instruction outgrew its on-chip slot: it takes the large path from now on
        c->mid_check_pending = false;
        for (size_t k = 0; k < c->h_ins.size(); ++k)
            if (c->h_ins_overflow[k]) { c->force_large[k] = 1; m = 1; }
        if (m) {
            const int rc = build_tables(c);
            if (rc != PFC_OK) return rc;
            large_mark_clear(c->large_buf); exact_mark_clear(c->exact_buf);   // the evaluation is repeated as a whole
            return 1;
        }
    }
    const int a = lg ? large_check(c->large_buf) : 0, b = ex ? exact_check(c->exact_buf) : 0;
    if (a < 0 || b < 0) return fail(PFC_E_CAPACITY, "candidate-pair / traction buffers cannot be grown far enough");
    return (a | b) ? 1 : 0;
}
#define PFC_REQUEUE_LOOP(body)                                                                                   \
    for (int attempt_ = 0;; ++attempt_) {                                                                        \
        body                                                                                                     \
        const int fit_ = evaluation_fits(c);                                                                     \
        if (fit_ < 0) return fit_;                                                                               \
        if (fit_ == 0) break;                                                                                    \
        if (attempt_ >= 8) return fail(PFC_E_CAPACITY, "candidate-pair / traction buffers kept overflowing");    \
    }

static int eval_device_once(pfc_ctx* c, const EvalIO& io_in) {
    EvalIO io = io_in;
    const int n_ins = c->scene.n_ins;
    if (c->keep_pairs) {
        c->dbg_cap = std::max(kSmallCap, small_cap(c->small_max_pairs));
        CU(c->d_dbg_pairs.ensure(size_t(2) * c->dbg_cap * io.n_env * n_ins));
        io.dbg_pairs = c->d_dbg_pairs.p;
        io.dbg_cap = c->dbg_cap;
        c->dbg_n_env = io.n_env;
    } else { io.dbg_pairs = nullptr; io.dbg_cap = 0; }
    int nl = 0;
    // Scenes that mix bristle and regularized instructions on the small path (test/pencil.jl): once the pair lists exist, the bristle
    // pipeline (reference-order points + patch passes, two long single-warp kernels) and the regularized narrow phase are independent
    // (disjoint instructions, disjoint outputs): the bristle pipeline runs on a second stream beside the narrow kernel.  Not when large
    // bristle instructions exist (their counts are published by the large path's finish kernel).
    const bool beside = c->exact_scene.n_bris > 0 && c->scene.n_small > 0 && !c->has_large_bristle && !c->timing && c->n_bristle < c->scene.n_ins;
    if (beside && !c->stream2) {
        CU(cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    }
    if (c->scene.n_small > 0) {
        CU(c->d_small_pairs.ensure(size_t(small_cap(c->small_max_pairs)) * io.n_env * n_ins + kSmallPairsSlack));
        CU(launch_eval_small_f64(c->scene, io, c->small_max_pairs, c->d_small_pairs.p, c->stream, &nl, c->timing ? c->ev : nullptr, beside ? c->ev_fork : nullptr));
        c->ev_valid = c->timing;
    }
    if (beside) {
        CU(cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
        int rc = eval_bristle_exact(c, io.n_env, io.X, io.twist, io.s, io.wrench, io.sdot, io.n_pairs, io.flags, io.params, 0, false, &nl, c->stream2);
        if (rc != PFC_OK) return rc;
        CU(cudaEventRecord(c->ev_join, c->stream2));
    }
    if (c->large_scene.n_large > 0) {
        if (c->shard_world > 1) return fail(PFC_E_ARG, "this context is sharded: use pfc_eval_sharded_begin / _step");
        CU(large_broad_phase(c->scene, c->large_scene, io, c->large_buf, c->stream, &nl));
        CU(large_narrow_stage(c->scene, c->large_scene, io, c->large_buf, 0, 0, c->stream, &nl));
    }
    if (beside) {
        CU(cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    } else {   // bristle instructions (small and large): reference-order pipeline
        int rc = eval_bristle_exact(c, io.n_env, io.X, io.twist, io.s, io.wrench, io.sdot, io.n_pairs, io.flags, io.params, 0, false, &nl);
        if (rc != PFC_OK) return rc;
    }
    if (c->n_mid > 0) {
        CU(cudaMemcpyAsync(c->h_ins_overflow, c->d_ins_overflow.p, sizeof(int) * c->h_ins.size(), cudaMemcpyDeviceToHost, c->stream));
        c->mid_check_pending = true;
    }
    c->launches += nl;
    c->last_X = io.X; c->last_tw = io.twist; c->last_params = io.params;
    // the pair lists now belong to this evaluation: pfc_eval_dual6(X_bp = NULL) may reuse them only together with the library's own
    // count / flag arrays (set again by the host-pointer entry points after a successful evaluation)
    c->lists_n_env = -1;
    if (c->keep_pairs) {
        CU(c->d_last_np.ensure(size_t(io.n_env) * n_ins));
        CU(cudaMemcpyAsync(c->d_last_np.p, io.n_pairs, sizeof(long long) * io.n_env * n_ins, cudaMemcpyDeviceToDevice, c->stream));
    }
    return PFC_OK;
}

// Scenes with large or bristle instructions queue dozens of short kernels per evaluation (breadth-first levels, radix passes, ...): once
// the same evaluation -- same entry point, batch size and buffers, nothing reallocated since -- has run eagerly, its launch sequence is
// captured into a CUDA graph and replayed (one launch instead of ~45; the kernels read every data-dependent size from the device).
// enqueue() must queue one complete evaluation on c->stream and return PFC_OK.
static int run_evaluation(pfc_ctx* c, unsigned long long key, const std::function<int()>& enqueue) {
    pfc_ctx::GraphCache& g = c->graph;
    const bool want_graph = !g.disabled && !c->timing && !c->keep_pairs && (c->large_buf || c->exact_buf);
    for (int attempt = 0;; ++attempt) {
        const unsigned long long gen = alloc_generation().load();
        bool replayed = false;
        if (want_graph && attempt == 0 && g.key == key && g.gen == gen) {
            if (g.exec) {
                if (cudaGraphLaunch(g.exec, c->stream) == cudaSuccess) { replayed = true; c->launches += g.launches; }
                else { cudaGetLastError(); cudaGraphExecDestroy(g.exec); g.exec = nullptr; g.disabled = true; }
            } else if (g.seen) {   // second identical evaluation: capture it
                cudaGraph_t graph = nullptr;
                const long long l0 = c->launches;
                if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                    const int rc = enqueue();
                    const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
                    if (rc == PFC_OK && e == cudaSuccess && graph && alloc_generation().load() == gen &&
                        cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess && cudaGraphLaunch(g.exec, c->stream) == cudaSuccess) {
                        g.launches = int(c->launches - l0);
                        replayed = true;
                    } else {
                        cudaGetLastError();
                        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
                        g.disabled = true;   // this context's evaluations do not capture: stay eager
                        c->launches = l0;
                    }
                    if (graph) cudaGraphDestroy(graph);
                } else { cudaGetLastError(); g.disabled = true; }
            }
        }
        if (replayed) {
            large_mark_pending(c->large_buf);
            exact_mark_pending(c->exact_buf);
            if (c->n_mid > 0) c->mid_check_pending = true;
        } else {
            const int rc = enqueue();
            if (rc != PFC_OK) return rc;
            if (want_graph) {
                if (g.key != key || g.gen != alloc_generation().load()) { if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; } g.seen = false; }
                g.key = key; g.gen = alloc_generation().load(); g.seen = true;
            }
        }
        const int fit = evaluation_fits(c);
        if (fit < 0) return fit;
        if (fit == 0) return PFC_OK;
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }   // buffers grow: the captured pointers are stale
        g.seen = false; g.gen = ~0ull;
        if (attempt >= 8) return fail(PFC_E_CAPACITY, "candidate-pair / traction buffers kept overflowing");
    }
}
static unsigned long long eval_key(int kind, const pfc_ctx* c, const EvalIO& io) {
    unsigned long long h = 1469598103934665603ull;
    auto mix = [&](unsigned long long v) { h ^= v; h *= 1099511628211ull; };
    mix((unsigned long long)kind); mix((unsigned long long)io.n_env); mix((unsigned long long)(uintptr_t)io.X); mix((unsigned long long)(uintptr_t)io.twist);
    mix((unsigned long long)(uintptr_t)io.s); mix((unsigned long long)(uintptr_t)io.wrench); mix((unsigned long long)(uintptr_t)io.sdot);
    mix((unsigned long long)(uintptr_t)io.n_pairs); mix((unsigned long long)(uintptr_t)io.flags); mix((unsigned long long)c->shard_rank * 64 + c->shard_world);
    mix((unsigned long long)(uintptr_t)io.params);   // (a table's buffer, or none: a graph never replays with another table)
    return h ? h : 1;
}

static int eval_device(pfc_ctx* c, const EvalIO& io) {
    return run_evaluation(c, eval_key(1, c, io), [&]() { return eval_device_once(c, io); });
}

// A small-path scene queues a handful of short operations per host-pointer call (copies in, two to four kernels, copies out); launched
// one by one the GPU waits for the host between them (the copies and kernels of a 512-environment batch last 3-30 us each).  When the same
// call -- same batch size, same buffers, nothing reallocated since -- comes again, its operations are captured into a CUDA graph and
// replayed with one launch.  (Pageable caller buffers cannot be captured: the capture fails once and the context stays with plain
// launches.)  Scenes with large / mid-size / bristle instructions are left to run_evaluation: their evaluations synchronise to check
// buffer sizes.  enqueue() queues the whole call on c->stream (no synchronisation) and returns PFC_OK.
static int run_host_call(pfc_ctx* c, pfc_ctx::GraphCache& g, unsigned long long key, const std::function<int()>& enqueue) {
    static const bool host_graph_off = getenv("PFC_NO_HOST_GRAPH") != nullptr;   // (experiment switch)
    const bool graphable = !host_graph_off && !g.disabled && !c->timing && !c->keep_pairs && !c->large_buf && !c->exact_buf && c->n_mid == 0;
    if (!graphable) return enqueue();
    const unsigned long long gen = alloc_generation().load();
    if (g.key == key && g.gen == gen) {
        if (g.exec) {
            if (cudaGraphLaunch(g.exec, c->stream) == cudaSuccess) { c->launches += g.launches; return PFC_OK; }
            cudaGetLastError(); cudaGraphExecDestroy(g.exec); g.exec = nullptr; g.disabled = true;
        } else if (g.seen) {
            cudaGraph_t graph = nullptr;
            const long long l0 = c->launches;
            if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const int rc = enqueue();
                const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
                bool ok = rc == PFC_OK && e == cudaSuccess && graph && alloc_generation().load() == gen && cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess &&
                          cudaGraphLaunch(g.exec, c->stream) == cudaSuccess;
                if (graph) cudaGraphDestroy(graph);
                if (ok) { g.launches = int(c->launches - l0); return PFC_OK; }
                cudaGetLastError();
                if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
                g.disabled = true;
                c->launches = l0;
            } else { cudaGetLastError(); g.disabled = true; }
        }
    }
    const int rc = enqueue();
    if (rc != PFC_OK) return rc;
    if (g.exec && (g.key != key || g.gen != alloc_generation().load())) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    g.key = key; g.gen = alloc_generation().load(); g.seen = true;   // everything this call needs is allocated now: the next identical one is captured
    return PFC_OK;
}

// ---- small host-pointer calls: copies through a pinned arena ----------------------------------------------------------------
constexpr size_t kArenaBytes = 256 << 10;
static void arena_reset(pfc_ctx* c) {
    if (!c->h_arena && cudaHostAlloc(reinterpret_cast<void**>(&c->h_arena), kArenaBytes, cudaHostAllocDefault) == cudaSuccess) c->arena_cap = kArenaBytes;
    c->arena_used = 0;
    c->arena_out.clear();
}
static void* arena_take(pfc_ctx* c, size_t bytes) {
    const size_t a = (c->arena_used + 63) & ~size_t(63);
    if (!c->h_arena || a + bytes > c->arena_cap) return nullptr;
    c->arena_used = a + bytes;
    return c->h_arena + a;
}
// host -> device on the context's stream; small transfers go through the arena
static cudaError_t copy_in(pfc_ctx* c, void* dev, const void* host, size_t bytes) {
    if (void* p = arena_take(c, bytes)) { std::memcpy(p, host, bytes); host = p; }
    return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, c->stream);
}
// device -> host; small transfers land in the arena and are handed to the caller's buffer by copy_out_finish (after the stream sync)
static cudaError_t copy_out(pfc_ctx* c, void* host, const void* dev, size_t bytes) {
    if (void* p = arena_take(c, bytes)) { c->arena_out.push_back({host, p, bytes}); host = p; }
    return cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, c->stream);
}
static void copy_out_finish(pfc_ctx* c) {
    for (const auto& o : c->arena_out) std::memcpy(o.dst, o.src, o.bytes);
    c->arena_out.clear();
}

// ---- per-environment contact parameters ------------------------------------------------------------------------------------
// the table of the context (nullptr while none is set) and the batch size it imposes on every evaluation
static const InsParam* ctx_params(const pfc_ctx* c) { return c->params_n_env > 0 ? c->d_params.p : nullptr; }
static int params_check(const pfc_ctx* c, const char* who, int64_t n_env) {
    if (c->params_n_env > 0 && n_env != c->params_n_env)
        return fail(PFC_E_ARG, std::string(who) + ": n_env differs from the batch of the contact-parameter table (pfc_set_contact_params)");
    return PFC_OK;
}

int pfc_set_contact_params(pfc_ctx* c, int64_t n_env, const double* params) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_set_contact_params: call after pfc_finalize");
    if (n_env < 0 || n_env > c->max_env) return fail(PFC_E_ARG, "pfc_set_contact_params: n_env must be in 0..max_env");
    if (n_env > 0 && !params) return fail(PFC_E_ARG, "pfc_set_contact_params: params is NULL");
    CU(cudaSetDevice(c->device));
    if (n_env == 0) {   // back to the scene's own values (the buffer is kept for the next table)
        c->params_n_env = 0;
        return PFC_OK;
    }
    const size_t ni = c->ins.size();
    std::vector<InsParam> rows(size_t(n_env) * ni);
    for (int64_t e = 0; e < n_env; ++e)
        for (size_t k = 0; k < ni; ++k) {
            const double* v = params + 8 * (size_t(e) * ni + k);
            const HostIns& h = c->ins[k];
            const bool tet1 = c->mesh[h.mesh_1].kind == 1;
            const int n_q = h.model == 0 ? 3 : 5;   // the entries the instruction's model uses
            bool finite = std::isfinite(v[0]) && std::isfinite(v[2]) && (!tet1 || std::isfinite(v[1]));
            for (int j = 0; j < n_q; ++j) finite = finite && std::isfinite(v[3 + j]);
            if (!finite)
                return fail(PFC_E_ARG, "pfc_set_contact_params: non-finite entry (environment " + std::to_string(e) + ", instruction " + std::to_string(k) + ")");
            rows[size_t(e) * ni + k] = derive_contact_params(h.model, v[0], tet1 ? v[1] : 0.0, v[2], v + 3);
        }
    // in stream order behind the evaluations already queued (they read the previous table), and complete before `rows` goes
    if (rows.size() > c->d_params.n) {
        c->params_n_env = 0;   // (growing frees the previous table: should the allocation fail, no table is left in force)
        CU(c->d_params.ensure(rows.size()));
    }
    CU(cudaMemcpyAsync(c->d_params.p, rows.data(), sizeof(InsParam) * rows.size(), cudaMemcpyHostToDevice, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->params_n_env = n_env;
    return PFC_OK;
}

int pfc_eval_f64_device(pfc_ctx* c, int64_t n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot,
                        int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_eval_f64_device: context not finalized");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_f64_device: negative n_env");
    { const int rc = params_check(c, "pfc_eval_f64_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!X || !twist || !wrench || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_eval_f64_device: NULL buffer");
    if (c->n_bristle > 0 && (!s || !sdot)) return fail(PFC_E_ARG, "pfc_eval_f64_device: bristle instructions need s and sdot");
    CU(cudaSetDevice(c->device));
    EvalIO io{};
    io.n_env = n_env; io.X = X; io.twist = twist; io.s = s; io.wrench = wrench; io.sdot = sdot;
    io.n_pairs = reinterpret_cast<long long*>(n_pairs); io.flags = flags; io.params = ctx_params(c);
    return eval_device(c, io);
}

int pfc_eval_f64(pfc_ctx* c, int64_t n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot, int64_t* n_pairs,
                 int32_t* flags) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_eval_f64: context not finalized");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_f64: negative n_env");
    { const int rc = params_check(c, "pfc_eval_f64", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!X || !twist || !wrench) return fail(PFC_E_ARG, "pfc_eval_f64: NULL buffer");
    if (c->n_bristle > 0 && (!s || !sdot)) return fail(PFC_E_ARG, "pfc_eval_f64: bristle instructions need s and sdot");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle);
    arena_reset(c);
    // (Measured and rejected: letting the kernels of a single small scene read X / twist straight from the pinned arena and write the
    // wrenches into it -- zero-copy over PCIe instead of five cudaMemcpyAsync calls: no gain on test/boxes.jl (69 vs 67 us per call), and
    // scenes whose large instructions re-read X in every thread got slower, 316 -> 402 us on the spoon.)
    const size_t bX = sizeof(double) * 16 * ne * ni, bT = sizeof(double) * 6 * ne * ni, bS = sizeof(double) * 6 * ne * nb;
    const size_t bW = bT, bD = bS, bN = sizeof(long long) * ne * ni, bF = (sizeof(int32_t) * ne * ni + 7) & ~size_t(7);
    EvalIO io{};
    io.n_env = n_env; io.params = ctx_params(c);
    std::vector<int32_t> fl_local;
    int32_t* fl = flags;
    if (!fl) { fl_local.resize(ne * ni); fl = fl_local.data(); }
    unsigned char* h_in = (bX + bT + bS + bW + bD + bN + bF <= 32768) ? static_cast<unsigned char*>(arena_take(c, bX + bT + bS)) : nullptr;
    unsigned char* h_out = h_in ? static_cast<unsigned char*>(arena_take(c, bW + bD + bN + bF)) : nullptr;
    if (h_in && h_out) {
        // One small scene per call (the reference's own use: Radau on a single scene): every input in one block and every output in one
        // block, so the call costs one copy each way instead of three in and four out (each a few microseconds of copy-engine latency).
        CU(c->d_pack_in.ensure(bX + bT + bS)); CU(c->d_pack_out.ensure(bW + bD + bN + bF));
        std::memcpy(h_in, X, bX); std::memcpy(h_in + bX, twist, bT);
        if (nb) std::memcpy(h_in + bX + bT, s, bS);
        unsigned char* di = c->d_pack_in.p; unsigned char* dn = c->d_pack_out.p;
        io.X = reinterpret_cast<const double*>(di); io.twist = reinterpret_cast<const double*>(di + bX); io.s = nb ? reinterpret_cast<const double*>(di + bX + bT) : nullptr;
        io.wrench = reinterpret_cast<double*>(dn); io.sdot = nb ? reinterpret_cast<double*>(dn + bW) : nullptr;
        io.n_pairs = reinterpret_cast<long long*>(dn + bW + bD); io.flags = reinterpret_cast<int*>(dn + bW + bD + bN);
        auto enqueue = [&]() -> int {
            CU(cudaMemcpyAsync(c->d_pack_in.p, h_in, bX + bT + bS, cudaMemcpyHostToDevice, c->stream));
            const int rc = eval_device(c, io);
            if (rc != PFC_OK) return rc;
            CU(cudaMemcpyAsync(h_out, dn, bW + bD + bN + bF, cudaMemcpyDeviceToHost, c->stream));
            return PFC_OK;
        };
        unsigned long long key = 1469598103934665603ull;
        auto mix = [&](unsigned long long v) { key ^= v; key *= 1099511628211ull; };
        mix(6ull); mix((unsigned long long)n_env); mix((unsigned long long)(uintptr_t)h_in); mix((unsigned long long)(uintptr_t)h_out);
        mix((unsigned long long)(uintptr_t)di); mix((unsigned long long)(uintptr_t)dn); mix((unsigned long long)(uintptr_t)io.params);
        { const int rc = run_host_call(c, c->graph_pack, key, enqueue); if (rc != PFC_OK) return rc; }
        CU(cudaStreamSynchronize(c->stream));
        std::memcpy(wrench, h_out, bW);
        if (nb) std::memcpy(sdot, h_out + bW, bD);
        if (n_pairs) std::memcpy(n_pairs, h_out + bW + bD, bN);
        std::memcpy(fl, h_out + bW + bD + bN, sizeof(int32_t) * ne * ni);
    } else {
        CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni)); CU(c->d_w.ensure(6 * ne * ni));
        CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
        if (nb) { CU(c->d_s.ensure(6 * ne * nb)); CU(c->d_sd.ensure(6 * ne * nb)); }
        CU(copy_in(c, c->d_X.p, X, bX));
        CU(copy_in(c, c->d_tw.p, twist, bT));
        if (nb) CU(copy_in(c, c->d_s.p, s, bS));
        io.X = c->d_X.p; io.twist = c->d_tw.p; io.s = nb ? c->d_s.p : nullptr; io.wrench = c->d_w.p;
        io.sdot = nb ? c->d_sd.p : nullptr; io.n_pairs = c->d_np.p; io.flags = c->d_fl.p;
        int rc = eval_device(c, io);
        if (rc != PFC_OK) return rc;
        CU(copy_out(c, wrench, c->d_w.p, bW));
        if (nb) CU(copy_out(c, sdot, c->d_sd.p, bD));
        if (n_pairs) CU(copy_out(c, n_pairs, c->d_np.p, bN));
        CU(copy_out(c, fl, c->d_fl.p, sizeof(int32_t) * ne * ni));
        CU(cudaStreamSynchronize(c->stream));
        copy_out_finish(c);
    }
    c->lists_np = io.n_pairs; c->lists_fl = io.flags;
    c->lists_n_env = n_env;  // d_np / d_fl / pair lists of this evaluation can be reused by pfc_eval_dual6(X_bp = NULL)
    for (size_t k = 0; k < ne * ni; ++k) {
        if (fl[k] & PFC_FLAG_NONFINITE) return fail(PFC_E_NONFINITE, "Non-finite vertex likely");
        if (fl[k] & PFC_FLAG_OVERFLOW) return fail(PFC_E_CAPACITY, "candidate-pair capacity exceeded");
    }
    return PFC_OK;
}

// ---- one large scene split over several GPUs ------------------------------------------------------------------
// queues this rank's share of a split evaluation (no synchronisation; evaluation_fits() must be asked afterwards)
static int sharded_enqueue(pfc_ctx* c, const EvalIO& io) {
    int nl = 0;
    if (c->scene.n_small > 0) {  // small instructions are cheap: every rank evaluates them completely
        CU(c->d_small_pairs.ensure(size_t(small_cap(c->small_max_pairs)) * io.n_env * c->scene.n_ins + kSmallPairsSlack));
        CU(launch_eval_small_f64(c->scene, io, c->small_max_pairs, c->d_small_pairs.p, c->stream, &nl, nullptr));
    }
    // every rank runs the shared breadth-first levels, then traverses and lists only the sub-trees whose hash falls on it: disjoint pair
    // lists.  Bristle instructions are the exception: their sums run sequentially over the whole TractionCache list (pfc_exact.cuh), so
    // every rank lists and evaluates them completely -- identical bits on every rank, nothing to exchange.
    CU(large_broad_phase(c->scene, c->large_scene, io, c->large_buf, c->stream, &nl, c->shard_rank, c->shard_world));
    CU(large_narrow_stage(c->scene, c->large_scene, io, c->large_buf, c->shard_world > 1, 0, c->stream, &nl));
    int rc = eval_bristle_exact(c, io.n_env, io.X, io.twist, io.s, io.wrench, io.sdot, io.n_pairs, io.flags, nullptr, 0, false, &nl);
    if (rc != PFC_OK) return rc;
    if (c->n_mid > 0) {
        CU(cudaMemcpyAsync(c->h_ins_overflow, c->d_ins_overflow.p, sizeof(int) * c->h_ins.size(), cudaMemcpyDeviceToHost, c->stream));
        c->mid_check_pending = true;
    }
    c->launches += nl;
    c->sharded_io = io;
    c->sharded_stage = 0;
    c->lists_n_env = -1;
    if (c->keep_pairs) c->dbg_n_env = io.n_env;   // (pfc_get_pairs: the large instructions' lists live in the large path's buffers)
    c->last_X = io.X; c->last_tw = io.twist;
    return PFC_OK;
}

int pfc_eval_sharded_begin(pfc_ctx* c, int64_t n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot,
                           int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: context not finalized");
    if (c->params_n_env > 0) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: per-environment contact parameters are not supported by the sharded protocol");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: negative n_env");
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!X || !twist || !wrench || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: NULL buffer");
    if (c->n_bristle > 0 && (!s || !sdot)) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: bristle instructions need s and sdot");
    if (c->large_scene.n_large == 0) return fail(PFC_E_ARG, "pfc_eval_sharded_begin: the scene has no large instruction to split");
    CU(cudaSetDevice(c->device));
    EvalIO io{};
    io.n_env = n_env; io.X = X; io.twist = twist; io.s = s; io.wrench = wrench; io.sdot = sdot;
    io.n_pairs = reinterpret_cast<long long*>(n_pairs); io.flags = flags;
    // one synchronisation at the end of what was queued: the traversal's and the bristle pipeline's buffers grow after the fact
    const int rc = run_evaluation(c, eval_key(2, c, io), [&]() { return sharded_enqueue(c, io); });
    if (rc != PFC_OK) return rc;
    // host-side state of the evaluation in flight (a replayed CUDA graph does not pass through sharded_enqueue)
    c->sharded_io = io;
    c->sharded_stage = 0;
    c->lists_n_env = -1;
    if (c->keep_pairs) c->dbg_n_env = io.n_env;
    c->last_X = io.X; c->last_tw = io.twist;
    return PFC_OK;
}

int pfc_eval_sharded_partials(pfc_ctx* c, double** dev_ptr, int64_t* count) {
    if (!c || c->sharded_stage < 0 || !dev_ptr || !count) return fail(PFC_E_ARG, "pfc_eval_sharded_partials: no sharded evaluation in flight");
    *dev_ptr = c->shard_world > 1 ? large_part_buffer(c->large_buf) : nullptr;
    *count = c->shard_world > 1 ? int64_t(kLargePartStride) * c->sharded_io.n_env * c->large_scene.n_large : 0;
    return PFC_OK;
}

int pfc_eval_sharded_step(pfc_ctx* c, int* more) {
    if (!c || c->sharded_stage < 0 || !more) return fail(PFC_E_ARG, "pfc_eval_sharded_step: no sharded evaluation in flight");
    CU(cudaSetDevice(c->device));
    int nl = 0;
    if (c->shard_world > 1)  // the caller has summed the partial buffer over the ranks: apply it
        CU(large_narrow_stage(c->scene, c->large_scene, c->sharded_io, c->large_buf, 1, 1, c->stream, &nl));
    c->sharded_stage = -1;   // one exchange per evaluation (regularized sums; bristle instructions are not split)
    *more = 0;
    c->launches += nl;
    return PFC_OK;
}

// ---- library-owned collective (SURVEY.md section 8b "pfc_group") -------------------------------------------------------------
// The exchange of a split scene: every rank's per-instruction partial sums (8 doubles per large instruction) are ALL-GATHERED over NCCL
// and added in rank order by sum_ranks_kernel, so every rank holds the same bits; then the sums are applied.  All on the context's stream.
static int sharded_exchange_and_finish(pfc_ctx* c) {
    NcclApi& n = nccl_api();
    const long long count = (long long)kLargePartStride * c->sharded_io.n_env * c->large_scene.n_large;
    if (c->shard_world > 1) {
        double* part = large_part_buffer(c->large_buf);
        CU(c->d_gather.ensure(size_t(count) * c->shard_world));
        NC(n.AllGather(part, c->d_gather.p, size_t(count), ncclDouble, c->comm, c->stream));
        sum_ranks_kernel<<<(unsigned)std::min<long long>((count + 255) / 256, 1024), 256, 0, c->stream>>>(c->d_gather.p, c->shard_world, count, part);
        CU(cudaGetLastError());
        c->launches += 1;
    }
    int more = 0;
    return pfc_eval_sharded_step(c, &more);
}

int pfc_comm_unique_id(void* id128) {
    if (!id128) return fail(PFC_E_ARG, "pfc_comm_unique_id: NULL buffer");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(PFC_E_CUDA, n.error);
    static_assert(sizeof(ncclUniqueId) == 128, "the unique id is handed over as 128 bytes");
    NC(n.GetUniqueId(reinterpret_cast<ncclUniqueId*>(id128)));
    return PFC_OK;
}

int pfc_comm_init_rank(pfc_ctx* c, const void* id128, int rank, int world) {
    if (!c || !id128 || world < 1 || rank < 0 || rank >= world) return fail(PFC_E_ARG, "pfc_comm_init_rank: bad argument");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(PFC_E_CUDA, n.error);
    CU(cudaSetDevice(c->device));
    if (c->comm) { n.CommDestroy(c->comm); c->comm = nullptr; }
    ncclUniqueId id;
    std::memcpy(&id, id128, sizeof id);
    NC(n.CommInitRank(&c->comm, world, id, rank));
    c->shard_rank = rank; c->shard_world = world;
    return PFC_OK;
}

int pfc_eval_sharded_f64_device(pfc_ctx* c, int64_t n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot,
                                int64_t* n_pairs, int32_t* flags) {
    if (c && c->params_n_env > 0) return fail(PFC_E_ARG, "pfc_eval_sharded_f64_device: per-environment contact parameters are not supported by the sharded protocol");
    if (!c || !c->comm) return fail(PFC_E_ARG, "pfc_eval_sharded_f64_device: pfc_comm_init_rank (or pfc_group_create) first");
    int rc = pfc_eval_sharded_begin(c, n_env, X, twist, s, wrench, sdot, n_pairs, flags);
    if (rc != PFC_OK || n_env == 0) return rc;
    return sharded_exchange_and_finish(c);
}

struct pfc_group {
    std::vector<pfc_ctx*> ctx;
};

int pfc_group_create(int n_dev, const int* devices, pfc_group** out) {
    if (n_dev < 1 || !devices || !out) return fail(PFC_E_ARG, "pfc_group_create: bad argument");
    NcclApi& n = nccl_api();
    if (!n.ok()) return fail(PFC_E_CUDA, n.error);
    pfc_group* g = new pfc_group();
    for (int r = 0; r < n_dev; ++r) {
        pfc_ctx* c = nullptr;
        const int rc = pfc_create(devices[r], &c);
        if (rc != PFC_OK) { for (pfc_ctx* x : g->ctx) pfc_destroy(x); delete g; return rc; }
        c->shard_rank = r; c->shard_world = n_dev;
        g->ctx.push_back(c);
    }
    std::vector<ncclComm_t> comms(n_dev);
    ncclResult_t r_ = n.CommInitAll(comms.data(), n_dev, devices);   // one process, one communicator rank per device
    if (r_ != ncclSuccess) { for (pfc_ctx* x : g->ctx) pfc_destroy(x); delete g; return fail(PFC_E_CUDA, std::string("ncclCommInitAll: ") + n.GetErrorString(r_)); }
    for (int r = 0; r < n_dev; ++r) g->ctx[r]->comm = comms[r];
    *out = g;
    return PFC_OK;
}
int pfc_group_destroy(pfc_group* g) {
    if (!g) return PFC_OK;
    for (pfc_ctx* c : g->ctx) pfc_destroy(c);
    delete g;
    return PFC_OK;
}
int pfc_group_size(pfc_group* g) { return g ? int(g->ctx.size()) : 0; }
pfc_ctx* pfc_group_ctx(pfc_group* g, int rank) { return (g && rank >= 0 && rank < int(g->ctx.size())) ? g->ctx[rank] : nullptr; }

// scene description: the same calls on every device of the group
int pfc_group_add_mesh(pfc_group* g, int kind, int64_t n_point, const double* xyz, int64_t n_prim, const int32_t* idx, const double* eps, double Ebar,
                       int64_t n_node, const double* node_c, const double* node_e, const double* node_R, const int32_t* node_left,
                       const int32_t* node_right, const int32_t* node_leaf_id, int* mesh_id_out) {
    if (!g) return fail(PFC_E_ARG, "pfc_group_add_mesh: NULL group");
    for (pfc_ctx* c : g->ctx) {
        const int rc = pfc_add_mesh(c, kind, n_point, xyz, n_prim, idx, eps, Ebar, n_node, node_c, node_e, node_R, node_left, node_right, node_leaf_id, mesh_id_out);
        if (rc != PFC_OK) return rc;
    }
    return PFC_OK;
}
int pfc_group_add_instruction(pfc_group* g, int mesh_1, int mesh_2, double chi, int model, const double* params, int n_quad_rule, int* ins_id_out) {
    if (!g) return fail(PFC_E_ARG, "pfc_group_add_instruction: NULL group");
    for (pfc_ctx* c : g->ctx) { const int rc = pfc_add_instruction(c, mesh_1, mesh_2, chi, model, params, n_quad_rule, ins_id_out); if (rc != PFC_OK) return rc; }
    return PFC_OK;
}
int pfc_group_finalize(pfc_group* g, int64_t max_env) {
    if (!g) return fail(PFC_E_ARG, "pfc_group_finalize: NULL group");
    for (pfc_ctx* c : g->ctx) { const int rc = pfc_finalize(c, max_env); if (rc != PFC_OK) return rc; }
    return PFC_OK;
}

// forceAllElasticIntersections! for a scene split over the group's devices.  Host pointers, as pfc_eval_f64; synchronous at return.
int pfc_group_eval_f64(pfc_group* g, int64_t n_env, const double* X, const double* twist, const double* s, double* wrench, double* sdot, int64_t* n_pairs,
                       int32_t* flags) {
    if (!g || g->ctx.empty()) return fail(PFC_E_ARG, "pfc_group_eval_f64: NULL group");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_group_eval_f64: negative n_env");
    if (n_env == 0) return PFC_OK;
    if (!X || !twist || !wrench) return fail(PFC_E_ARG, "pfc_group_eval_f64: NULL buffer");
    pfc_ctx* c0 = g->ctx[0];
    if (!c0->finalized) return fail(PFC_E_ARG, "pfc_group_eval_f64: pfc_group_finalize first");
    if (c0->n_bristle > 0 && (!s || !sdot)) return fail(PFC_E_ARG, "pfc_group_eval_f64: bristle instructions need s and sdot");
    for (pfc_ctx* c : g->ctx)
        if (c->params_n_env > 0) return fail(PFC_E_ARG, "pfc_group_eval_f64: per-environment contact parameters are not supported by the group protocol");
    if (g->ctx.size() == 1 || c0->large_scene.n_large == 0)   // nothing to split: the plain evaluation on the first device
        return pfc_eval_f64(c0, n_env, X, twist, s, wrench, sdot, n_pairs, flags);
    NcclApi& n = nccl_api();
    const size_t ne = size_t(n_env), ni = size_t(c0->scene.n_ins), nb = size_t(c0->n_bristle);
    std::vector<EvalIO> ios(g->ctx.size());
    // 1. every device: inputs in, its share of the traversal / narrow phase queued
    for (size_t r = 0; r < g->ctx.size(); ++r) {
        pfc_ctx* c = g->ctx[r];
        CU(cudaSetDevice(c->device));
        CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni)); CU(c->d_w.ensure(6 * ne * ni)); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
        if (nb) { CU(c->d_s.ensure(6 * ne * nb)); CU(c->d_sd.ensure(6 * ne * nb)); }
        CU(cudaMemcpyAsync(c->d_X.p, X, sizeof(double) * 16 * ne * ni, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(c->d_tw.p, twist, sizeof(double) * 6 * ne * ni, cudaMemcpyHostToDevice, c->stream));
        if (nb) CU(cudaMemcpyAsync(c->d_s.p, s, sizeof(double) * 6 * ne * nb, cudaMemcpyHostToDevice, c->stream));
        EvalIO& io = ios[r];
        io = EvalIO{};
        io.n_env = n_env; io.X = c->d_X.p; io.twist = c->d_tw.p; io.s = nb ? c->d_s.p : nullptr; io.wrench = c->d_w.p; io.sdot = nb ? c->d_sd.p : nullptr;
        io.n_pairs = c->d_np.p; io.flags = c->d_fl.p;
        const int rc = sharded_enqueue(c, io);
        if (rc != PFC_OK) return rc;
    }
    // 2. did everything fit?  (a device whose buffers overflowed repeats its own share; the others wait at the exchange)
    for (size_t r = 0; r < g->ctx.size(); ++r) {
        pfc_ctx* c = g->ctx[r];
        CU(cudaSetDevice(c->device));
        for (int attempt = 0;; ++attempt) {
            const int fit = evaluation_fits(c);
            if (fit < 0) return fit;
            if (fit == 0) break;
            if (attempt >= 8) return fail(PFC_E_CAPACITY, "candidate-pair / traction buffers kept overflowing");
            const int rc = sharded_enqueue(c, ios[r]);
            if (rc != PFC_OK) return rc;
        }
    }
    // 3. the exchange: all-gather of the partial sums, rank-order sum, apply
    const long long count = (long long)kLargePartStride * n_env * c0->large_scene.n_large;
    for (pfc_ctx* c : g->ctx) { CU(cudaSetDevice(c->device)); CU(c->d_gather.ensure(size_t(count) * g->ctx.size())); }
    NC(n.GroupStart());
    for (pfc_ctx* c : g->ctx) {
        const ncclResult_t r_ = n.AllGather(large_part_buffer(c->large_buf), c->d_gather.p, size_t(count), ncclDouble, c->comm, c->stream);
        if (r_ != ncclSuccess) { n.GroupEnd(); return fail(PFC_E_CUDA, std::string("ncclAllGather: ") + n.GetErrorString(r_)); }
    }
    NC(n.GroupEnd());
    for (pfc_ctx* c : g->ctx) {
        CU(cudaSetDevice(c->device));
        sum_ranks_kernel<<<(unsigned)std::min<long long>((count + 255) / 256, 1024), 256, 0, c->stream>>>(c->d_gather.p, c->shard_world, count, large_part_buffer(c->large_buf));
        CU(cudaGetLastError());
        c->launches += 1;
        int more = 0;
        const int rc = pfc_eval_sharded_step(c, &more);
        if (rc != PFC_OK) return rc;
    }
    // 4. results: every device holds the same wrench; the first one hands them over
    CU(cudaSetDevice(c0->device));
    CU(cudaMemcpyAsync(wrench, c0->d_w.p, sizeof(double) * 6 * ne * ni, cudaMemcpyDeviceToHost, c0->stream));
    if (nb) CU(cudaMemcpyAsync(sdot, c0->d_sd.p, sizeof(double) * 6 * ne * nb, cudaMemcpyDeviceToHost, c0->stream));
    if (n_pairs) CU(cudaMemcpyAsync(n_pairs, c0->d_np.p, sizeof(long long) * ne * ni, cudaMemcpyDeviceToHost, c0->stream));
    std::vector<int32_t> fl_local;
    int32_t* fl = flags;
    if (!fl) { fl_local.resize(ne * ni); fl = fl_local.data(); }
    CU(cudaMemcpyAsync(fl, c0->d_fl.p, sizeof(int32_t) * ne * ni, cudaMemcpyDeviceToHost, c0->stream));
    for (pfc_ctx* c : g->ctx) { CU(cudaSetDevice(c->device)); CU(cudaStreamSynchronize(c->stream)); }
    for (size_t k = 0; k < ne * ni; ++k) {
        if (fl[k] & PFC_FLAG_NONFINITE) return fail(PFC_E_NONFINITE, "Non-finite vertex likely");
        if (fl[k] & PFC_FLAG_OVERFLOW) return fail(PFC_E_CAPACITY, "candidate-pair capacity exceeded");
    }
    return PFC_OK;
}

int pfc_eval_dual6(pfc_ctx* c, int64_t n_env, const double* X_bp, const double* X7, const double* twist7, const double* s7, double* wrench7,
                   double* sdot7, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_eval_dual6: context not finalized");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_dual6: negative n_env");
    { const int rc = params_check(c, "pfc_eval_dual6", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!X7 || !twist7 || !wrench7) return fail(PFC_E_ARG, "pfc_eval_dual6: NULL buffer");
    if (c->n_bristle > 0 && (!s7 || !sdot7)) return fail(PFC_E_ARG, "pfc_eval_dual6: bristle instructions need s7 and sdot7");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle);
    arena_reset(c);
    if (X_bp) {  // traverse with the Float64 transform (calcTriTetIntersections! always uses m.float)
        CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
        CU(copy_in(c, c->d_X.p, X_bp, sizeof(double) * 16 * ne * ni));
    } else if (c->lists_n_env != n_env || !c->lists_np || !c->lists_fl) {
        return fail(PFC_E_ARG, "pfc_eval_dual6: X_bp is NULL but no pair lists of a previous pfc_eval_f64 with the same n_env exist");
    }
    CU(c->d_X7.ensure(112 * ne * ni)); CU(c->d_tw7.ensure(42 * ne * ni)); CU(c->d_w7.ensure(42 * ne * ni)); CU(c->d_dual_ticket.ensure(1));
    if (nb) { CU(c->d_s7.ensure(42 * ne * nb)); CU(c->d_sd7.ensure(42 * ne * nb)); }
    CU(copy_in(c, c->d_X7.p, X7, sizeof(double) * 112 * ne * ni));
    CU(copy_in(c, c->d_tw7.p, twist7, sizeof(double) * 42 * ne * ni));
    if (nb) CU(copy_in(c, c->d_s7.p, s7, sizeof(double) * 42 * ne * nb));
    // pair counts / flags: this call's own traversal, or where the previous Float64 evaluation left them
    long long* const np_d = X_bp ? c->d_np.p : c->lists_np;
    int* const fl_d = X_bp ? c->d_fl.p : c->lists_fl;
    PFC_REQUEUE_LOOP({
        int nl = 0;
        if (X_bp) {
            EvalIO io{};
            io.n_env = n_env; io.X = c->d_X.p; io.n_pairs = c->d_np.p; io.flags = c->d_fl.p;
            if (c->scene.n_small > 0) {
                CU(c->d_small_pairs.ensure(size_t(small_cap(c->small_max_pairs)) * ne * ni + kSmallPairsSlack));
                CU(launch_broad_small_only(c->scene, io, c->small_max_pairs, c->d_small_pairs.p, c->stream, &nl));
            }
            if (c->large_scene.n_large > 0) {
                CU(large_broad_phase(c->scene, c->large_scene, io, c->large_buf, c->stream, &nl));
                CU(large_write_counts(c->scene, c->large_scene, io, c->large_buf, c->stream));
                nl += 1;
            }
        }
        CU(launch_eval_dual6(c->scene, n_env, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->d_w7.p, nb ? c->d_sd7.p : nullptr, np_d, fl_d,
                             c->d_small_pairs.p, small_cap(c->small_max_pairs), c->large_scene.n_large > 0 ? c->large_buf : nullptr, c->d_large_index.p,
                             c->large_scene.n_large, ctx_params(c), c->stream, c->d_dual_ticket.p));
        {   // bristle instructions on Duals, in the reference's operation order
            int rc = eval_bristle_exact(c, n_env, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->d_w7.p, nb ? c->d_sd7.p : nullptr, np_d, fl_d, ctx_params(c),
                                        1, false, &nl);
            if (rc != PFC_OK) return rc;
        }
        c->launches += nl + 1;
    })
    if (X_bp) { c->lists_n_env = n_env; c->lists_np = c->d_np.p; c->lists_fl = c->d_fl.p; }
    CU(copy_out(c, wrench7, c->d_w7.p, sizeof(double) * 42 * ne * ni));
    if (nb) CU(copy_out(c, sdot7, c->d_sd7.p, sizeof(double) * 42 * ne * nb));
    if (n_pairs) CU(copy_out(c, n_pairs, np_d, sizeof(long long) * ne * ni));
    std::vector<int32_t> fl_local;
    int32_t* fl = flags;
    if (!fl) { fl_local.resize(ne * ni); fl = fl_local.data(); }
    CU(copy_out(c, fl, fl_d, sizeof(int32_t) * ne * ni));
    CU(cudaStreamSynchronize(c->stream));
    copy_out_finish(c);
    for (size_t k = 0; k < ne * ni; ++k) {
        if (fl[k] & PFC_FLAG_NONFINITE) return fail(PFC_E_NONFINITE, "Non-finite vertex likely");
        if (fl[k] & PFC_FLAG_OVERFLOW) return fail(PFC_E_CAPACITY, "candidate-pair capacity exceeded");
    }
    return PFC_OK;
}

int pfc_set_debug(pfc_ctx* c, int keep_pairs) {
    if (!c) return fail(PFC_E_ARG, "pfc_set_debug: NULL context");
    c->keep_pairs = keep_pairs != 0;
    return PFC_OK;
}

int pfc_get_pairs(pfc_ctx* c, int64_t env, int ins, int32_t* pairs, int64_t cap, int64_t* n_out) {
    if (!c || !c->finalized || !c->keep_pairs) return fail(PFC_E_ARG, "pfc_get_pairs: call pfc_set_debug(ctx, 1) before evaluating");
    if (env < 0 || env >= c->dbg_n_env || ins < 0 || ins >= c->scene.n_ins) return fail(PFC_E_ARG, "pfc_get_pairs: index out of range");
    if (c->h_ins[ins].small && !c->d_dbg_pairs.p) return fail(PFC_E_ARG, "pfc_get_pairs: call pfc_set_debug(ctx, 1) before evaluating");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    const int64_t ei = env * c->scene.n_ins + ins;
    if (!c->h_ins[ins].small) {
        const int li = int(std::find(c->large_ins_host.begin(), c->large_ins_host.end(), ins) - c->large_ins_host.begin());
        long long nn = 0;
        CU(large_get_pairs(c->large_buf, int(env * c->large_scene.n_large + li), pairs, cap, &nn, c->stream));
        if (n_out) *n_out = nn;
        return PFC_OK;
    }
    long long n = 0;
    CU(cudaMemcpy(&n, c->d_last_np.p + ei, sizeof(long long), cudaMemcpyDeviceToHost));
    if (n_out) *n_out = n;
    const int64_t m = std::min<int64_t>(std::min<int64_t>(n, cap), c->dbg_cap);
    if (pairs && m > 0) CU(cudaMemcpy(pairs, c->d_dbg_pairs.p + 2 * int64_t(c->dbg_cap) * ei, sizeof(int32_t) * 2 * m, cudaMemcpyDeviceToHost));
    return PFC_OK;
}

int pfc_get_traction(pfc_ctx* c, int64_t env, int ins, double* out, int64_t cap_points, int64_t* n_out) {
    if (!c || !c->finalized || !c->keep_pairs || !c->d_dbg_pairs.p) return fail(PFC_E_ARG, "pfc_get_traction: call pfc_set_debug(ctx, 1) before evaluating");
    if (env < 0 || env >= c->dbg_n_env || ins < 0 || ins >= c->scene.n_ins) return fail(PFC_E_ARG, "pfc_get_traction: index out of range");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    const int64_t ei = env * c->scene.n_ins + ins;
    long long n = 0;
    CU(cudaMemcpy(&n, c->d_last_np.p + ei, sizeof(long long), cudaMemcpyDeviceToHost));
    const int cap = int(std::max<int64_t>(cap_points, 1));
    DevBuf<double> d_out; DevBuf<int> d_n;
    CU(d_out.ensure(size_t(8) * cap)); CU(d_n.ensure(1));
    EvalIO io{};
    io.X = c->last_X; io.twist = c->last_tw; io.params = c->last_params;
    const int* d_pairs = c->d_dbg_pairs.p + 2 * int64_t(c->dbg_cap) * ei;
    DevBuf<int> d_tmp;
    if (!c->h_ins[ins].small) {  // large instruction: fetch its sorted pair list and stage it as (a, b) ints
        const int li = int(std::find(c->large_ins_host.begin(), c->large_ins_host.end(), ins) - c->large_ins_host.begin());
        std::vector<int> hp(size_t(2) * std::max<long long>(n, 1));
        long long nn = 0;
        CU(large_get_pairs(c->large_buf, int(env * c->large_scene.n_large + li), hp.data(), n, &nn, c->stream));
        CU(d_tmp.ensure(hp.size()));
        CU(cudaMemcpy(d_tmp.p, hp.data(), hp.size() * sizeof(int), cudaMemcpyHostToDevice));
        d_pairs = d_tmp.p;
    }
    CU(launch_dump_traction(c->scene, io, env, ins, d_pairs, n, d_out.p, cap, d_n.p, c->stream));
    c->launches += 1;
    int np = 0;
    CU(cudaMemcpyAsync(&np, d_n.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (n_out) *n_out = np;
    const int m = std::min(np, cap);
    if (out && m > 0 && cap_points > 0) CU(cudaMemcpy(out, d_out.p, sizeof(double) * 8 * m, cudaMemcpyDeviceToHost));
    d_out.release(); d_n.release(); d_tmp.release();
    return PFC_OK;
}


// ---- device-side prologue / epilogue (floating-joint scenes) ----------------------------------------------------
int pfc_set_bodies(pfc_ctx* c, int n_body, const int32_t* joint_type, const int32_t* q0, const int32_t* v0, const double* pose,
                   const int32_t* mesh_body, int nq, int nv) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_set_bodies: call after pfc_finalize");
    if (n_body < 1 || !joint_type || !q0 || !v0 || !mesh_body || nq < 0 || nv < 0) return fail(PFC_E_ARG, "pfc_set_bodies: bad argument");
    c->h_bodies.assign(n_body, BodyDev{});
    for (int b = 0; b < n_body; ++b) {
        BodyDev& d = c->h_bodies[b];
        if (joint_type[b] != 0 && joint_type[b] != 1)
            return fail(PFC_E_ARG, "pfc_set_bodies: only world-attached bodies (0) and SPQuatFloating joints (1) are handled on the device; "
                                   "use pfc_eval_f64 with host kinematics for other joints");
        d.joint = joint_type[b]; d.q0 = q0[b]; d.v0 = v0[b];
        if (d.joint == 1 && (d.q0 < 0 || d.q0 + 6 > nq || d.v0 < 0 || d.v0 + 6 > nv)) return fail(PFC_E_ARG, "pfc_set_bodies: joint offsets out of range");
        for (int i = 0; i < 9; ++i) d.pose_R[i] = pose ? pose[12 * b + i] : (i % 4 == 0 ? 1.0 : 0.0);
        for (int i = 0; i < 3; ++i) d.pose_t[i] = pose ? pose[12 * b + 9 + i] : 0.0;
    }
    const int n_mesh = int(c->mesh.size()), n_ins = int(c->ins.size());
    c->h_mesh_body.assign(mesh_body, mesh_body + n_mesh);
    for (int m = 0; m < n_mesh; ++m) if (mesh_body[m] < 0 || mesh_body[m] >= n_body) return fail(PFC_E_ARG, "pfc_set_bodies: mesh_body out of range");
    std::vector<int> ins_body(2 * std::max(n_ins, 1)), ptr(n_body + 1, 0), lst;
    for (int k = 0; k < n_ins; ++k) { ins_body[2 * k] = mesh_body[c->ins[k].mesh_1]; ins_body[2 * k + 1] = mesh_body[c->ins[k].mesh_2]; }
    for (int b = 0; b < n_body; ++b) {   // Python / Julia order: for every instruction, body 2 first, then body 1
        for (int k = 0; k < n_ins; ++k) {
            if (ins_body[2 * k + 1] == b) lst.push_back((k << 1) | 1);
            if (ins_body[2 * k] == b) lst.push_back((k << 1) | 0);
        }
        ptr[b + 1] = int(lst.size());
    }
    CU(cudaSetDevice(c->device));
    CU(c->d_bodies.ensure(n_body)); CU(c->d_ins_body.ensure(ins_body.size())); CU(c->d_body_ins_ptr.ensure(ptr.size())); CU(c->d_body_ins.ensure(std::max<size_t>(lst.size(), 1)));
    CU(cudaMemcpy(c->d_bodies.p, c->h_bodies.data(), sizeof(BodyDev) * n_body, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_ins_body.p, ins_body.data(), sizeof(int) * ins_body.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_body_ins_ptr.p, ptr.data(), sizeof(int) * ptr.size(), cudaMemcpyHostToDevice));
    if (!lst.empty()) CU(cudaMemcpy(c->d_body_ins.p, lst.data(), sizeof(int) * lst.size(), cudaMemcpyHostToDevice));
    c->state.bodies = c->d_bodies.p; c->state.ins_body = c->d_ins_body.p; c->state.body_ins_ptr = c->d_body_ins_ptr.p; c->state.body_ins = c->d_body_ins.p;
    c->state.n_body = n_body; c->state.nq = nq; c->state.nv = nv; c->state.n_x = nq + nv + 6 * c->n_bristle;
    c->has_bodies = true;
    return PFC_OK;
}

// one device word collects the error bits of an evaluation (or_error_flags); the host reads 4 bytes back
static cudaError_t status_begin(pfc_ctx* c) {
    cudaError_t e = c->d_status.ensure(1);
    if (e != cudaSuccess) return e;
    if (!c->h_status) { e = cudaHostAlloc(reinterpret_cast<void**>(&c->h_status), sizeof(int), cudaHostAllocDefault); if (e != cudaSuccess) return e; }
    return cudaMemsetAsync(c->d_status.p, 0, sizeof(int), c->stream);
}
static int status_end(pfc_ctx* c, int64_t n_env, bool copy_status = true) {
    if (copy_status) CU(cudaMemcpyAsync(c->h_status, c->d_status.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->lists_n_env = n_env; c->lists_np = c->d_np.p; c->lists_fl = c->d_fl.p;
    if (*c->h_status & PFC_FLAG_NONFINITE) return fail(PFC_E_NONFINITE, "Non-finite vertex likely");
    if (*c->h_status & PFC_FLAG_OVERFLOW) return fail(PFC_E_CAPACITY, "candidate-pair capacity exceeded");
    return PFC_OK;
}

static int eval_state_device(pfc_ctx* c, int64_t n_env, const double* x, double* f_gen, double* sdot, long long* n_pairs, int* flags, const InsParam* params,
                             int* status = nullptr) {
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle);
    CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni)); CU(c->d_w.ensure(6 * ne * ni));
    if (nb) CU(c->d_s.ensure(6 * ne * nb));
    double* dX = c->d_X.p;
    double* dtw = c->d_tw.p;
    double* dw = c->d_w.p;
    double* ds = nb ? c->d_s.p : nullptr;
    int nl = 0;
    CU(launch_state_prologue(c->state, n_env, int(ni), int(nb), x, dX, dtw, ds, c->stream, &nl));
    EvalIO io{};
    io.n_env = n_env; io.X = dX; io.twist = dtw; io.s = ds; io.wrench = dw;
    io.sdot = sdot; io.n_pairs = n_pairs; io.flags = flags; io.params = params;
    int rc = eval_device(c, io);
    if (rc != PFC_OK) return rc;
    CU(launch_state_epilogue(c->state, n_env, int(ni), x, dw, f_gen, c->stream, &nl, flags, status));
    c->launches += nl;
    return PFC_OK;
}

int pfc_eval_state_f64_device(pfc_ctx* c, int64_t n_env, const double* x, double* f_generalized, double* sdot, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_bodies) return fail(PFC_E_ARG, "pfc_eval_state_f64_device: pfc_finalize and pfc_set_bodies first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_state_f64_device: negative n_env");
    { const int rc = params_check(c, "pfc_eval_state_f64_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !f_generalized || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_eval_state_f64_device: NULL buffer");
    if (c->n_bristle > 0 && !sdot) return fail(PFC_E_ARG, "pfc_eval_state_f64_device: bristle instructions need sdot");
    CU(cudaSetDevice(c->device));
    return eval_state_device(c, n_env, x, f_generalized, sdot, reinterpret_cast<long long*>(n_pairs), flags, ctx_params(c));
}

int pfc_eval_state_f64(pfc_ctx* c, int64_t n_env, const double* x, double* f_generalized, double* sdot, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_bodies) return fail(PFC_E_ARG, "pfc_eval_state_f64: pfc_finalize and pfc_set_bodies first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_eval_state_f64: negative n_env");
    { const int rc = params_check(c, "pfc_eval_state_f64", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !f_generalized) return fail(PFC_E_ARG, "pfc_eval_state_f64: NULL buffer");
    if (c->n_bristle > 0 && !sdot) return fail(PFC_E_ARG, "pfc_eval_state_f64: bristle instructions need sdot");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(c->d_x.ensure(ne * nx)); CU(c->d_fgen.ensure(std::max<size_t>(ne * nv, 1))); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
    if (nb) CU(c->d_sd.ensure(6 * ne * nb));
    // everything the call queues: status word, inputs in, kernels, outputs out (the caller synchronises in status_end)
    auto enqueue = [&]() -> int {
        CU(status_begin(c));
        CU(cudaMemsetAsync(c->d_fgen.p, 0, sizeof(double) * ne * nv, c->stream));
        // (Splitting the batch in two and overlapping the copies of one half with the kernels of the other was measured on B200 and is
        // slower -- 379 vs 325 us for 4096 environments: half-size grids no longer fill the GPU and the extra launches / events cost more
        // than the ~50 us of copies they hide.)
        CU(cudaMemcpyAsync(c->d_x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
        int rc = eval_state_device(c, n_env, c->d_x.p, c->d_fgen.p, nb ? c->d_sd.p : nullptr, c->d_np.p, c->d_fl.p, ctx_params(c), c->d_status.p);
        if (rc != PFC_OK) return rc;
        CU(cudaMemcpyAsync(f_generalized, c->d_fgen.p, sizeof(double) * ne * nv, cudaMemcpyDeviceToHost, c->stream));
        if (nb) CU(cudaMemcpyAsync(sdot, c->d_sd.p, sizeof(double) * 6 * ne * nb, cudaMemcpyDeviceToHost, c->stream));
        if (n_pairs) CU(cudaMemcpyAsync(n_pairs, c->d_np.p, sizeof(long long) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
        if (flags) CU(cudaMemcpyAsync(flags, c->d_fl.p, sizeof(int32_t) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(c->h_status, c->d_status.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        return PFC_OK;
    };
    unsigned long long key = 1469598103934665603ull;
    auto mix = [&](unsigned long long v) { key ^= v; key *= 1099511628211ull; };
    mix(5ull); mix((unsigned long long)n_env); mix((unsigned long long)(uintptr_t)x); mix((unsigned long long)(uintptr_t)f_generalized);
    mix((unsigned long long)(uintptr_t)sdot); mix((unsigned long long)(uintptr_t)n_pairs); mix((unsigned long long)(uintptr_t)flags);
    mix((unsigned long long)(uintptr_t)ctx_params(c));
    { const int rc = run_host_call(c, c->graph_host, key, enqueue); if (rc != PFC_OK) return rc; }
    return status_end(c, n_env, false);
}

// inverse of a symmetric positive definite 6x6 by Cholesky (what the reference does per evaluation with cholesky!/ldiv!)
static bool spd6_inverse(const double* H, double* inv) {
    double L[36] = {0};
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) {
            double a = H[6 * i + j];
            for (int k = 0; k < j; ++k) a -= L[6 * i + k] * L[6 * j + k];
            if (i == j) { if (!(a > 0.0)) return false; L[6 * i + i] = std::sqrt(a); }
            else L[6 * i + j] = a / L[6 * j + j];
        }
    for (int c = 0; c < 6; ++c) {   // solve L L' x = e_c
        double y[6], x[6];
        for (int i = 0; i < 6; ++i) { double a = (i == c) ? 1.0 : 0.0; for (int k = 0; k < i; ++k) a -= L[6 * i + k] * y[k]; y[i] = a / L[6 * i + i]; }
        for (int i = 5; i >= 0; --i) { double a = y[i]; for (int k = i + 1; k < 6; ++k) a -= L[6 * k + i] * x[k]; x[i] = a / L[6 * i + i]; }
        for (int i = 0; i < 6; ++i) inv[6 * i + c] = x[i];
    }
    return true;
}

int pfc_set_dynamics(pfc_ctx* c, int n_body, const double* spatial_inertia, const double* gravity) {
    if (!c || !c->has_bodies) return fail(PFC_E_ARG, "pfc_set_dynamics: call after pfc_set_bodies");
    if (n_body != c->state.n_body || !spatial_inertia || !gravity) return fail(PFC_E_ARG, "pfc_set_dynamics: bad argument");
    std::vector<double> H(36 * size_t(n_body), 0.0), Hi(36 * size_t(n_body), 0.0);
    for (int b = 0; b < n_body; ++b) {
        if (c->h_bodies[b].joint == 0) continue;
        for (int i = 0; i < 36; ++i) H[36 * b + i] = spatial_inertia[36 * b + i];
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < i; ++j)
                if (std::fabs(H[36 * b + 6 * i + j] - H[36 * b + 6 * j + i]) > 1e-12 * (std::fabs(H[36 * b + 6 * i + i]) + std::fabs(H[36 * b + 6 * j + j])))
                    return fail(PFC_E_ARG, "pfc_set_dynamics: spatial inertia is not symmetric");
        if (!spd6_inverse(&H[36 * b], &Hi[36 * b])) return fail(PFC_E_ARG, "pfc_set_dynamics: spatial inertia is not positive definite");
    }
    CU(cudaSetDevice(c->device));
    CU(c->d_H.ensure(H.size())); CU(c->d_Hinv.ensure(Hi.size()));
    CU(cudaMemcpy(c->d_H.p, H.data(), sizeof(double) * H.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->d_Hinv.p, Hi.data(), sizeof(double) * Hi.size(), cudaMemcpyHostToDevice));
    c->dyn.H = c->d_H.p; c->dyn.Hinv = c->d_Hinv.p;
    for (int i = 0; i < 3; ++i) c->dyn.gravity[i] = gravity[i];
    c->has_dynamics = true;
    return PFC_OK;
}

static int calcxd_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, const InsParam* params, double* xdot, long long* n_pairs, int* flags,
                         int* status = nullptr) {
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle);
    CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni)); CU(c->d_w.ensure(6 * ne * ni));
    if (nb) { CU(c->d_s.ensure(6 * ne * nb)); CU(c->d_sd.ensure(6 * ne * nb)); }
    int nl = 0;
    CU(launch_state_prologue(c->state, n_env, int(ni), int(nb), x, c->d_X.p, c->d_tw.p, nb ? c->d_s.p : nullptr, c->stream, &nl));
    EvalIO io{};
    io.n_env = n_env; io.X = c->d_X.p; io.twist = c->d_tw.p; io.s = nb ? c->d_s.p : nullptr; io.wrench = c->d_w.p;
    io.sdot = nb ? c->d_sd.p : nullptr; io.n_pairs = n_pairs; io.flags = flags; io.params = params;
    int rc = eval_device(c, io);
    if (rc != PFC_OK) return rc;
    CU(launch_state_dynamics(c->state, c->dyn, n_env, int(ni), int(nb), x, c->d_w.p, tau_ext, nb ? c->d_sd.p : nullptr, xdot, c->stream, &nl, flags, status));
    c->launches += nl;
    return PFC_OK;
}

int pfc_calcxd_f64_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, double* xdot, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_f64_device: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_f64_device: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_f64_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !xdot || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_calcxd_f64_device: NULL buffer");
    CU(cudaSetDevice(c->device));
    return calcxd_device(c, n_env, x, tau_ext, ctx_params(c), xdot, reinterpret_cast<long long*>(n_pairs), flags);
}

int pfc_calcxd_f64(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, double* xdot, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_f64: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_f64: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_f64", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !xdot) return fail(PFC_E_ARG, "pfc_calcxd_f64: NULL buffer");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(c->d_x.ensure(ne * nx)); CU(c->d_xdot.ensure(ne * nx)); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
    CU(cudaMemcpyAsync(c->d_x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
    if (tau_ext) {
        CU(c->d_tau.ensure(std::max<size_t>(ne * nv, 1)));
        CU(cudaMemcpyAsync(c->d_tau.p, tau_ext, sizeof(double) * ne * nv, cudaMemcpyHostToDevice, c->stream));
    }
    CU(cudaMemsetAsync(c->d_xdot.p, 0, sizeof(double) * ne * nx, c->stream));
    CU(status_begin(c));
    int rc = calcxd_device(c, n_env, c->d_x.p, tau_ext ? c->d_tau.p : nullptr, ctx_params(c), c->d_xdot.p, c->d_np.p, c->d_fl.p, c->d_status.p);
    if (rc != PFC_OK) return rc;
    CU(cudaMemcpyAsync(xdot, c->d_xdot.p, sizeof(double) * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    if (n_pairs) CU(cudaMemcpyAsync(n_pairs, c->d_np.p, sizeof(long long) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    if (flags) CU(cudaMemcpyAsync(flags, c->d_fl.p, sizeof(int32_t) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    return status_end(c, n_env);
}

// The Float64 part the seed chunks of a Jacobian share: candidate-pair lists, the wrenches of the regularized instructions (problems whose
// inputs do not depend on a chunk's seeds copy them) and, for the small instructions, the pairs that survive the Float64 clip.
// Expects the Float64 boundary arrays in c->d_X / c->d_tw.
static int dual_shared_f64(pfc_ctx* c, int64_t n_env, long long* n_pairs, int* flags, const InsParam* params, DualShared* sh, int* nl) {
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins);
    CU(c->d_w.ensure(6 * ne * ni));
    EvalIO io{};
    io.n_env = n_env; io.X = c->d_X.p; io.twist = c->d_tw.p; io.wrench = c->d_w.p; io.n_pairs = n_pairs; io.flags = flags; io.params = params;
    sh->surv_pairs = nullptr; sh->surv_n = nullptr; sh->w_f64 = c->d_w.p;
    if (c->scene.n_small > 0) {
        const int cap = small_cap(c->small_max_pairs);
        CU(c->d_small_pairs.ensure(size_t(cap) * ne * ni + kSmallPairsSlack));
        CU(launch_eval_small_f64(c->scene, io, c->small_max_pairs, c->d_small_pairs.p, c->stream, nl, nullptr));
        CU(c->d_surv.ensure(size_t(cap) * ne * ni)); CU(c->d_surv_n.ensure(ne * ni));
        CU(launch_dual_prefilter(c->scene, n_env, c->d_X.p, n_pairs, c->d_small_pairs.p, cap, c->d_surv.p, c->d_surv_n.p, params, c->stream));
        *nl += 1;
        sh->surv_pairs = c->d_surv.p; sh->surv_n = c->d_surv_n.p;
    }
    if (c->large_scene.n_large > 0) {
        if (c->shard_world > 1) return fail(PFC_E_ARG, "this context is sharded: the Jacobian mode needs an unsharded context");
        CU(large_broad_phase(c->scene, c->large_scene, io, c->large_buf, c->stream, nl));
        CU(large_narrow_stage(c->scene, c->large_scene, io, c->large_buf, 0, 0, c->stream, nl));
    }
    if (c->n_mid > 0) {
        CU(cudaMemcpyAsync(c->h_ins_overflow, c->d_ins_overflow.p, sizeof(int) * c->h_ins.size(), cudaMemcpyDeviceToHost, c->stream));
        c->mid_check_pending = true;
    }
    c->lists_n_env = -1;   // the lists belong to caller-owned count / flag arrays: not reusable by pfc_eval_dual6(X_bp = NULL)
    return PFC_OK;
}

// calcXd! in Jacobian mode for the same scenes: x (Float64) with Dual seeds on x[seed_start .. seed_start + 6) -> x_dot as 7 doubles per
// entry (value, then d x_dot / d x[seed_start + k]).  Device pipeline: Float64 prologue + broad phase (the reference always traverses
// with m.float), Dual prologue, Dual narrow phase / friction (pfc_dual.cu), Dual J' w and rigid-body terms.
static int calcxd_dual6_device_once(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, const InsParam* params, int seed_start, double* xdot7,
                                    long long* n_pairs, int* flags, int* status) {
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle);
    CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni));
    CU(c->d_X7.ensure(112 * ne * ni)); CU(c->d_tw7.ensure(42 * ne * ni)); CU(c->d_w7.ensure(42 * ne * ni)); CU(c->d_dual_ticket.ensure(1));
    if (nb) { CU(c->d_s.ensure(6 * ne * nb)); CU(c->d_s7.ensure(42 * ne * nb)); CU(c->d_sd7.ensure(42 * ne * nb)); }
    int nl = 0;
    // Float64 boundary arrays -> candidate-pair lists, Float64 wrenches, survivors of the Float64 clip
    CU(launch_state_prologue(c->state, n_env, int(ni), int(nb), x, c->d_X.p, c->d_tw.p, nb ? c->d_s.p : nullptr, c->stream, &nl));
    DualShared shared{};
    { const int rc = dual_shared_f64(c, n_env, n_pairs, flags, params, &shared, &nl); if (rc != PFC_OK) return rc; }
    // Dual boundary arrays, Dual contact wrenches, Dual rigid-body terms
    CU(launch_state_prologue_dual6(c->state, n_env, int(ni), int(nb), x, seed_start, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->stream, &nl));
    CU(launch_eval_dual6(c->scene, n_env, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->d_w7.p, nb ? c->d_sd7.p : nullptr, n_pairs, flags,
                         c->d_small_pairs.p, small_cap(c->small_max_pairs), c->large_scene.n_large > 0 ? c->large_buf : nullptr, c->d_large_index.p,
                         c->large_scene.n_large, params, c->stream, c->d_dual_ticket.p, 0, &shared));
    {
        int rc = eval_bristle_exact(c, n_env, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->d_w7.p, nb ? c->d_sd7.p : nullptr, n_pairs, flags, params, 1, false,
                                    &nl);
        if (rc != PFC_OK) return rc;
    }
    CU(launch_state_dynamics_dual6(c->state, c->dyn, n_env, int(ni), int(nb), x, seed_start, c->d_w7.p, tau_ext, nb ? c->d_sd7.p : nullptr, xdot7,
                                   c->stream, &nl, flags, status));
    c->launches += nl + 1;
    return PFC_OK;
}
static int calcxd_dual6_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, const InsParam* params, int seed_start, double* xdot7,
                               long long* n_pairs, int* flags, int* status) {
    PFC_REQUEUE_LOOP({ const int rc_ = calcxd_dual6_device_once(c, n_env, x, tau_ext, params, seed_start, xdot7, n_pairs, flags, status); if (rc_ != PFC_OK) return rc_; })
    return PFC_OK;
}

int pfc_calcxd_dual6_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, int seed_start, double* xdot7, int64_t* n_pairs,
                            int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_dual6_device: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_dual6_device: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_dual6_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !xdot7 || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_calcxd_dual6_device: NULL buffer");
    if (seed_start < 0 || seed_start >= c->state.n_x) return fail(PFC_E_ARG, "pfc_calcxd_dual6_device: seed_start out of range");
    CU(cudaSetDevice(c->device));
    return calcxd_dual6_device(c, n_env, x, tau_ext, ctx_params(c), seed_start, xdot7, reinterpret_cast<long long*>(n_pairs), flags, nullptr);
}

int pfc_calcxd_dual6(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, int seed_start, double* xdot7, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_dual6: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_dual6: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_dual6", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !xdot7) return fail(PFC_E_ARG, "pfc_calcxd_dual6: NULL buffer");
    if (seed_start < 0 || seed_start >= c->state.n_x) return fail(PFC_E_ARG, "pfc_calcxd_dual6: seed_start out of range");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(c->d_x.ensure(ne * nx)); CU(c->d_xdot.ensure(7 * ne * nx)); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
    CU(cudaMemcpyAsync(c->d_x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
    if (tau_ext) {
        CU(c->d_tau.ensure(std::max<size_t>(ne * nv, 1)));
        CU(cudaMemcpyAsync(c->d_tau.p, tau_ext, sizeof(double) * ne * nv, cudaMemcpyHostToDevice, c->stream));
    }
    CU(cudaMemsetAsync(c->d_xdot.p, 0, sizeof(double) * 7 * ne * nx, c->stream));
    CU(status_begin(c));
    int rc = calcxd_dual6_device(c, n_env, c->d_x.p, tau_ext ? c->d_tau.p : nullptr, ctx_params(c), seed_start, c->d_xdot.p, c->d_np.p, c->d_fl.p, c->d_status.p);
    if (rc != PFC_OK) return rc;
    CU(cudaMemcpyAsync(xdot7, c->d_xdot.p, sizeof(double) * 7 * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    if (n_pairs) CU(cudaMemcpyAsync(n_pairs, c->d_np.p, sizeof(long long) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    if (flags) CU(cudaMemcpyAsync(flags, c->d_fl.p, sizeof(int32_t) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    int rc2 = status_end(c, n_env);
    c->lists_n_env = -1;
    return rc2;
}

// The whole Jacobian of calcXd! (calcJacobian!, /root/reference/src/radau/radau_functions.jl:2-26: ceil(n_x / 6) passes of calcXd! on
// Dual{6} states, the candidate-pair lists always from the Float64 state).  Here the Float64 kinematics and the broad phase run ONCE; the
// seed chunks are a grid axis of the Dual kernels ("environment" (g, env) = chunk g of real environment env) as far as the work space
// allows, and the rigid-body kernel writes the partials straight into jac[env][row][col].  Scenes with bristle instructions go chunk by
// chunk (their reference-order pipeline is sized per real environment) but still share the broad phase.
static int jacobian_device_once(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, const InsParam* params, double* jac, double* xdot,
                                long long* n_pairs, int* flags, int* status) {
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nb = size_t(c->n_bristle), nx = size_t(c->state.n_x);
    const int n_chunk = int((nx + 5) / 6);
    // chunks per pass: all of them if the Dual boundary arrays (196 doubles per (chunk, environment, instruction)) stay below 1 GiB
    int G = 1;
    if (nb == 0) G = int(std::max<size_t>(1, std::min<size_t>(size_t(n_chunk), (size_t(1) << 30) / std::max<size_t>(1, ne * ni * 196 * sizeof(double)))));
    const size_t nv_env = ne * size_t(G);
    CU(c->d_X.ensure(16 * ne * ni)); CU(c->d_tw.ensure(6 * ne * ni));
    CU(c->d_X7.ensure(112 * nv_env * ni)); CU(c->d_tw7.ensure(42 * nv_env * ni)); CU(c->d_w7.ensure(42 * nv_env * ni)); CU(c->d_dual_ticket.ensure(1));
    if (nb) { CU(c->d_s.ensure(6 * ne * nb)); CU(c->d_s7.ensure(42 * ne * nb)); CU(c->d_sd7.ensure(42 * ne * nb)); }
    int nl = 0;
    CU(launch_state_prologue(c->state, n_env, int(ni), int(nb), x, c->d_X.p, c->d_tw.p, nb ? c->d_s.p : nullptr, c->stream, &nl));
    DualShared shared{};
    { const int rc = dual_shared_f64(c, n_env, n_pairs, flags, params, &shared, &nl); if (rc != PFC_OK) return rc; }
    for (int g0 = 0; g0 < n_chunk; g0 += G) {
        const int g = std::min(G, n_chunk - g0);
        const long long n_virtual = n_env * g;
        CU(launch_state_prologue_dual6(c->state, n_virtual, int(ni), int(nb), x, 6 * g0, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->stream, &nl, n_env));
        CU(launch_eval_dual6(c->scene, n_virtual, c->d_X7.p, c->d_tw7.p, nb ? c->d_s7.p : nullptr, c->d_w7.p, nb ? c->d_sd7.p : nullptr, n_pairs, flags,
                             c->d_small_pairs.p, small_cap(c->small_max_pairs), c->large_scene.n_large > 0 ? c->large_buf : nullptr, c->d_large_index.p,
                             c->large_scene.n_large, params, c->stream, c->d_dual_ticket.p, n_env, &shared));
        nl += 1;
        if (nb) {
            int rc = eval_bristle_exact(c, n_env, c->d_X7.p, c->d_tw7.p, c->d_s7.p, c->d_w7.p, c->d_sd7.p, n_pairs, flags, params, 1, false, &nl);
            if (rc != PFC_OK) return rc;
        }
        CU(launch_state_dynamics_dual6(c->state, c->dyn, n_virtual, int(ni), int(nb), x, 6 * g0, c->d_w7.p, tau_ext, nb ? c->d_sd7.p : nullptr,
                                       g0 == 0 ? xdot : nullptr, c->stream, &nl, flags, status, n_env, jac));
    }
    c->launches += nl;
    return PFC_OK;
}
static int jacobian_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, const InsParam* params, double* jac, double* xdot,
                           long long* n_pairs, int* flags, int* status) {
    PFC_REQUEUE_LOOP({ const int rc_ = jacobian_device_once(c, n_env, x, tau_ext, params, jac, xdot, n_pairs, flags, status); if (rc_ != PFC_OK) return rc_; })
    return PFC_OK;
}

int pfc_calcxd_jacobian_device(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, double* jac, double* xdot, int64_t* n_pairs,
                               int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_jacobian_device: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_jacobian_device: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_jacobian_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !jac || !n_pairs || !flags) return fail(PFC_E_ARG, "pfc_calcxd_jacobian_device: NULL buffer");
    CU(cudaSetDevice(c->device));
    return jacobian_device(c, n_env, x, tau_ext, ctx_params(c), jac, xdot, reinterpret_cast<long long*>(n_pairs), flags, nullptr);
}

int pfc_calcxd_jacobian(pfc_ctx* c, int64_t n_env, const double* x, const double* tau_ext, double* jac, double* xdot, int64_t* n_pairs, int32_t* flags) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_calcxd_jacobian: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_calcxd_jacobian: negative n_env");
    { const int rc = params_check(c, "pfc_calcxd_jacobian", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;   // an empty batch is a no-op whatever the pointers are
    if (!x || !jac) return fail(PFC_E_ARG, "pfc_calcxd_jacobian: NULL buffer");
    CU(cudaSetDevice(c->device));
    const size_t ne = size_t(n_env), ni = size_t(c->scene.n_ins), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(c->d_x.ensure(ne * nx)); CU(c->d_jac.ensure(ne * nx * nx)); CU(c->d_xdot.ensure(ne * nx)); CU(c->d_np.ensure(ne * ni)); CU(c->d_fl.ensure(ne * ni));
    CU(cudaMemcpyAsync(c->d_x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
    if (tau_ext) {
        CU(c->d_tau.ensure(std::max<size_t>(ne * nv, 1)));
        CU(cudaMemcpyAsync(c->d_tau.p, tau_ext, sizeof(double) * ne * nv, cudaMemcpyHostToDevice, c->stream));
    }
    CU(status_begin(c));
    int rc = jacobian_device(c, n_env, c->d_x.p, tau_ext ? c->d_tau.p : nullptr, ctx_params(c), c->d_jac.p, c->d_xdot.p, c->d_np.p, c->d_fl.p, c->d_status.p);
    if (rc != PFC_OK) return rc;
    CU(cudaMemcpyAsync(jac, c->d_jac.p, sizeof(double) * ne * nx * nx, cudaMemcpyDeviceToHost, c->stream));
    if (xdot) CU(cudaMemcpyAsync(xdot, c->d_xdot.p, sizeof(double) * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    if (n_pairs) CU(cudaMemcpyAsync(n_pairs, c->d_np.p, sizeof(long long) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    if (flags) CU(cudaMemcpyAsync(flags, c->d_fl.p, sizeof(int32_t) * ne * ni, cudaMemcpyDeviceToHost, c->stream));
    int rc2 = status_end(c, n_env);
    c->lists_n_env = -1;
    return rc2;
}

int pfc_refit_mesh(pfc_ctx* c, int mesh_id, int64_t n_point, const double* xyz) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_refit_mesh: call after pfc_finalize");
    if (mesh_id < 0 || mesh_id >= int(c->mesh.size()) || !xyz) return fail(PFC_E_ARG, "pfc_refit_mesh: bad argument");
    HostMesh& m = c->mesh[mesh_id];
    if (n_point != m.n_point) return fail(PFC_E_ARG, "pfc_refit_mesh: the number of points must not change (same connectivity)");
    for (int64_t k = 0; k < 3 * n_point; ++k) if (!std::isfinite(xyz[k])) return fail(PFC_E_MESH, "pfc_refit_mesh: non-finite vertex");
    CU(cudaSetDevice(c->device));
    if (c->refit.size() < c->mesh.size()) c->refit.resize(c->mesh.size());
    pfc_ctx::RefitDev& r = c->refit[mesh_id];
    const int64_t n_node = int64_t(m.nodes.size());
    if (!r.ready) {   // connectivity, eps and the internal nodes grouped by depth (pre-order: parents come first)
        std::vector<int> depth(n_node, 0), order;
        int max_depth = 0;
        for (int64_t k = 0; k < n_node; ++k)
            if (m.nodes[k].kind >= 0) { depth[k + 1] = depth[m.nodes[k].right] = depth[k] + 1; max_depth = std::max(max_depth, depth[k]); }
        r.level_ptr.assign(max_depth + 2, 0);
        for (int64_t k = 0; k < n_node; ++k) if (m.nodes[k].kind >= 0) r.level_ptr[depth[k] + 1]++;
        for (int l = 0; l <= max_depth; ++l) r.level_ptr[l + 1] += r.level_ptr[l];
        order.resize(std::max<int>(r.level_ptr[max_depth + 1], 1));
        std::vector<int> cursor(r.level_ptr.begin(), r.level_ptr.end() - 1);
        for (int64_t k = 0; k < n_node; ++k) if (m.nodes[k].kind >= 0) order[cursor[depth[k]]++] = int(k);
        CU(r.idx.ensure(m.idx.size())); CU(r.level_nodes.ensure(order.size()));
        CU(cudaMemcpy(r.idx.p, m.idx.data(), sizeof(int) * m.idx.size(), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(r.level_nodes.p, order.data(), sizeof(int) * order.size(), cudaMemcpyHostToDevice));
        if (m.kind == 1) { CU(r.eps.ensure(m.eps.size())); CU(cudaMemcpy(r.eps.p, m.eps.data(), sizeof(double) * m.eps.size(), cudaMemcpyHostToDevice)); }
        r.ready = true;
    }
    CU(c->d_refit_xyz.ensure(3 * size_t(n_point))); CU(c->d_refit_aabb.ensure(6 * size_t(n_node)));
    CU(cudaMemcpyAsync(c->d_refit_xyz.p, xyz, sizeof(double) * 3 * n_point, cudaMemcpyHostToDevice, c->stream));
    CU(status_begin(c));
    int nl = 0;
    CU(launch_refit(m.kind, m.n_prim, n_node, r.idx.p, m.kind == 1 ? r.eps.p : nullptr, c->d_refit_xyz.p, m.kind == 0 ? c->d_tris.p + m.prim_base : nullptr,
                    m.kind == 1 ? c->d_tets.p + m.prim_base : nullptr, c->d_nodes.p + m.node_base, c->d_refit_aabb.p, r.level_nodes.p, r.level_ptr.data(),
                    int(r.level_ptr.size()) - 1, c->d_status.p, c->stream, &nl));
    c->launches += nl;
    CU(cudaMemcpyAsync(c->h_status, c->d_status.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    c->lists_n_env = -1;   // pair lists of earlier evaluations no longer describe this geometry
    if (*c->h_status & 1) return fail(PFC_E_MESH, "pfc_refit_mesh: inverted or degenerate tetrahedron (the mesh's device records are undefined until a successful refit)");
    m.xyz.assign(xyz, xyz + 3 * n_point);
    return PFC_OK;
}

int pfc_radau_inv_c_device(pfc_ctx* c, int64_t n_mat, int n, const double* neg_J, const double* shift, const int32_t* index, double* inv_c, int32_t* info) {
    if (!c) return fail(PFC_E_ARG, "pfc_radau_inv_c_device: NULL context");
    if (n_mat < 0 || n < 1 || n > 96 || !neg_J || !shift || !inv_c) return fail(PFC_E_ARG, "pfc_radau_inv_c_device: bad argument (1 <= n <= 96)");
    CU(cudaSetDevice(c->device));
    CU(launch_radau_inv_c(n_mat, n, neg_J, shift, index, inv_c, info, c->stream));
    c->launches += 1;
    return PFC_OK;
}

// ---- batched adaptive Radau IIA step (solveRadau, radau_solve.jl:1-34) ------------------------------------------------------------
int pfc_radau_init(pfc_ctx* c, int64_t n_env, int max_rule, double h0, double h_max, double tol_newton) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, "pfc_radau_init: pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (n_env < 0) return fail(PFC_E_ARG, "pfc_radau_init: negative n_env");
    { const int rc = params_check(c, "pfc_radau_init", n_env); if (rc != PFC_OK) return rc; }
    if (max_rule < 1 || max_rule > kRadauMaxRule) return fail(PFC_E_ARG, "pfc_radau_init: max_rule must be 1, 2 or 3");
    if (c->state.n_x < 1 || c->state.n_x > 96) return fail(PFC_E_ARG, "pfc_radau_init: the state must have 1 to 96 entries");
    if (!(std::isfinite(h0) && h0 > 0.0) || !(std::isfinite(h_max) && h_max > 0.0)) return fail(PFC_E_ARG, "pfc_radau_init: h0 and h_max must be finite and positive");
    if (!(tol_newton >= 0.0) || !std::isfinite(tol_newton)) return fail(PFC_E_ARG, "pfc_radau_init: tol_newton must be finite and >= 0");
    CU(cudaSetDevice(c->device));
    pfc_ctx::RadauState& r = c->radau;
    r.n_env = -1;   // not usable until everything below succeeded
    const size_t ne = size_t(n_env), nx = size_t(c->state.n_x), nv = size_t(c->state.nv), ni = size_t(c->scene.n_ins);
    const size_t s_max = size_t(2 * max_rule - 1), ns = std::max<size_t>(ne * s_max, 1), ne1 = std::max<size_t>(ne, 1);
    CU(r.env.ensure(ne1)); CU(r.X.ensure(ns * nx)); CU(r.Xp.ensure(ns * nx)); CU(r.Fp.ensure(ns * nx)); CU(r.taup.ensure(ns * std::max<size_t>(nv, 1)));
    CU(r.xx0.ensure(ne1 * nx)); CU(r.jac.ensure(ne1 * nx * nx)); CU(r.invc.ensure(ns * nx * nx * 2)); CU(r.shift.ensure(2 * ns));
    CU(r.index.ensure(ns)); CU(r.state_list.ensure(ns)); CU(r.env_list.ensure(ne1)); CU(r.state_pos.ensure(ne1)); CU(r.inv_base.ensure(ne1));
    CU(r.counts.ensure(4)); CU(r.info.ensure(1)); CU(r.flags.ensure(ne1 * ni)); CU(r.np.ensure(ne1 * ni)); CU(r.flags_stage.ensure(ns * ni));
    CU(r.np_stage.ensure(ns * ni));
    if (!r.h_counts) CU(cudaHostAlloc(reinterpret_cast<void**>(&r.h_counts), 8 * sizeof(int), cudaHostAllocDefault));
    std::vector<RadauEnv> h_env(ne1);
    for (auto& e : h_env) radau_env_reset(e, h0);
    CU(cudaMemcpy(r.env.p, h_env.data(), sizeof(RadauEnv) * ne1, cudaMemcpyHostToDevice));
    r.n_env = n_env; r.max_rule = max_rule; r.s_max = int(s_max); r.h_max = h_max; r.tol_newton = tol_newton;
    return PFC_OK;
}

static int radau_check(pfc_ctx* c, const char* who, int64_t n_env) {
    if (!c || !c->finalized || !c->has_dynamics) return fail(PFC_E_ARG, std::string(who) + ": pfc_finalize, pfc_set_bodies and pfc_set_dynamics first");
    if (c->radau.n_env < 0) return fail(PFC_E_ARG, std::string(who) + ": pfc_radau_init first");
    if (n_env != c->radau.n_env) return fail(PFC_E_ARG, std::string(who) + ": n_env differs from the one given to pfc_radau_init");
    return params_check(c, who, n_env);
}

static void radau_info_reset(pfc_ctx::RadauState& r) {
    r.rounds = 0; r.syncs = 0;
    for (double& v : r.ms) v = 0.0;
}

// One accepted step for every environment.  Host round trips: one per attempt round (how many environments are pending) and one per Newton
// iteration (how many stage states are still active); the error bits of every evaluation that counts ride along with them.
// The buffer set is the caller's: the context's own for pfc_radau_step, the compact sub-batch of a roll-out round; the work space is sized
// for pfc_radau_init's n_env, which n_env never exceeds.  The step info (rounds, synchronisations, phase times) is added to.
// params: the contact-parameter rows [env][ins] of these environments (or nullptr); they travel like tau_ext, gathered per stage state.
static int radau_step_device(pfc_ctx* c, int64_t n_env, RadauEnv* env, double* x, const double* tau_ext, const InsParam* params, double* t, double* h_taken,
                             int32_t* stats) {
    pfc_ctx::RadauState& r = c->radau;
    const int nx = c->state.n_x, nv = c->state.nv, ni = c->scene.n_ins;
    RadauBufs b{};
    b.n_env = n_env; b.nx = nx; b.nv = nv; b.n_ins = ni; b.s_max = r.s_max; b.max_rule = r.max_rule; b.h_max = r.h_max; b.tol_newton = r.tol_newton;
    b.env = env; b.x = x; b.tau = tau_ext; b.t = t; b.h_taken = h_taken; b.stats = stats;
    b.X = r.X.p; b.Xp = r.Xp.p; b.Fp = r.Fp.p; b.taup = r.taup.p; b.xx0 = r.xx0.p; b.jac = r.jac.p; b.invc = r.invc.p; b.shift = r.shift.p;
    b.index = r.index.p; b.state_list = r.state_list.p; b.env_list = r.env_list.p; b.state_pos = r.state_pos.p; b.inv_base = r.inv_base.p;
    b.counts = r.counts.p; b.bodies = c->d_bodies.p; b.n_body = c->state.n_body;
    if (params) {
        CU(r.paramp.ensure(std::max<size_t>(size_t(r.n_env) * r.s_max * ni, 1)));
        b.params = params; b.paramp = r.paramp.p;
    }
    // phase timing (pfc_set_timing): events around every phase, read after the step's last synchronisation
    std::vector<std::pair<int, int>> marks;   // (phase, index of its start event; the end event follows)
    std::vector<cudaEvent_t>& pool = r.ev_pool;
    auto mark = [&](int phase, bool start) -> cudaError_t {
        if (!c->timing) return cudaSuccess;
        if (start) marks.push_back({phase, int(marks.size() * 2)});
        const size_t k = marks.back().second + (start ? 0 : 1);
        while (pool.size() <= k) { cudaEvent_t ev; cudaError_t e = cudaEventCreate(&ev); if (e != cudaSuccess) return e; pool.push_back(ev); }
        return cudaEventRecord(pool[k], c->stream);
    };
    auto read_back = [&]() -> int {   // counts + status word to the host, one synchronisation; errors of the evaluations so far
        CU(cudaMemcpyAsync(r.h_counts, r.counts.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(r.h_counts + 4, c->d_status.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        r.syncs += 1;
        if (r.h_counts[4] & PFC_FLAG_NONFINITE) return fail(PFC_E_NONFINITE, "Non-finite vertex likely");
        if (r.h_counts[4] & PFC_FLAG_OVERFLOW) return fail(PFC_E_CAPACITY, "candidate-pair capacity exceeded");
        if (r.h_counts[2] & 2) return fail(PFC_E_STEP, "time step is too small, something is wrong");
        if (r.h_counts[2] & 1) return fail(PFC_E_STEP, "unacceptable h");
        return PFC_OK;
    };
    CU(status_begin(c));
    CU(cudaMemsetAsync(r.counts.p, 0, 4 * sizeof(int), c->stream));
    // calcJacobian! once per step: xx_0 and -J (a retry reuses them, radau_solve.jl:23-28)
    CU(mark(0, true));
    { const int rc = jacobian_device(c, n_env, x, tau_ext, params, r.jac.p, r.xx0.p, r.np.p, r.flags.p, nullptr); if (rc != PFC_OK) return rc; }
    CU(launch_radau_prepare(b, r.flags.p, c->d_status.p, c->stream));
    CU(mark(0, false));
    c->launches += 1;
    int mode = 2;
    for (;;) {
        CU(mark(3, true));
        CU(launch_radau_plan(b, mode, c->stream));
        CU(mark(3, false));
        c->launches += 1;
        { const int rc = read_back(); if (rc != PFC_OK) return rc; }
        long long n_states = r.h_counts[0], n_active = r.h_counts[1];
        if (n_states == 0) break;
        r.rounds += 1;
        mode = 1;
        // updateInvC!: one matrix per (pending environment, stage of its rule)
        CU(mark(2, true));
        CU(launch_radau_inv_c(n_states, nx, r.jac.p, r.shift.p, r.index.p, r.invc.p, r.info.p, c->stream));
        CU(mark(2, false));
        c->launches += 1;
        while (n_states > 0) {
            CU(mark(1, true));
            CU(launch_radau_gather(b, n_states, c->stream));
            CU(cudaMemsetAsync(r.Fp.p, 0, sizeof(double) * size_t(n_states) * nx, c->stream));
            { const int rc = calcxd_device(c, n_states, r.Xp.p, tau_ext ? r.taup.p : nullptr, params ? r.paramp.p : nullptr, r.Fp.p, r.np_stage.p, r.flags_stage.p,
                                          c->d_status.p); if (rc != PFC_OK) return rc; }
            CU(mark(1, false));
            CU(mark(3, true));
            CU(launch_radau_newton(b, n_active, c->stream));
            CU(launch_radau_plan(b, 0, c->stream));
            CU(mark(3, false));
            c->launches += 3;
            { const int rc = read_back(); if (rc != PFC_OK) return rc; }
            n_states = r.h_counts[0]; n_active = r.h_counts[1];
        }
        CU(mark(3, true));
        CU(launch_radau_controller(b, c->stream));
        CU(mark(3, false));
        c->launches += 1;
    }
    for (const auto& m : marks) {
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, pool[m.second], pool[m.second + 1]));
        r.ms[m.first] += ms;
    }
    return PFC_OK;
}

int pfc_radau_step_device(pfc_ctx* c, int64_t n_env, double* x, const double* tau_ext, double* t, double* h_taken, int32_t* stats) {
    { const int rc = radau_check(c, "pfc_radau_step_device", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;
    if (!x || !t || !h_taken) return fail(PFC_E_ARG, "pfc_radau_step_device: NULL buffer");
    CU(cudaSetDevice(c->device));
    radau_info_reset(c->radau);
    return radau_step_device(c, n_env, c->radau.env.p, x, tau_ext, ctx_params(c), t, h_taken, stats);
}

int pfc_radau_step(pfc_ctx* c, int64_t n_env, double* x, const double* tau_ext, double* t, double* h_taken, int32_t* stats) {
    { const int rc = radau_check(c, "pfc_radau_step", n_env); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;
    if (!x || !t || !h_taken) return fail(PFC_E_ARG, "pfc_radau_step: NULL buffer");
    CU(cudaSetDevice(c->device));
    pfc_ctx::RadauState& r = c->radau;
    const size_t ne = size_t(n_env), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(r.x.ensure(ne * nx)); CU(r.t.ensure(ne)); CU(r.h.ensure(ne)); CU(r.stats.ensure(4 * ne));
    if (tau_ext) CU(r.tau.ensure(std::max<size_t>(ne * nv, 1)));
    CU(cudaMemcpyAsync(r.x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(r.t.p, t, sizeof(double) * ne, cudaMemcpyHostToDevice, c->stream));
    if (tau_ext) CU(cudaMemcpyAsync(r.tau.p, tau_ext, sizeof(double) * ne * nv, cudaMemcpyHostToDevice, c->stream));
    radau_info_reset(r);
    const int rc = radau_step_device(c, n_env, r.env.p, r.x.p, tau_ext ? r.tau.p : nullptr, ctx_params(c), r.t.p, r.h.p, r.stats.p);
    if (rc != PFC_OK) { cudaStreamSynchronize(c->stream); return rc; }
    CU(cudaMemcpyAsync(x, r.x.p, sizeof(double) * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(t, r.t.p, sizeof(double) * ne, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h_taken, r.h.p, sizeof(double) * ne, cudaMemcpyDeviceToHost, c->stream));
    if (stats) CU(cudaMemcpyAsync(stats, r.stats.p, sizeof(int32_t) * 4 * ne, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return PFC_OK;
}

// ---- roll-outs through shared knot times: rounds of one step for every environment with a knot ahead and steps left ---------------
static int radau_rollout_check(pfc_ctx* c, const char* who, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps) {
    { const int rc = radau_check(c, who, n_env); if (rc != PFC_OK) return rc; }
    if (n_knot < 1 || !t_knot) return fail(PFC_E_ARG, std::string(who) + ": at least one knot time");
    for (int k = 0; k < n_knot; ++k) {
        if (!std::isfinite(t_knot[k])) return fail(PFC_E_ARG, std::string(who) + ": non-finite knot time");
        if (k > 0 && !(t_knot[k] - t_knot[k - 1] >= kRadauHMin)) return fail(PFC_E_ARG, std::string(who) + ": knot times must increase by at least h_min = 1e-8");
    }
    if (max_steps < 1) return fail(PFC_E_ARG, std::string(who) + ": max_steps must be at least 1");
    return PFC_OK;
}

// Host round trips: one per round (how many environments take a step), besides the step's own.  The first selection also checks every
// environment's distance to knot 0, before anything the caller sees is written.
static int radau_rollout_device(pfc_ctx* c, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps, double* x, const double* tau_ext,
                                double* t, double* x_knot, int32_t* stats) {
    pfc_ctx::RadauState& r = c->radau;
    const size_t ne = size_t(n_env), nx = size_t(c->state.n_x), nv = size_t(c->state.nv);
    CU(r.knots.ensure(size_t(n_knot))); CU(r.knot.ensure(ne)); CU(r.steps.ensure(ne)); CU(r.ro_stats.ensure(4 * ne)); CU(r.list.ensure(ne));
    CU(r.env_c.ensure(ne)); CU(r.x_c.ensure(ne * nx)); CU(r.tau_c.ensure(ne * std::max<size_t>(nv, 1))); CU(r.t_c.ensure(ne)); CU(r.h_c.ensure(ne));
    CU(r.h_save.ensure(ne)); CU(r.stats_c.ensure(4 * ne)); CU(r.ro_count.ensure(2));
    const InsParam* params = ctx_params(c);
    if (params) CU(r.params_c.ensure(ne * size_t(c->scene.n_ins)));
    RadauRolloutBufs b{};
    b.n_env = n_env; b.max_steps = max_steps; b.nx = int(nx); b.nv = int(nv); b.n_knot = n_knot;
    b.knots = r.knots.p; b.env = r.env.p; b.x = x; b.tau = tau_ext; b.t = t; b.x_knot = x_knot; b.knot = r.knot.p; b.steps = r.steps.p;
    b.stats = r.ro_stats.p; b.list = r.list.p; b.env_c = r.env_c.p; b.x_c = r.x_c.p; b.tau_c = r.tau_c.p; b.t_c = r.t_c.p; b.h_c = r.h_c.p;
    b.h_save = r.h_save.p; b.stats_c = r.stats_c.p; b.count = r.ro_count.p;
    b.params = params; b.params_c = params ? r.params_c.p : nullptr; b.n_ins = c->scene.n_ins;
    radau_info_reset(r);
    CU(cudaMemcpyAsync(r.knots.p, t_knot, sizeof(double) * n_knot, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(r.knot.p, 0, sizeof(int) * ne, c->stream));
    CU(cudaMemsetAsync(r.steps.p, 0, sizeof(int) * ne, c->stream));
    CU(cudaMemsetAsync(r.ro_stats.p, 0, sizeof(int) * 4 * ne, c->stream));
    for (int round = 0;; ++round) {
        CU(launch_radau_select(b, round == 0, c->stream));
        c->launches += 1;
        CU(cudaMemcpyAsync(r.h_counts + 5, r.ro_count.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        r.syncs += 1;
        if (r.h_counts[6]) return fail(PFC_E_ARG, "pfc_radau_rollout: t_knot[0] - t < h_min for some environment");
        if (round == 0 && x_knot) CU(cudaMemsetAsync(x_knot, 0xFF, sizeof(double) * n_knot * ne * nx, c->stream));   // all-ones bytes: a NaN
        const long long n_active = r.h_counts[5];
        if (n_active == 0) break;
        { const int rc = radau_step_device(c, n_active, r.env_c.p, r.x_c.p, tau_ext ? r.tau_c.p : nullptr, params ? r.params_c.p : nullptr, r.t_c.p, r.h_c.p,
                                           r.stats_c.p); if (rc != PFC_OK) return rc; }
        CU(launch_radau_finish(b, n_active, c->stream));
        c->launches += 1;
    }
    if (stats) CU(cudaMemcpyAsync(stats, r.ro_stats.p, sizeof(int32_t) * 4 * ne, cudaMemcpyDeviceToDevice, c->stream));
    return PFC_OK;
}

int pfc_radau_rollout_device(pfc_ctx* c, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps, double* x, const double* tau_ext, double* t,
                             double* x_knot, int32_t* stats) {
    { const int rc = radau_rollout_check(c, "pfc_radau_rollout_device", n_env, n_knot, t_knot, max_steps); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;
    if (!x || !t) return fail(PFC_E_ARG, "pfc_radau_rollout_device: NULL buffer");
    CU(cudaSetDevice(c->device));
    return radau_rollout_device(c, n_env, n_knot, t_knot, max_steps, x, tau_ext, t, x_knot, stats);
}

int pfc_radau_rollout(pfc_ctx* c, int64_t n_env, int n_knot, const double* t_knot, int64_t max_steps, double* x, const double* tau_ext, double* t,
                      double* x_knot, int32_t* stats) {
    { const int rc = radau_rollout_check(c, "pfc_radau_rollout", n_env, n_knot, t_knot, max_steps); if (rc != PFC_OK) return rc; }
    if (n_env == 0) return PFC_OK;
    if (!x || !t) return fail(PFC_E_ARG, "pfc_radau_rollout: NULL buffer");
    CU(cudaSetDevice(c->device));
    pfc_ctx::RadauState& r = c->radau;
    const size_t ne = size_t(n_env), nx = size_t(c->state.n_x), nv = size_t(c->state.nv), nk = size_t(n_knot);
    CU(r.x.ensure(ne * nx)); CU(r.t.ensure(ne)); CU(r.stats.ensure(4 * ne));
    if (tau_ext) CU(r.tau.ensure(std::max<size_t>(nk * ne * nv, 1)));
    if (x_knot) CU(r.x_knot.ensure(nk * ne * nx));
    CU(cudaMemcpyAsync(r.x.p, x, sizeof(double) * ne * nx, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(r.t.p, t, sizeof(double) * ne, cudaMemcpyHostToDevice, c->stream));
    if (tau_ext) CU(cudaMemcpyAsync(r.tau.p, tau_ext, sizeof(double) * nk * ne * nv, cudaMemcpyHostToDevice, c->stream));
    const int rc = radau_rollout_device(c, n_env, n_knot, t_knot, max_steps, r.x.p, tau_ext ? r.tau.p : nullptr, r.t.p, x_knot ? r.x_knot.p : nullptr,
                                        r.stats.p);
    if (rc != PFC_OK) { cudaStreamSynchronize(c->stream); return rc; }
    CU(cudaMemcpyAsync(x, r.x.p, sizeof(double) * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(t, r.t.p, sizeof(double) * ne, cudaMemcpyDeviceToHost, c->stream));
    if (x_knot) CU(cudaMemcpyAsync(x_knot, r.x_knot.p, sizeof(double) * nk * ne * nx, cudaMemcpyDeviceToHost, c->stream));
    if (stats) CU(cudaMemcpyAsync(stats, r.stats.p, sizeof(int32_t) * 4 * ne, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return PFC_OK;
}

int pfc_radau_step_info(pfc_ctx* c, double* ms, int64_t* counts) {
    if (!c || c->radau.n_env < 0) return fail(PFC_E_ARG, "pfc_radau_step_info: pfc_radau_init first");
    if (ms) for (int k = 0; k < 4; ++k) ms[k] = c->radau.ms[k];
    if (counts) { counts[0] = c->radau.rounds; counts[1] = c->radau.syncs; }
    return PFC_OK;
}

int pfc_get_boundary(pfc_ctx* c, int64_t n_env, double* X, double* twist, double* wrench) {
    if (!c || !c->finalized) return fail(PFC_E_ARG, "pfc_get_boundary: context not finalized");
    const size_t n = size_t(n_env) * size_t(c->scene.n_ins);
    if (c->d_X.n < 16 * n || c->d_tw.n < 6 * n || c->d_w.n < 6 * n) return fail(PFC_E_ARG, "pfc_get_boundary: no evaluation of that size has run");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    if (X) CU(cudaMemcpy(X, c->d_X.p, sizeof(double) * 16 * n, cudaMemcpyDeviceToHost));
    if (twist) CU(cudaMemcpy(twist, c->d_tw.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost));
    if (wrench) CU(cudaMemcpy(wrench, c->d_w.p, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost));
    return PFC_OK;
}

int pfc_set_shard(pfc_ctx* c, int rank, int world) {
    if (!c || world < 1 || rank < 0 || rank >= world) return fail(PFC_E_ARG, "pfc_set_shard: bad rank/world");
    c->shard_rank = rank; c->shard_world = world;
    return PFC_OK;
}

int pfc_sync(pfc_ctx* c) {
    if (!c) return fail(PFC_E_ARG, "pfc_sync: NULL context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return PFC_OK;
}

int pfc_measure_fp64_peak(pfc_ctx* c, double* tflops) {
    if (!c || !tflops) return fail(PFC_E_ARG, "pfc_measure_fp64_peak: NULL argument");
    CU(cudaSetDevice(c->device));
    CU(measure_fp64_peak(c->stream, tflops));
    c->launches += 5;
    return PFC_OK;
}

int pfc_set_timing(pfc_ctx* c, int on) {
    if (!c) return fail(PFC_E_ARG, "pfc_set_timing: NULL context");
    CU(cudaSetDevice(c->device));
    if (on && !c->ev[0]) for (int k = 0; k < 8; ++k) CU(cudaEventCreate(&c->ev[k]));
    c->timing = on != 0;
    c->ev_valid = false;
    return PFC_OK;
}

int pfc_kernel_times(pfc_ctx* c, double* ms, int n) {
    if (!c || !ms || n < 2) return fail(PFC_E_ARG, "pfc_kernel_times: bad argument");
    if (!c->ev_valid) return fail(PFC_E_ARG, "pfc_kernel_times: enable pfc_set_timing and evaluate first");
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->ev[2]));
    float a = 0, b = 0;
    CU(cudaEventElapsedTime(&a, c->ev[0], c->ev[1]));
    CU(cudaEventElapsedTime(&b, c->ev[1], c->ev[2]));
    ms[0] = a; ms[1] = b;
    for (int k = 2; k < n; ++k) ms[k] = 0.0;
    return PFC_OK;
}

void* pfc_stream(pfc_ctx* c) { return c ? (void*)c->stream : nullptr; }
int64_t pfc_launch_count(pfc_ctx* c) { return c ? c->launches : 0; }
int pfc_counters(pfc_ctx* c, int64_t* a, int64_t* b) {
    if (!c) return fail(PFC_E_ARG, "pfc_counters: NULL context");
    if (a) *a = c->large_buf ? (int64_t)large_last_tests(c->large_buf) : 0;
    if (b) *b = c->large_buf ? (int64_t)large_last_pairs(c->large_buf) : 0;
    return PFC_OK;
}

}  // extern "C"
