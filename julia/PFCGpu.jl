# PFCGpu.jl -- the reference-side binding of libpfc_b200.so (include/pfc.h).
#
# NOT RUNNABLE IN THE BUILD ENVIRONMENT (no Julia in the image); written against the pinned
# Manifest of ryanelandt/PressureFieldContact.jl (Julia >= 1.1, RigidBodyDynamics 1.4.0) for a
# maintainer to drop next to src/PressureFieldContact.jl.  It replaces ONLY
# forceAllElasticIntersections!(m, tm) (src/contact_algorithms_non_friction.jl:60-68); rigid-body
# kinematics, the controller, the Cholesky solve and Radau stay exactly as they are.
#
#   m = MechanismScenario(de = PFCGpu.calcXd_gpu!)   # plug-in point: src/mechanism_scenario.jl:181
#   ... add_contact! / add_body_contact! / add_friction_*! ... ; finalize!(m)
#   PFCGpu.finalize_gpu!(m)                          # one-time upload of meshes, trees, instructions
#   integrate_scenario_radau(Radau_for_MechanismScenario(m), t_final = 5.0)
module PFCGpu

using PressureFieldContact
using PressureFieldContact: MechanismScenario, TypedMechanismScenario, ContactInstructions, Regularized, Bristle,
    refreshJacobians!, refreshBodyBodyTransform!, refreshBodyBodyCache!, addGeneralizedForcesThirdLaw!,
    get_bristle_d0, get_bristle_d1, get_tree, get_c_prop, sum_all_forces!, as_static_vector
using PressureFieldContact.Binary_BB_Trees: bin_BB_Tree, OBB, is_leaf
using RigidBodyDynamics
using RigidBodyDynamics.Spatial: Wrench, angular, linear
using ForwardDiff: Dual, value, partials
using StaticArrays
using LinearAlgebra

const LIB = get(ENV, "PFC_B200_LIB", "libpfc_b200.so")
const CTX = IdDict{MechanismScenario,Ptr{Cvoid}}()

check(rc::Cint) = rc == 0 || error("pfc: " * unsafe_string(ccall((:pfc_last_error, LIB), Cstring, ())))

# --- one-time upload -------------------------------------------------------------------------------------------
"Pre-order flattening of bin_BB_Tree (src/obb/tree_types.jl:1-16): node 0 is the root; 0-based ids; -1 = none."
function flatten(tree::bin_BB_Tree{OBB})
    c = Float64[]; e = Float64[]; R = Float64[]; left = Int32[]; right = Int32[]; leaf = Int32[]
    function visit(t)
        k = length(left)
        append!(c, t.box.c); append!(e, t.box.e); append!(R, t.box.R[:])    # R column-major, as SMatrix stores it
        push!(left, -1); push!(right, -1); push!(leaf, is_leaf(t) ? Int32(t.id - 1) : Int32(-1))
        if !is_leaf(t)
            left[k + 1] = visit(t.node_1)
            right[k + 1] = visit(t.node_2)
        end
        return Int32(k)
    end
    visit(tree)
    return c, e, R, left, right, leaf
end

function finalize_gpu!(m::MechanismScenario; device::Integer = 0, max_env::Integer = 1)
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:pfc_create, LIB), Cint, (Cint, Ref{Ptr{Cvoid}}), device, ref))
    ctx = ref[]
    for id in m.mesh_ids                                      # MeshCache: src/structs.jl:33-54
        mc = m.MeshCache[id]
        eM = mc.mesh
        xyz = collect(Iterators.flatten(eM.point))
        is_tet = eM.tet !== nothing
        idx = Int32.(collect(Iterators.flatten(is_tet ? eM.tet : eM.tri)) .- 1)
        c, e, R, l, r, leaf = flatten(get_tree(mc))
        eps_ptr = is_tet ? pointer(eM.ϵ) : Ptr{Float64}(C_NULL)
        out = Ref{Cint}(-1)
        GC.@preserve xyz idx c e R l r leaf eM check(ccall((:pfc_add_mesh, LIB), Cint,
            (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ref{Cint}),
            ctx, is_tet ? 1 : 0, length(eM.point), xyz, is_tet ? length(eM.tet) : length(eM.tri), idx, eps_ptr,
            is_tet ? get_c_prop(mc).Ē : 0.0, length(l), c, e, R, l, r, leaf, out))
        @assert out[] == Int(id) - 1
    end
    for ci in m.ContactInstructions                           # src/mechanism_scenario.jl:36-49
        fm = ci.FrictionModel
        model, params = fm isa Regularized ? (0, [fm.μs, fm.μd, fm.v_c]) : (1, [fm.τ, fm.k̄, fm.μs, fm.μd, fm.magic])
        n_quad_rule = length(ci.quad.w) == 1 ? 1 : 2
        check(ccall((:pfc_add_instruction, LIB), Cint, (Ptr{Cvoid}, Cint, Cint, Float64, Cint, Ptr{Float64}, Cint, Ptr{Cint}),
            ctx, Int(ci.id_1) - 1, Int(ci.id_2) - 1, ci.χ, model, params, n_quad_rule, C_NULL))
    end
    check(ccall((:pfc_finalize, LIB), Cint, (Ptr{Cvoid}, Int64), ctx, max_env))
    CTX[m] = ctx
    return nothing
end

# --- per-evaluation boundary arrays (host kinematics stay with RigidBodyDynamics) -----------------------------
function boundary!(X::Matrix{T}, tw::Matrix{T}, m::MechanismScenario, tm::TypedMechanismScenario{T}) where {T}
    for (k, ci) in enumerate(m.ContactInstructions)
        refreshBodyBodyCache!(m, tm, ci)                      # src/contact_algorithms_non_friction.jl:117-134
        b = tm.bodyBodyCache
        X[:, k] .= SMatrix{4,4,T,16}(b.x_r²_r¹)[:]            # column-major 4x4
        tw[:, k] .= as_static_vector(b.twist_r²_r¹_r²)        # angular first (src/utility.jl:13-14)
    end
end

"Drop-in for forceAllElasticIntersections!(m, tm), Float64 mode."
function force_all_gpu!(m::MechanismScenario, tm::TypedMechanismScenario{Float64})
    ctx = CTX[m]
    n_ins = length(m.ContactInstructions)
    X = Matrix{Float64}(undef, 16, n_ins); tw = Matrix{Float64}(undef, 6, n_ins)
    refreshJacobians!(m, tm)
    tm.f_generalized .= 0.0
    boundary!(X, tw, m, tm)
    w = Matrix{Float64}(undef, 6, n_ins)
    s = tm.s.parent; sdot = tm.ṡ.parent
    GC.@preserve X tw w s sdot check(ccall((:pfc_eval_f64, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        ctx, 1, X, tw, isempty(s) ? C_NULL : pointer(s), w, isempty(sdot) ? C_NULL : pointer(sdot), C_NULL, C_NULL))
    apply_wrenches!(m, tm, w)
end

"Jacobian chunks: every Dual{Nothing,Float64,6} is 7 doubles (value, partials); the broad phase uses m.float's state (R8)."
function force_all_gpu!(m::MechanismScenario, tm::TypedMechanismScenario{Dual{Nothing,Float64,6}})
    ctx = CTX[m]; TD = Dual{Nothing,Float64,6}
    n_ins = length(m.ContactInstructions)
    Xf = Matrix{Float64}(undef, 16, n_ins); twf = Matrix{Float64}(undef, 6, n_ins)
    boundary!(Xf, twf, m, m.float)                            # src/contact_algorithms_non_friction.jl:94-101
    X = Matrix{TD}(undef, 16, n_ins); tw = Matrix{TD}(undef, 6, n_ins)
    refreshJacobians!(m, tm)
    tm.f_generalized .= zero(TD)
    boundary!(X, tw, m, tm)
    w = Matrix{TD}(undef, 6, n_ins)
    s = tm.s.parent; sdot = tm.ṡ.parent                        # isbits Duals are laid out as 7 contiguous Float64
    GC.@preserve Xf X tw w s sdot check(ccall((:pfc_eval_dual6, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        ctx, 1, Xf, pointer(X), pointer(tw), isempty(s) ? C_NULL : pointer(s), pointer(w), isempty(sdot) ? C_NULL : pointer(sdot), C_NULL, C_NULL))
    apply_wrenches!(m, tm, w)
end

function apply_wrenches!(m, tm::TypedMechanismScenario{T}, w::Matrix{T}) where {T}
    for (k, ci) in enumerate(m.ContactInstructions)
        all(iszero, view(w, :, k)) && continue
        refreshBodyBodyTransform!(m, tm, ci)                  # sets bodyBodyCache.mesh_1/2 and x_rʷ_r²
        frame = tm.bodyBodyCache.mesh_2.FrameID
        wrench = Wrench(frame, SVector{3,T}(w[1, k], w[2, k], w[3, k]), SVector{3,T}(w[4, k], w[5, k], w[6, k]))
        addGeneralizedForcesThirdLaw!(wrench, tm, ci)         # src/contact_algorithms_non_friction.jl:267-273
    end
    return nothing
end

"calcXd! (src/contact_algorithms_non_friction.jl:18-38) with the contact-wrench evaluation on the GPU."
function calcXd_gpu!(xx::AbstractVector{T}, x::AbstractVector{T}, m::MechanismScenario, t::Float64 = 0.0) where {T}
    tm = T == Float64 ? m.float : m.dual
    state = tm.state
    copyto!(tm, x)
    H = tm.result.massmatrix
    mass_matrix!(H, state)
    dynamics_bias!(tm.result, state)
    configuration_derivative!(tm.result.q̇, state)
    force_all_gpu!(m, tm)
    (m.continuous_controller == nothing) || m.continuous_controller(tm, t)
    sum_all_forces!(m, tm)
    chol_fact = LinearAlgebra.cholesky!(H)
    ldiv!(tm.result.v̇.parent, chol_fact, tm.rhs)
    copyto!(xx, tm, tm.result)
    return nothing
end

# --- batched roll-outs of floating-body scenes: states in, x_dot (and Jacobian chunks) out, no host RigidBodyDynamics in the loop ---------
"""
    finalize_floating_gpu!(m)

After `finalize_gpu!`: describes the mechanism to the device (`pfc_set_bodies`, `pfc_set_dynamics`).  Every non-root body must sit on an
`SPQuatFloating` joint attached to the world (what `add_body_contact!` creates by default, src/mechanism_scenario.jl:279-289).
"""
function finalize_floating_gpu!(m::MechanismScenario)
    ctx = CTX[m]
    mech = m.float.state.mechanism
    bs = collect(bodies(mech))
    nb = length(bs)
    jt = zeros(Int32, nb); q0 = zeros(Int32, nb); v0 = zeros(Int32, nb); pose = zeros(Float64, 12, nb); H = zeros(Float64, 36, nb)
    for (k, b) in enumerate(bs)
        pose[[1, 5, 9], k] .= 1.0
        isroot(b, mech) && continue
        j = joint_to_parent(b, mech)
        (joint_type(j) isa SPQuatFloating && isroot(predecessor(j, mech), mech)) || error("finalize_floating_gpu!: only SPQuatFloating joints on the world")
        jt[k] = 1
        q0[k] = first(parentindexes(configuration(m.float.state, j))[1]) - 1
        v0[k] = first(parentindexes(velocity(m.float.state, j))[1]) - 1
        tf = joint_to_predecessor(j)                                         # joint pose on the world: R row-major, then t
        pose[1:9, k] .= vec(transpose(rotation(tf))); pose[10:12, k] .= translation(tf)
        I = spatial_inertia(b)                                               # about the body origin, body frame
        c = I.cross_part; cx = [0 -c[3] c[2]; c[3] 0 -c[1]; -c[2] c[1] 0]
        H[:, k] .= vec(transpose([Matrix(I.moment) cx; transpose(cx) I.mass * Matrix(1.0LinearAlgebra.I, 3, 3)]))
    end
    mesh_body = Int32[findfirst(b -> BodyID(b) == m.MeshCache[id].BodyID, bs) - 1 for id in m.mesh_ids]
    nq, nv = num_positions(mech), num_velocities(mech)
    GC.@preserve jt q0 v0 pose mesh_body check(ccall((:pfc_set_bodies, LIB), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Cint, Cint), ctx, nb, jt, q0, v0, pose, mesh_body, nq, nv))
    g = Vector{Float64}(mech.gravitational_acceleration.v)
    GC.@preserve H g check(ccall((:pfc_set_dynamics, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}), ctx, nb, H, g))
    return nothing
end

"Per-environment contact parameters (pfc_set_contact_params): `params[:, ins, env]` = (chi, Ebar_1, Ebar_2, q0..q4) with q = (mu_s, mu_d,
v_c, -, -) for a regularized instruction and (tau, k_bar, mu_s, mu_d, magic) for a bristle one; every batched call then takes
n_env = size(params, 3).  `nothing` clears the table."
function set_contact_params!(m::MechanismScenario, params::Union{Array{Float64,3},Nothing})
    if params === nothing
        check(ccall((:pfc_set_contact_params, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}), CTX[m], 0, C_NULL))
    else
        size(params, 1) == 8 || error("params must be 8 x n_ins x n_env")
        GC.@preserve params check(ccall((:pfc_set_contact_params, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}), CTX[m], size(params, 3), params))
    end
    return nothing
end

"Per-environment body parameters (pfc_set_body_params), after `finalize_floating_gpu!`: `H[:, body, env]` = the body's 6x6 spatial inertia
as `finalize_floating_gpu!` lays it out (`vec(transpose(M))`, M = [moment cx; cx' mass I] about the body origin in the body frame; columns of
the root are ignored), `g[:, env]` = gravity in the world frame; the calcXd!, Jacobian and Radau calls then take n_env = size(H, 3).
`nothing` clears the table."
function set_body_params!(m::MechanismScenario, H::Union{Array{Float64,3},Nothing}, g::Union{Matrix{Float64},Nothing}=nothing)
    if H === nothing
        check(ccall((:pfc_set_body_params, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}), CTX[m], 0, C_NULL, C_NULL))
    else
        nb = length(collect(bodies(m.float.state.mechanism)))
        (size(H, 1) == 36 && size(H, 2) == nb) || error("H must be 36 x n_body x n_env")
        (g !== nothing && size(g) == (3, size(H, 3))) || error("g must be 3 x n_env")
        GC.@preserve H g check(ccall((:pfc_set_body_params, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}), CTX[m], size(H, 3), H, g))
    end
    return nothing
end

"Continuous affine state feedback inside calcXd! (pfc_set_feedback), after `finalize_floating_gpu!`: calcXd! of environment `env` uses
`tau_ext + K[:, :, env, seg]' * (x_ref[:, env, seg] - x[1:nq+nv, env])`, with `K[:, i, env, seg]` the gains of generalized force `i`
((nq + nv) x nv x n_env x n_seg: column-major, so the bytes are pfc.h's K[seg][env][nv][nq + nv]) and `x_ref` (nq + nv) x n_env x n_seg.
Roll-outs use segment k on the k-th knot interval (n_seg = 1 or n_knot); the other calls use segment 1.  `nothing` clears the table."
function set_feedback!(m::MechanismScenario, K::Union{Array{Float64,4},Nothing}, x_ref::Union{Array{Float64,3},Nothing}=nothing)
    if K === nothing
        check(ccall((:pfc_set_feedback, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Ptr{Float64}, Ptr{Float64}), CTX[m], 0, 0, C_NULL, C_NULL))
    else
        (x_ref !== nothing && size(x_ref) == (size(K, 1), size(K, 3), size(K, 4))) || error("x_ref must be (nq + nv) x n_env x n_seg")
        GC.@preserve K x_ref check(ccall((:pfc_set_feedback, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Ptr{Float64}, Ptr{Float64}),
                                         CTX[m], size(K, 3), size(K, 4), K, x_ref))
    end
    return nothing
end

"forceAllElasticIntersections! for a batch of states `x[:, env]`: generalized forces `f[:, env]` and `sdot` (pfc_eval_state_f64)."
function force_all_batch_gpu!(f::Matrix{Float64}, sdot::Matrix{Float64}, m::MechanismScenario, x::Matrix{Float64})
    GC.@preserve x f sdot check(ccall((:pfc_eval_state_f64, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        CTX[m], size(x, 2), x, f, isempty(sdot) ? C_NULL : pointer(sdot), C_NULL, C_NULL))
    return nothing
end

"calcXd! for a batch of states `x[:, env]` entirely on the device (pfc_calcxd_f64)."
function calcXd_batch_gpu!(xx::Matrix{Float64}, m::MechanismScenario, x::Matrix{Float64})
    GC.@preserve x xx check(ccall((:pfc_calcxd_f64, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}), CTX[m], size(x, 2), x, C_NULL, xx, C_NULL, C_NULL))
    return nothing
end

"One Jacobian chunk of calcXd! for a batch: `xx7[1, i, env]` = x_dot[i], `xx7[1 + k, i, env]` = d x_dot[i] / d x[seed + k] (seed is 1-based here)."
function calcXd_chunk_batch_gpu!(xx7::Array{Float64,3}, m::MechanismScenario, x::Matrix{Float64}, seed::Integer)
    GC.@preserve x xx7 check(ccall((:pfc_calcxd_dual6, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        CTX[m], size(x, 2), x, C_NULL, seed - 1, xx7, C_NULL, C_NULL))
    return nothing
end

"The whole Jacobian of calcXd! for a batch in one call: `jac[j, i, env]` = d x_dot[i] / d x[j] (the C layout is row-major [env][i][j]);
`xx[:, env]` = calcXd!(x[:, env]).  calcJacobian! (src/radau/radau_functions.jl:2-26) stores `-transpose(jac[:, :, env])`."
function calcJacobian_batch_gpu!(jac::Array{Float64,3}, xx::Matrix{Float64}, m::MechanismScenario, x::Matrix{Float64})
    GC.@preserve x xx jac check(ccall((:pfc_calcxd_jacobian, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        CTX[m], size(x, 2), x, C_NULL, jac, xx, C_NULL, C_NULL))
    return nothing
end

"Resets the batched Radau integrator of the context (pfc_radau_init): n_env environments, h = h0, rule 1 (RadauStep / RadauRule),
at most `max_rule` (NR) rules, the reference's tolerances."
function radau_init!(m::MechanismScenario, n_env::Integer; max_rule::Integer = 2, h0::Float64 = 1.0e-4, h_max::Float64 = 0.01,
                     tol_newton::Float64 = 1.0e-16)
    check(ccall((:pfc_radau_init, LIB), Cint, (Ptr{Cvoid}, Int64, Cint, Float64, Float64, Float64), CTX[m], n_env, max_rule, h0, h_max, tol_newton))
    return nothing
end

"One accepted Radau step (solveRadau + principal_value!) of every environment `x[:, env]` (pfc_radau_step, host arrays; pfc_radau_step_device
for `CuArray`s): `x` and `t` in place, `h_taken[env]` out; `tau_ext[:, env]` is held over the step.  Returns `stats[:, env]` = stages of the
accepted attempt, its Newton iterations, rejected attempts, stage evaluations."
function radau_step_batch_gpu!(m::MechanismScenario, x::Matrix{Float64}, t::Vector{Float64}, h_taken::Vector{Float64};
                               tau_ext::Union{Nothing,Matrix{Float64}} = nothing)
    stats = zeros(Int32, 4, size(x, 2))
    tau = tau_ext === nothing ? C_NULL : tau_ext
    GC.@preserve x t h_taken tau_ext stats check(ccall((:pfc_radau_step, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}), CTX[m], size(x, 2), x, tau, t, h_taken, stats))
    return stats
end

"Every environment `x[:, env]` from `t[env]` through the shared knot times `t_knot` (pfc_radau_rollout, host arrays): `tau_ext[:, env, k]`
acts on `(t_knot[k-1], t_knot[k]]`, `x_knot[:, env, k]` gets the state at knot k (NaN if the environment ran out of `max_steps` accepted
steps first), `x` and `t` advance in place.  Returns `stats[:, env]` = knots reached, accepted steps, rejected attempts, stage evaluations.
Written against include/pfc.h; not run (no Julia in the build environment)."
function radau_rollout_batch_gpu!(m::MechanismScenario, x::Matrix{Float64}, t::Vector{Float64}, t_knot::Vector{Float64},
                                  x_knot::Array{Float64,3}; tau_ext::Union{Nothing,Array{Float64,3}} = nothing, max_steps::Integer = 1000)
    stats = zeros(Int32, 4, size(x, 2))
    tau = tau_ext === nothing ? C_NULL : tau_ext
    GC.@preserve x t t_knot x_knot tau_ext stats check(ccall((:pfc_radau_rollout, LIB), Cint,
        (Ptr{Cvoid}, Int64, Cint, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        CTX[m], size(x, 2), length(t_knot), t_knot, max_steps, x, tau, t, x_knot, stats))
    return stats
end

"Moved vertices of mesh `id` (same connectivity): the device rebuilds the mesh's primitive records and refits its tree (pfc_refit_mesh)."
function refit_mesh_gpu!(m::MechanismScenario, id::MeshID, point::Vector{SVector{3,Float64}})
    xyz = collect(Iterators.flatten(point))
    GC.@preserve xyz check(ccall((:pfc_refit_mesh, LIB), Cint, (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}), CTX[m], Int(id) - 1, length(point), xyz))
    return nothing
end

# ---- one very large scene split over several GPUs of this process: the library owns the NCCL communicator (pfc_group) ----------------
"Creates a group over `devices` (0-based CUDA ordinals) and uploads the scene of `m` to every device (the walk of finalize_gpu!)."
function finalize_group_gpu!(m::MechanismScenario, devices::Vector{Int32})
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:pfc_group_create, LIB), Cint, (Cint, Ptr{Int32}, Ref{Ptr{Cvoid}}), length(devices), devices, ref))
    g = ref[]
    for id in m.mesh_ids
        mc = m.MeshCache[id]
        eM = mc.mesh
        xyz = collect(Iterators.flatten(eM.point))
        is_tet = eM.tet !== nothing
        idx = Int32.(collect(Iterators.flatten(is_tet ? eM.tet : eM.tri)) .- 1)
        c, e, R, l, r, leaf = flatten(get_tree(mc))
        eps_ptr = is_tet ? pointer(eM.ϵ) : Ptr{Float64}(C_NULL)
        out = Ref{Cint}(-1)
        GC.@preserve xyz idx c e R l r leaf eM check(ccall((:pfc_group_add_mesh, LIB), Cint,
            (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Int64, Ptr{Int32}, Ptr{Float64}, Float64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ref{Cint}),
            g, is_tet ? 1 : 0, length(eM.point), xyz, is_tet ? length(eM.tet) : length(eM.tri), idx, eps_ptr,
            is_tet ? get_c_prop(mc).Ē : 0.0, length(l), c, e, R, l, r, leaf, out))
    end
    for ci in m.ContactInstructions
        fm = ci.FrictionModel
        model, params = fm isa Regularized ? (0, [fm.μs, fm.μd, fm.v_c]) : (1, [fm.τ, fm.k̄, fm.μs, fm.μd, fm.magic])
        n_quad_rule = length(ci.quad.w) == 1 ? 1 : 2
        check(ccall((:pfc_group_add_instruction, LIB), Cint, (Ptr{Cvoid}, Cint, Cint, Float64, Cint, Ptr{Float64}, Cint, Ptr{Cint}),
            g, Int(ci.id_1) - 1, Int(ci.id_2) - 1, ci.χ, model, params, n_quad_rule, C_NULL))
    end
    check(ccall((:pfc_group_finalize, LIB), Cint, (Ptr{Cvoid}, Int64), g, 1))
    return g
end

"forceAllElasticIntersections! with the candidate-pair lists split over the group's GPUs: same arrays as pfc_eval_f64."
function eval_group_gpu!(g::Ptr{Cvoid}, X::Matrix{Float64}, tw::Matrix{Float64}, s, w::Matrix{Float64}, sdot)
    GC.@preserve X tw s w sdot check(ccall((:pfc_group_eval_f64, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
        g, 1, X, tw, s === nothing ? C_NULL : pointer(s), w, sdot === nothing ? C_NULL : pointer(sdot), C_NULL, C_NULL))
    return nothing
end

end # module
