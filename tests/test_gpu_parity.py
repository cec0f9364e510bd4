"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Bars: candidate-pair lists bit-exact (same pairs, same order); flags equal;
wrenches and bristle state derivatives within 1e-9 relative (SURVEY.md H7 definition: per force /
torque 3-vector, ||delta||_inf / ||ref||_inf, with an absolute floor for halves that vanish by symmetry)."""
import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import _sphere_scene, _sphere_states, _tet_tet_scene, boxes_env_states, rot_z, scene_boxes, wrench_rel_err
from oracle import orc
from pfc_b200 import geometry as G
from pfc_b200 import scenario as S

pytestmark = pytest.mark.gpu
TOL = 1.0e-9


def _ctx():
    from pfc_b200 import capi
    return capi.Context(0)


def _both(build, n_env=1):
    m_gpu = build(_ctx(), n_env)
    m_cpu = build(orc.OracleContext(), n_env)
    return m_gpu, m_cpu


def _compare(m_gpu, m_cpu, X, tw, s=None, pairs=True, floor=1e-9):
    """Every instruction -- regularized and bristle alike -- is held to TOL = 1e-9 on its wrench, and s-dot to 1e-9 as well: the
    bristle instructions run in the reference's operation order on the device (csrc/pfc_exact.cuh), which makes the ill-conditioned
    K^(-1/2) of the bristle model reproducible.  Candidate-pair lists are compared for EVERY (environment, instruction)."""
    g = m_gpu.backend.eval_f64(X, tw, s, keep=pairs)
    c = m_cpu.backend.eval_f64(X, tw, s, keep=pairs)
    assert (g["n_pairs"] == c["n_pairs"]).all()
    assert (g["flags"] == c["flags"]).all()
    scale = max(np.abs(c["wrench"]).max(), 1e-300)
    assert wrench_rel_err(g["wrench"], c["wrench"], floor=floor * scale) <= TOL
    if s is not None:
        sc = max(np.abs(c["sdot"]).max(), 1e-300)
        assert wrench_rel_err(g["sdot"], c["sdot"], floor=floor * sc) <= TOL
    if pairs:
        n_env, n_ins = c["n_pairs"].shape
        for e in range(n_env):
            for k in range(n_ins):
                assert (m_gpu.backend.get_pairs(e, k) == m_cpu.backend.get_pairs(e, k)).all(), (e, k)
    return g, c


def test_boxes_batch_parity():
    """Config C1/C3: test/boxes.jl scene, randomized settled-stack states."""
    n_env = 256
    m_gpu, m_cpu = _both(lambda b, n: scene_boxes(b, n)[0], n_env)
    x = boxes_env_states(m_gpu, n_env)
    X, tw, _ = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw)
    assert (c["flags"] & 1).sum() > n_env  # plenty of contacts in the sample
    assert c["n_pairs"].max() <= 144
    # traction lists (the reference's TractionCache) of one environment, point by point
    for k in range(4):
        tg, tc = m_gpu.backend.get_traction(3, k), m_cpu.backend.get_traction(3, k)
        assert tg.shape == tc.shape
        if len(tc):
            assert np.allclose(tg, tc, rtol=1e-9, atol=1e-12 * np.abs(tc).max())


def test_boxes_initial_state_no_contact():
    """test/boxes.jl:42-45 initial state: boxes spaced 3 r apart, nothing touches; wrenches are zero."""
    m_gpu, m_cpu = _both(lambda b, n: scene_boxes(b, n)[0])
    X, tw, _ = S.boundary_arrays(m_gpu, S.get_state(m_gpu))
    g, c = _compare(m_gpu, m_cpu, X, tw)
    assert (g["wrench"] == 0).all() and (g["flags"] == 0).all()


def _normal_scene(k_quad_rule):
    def build(backend, n_env):
        r = 0.05
        m = S.MechanismScenario()
        id_plane = S.add_contact(m, "plane", G.as_tet_eMesh(G.eMesh_half_plane()), c_prop=S.ContactProperties(1.0e9))
        eM_box = G.transform(G.as_tri_eMesh(G.eMesh_box(r)), t=(0.0, 0.0, r))
        body, _, id_box = S.add_body_contact(m, "box", eM_box, i_prop=S.InertiaProperties(400.0, d=0.09))
        S.add_friction_bristle(m, id_box, id_plane, mu_d=0.3, chi=0.6, k_bar=1.0e6, tau=0.03, n_quad_rule=k_quad_rule)
        S.finalize(m, backend, n_env)
        m.box_body = body
        return m
    return build


@pytest.mark.parametrize("k_quad_rule", [1, 2])
def test_normal_wrench_kat_on_gpu(k_quad_rule):
    """test/test_normal.jl through the CUDA path: analytic answer AND oracle parity (bristle model)."""
    m_gpu, m_cpu = _both(_normal_scene(k_quad_rule))
    r, p_pos = 0.05, (0.1, 0.2)
    pene = 0.1 * r
    for m in (m_gpu, m_cpu):
        S.set_state_spq(m, m.box_body, trans=(p_pos[0], p_pos[1], -pene))
    X, tw, s = S.boundary_arrays(m_gpu, S.get_state(m_gpu))
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(1, 1, 6))
    check = 1.0e9 * pene * r ** 2 * 4
    f3 = np.array([0.0, 0.0, check])
    assert np.allclose(g["wrench"][0, 0], -np.concatenate([np.cross([p_pos[0], p_pos[1], 0.0], f3), f3]), rtol=1e-10)


def test_bristle_sliding_batch():
    """Bristle friction with non-zero bristle state, sliding and spinning box: wrench and s-dot."""
    n_env = 64
    m_gpu, m_cpu = _both(_normal_scene(2), n_env)
    rng = np.random.default_rng(42)
    x = np.zeros((n_env, S.num_x(m_gpu)))
    r = 0.05
    for e in range(n_env):
        x[e, 0:3] = rng.uniform(-0.03, 0.03, 3)
        x[e, 3:6] = [rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2), -rng.uniform(0.0, 0.1) * r]
        x[e, 6:9] = rng.uniform(-1, 1, 3)
        x[e, 9:12] = rng.uniform(-0.1, 0.1, 3)
        x[e, 12:18] = rng.uniform(-1, 1, 6) * np.array([1e-3, 1e-3, 1e-3, 1e-5, 1e-5, 1e-5])
    x[0, 3:6] = [0, 0, 0.01]  # one environment out of contact: no_contact!(::Bristle)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))
    assert c["flags"][0, 0] == 0 and np.allclose(g["sdot"][0, 0], -x[0, 12:18] / 0.03)
    assert (c["flags"][1:, 0] & 1).all()


def test_tet_tet_batch_parity():
    """test/test_vol_vol.jl-style volumetric contact (tet-tet), regularized and bristle."""
    n_env = 128
    m_gpu, m_cpu = _both(_tet_tet_scene, n_env)
    rng = np.random.default_rng(7)
    r = 0.05
    x = np.zeros((n_env, S.num_x(m_gpu)))
    nq = m_gpu.nq
    for e in range(n_env):
        x[e, 0:3] = rng.uniform(-0.05, 0.05, 3)
        x[e, 3:6] = [rng.uniform(-0.01, 0.01), rng.uniform(-0.01, 0.01), r - rng.uniform(0, 0.004)]
        x[e, 6:9] = rng.uniform(-0.05, 0.05, 3)
        x[e, 9:12] = [rng.uniform(-0.03, 0.03), rng.uniform(-0.03, 0.03), 3 * r - rng.uniform(0, 0.008)]
        x[e, nq:nq + 12] = rng.uniform(-1, 1, 12) * 0.2
        x[e, nq + 12:] = rng.uniform(-1, 1, 6) * 1e-4
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))   # nearly flat box-box patches: rank-deficient stiffness
    assert (c["flags"] & 1).sum() > n_env


def _single_pair_scene(kind1):
    """One primitive against one tetrahedron: every environment is one random clip problem."""
    def build(backend, n_env):
        rng = np.random.default_rng(2024)
        m = S.MechanismScenario()
        while True:
            t2 = rng.standard_normal((4, 3)) * 0.1
            if G.tet_volume(t2) > 1e-5:
                break
        tet2 = G.eMesh(t2, None, [[0, 1, 2, 3]], [0.0, 0.0, 0.0, 1.0])
        id2 = S.add_contact(m, "tet2", tet2, c_prop=S.ContactProperties(1.0e6))
        if kind1 == 0:
            tri = G.eMesh(rng.standard_normal((3, 3)) * 0.2, [[0, 1, 2]])
            b = S.add_body_contact(m, "tri", tri, i_prop=S.InertiaProperties(400.0, d=0.01), tree=G.eMesh_to_tree(tri))
        else:
            while True:
                t1 = rng.standard_normal((4, 3)) * 0.1
                if G.tet_volume(t1) > 1e-5:
                    break
            b = S.add_body_contact(m, "tet1", G.eMesh(t1, None, [[0, 1, 2, 3]], [0.0, 1.0, 0.0, 0.0]), i_prop=S.InertiaProperties(400.0),
                                   c_prop=S.ContactProperties(2.0e6))
        S.add_friction_regularize(m, b[2], id2, mu_s=0.5, mu_d=0.3, chi=0.4, v_tol=1e-2, n_quad_rule=2)
        S.finalize(m, backend, n_env)
        return m
    return build


@pytest.mark.parametrize("kind1", [0, 1])
def test_random_single_pair_clip_stress(kind1):
    """Thousands of random relative poses of one triangle / tetrahedron against one tetrahedron:
    exercises every arity of the clipper (3..8 vertices) and every plane-tet case."""
    n_env = 8192
    m_gpu, m_cpu = _both(_single_pair_scene(kind1), n_env)
    rng = np.random.default_rng(99)
    x = np.zeros((n_env, S.num_x(m_gpu)))
    x[:, 0:3] = rng.uniform(-0.6, 0.6, (n_env, 3))
    x[:, 3:6] = rng.uniform(-0.12, 0.12, (n_env, 3))
    x[:, 6:12] = rng.uniform(-1, 1, (n_env, 6))
    X, tw, _ = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, pairs=False, floor=1e-7)
    assert (c["flags"] & 1).sum() > n_env // 20
    assert (c["n_pairs"] == 0).any() and (c["n_pairs"] == 1).any()


def test_sphere_small_path():
    """Curved meshes on the small path: icosahedron-level spheres (20 x 20 leaf pairs), tri-tet and tet-tet."""
    def build(backend, n_env):
        m = S.MechanismScenario()
        sph = G.eMesh_sphere(0.05, 1)
        ground = S.add_contact(m, "ground", G.as_tet_eMesh(G.eMesh_sphere(0.08, 1)), c_prop=S.ContactProperties(2.0e6))
        b1 = S.add_body_contact(m, "s_tri", G.as_tri_eMesh(sph), i_prop=S.InertiaProperties(400.0, d=0.01))
        b2 = S.add_body_contact(m, "s_tet", G.as_tet_eMesh(sph), i_prop=S.InertiaProperties(400.0), c_prop=S.ContactProperties(1.0e6))
        S.add_friction_regularize(m, b1[2], ground, mu_d=0.3, chi=0.5, n_quad_rule=1)
        S.add_friction_regularize(m, b2[2], ground, mu_d=0.3, chi=0.5, n_quad_rule=2)
        S.add_friction_bristle(m, b1[2], b2[2], mu_d=0.4, k_bar=2.0e4, tau=0.05, n_quad_rule=2)
        S.finalize(m, backend, n_env)
        return m
    n_env = 96
    m_gpu, m_cpu = _both(build, n_env)
    rng = np.random.default_rng(5)
    x = np.zeros((n_env, S.num_x(m_gpu)))
    nq = m_gpu.nq
    for e in range(n_env):
        d1 = rng.standard_normal(3); d1 /= np.linalg.norm(d1)
        d2 = rng.standard_normal(3); d2 /= np.linalg.norm(d2)
        x[e, 0:3] = rng.uniform(-0.3, 0.3, 3)
        x[e, 3:6] = d1 * rng.uniform(0.10, 0.128)
        x[e, 6:9] = rng.uniform(-0.3, 0.3, 3)
        x[e, 9:12] = x[e, 3:6] + d2 * rng.uniform(0.07, 0.098) if e % 2 else d2 * rng.uniform(0.10, 0.128)
        x[e, nq:nq + 12] = rng.uniform(-1, 1, 12) * 0.3
        x[e, nq + 12:] = rng.uniform(-1, 1, 6) * 1e-4
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))  # tiny patches: rank-deficient stiffness
    assert (c["flags"] & 1).sum() > n_env // 2


def test_determinism_bitwise():
    """Fixed-order reduction: two evaluations of the same batch are bitwise identical."""
    n_env = 512
    m_gpu = scene_boxes(_ctx(), n_env)[0]
    X, tw, _ = S.boundary_arrays(m_gpu, boxes_env_states(m_gpu, n_env))
    a = m_gpu.backend.eval_f64(X, tw, None)
    b = m_gpu.backend.eval_f64(X, tw, None)
    assert (a["wrench"].view(np.int64) == b["wrench"].view(np.int64)).all()


# ---- large path (traversal + DFS-key sort + per-pair narrow phase) ------------------------
@pytest.fixture
def force_large_path(monkeypatch):
    """Trees of a few hundred leaves normally take the on-chip path with a bounded pair-list slot (build_tables in csrc/pfc_api.cu);
    these tests are about the multi-kernel large path, so that class is switched off while their scenes are built."""
    monkeypatch.setenv("PFC_MID_LEAVES", "0")


def test_large_path_spheres(force_large_path):
    """Instructions too big for the on-chip path (320 x 180 and 320 x 320 leaf pairs): the pair lists
    must come back in exactly the reference's traversal order after the DFS-key sort."""
    n_env = 6
    m_gpu, m_cpu = _both(_sphere_scene(), n_env)
    x = _sphere_states(m_gpu, n_env, 11)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))
    n_tests, n_large_pairs = m_gpu.backend.counters()  # the large path's own counters: it really ran
    assert n_large_pairs == int(c["n_pairs"][:, :3].sum()) and n_tests > n_large_pairs > 500
    assert (c["flags"][:, :3] & 1).sum() >= n_env
    # traction lists of a large instruction, point by point, in order
    e = int(np.argmax(c["n_pairs"][:, 0]))
    tg, tc = m_gpu.backend.get_traction(e, 0), m_cpu.backend.get_traction(e, 0)
    assert tg.shape == tc.shape and len(tc) > 0
    assert np.allclose(tg, tc, rtol=1e-9, atol=1e-12 * np.abs(tc).max())


def test_large_path_many_envs_deterministic(force_large_path):
    """Large path over a batch of environments; two runs are bitwise identical although the traversal
    appends pairs with atomics (the sort and the fixed-order reductions remove the nondeterminism)."""
    n_env = 48
    m_gpu, m_cpu = _both(_sphere_scene(3, 3, with_small=False), n_env)
    x = _sphere_states(m_gpu, n_env, 12, with_small=False)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6), pairs=False)
    g2 = m_gpu.backend.eval_f64(X, tw, s.reshape(n_env, 1, 6))
    assert (g["wrench"].view(np.int64) == g2["wrench"].view(np.int64)).all()
    assert (g["n_pairs"] == g2["n_pairs"]).all()
    a, b = m_gpu.backend.counters()
    assert b == int(c["n_pairs"].sum()) and a > b


def test_large_path_no_contact_and_empty(force_large_path):
    """Far-apart bodies: the root boxes are disjoint, pair lists are empty, wrenches zero, bristle s-dot = -s / tau."""
    n_env = 3
    m_gpu, m_cpu = _both(_sphere_scene(2, 2, with_small=False), n_env)
    x = _sphere_states(m_gpu, n_env, 13, with_small=False)
    x[:, 3:6] = [1.0, 0.0, 0.0]
    x[:, 9:12] = [0.0, 1.0, 0.0]
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))
    assert (g["n_pairs"] == 0).all() and (g["wrench"] == 0).all()


def test_sharded_large_scene_two_ranks_on_one_gpu(force_large_path):
    """The multi-GPU split of one large scene, emulated with two contexts (rank 0 and 1 of world 2) on
    one GPU: each traverses and evaluates the sub-trees whose hash falls on it (disjoint pair lists), the
    partial buffers are summed (what the NCCL allreduce does), and both end with the same wrench / s-dot /
    pair counts as the unsharded evaluation."""
    import torch
    from pfc_b200 import capi, parallel
    n_env = 2
    build = _sphere_scene(4, 3, with_small=True)
    ref = build(capi.Context(0), n_env)
    ranks = []
    for r in range(2):
        ctx = capi.Context(0)
        ctx_m = build(ctx, n_env)
        ctx.set_shard(r, 2)
        ranks.append((ctx, ctx_m))
    x = _sphere_states(ref, n_env, 21)
    X, tw, s = S.boundary_arrays(ref, x)
    full = ref.backend.eval_f64(X, tw, s.reshape(n_env, 1, 6))
    dev = torch.device("cuda", 0)
    n_ins = ref.backend.n_ins
    bufs = []
    for ctx, _ in ranks:
        b = dict(X=torch.from_numpy(X).to(dev), tw=torch.from_numpy(tw).to(dev), s=torch.from_numpy(s.reshape(n_env, 1, 6).copy()).to(dev),
                 w=torch.zeros((n_env, n_ins, 6), dtype=torch.float64, device=dev), sd=torch.zeros((n_env, 1, 6), dtype=torch.float64, device=dev),
                 np_=torch.zeros((n_env, n_ins), dtype=torch.int64, device=dev), fl=torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev))
        bufs.append(b)
        ctx.eval_sharded_begin(n_env, b["X"].data_ptr(), b["tw"].data_ptr(), b["s"].data_ptr(), b["w"].data_ptr(), b["sd"].data_ptr(),
                               b["np_"].data_ptr(), b["fl"].data_ptr())
    n_exchange = 0
    while True:
        parts = []
        for ctx, _ in ranks:
            ctx.sync()
            ptr, count = ctx.eval_sharded_partials()
            assert count == 8 * n_env * 3   # 6 sums + point count + pair count per (environment, large instruction)
            parts.append((ptr, count))
        # the "allreduce": sum the two device buffers and write the sum back into both
        import ctypes
        cudart = ctypes.CDLL("libcudart.so")
        host = [np.zeros(c) for _, c in parts]
        for h, (ptr, c) in zip(host, parts):
            assert cudart.cudaMemcpy(h.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(ptr), ctypes.c_size_t(8 * c), 2) == 0
        total = host[0] + host[1]
        for ptr, c in parts:
            assert cudart.cudaMemcpy(ctypes.c_void_p(ptr), total.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(8 * c), 1) == 0
        n_exchange += 1
        more = [ctx.eval_sharded_step() for ctx, _ in ranks]
        assert more[0] == more[1]
        if not more[0]:
            break
    assert n_exchange == 1  # one exchange: the regularized sums (bristle instructions are never split: every rank evaluates them whole)
    for (ctx, _), b in zip(ranks, bufs):
        ctx.sync()
        w = b["w"].cpu().numpy()
        scale = np.abs(full["wrench"]).max()
        assert wrench_rel_err(w, full["wrench"], floor=1e-9 * scale) <= 1e-11   # same traction points, different association only
        assert (b["np_"].cpu().numpy() == full["n_pairs"]).all()
        assert ((b["fl"].cpu().numpy() & 1) == (full["flags"] & 1)).all()
        assert np.array_equal(b["sd"].cpu().numpy(), full["sdot"])   # bristle: the same sequential sums on every rank, bit for bit
    assert parallel.env_range(10, 1, 3) == (3, 6)


# ---- Jacobian mode: Dual{Nothing,Float64,6} ---------------------------------------------------------------
def _dual_inputs(m, x, seed_start):
    X0, X7, tw7, s7 = S.boundary_arrays_dual6(m, x, seed_start)
    return X0, X7, tw7, (s7 if m.n_bristle else None)


def _rel7(a, b, floor):
    """max relative error per 3-vector half; value and each partial are scaled separately, but a partial that is
    pure rounding noise (below 1e-6 of the array's overall scale) is measured against that overall scale;
    `floor` is the fraction of a partial's scale below which a force/torque half is measured against the scale itself"""
    a, b = np.asarray(a), np.asarray(b)
    worst = 0.0
    overall = max(np.abs(b).max(), 1e-300)
    for d in range(7):
        worst = max(worst, wrench_rel_err(a[..., d], b[..., d], floor=floor * max(np.abs(b[..., d]).max(), 1e-6 * overall)))
    return worst


def test_dual6_boxes_matches_oracle_and_finite_differences():
    """Jacobian chunks on the test/boxes.jl scene (regularized friction): value + 6 partials of every
    wrench against the Dual oracle (1e-9) and against central differences of the Float64 path."""
    m_gpu, m_cpu = _both(lambda b, n: scene_boxes(b, n)[0])
    x = boxes_env_states(m_gpu, 3)[2]
    for seed_start in (6, 27, 33):     # box 2 pose, box 1 velocity, box 2/3 velocity
        X0, X7, tw7, _ = _dual_inputs(m_gpu, x, seed_start)
        g = m_gpu.backend.eval_dual6(X0, X7, tw7)
        c = m_cpu.backend.eval_dual6(X0, X7, tw7)
        assert (g["n_pairs"] == c["n_pairs"]).all() and (g["flags"] == c["flags"]).all()
        assert _rel7(g["wrench"], c["wrench"], 1e-3) <= TOL
        assert np.abs(c["wrench"][..., 1:]).max() > 0
        # finite differences of the Float64 path through the same C ABI
        h = 1e-7
        for d in range(6):
            xp, xm = x.copy(), x.copy()
            xp[seed_start + d] += h
            xm[seed_start + d] -= h
            Xp, twp, _ = S.boundary_arrays(m_gpu, xp)
            Xm, twm, _ = S.boundary_arrays(m_gpu, xm)
            fd = (m_gpu.backend.eval_f64(Xp, twp)["wrench"] - m_gpu.backend.eval_f64(Xm, twm)["wrench"]) / (2 * h)
            an = g["wrench"][..., 1 + d]
            assert np.allclose(an, fd, rtol=2e-4, atol=2e-5 * max(np.abs(fd).max(), 1.0)), (seed_start, d)
    # reuse of the previous Float64 pair lists (X_bp = NULL): same answer
    Xf, twf, _ = S.boundary_arrays(m_gpu, x)
    m_gpu.backend.eval_f64(Xf, twf)
    X0, X7, tw7, _ = _dual_inputs(m_gpu, x, 6)
    g1 = m_gpu.backend.eval_dual6(None, X7, tw7)
    g2 = m_gpu.backend.eval_dual6(X0, X7, tw7)
    assert np.array_equal(g1["wrench"], g2["wrench"])


def test_dual6_bristle_and_tet_tet():
    """Dual mode through the bristle model (K̄^(-1/2) differentiated by the Daleckii-Krein formula) and tet-tet clipping."""
    m_gpu, m_cpu = _both(_tet_tet_scene)
    rng = np.random.default_rng(3)
    r = 0.05
    x = np.zeros(S.num_x(m_gpu))
    nq = m_gpu.nq
    x[0:3] = rng.uniform(-0.05, 0.05, 3)
    x[3:6] = [0.004, -0.003, r - 0.003]
    x[6:9] = rng.uniform(-0.05, 0.05, 3)
    x[9:12] = [0.01, 0.02, 3 * r - 0.006]
    x[nq:nq + 12] = rng.uniform(-1, 1, 12) * 0.2
    x[nq + 12:] = rng.uniform(-1, 1, 6) * 1e-4
    for seed_start in (0, 6, 18, 24):   # poses, velocities, bristle state
        X0, X7, tw7, s7 = _dual_inputs(m_gpu, x, seed_start)
        g = m_gpu.backend.eval_dual6(X0, X7, tw7, s7)
        c = m_cpu.backend.eval_dual6(X0, X7, tw7, s7)
        assert (g["n_pairs"] == c["n_pairs"]).all() and (g["flags"] == c["flags"]).all()
        # regularized instructions (0, 1) and the bristle instruction (2, evaluated in the reference's operation order) alike
        assert _rel7(g["wrench"], c["wrench"], 1e-3) <= TOL
        assert _rel7(g["sdot"], c["sdot"], 1e-3) <= TOL


# ---- config C2: the pencil gripper and the spoon, bristle friction, sampled states ------------------------------
# halves of a wrench that vanish by symmetry (the pad-pad torque about the r2 origin) carry eps * |F| * L rounding noise:
# they are compared against 1e-6 of the largest wrench component instead of against themselves
C2_FLOOR = 1.0e-6
def test_c2_pencil_bristle_sampled_states():
    """test/pencil.jl with is_bristle = true (SURVEY.md section 8d, C2): wrench / s-dot / pair-list parity on sampled
    states of the task (the 1000-step Radau state parity needs the integrator and RigidBodyDynamics: out of scope)."""
    from pfc_b200 import scenes
    m_gpu, bodies = scenes.scene_c2_pencil(True, _ctx())
    m_cpu, _ = scenes.scene_c2_pencil(True, orc.OracleContext())
    xs = scenes.pencil_sample_states(m_gpu, bodies, 12)
    n_contact = 0
    for x in xs:
        X, tw, s = S.boundary_arrays(m_gpu, x)
        g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(1, m_gpu.n_bristle, 6), floor=C2_FLOOR)
        n_contact += int((c["flags"] & 1).sum())
        # the generalized forces the reference would add (J' w through the arm's joints) agree as well
        f_g = S.generalized_forces(m_gpu, x, g["wrench"][0])
        f_c = S.generalized_forces(m_cpu, x, c["wrench"][0])
        assert np.abs(f_g - f_c).max() <= TOL * max(np.abs(f_c).max(), 1e-300)
    assert n_contact >= 16  # pad-pencil (bristle), pencil-plane and pad-pad (tet-tet) contacts are all exercised


def test_c2_spoon_bristle_sampled_states():
    """test/spoon.jl re-expressed (R5): 5004-triangle spoon surface clamped between two compliant boxes, two
    bristle instructions, quadrature rule 1 (large-instruction path: 5004 x 12 leaf pairs)."""
    from pfc_b200 import scenes
    m_gpu, bodies = scenes.scene_c2_spoon(_ctx())
    m_cpu, _ = scenes.scene_c2_spoon(orc.OracleContext())
    xs = scenes.spoon_sample_states(m_gpu, bodies, 6)
    n_contact = 0
    for x in xs:
        X, tw, s = S.boundary_arrays(m_gpu, x)
        g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(1, m_gpu.n_bristle, 6), floor=C2_FLOOR)
        n_contact += int((c["flags"] & 1).sum())
    assert n_contact >= 8


# ---- state-level entry point: kinematics prologue and J' w epilogue on the device (SURVEY.md section 8f, rank 1) ----------
def test_state_entry_point_boxes_batch():
    """pfc_eval_state_f64 on 256 boxes.jl environments: the boundary arrays the device computes from x agree with the host
    mirror of RigidBodyDynamics (1e-13); fed to the oracle they give bit-exact pair counts / flags and wrenches within 1e-9;
    the generalized forces equal addGeneralizedForcesThirdLaw! applied on the host to the oracle's wrenches."""
    n_env = 256
    m_gpu, m_cpu = _both(lambda b, n: scene_boxes(b, max_env=n)[0], n_env)
    assert m_gpu.device_kinematics
    x = boxes_env_states(m_gpu, n_env)
    out = S.force_all_elastic_intersections_batch(m_gpu, x)
    X_d, tw_d, w_d = m_gpu.backend.get_boundary(n_env)
    X_h, tw_h, _ = S.boundary_arrays(m_gpu, x)
    assert np.abs(X_d - X_h).max() <= 1e-13 and np.abs(tw_d - tw_h).max() <= 1e-13 * max(1.0, np.abs(tw_h).max())
    c = m_cpu.backend.eval_f64(X_d, tw_d)
    assert (out["n_pairs"] == c["n_pairs"]).all() and (out["flags"] == c["flags"]).all()
    scale = np.abs(c["wrench"]).max()
    assert wrench_rel_err(w_d, c["wrench"], floor=1e-9 * scale) <= TOL
    f_ref = np.array([S.generalized_forces(m_cpu, x[e], c["wrench"][e]) for e in range(n_env)])
    assert np.abs(out["f_generalized"] - f_ref).max() <= TOL * np.abs(f_ref).max()
    assert (c["flags"] & 1).sum() > n_env
    # same numbers as the boundary-level entry point fed with the device's own boundary arrays
    g = m_gpu.backend.eval_f64(X_d, tw_d)
    assert np.array_equal(g["wrench"], w_d)


def test_state_entry_point_replayed_graph_follows_the_inputs():
    """From its third identical invocation (same batch size, same pinned caller buffers) pfc_eval_state_f64 is a replayed CUDA graph:
    the results must follow the CONTENT of the buffers, call after call, and equal what a fresh context computes from the same states."""
    import torch
    n_env = 64
    m_gpu = scene_boxes(_ctx(), max_env=n_env)[0]
    m_ref = scene_boxes(_ctx(), max_env=n_env)[0]
    nx = S.num_x(m_gpu)
    x_p = torch.zeros((n_env, nx), dtype=torch.float64).pin_memory()
    f_p = torch.zeros((n_env, m_gpu.nv), dtype=torch.float64).pin_memory()
    np_p = torch.zeros((n_env, 4), dtype=torch.int64).pin_memory()
    fl_p = torch.zeros((n_env, 4), dtype=torch.int32).pin_memory()
    for it in range(6):
        x = boxes_env_states(m_gpu, n_env, start=1000 * it)     # other states every call, same buffers
        x_p.copy_(torch.from_numpy(x))
        f_p.fill_(float("nan"))
        m_gpu.backend.eval_state_f64_ptr(n_env, x_p.data_ptr(), f_p.data_ptr(), None, np_p.data_ptr(), fl_p.data_ptr())
        want = S.force_all_elastic_intersections_batch(m_ref, x)   # numpy path: new buffers every call, never a graph
        assert np.array_equal(f_p.numpy(), want["f_generalized"]), it
        assert np.array_equal(np_p.numpy(), want["n_pairs"]) and np.array_equal(fl_p.numpy(), want["flags"])
    assert (fl_p.numpy() & 1).any()


def test_state_entry_point_bristle_and_rejects_chains():
    """Bristle states ride along in x (s-dot comes back); scenes with revolute / prismatic chains are refused."""
    n_env = 32
    m_gpu, m_cpu = _both(_normal_scene(2), n_env)
    rng = np.random.default_rng(7)
    x = np.zeros((n_env, S.num_x(m_gpu)))
    for e in range(n_env):
        x[e, 0:3] = rng.uniform(-0.03, 0.03, 3)
        x[e, 3:6] = [rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2), -rng.uniform(0.01, 0.1) * 0.05]
        x[e, 6:12] = rng.uniform(-0.1, 0.1, 6)
        x[e, 12:18] = rng.uniform(-1, 1, 6) * np.array([1e-3, 1e-3, 1e-3, 1e-5, 1e-5, 1e-5])
    out = S.force_all_elastic_intersections_batch(m_gpu, x)
    X_d, tw_d, w_d = m_gpu.backend.get_boundary(n_env)
    c = m_cpu.backend.eval_f64(X_d, tw_d, x[:, 12:18].reshape(n_env, 1, 6))
    assert (out["flags"] == c["flags"]).all() and (c["flags"] & 1).all()
    assert wrench_rel_err(out["sdot"], c["sdot"], floor=1e-9 * np.abs(c["sdot"]).max()) <= TOL
    f_ref = np.array([S.generalized_forces(m_cpu, x[e], c["wrench"][e]) for e in range(n_env)])
    assert np.abs(out["f_generalized"] - f_ref).max() <= TOL * np.abs(f_ref).max()
    from pfc_b200 import scenes
    m_chain, _ = scenes.scene_c2_pencil(True, _ctx())
    assert not m_chain.device_kinematics
    with pytest.raises(RuntimeError):
        S.force_all_elastic_intersections_batch(m_chain, S.get_state(m_chain))


# ---- mid-size trees on the on-chip path, and what happens when their pair-list slot is too small -------------------------
def test_mid_size_instructions_take_the_small_path_and_overflow_moves_them_to_the_large_path():
    """Spheres of 320 / 180 primitives: 57 600 possible leaf pairs, far more than the 1024-entry slot of the on-chip path, but a
    contact patch lists a few hundred.  (1) Shallow contacts: evaluated by the two small-path kernels (the large path's counters stay
    zero), results equal to the oracle's.  (2) A deep overlap (sphere inside sphere) overflows the slot: the library moves the
    instruction to the large path and repeats the evaluation by itself -- same parity bars, and from then on the large path runs."""
    n_env = 3
    m_gpu, m_cpu = _both(_sphere_scene(3, 2, with_small=False), n_env)      # 180 / 80 primitives: 14 400 possible leaf pairs
    x = _sphere_states(m_gpu, n_env + 1, 31, with_small=False)[1:]          # (the first sample is a deep contact: 513 pairs, a frontier beyond the slot)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))
    assert 0 < c["n_pairs"].max() < 512 and (c["flags"] & 1).sum() >= n_env
    assert m_gpu.backend.counters() == (0, 0)          # nothing went through the large path
    m_gpu, m_cpu = _both(_sphere_scene(4, 3, with_small=False), n_env)      # 320 / 180 primitives
    x = _sphere_states(m_gpu, n_env, 31, with_small=False)
    x[:, 3:6] = [0.0, 0.0, 0.012]                       # both spheres almost concentric with the ground sphere: thousands of candidate pairs
    x[:, 9:12] = [0.0, 0.004, -0.01]
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, c = _compare(m_gpu, m_cpu, X, tw, s.reshape(n_env, 1, 6))
    assert c["n_pairs"].max() > 1024
    n_tests, n_large_pairs = m_gpu.backend.counters()
    assert n_large_pairs > 1024 and n_tests > n_large_pairs   # the overflowing instructions now run on the large path
