"""The Float64 path at the batch sizes the benchmark runs and at every launch shape the small-path launchers pick, each against the CPU
oracle for EVERY environment.

The launchers choose by batch size (csrc/pfc_small.cu): the broad kernel takes P = 1, 2 or 4 problems per warp for n_prob = n_env * n_small
up to 16 n_sm, up to 32 n_sm and above (P = 1 whenever the pair-list slot holds more than 256 entries); the narrow tile kernel runs one CTA
per tile of 4 problems on at most 4 CTAs per SM and, once there are more tiles than that, CTAs draw further tiles from a ticket counter.
The thresholds here are computed from the device's SM count, and every test asserts, from the kernels it saw launched, that its sizes
reached the variant it is about."""
import re

import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import _sphere_scene, _sphere_states, _tet_tet_scene, boxes_env_states, kernel_grids, scene_boxes, wrench_rel_err
from oracle import orc
from pfc_b200 import dynamics as D
from pfc_b200 import parallel
from pfc_b200 import scenario as S

pytestmark = pytest.mark.gpu
TOL = 1.0e-9
N_BENCH = 4096           # bench.py's batch: 4096 environments at N = 1, env_range(4096, r, N) per GPU at N = 2, 4, 8
BOXES_SMALL = 4          # small instructions of test/boxes.jl: one narrow tile (4 problems) per environment
TILE_P, TILES_PER_SM = 4, 4


def _n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _broad_p(n_prob, n_sm):
    """Problems per warp of the small-path broad kernel for slots of <= 256 entries (launch_broad)."""
    return 1 if n_prob <= 16 * n_sm else (2 if n_prob <= 32 * n_sm else 4)


def _launched(kernels, name):
    hits = [(n, g) for n, g in kernels if re.search(r"\b" + name + r"\b", n)]
    assert hits, f"{name} was not launched: {[n for n, _ in kernels]}"
    return hits


def _broad_variant(kernels):
    (name, _), = _launched(kernels, "broad_tile_kernel")
    return int(re.search(r"broad_tile_kernel<(\d+)", name).group(1))


def _narrow_grid(kernels):
    (_, grid), = _launched(kernels, "narrow_tile_kernel")
    return grid


def _device_eval(ctx, X, tw, s=None):
    """pfc_eval_f64_device on torch device buffers (outputs pre-filled with values the library must overwrite), a sync on the context's
    stream; returns host copies and the kernels launched.  The profiled call is the second at this size: the first may grow the context's
    work buffers and repeat itself."""
    import torch
    dev = torch.device("cuda", 0)
    n_env, n_ins, nb = X.shape[0], ctx.n_ins, ctx.n_bristle
    b = dict(X=torch.from_numpy(np.ascontiguousarray(X)).to(dev), tw=torch.from_numpy(np.ascontiguousarray(tw)).to(dev),
             s=torch.from_numpy(np.ascontiguousarray(s).reshape(n_env, nb, 6)).to(dev) if nb else None,
             w=torch.full((n_env, n_ins, 6), float("nan"), dtype=torch.float64, device=dev),
             sd=torch.full((n_env, nb, 6), float("nan"), dtype=torch.float64, device=dev) if nb else None,
             np_=torch.full((n_env, n_ins), -1, dtype=torch.int64, device=dev), fl=torch.full((n_env, n_ins), 0x7f000000, dtype=torch.int32, device=dev))
    p = lambda t: None if t is None else t.data_ptr()

    def run():
        ctx.eval_f64_device(n_env, p(b["X"]), p(b["tw"]), p(b["s"]), p(b["w"]), p(b["sd"]), p(b["np_"]), p(b["fl"]))
        ctx.sync()
    torch.cuda.synchronize()
    run()
    b["w"].fill_(float("nan"))
    b["np_"].fill_(-1)
    b["fl"].fill_(0x7f000000)
    if nb:
        b["sd"].fill_(float("nan"))
    kernels = kernel_grids(run)
    out = dict(wrench=b["w"].cpu().numpy(), sdot=b["sd"].cpu().numpy() if nb else None, n_pairs=b["np_"].cpu().numpy(), flags=b["fl"].cpu().numpy())
    return out, kernels


def _check(g, c, sdot=False):
    """n_pairs and flags equal, wrench (and s-dot) within 1e-9 per 3-vector (test_gpu_parity's floor: 1e-9 of the batch's largest)."""
    assert np.array_equal(g["n_pairs"], c["n_pairs"])
    assert np.array_equal(g["flags"], c["flags"])
    assert wrench_rel_err(g["wrench"], c["wrench"], floor=1e-9 * max(np.abs(c["wrench"]).max(), 1e-300)) <= TOL
    if sdot:
        assert wrench_rel_err(g["sdot"], c["sdot"], floor=1e-9 * max(np.abs(c["sdot"]).max(), 1e-300)) <= TOL


# ---- test/boxes.jl at every broad-kernel variant and ticket regime, and at the benchmark's partitions ------------------------------------
@pytest.fixture(scope="module")
def boxes():
    """States of global environments 0..4095 seeded by their index (as bench.py seeds them), their boundary arrays, and the multi-threaded
    oracle's results for all of them (kept pair lists included)."""
    from pfc_b200 import capi
    m_host = scene_boxes(None)[0]
    x = boxes_env_states(m_host, N_BENCH)
    X, tw, _ = S.boundary_arrays(m_host, x)
    octx = orc.OracleContext(n_threads=orc.lib().orc_max_threads())
    m_cpu = scene_boxes(octx)[0]
    ref = octx.eval_f64(X, tw, keep=True)
    gpu = scene_boxes(capi.Context(0), max_env=N_BENCH)[0]
    keep = scene_boxes(capi.Context(0), max_env=N_BENCH)[0]
    return dict(x=x, X=X, tw=tw, ref=ref, octx=octx, m_cpu=m_cpu, gpu=gpu.backend, m_gpu=gpu, keep=keep.backend)


# threshold sizes (environments [0, n)) and the benchmark's partitions: env_range(4096, r, w) for w = 1, 2, 4, 8
SHAPES = ["1", "4sm", "4sm+1", "8sm", "8sm+1"] + [f"w{w}r{r}" for w in (1, 2, 4, 8) for r in range(w)]


def _shape_range(shape, n_sm):
    if shape.startswith("w"):
        w, r = map(int, shape[1:].split("r"))
        return parallel.env_range(N_BENCH, r, w)
    n = {"1": 1, "4sm": 4 * n_sm, "4sm+1": 4 * n_sm + 1, "8sm": 8 * n_sm, "8sm+1": 8 * n_sm + 1}[shape]
    assert n <= N_BENCH
    return 0, n


@pytest.mark.parametrize("shape", SHAPES)
def test_boxes_batch_shape_matches_oracle(boxes, shape):
    """Every environment of the batch, through pfc_eval_f64_device and pfc_eval_f64: pair counts and flags equal to the oracle's, wrenches
    within 1e-9; candidate-pair lists, in order, of the first and last environment and of 64 spread over the batch.  The threshold sizes sit
    on either side of the broad kernel's P = 1 / 2 and P = 2 / 4 cutoffs, which (4 boxes.jl problems per environment, 4 narrow tiles per SM)
    are also the sizes where the narrow tile kernel starts drawing tiles from its ticket counter (4 n_sm + 1 environments)."""
    n_sm = _n_sm()
    lo, hi = _shape_range(shape, n_sm)
    n = hi - lo
    p_want = _broad_p(BOXES_SMALL * n, n_sm)
    if shape in ("1", "4sm"):
        assert p_want == 1
    elif shape in ("4sm+1", "8sm"):
        assert p_want == 2
    elif shape == "8sm+1":
        assert p_want == 4
    if shape in ("4sm", "8sm"):   # the last size of its variant
        assert _broad_p(BOXES_SMALL * (n + 1), n_sm) == p_want + (1 if p_want == 1 else 2)
    X, tw = boxes["X"][lo:hi], boxes["tw"][lo:hi]
    ref = {k: boxes["ref"][k][lo:hi] for k in ("wrench", "n_pairs", "flags")}
    ctx = boxes["gpu"]
    g, kernels = _device_eval(ctx, X, tw)
    assert _broad_variant(kernels) == p_want
    grid = _narrow_grid(kernels)
    assert grid == min(n, TILES_PER_SM * n_sm)          # one tile per environment, at most 4 resident CTAs per SM
    if shape == "4sm+1" or n > 4 * n_sm:
        assert n > grid                                  # tiles beyond the resident CTAs: drawn from the ticket counter
    _check(g, ref)
    assert (ref["flags"] & 1).sum() > n
    h = ctx.eval_f64(X, tw)
    _check(h, ref)
    assert np.array_equal(h["wrench"], g["wrench"]) and np.array_equal(h["n_pairs"], g["n_pairs"]) and np.array_equal(h["flags"], g["flags"])
    # candidate-pair lists in the reference's order, on a context that keeps them
    boxes["keep"].eval_f64(X, tw, keep=True)
    envs = np.unique(np.concatenate([[0, n - 1], np.linspace(0, n - 1, 64).astype(int)]))
    for e in envs:
        for k in range(ctx.n_ins):
            assert np.array_equal(boxes["keep"].get_pairs(int(e), k), boxes["octx"].get_pairs(lo + int(e), k)), (shape, e, k)


def test_boxes_batch_invariance_bit_for_bit(boxes):
    """Each boxes.jl environment fills exactly one narrow tile and every sum has a fixed order, so environment e of the 4096 batch must come
    out bit for bit as when it is evaluated alone (n_env = 1: broad P = 1, one tile, no ticket) -- wrench, pair counts and flags, all 4096."""
    import torch
    ctx = boxes["gpu"]
    g, kernels = _device_eval(ctx, boxes["X"], boxes["tw"])
    assert _broad_variant(kernels) == 4 and _narrow_grid(kernels) < N_BENCH
    dev = torch.device("cuda", 0)
    n_ins = ctx.n_ins
    Xd, twd = torch.from_numpy(boxes["X"]).to(dev), torch.from_numpy(boxes["tw"]).to(dev)
    w1 = torch.full((N_BENCH, n_ins, 6), float("nan"), dtype=torch.float64, device=dev)
    np1 = torch.full((N_BENCH, n_ins), -1, dtype=torch.int64, device=dev)
    fl1 = torch.full((N_BENCH, n_ins), 0x7f000000, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    for e in range(N_BENCH):   # one environment per call, queued on the context's stream
        ctx.eval_f64_device(1, Xd[e].data_ptr(), twd[e].data_ptr(), None, w1[e].data_ptr(), None, np1[e].data_ptr(), fl1[e].data_ptr())
    ctx.sync()
    w1 = w1.cpu().numpy()
    same = (w1.view(np.int64) == g["wrench"].view(np.int64)).all(axis=(1, 2))
    assert same.all(), f"{int((~same).sum())} environments differ, first {np.flatnonzero(~same)[:8]}"
    assert np.array_equal(np1.cpu().numpy(), g["n_pairs"]) and np.array_equal(fl1.cpu().numpy(), g["flags"])


# ---- tiles that span environments: three small instructions per environment (one of them bristle) ------------------------------------------
def _tet_tet_states(m, n_env, seed):
    """test_tet_tet_batch_parity's state distribution: box_1 resting on the plane, box_2 on box_1, random twists and bristle state."""
    rng = np.random.default_rng(seed)
    r, nq = 0.05, m.nq
    x = np.zeros((n_env, S.num_x(m)))
    x[:, 0:3] = rng.uniform(-0.05, 0.05, (n_env, 3))
    x[:, 3:5] = rng.uniform(-0.01, 0.01, (n_env, 2))
    x[:, 5] = r - rng.uniform(0, 0.004, n_env)
    x[:, 6:9] = rng.uniform(-0.05, 0.05, (n_env, 3))
    x[:, 9:11] = rng.uniform(-0.03, 0.03, (n_env, 2))
    x[:, 11] = 3 * r - rng.uniform(0, 0.008, n_env)
    x[:, nq:nq + 12] = rng.uniform(-1, 1, (n_env, 12)) * 0.2
    x[:, nq + 12:] = rng.uniform(-1, 1, (n_env, 6)) * 1e-4
    return x


@pytest.mark.parametrize("n_env", [101, 4097])
def test_tiles_spanning_environments_match_oracle(n_env):
    """_tet_tet_scene has 3 small instructions, so with n_env * 3 % 4 != 0 the 4-problem tiles of the broad and narrow kernels straddle
    environments, and the last tile is partial.  101 environments (76 tiles) all fit the resident CTAs; 4097 (3073 tiles) draw most of theirs
    from the ticket counter.  Wrenches and the bristle instruction's s-dot (pfc_exact.cu at a batch size it is not otherwise run at) within
    1e-9 of the oracle, pair counts and flags equal."""
    from pfc_b200 import capi
    n_sm = _n_sm()
    m_gpu = _tet_tet_scene(capi.Context(0), n_env)
    m_cpu = _tet_tet_scene(orc.OracleContext(n_threads=orc.lib().orc_max_threads()), n_env)
    n_prob = 3 * n_env
    n_tile = (n_prob + TILE_P - 1) // TILE_P
    assert n_prob % TILE_P != 0
    x = _tet_tet_states(m_gpu, n_env, 17)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    g, kernels = _device_eval(m_gpu.backend, X, tw, s)
    grid = _narrow_grid(kernels)
    assert grid == min(n_tile, TILES_PER_SM * n_sm)
    assert (n_tile > grid) == (n_env > 1000)
    assert _broad_variant(kernels) == _broad_p(n_prob, n_sm)
    _launched(kernels, "exact_bristle_kernel")
    c = m_cpu.backend.eval_f64(X, tw, s.reshape(n_env, 1, 6))
    _check(g, c, sdot=True)
    assert (c["flags"] & 1).sum() > n_env


# ---- mid-size trees (slots of 1024 entries) in a batch above the P = 2 cutoff: the broad kernel must stay at P = 1 -----------------------------
def _shallow_sphere_states(m, n_env, seed):
    """_sphere_states with every overlap made shallow (2 to 6 mm): the s_tri sphere on the ground sphere, the s_tet sphere on the ground
    sphere (even environments, opposite side) or on the s_tri sphere (odd ones, radially outward) -- contact patches of at most ~100
    candidate pairs, whose frontiers fit the on-chip slot."""
    x = _sphere_states(m, n_env, seed, with_small=False)
    rng = np.random.default_rng(seed + 1)
    unit = lambda v: v / np.linalg.norm(v)
    for e in range(n_env):
        d1, d2 = unit(x[e, 3:6]), unit(rng.standard_normal(3))
        x[e, 3:6] = d1 * rng.uniform(0.104, 0.108)
        if e % 2:
            x[e, 9:12] = x[e, 3:6] + unit(d1 + 0.5 * d2) * rng.uniform(0.094, 0.098)
        else:
            x[e, 9:12] = unit(-d1 + 0.5 * d2) * rng.uniform(0.104, 0.108)
    return x


def test_mid_size_trees_above_the_p2_cutoff_stay_at_one_problem_per_warp():
    """_sphere_scene(3, 2): three mid-size instructions (180 / 80 primitives, pair-list slots of 1024 entries) in a batch with
    n_prob > 32 n_sm, where boxes.jl-size slots would take P = 4: the launcher's cap > 256 override must keep P = 1.  Oracle parity for every
    environment, and nothing moved to the large path (counters() == (0, 0): no slot overflowed)."""
    from pfc_b200 import capi
    n_sm = _n_sm()
    n_env = 32 * n_sm // 3 + 1
    assert 3 * n_env > 32 * n_sm and _broad_p(3 * n_env, n_sm) == 4
    build = _sphere_scene(3, 2, with_small=False)
    m_gpu = build(capi.Context(0), n_env)
    m_cpu = build(orc.OracleContext(n_threads=orc.lib().orc_max_threads()), n_env)
    x = _shallow_sphere_states(m_gpu, n_env, 41)
    X, tw, s = S.boundary_arrays(m_gpu, x)
    c = m_cpu.backend.eval_f64(X, tw, s.reshape(n_env, 1, 6))
    assert c["n_pairs"].max() < 256 and ((c["flags"] & 1).sum(axis=0) > n_env // 4).all()
    g, kernels = _device_eval(m_gpu.backend, X, tw, s)
    assert _broad_variant(kernels) == 1
    assert m_gpu.backend.counters() == (0, 0)
    _check(g, c, sdot=True)


# ---- state level at the benchmark's size ------------------------------------------------------------------------------------------------
def test_state_entry_point_pinned_graph_at_4096(boxes):
    """pfc_eval_state_f64 with pinned buffers, called three times with the same buffers (from the third identical call the host graph is
    replayed): the same bits every call, pair counts and flags equal to the oracle's, and every environment's generalized forces within 1e-9
    of addGeneralizedForcesThirdLaw! applied on the host to the oracle's wrenches."""
    import torch
    m_gpu, ctx = boxes["m_gpu"], boxes["gpu"]
    n_ins = ctx.n_ins
    x_p = torch.from_numpy(boxes["x"]).pin_memory()
    f_p = torch.zeros((N_BENCH, m_gpu.nv), dtype=torch.float64).pin_memory()
    np_p = torch.zeros((N_BENCH, n_ins), dtype=torch.int64).pin_memory()
    fl_p = torch.zeros((N_BENCH, n_ins), dtype=torch.int32).pin_memory()
    outs = []
    for _ in range(3):
        f_p.fill_(float("nan"))
        np_p.fill_(-1)
        ctx.eval_state_f64_ptr(N_BENCH, x_p.data_ptr(), f_p.data_ptr(), None, np_p.data_ptr(), fl_p.data_ptr())
        outs.append((f_p.numpy().copy(), np_p.numpy().copy(), fl_p.numpy().copy()))
    for f, n_pairs, flags in outs[1:]:
        assert np.array_equal(f.view(np.int64), outs[0][0].view(np.int64))
        assert np.array_equal(n_pairs, outs[0][1]) and np.array_equal(flags, outs[0][2])
    f, n_pairs, flags = outs[-1]
    ref = boxes["ref"]
    assert np.array_equal(n_pairs, ref["n_pairs"]) and np.array_equal(flags, ref["flags"])
    m_cpu, x = boxes["m_cpu"], boxes["x"]
    f_ref = np.array([S.generalized_forces(m_cpu, x[e], ref["wrench"][e]) for e in range(N_BENCH)])
    scale = np.maximum(np.abs(f_ref).max(axis=1), 1e-300)
    err = np.abs(f - f_ref).max(axis=1) / scale
    assert (err <= TOL).all(), (int(np.argmax(err)), float(err.max()))


def test_calcxd_device_at_4096(boxes):
    """pfc_calcxd_f64_device on the 4096 batch: every row bit for bit equal to the same environment evaluated alone, and 256 rows spread over
    the batch within 1e-9 (per 3-vector) of calcXd! on the host with the oracle's contact wrenches."""
    import torch
    m_gpu, ctx = boxes["m_gpu"], boxes["gpu"]
    assert m_gpu.device_dynamics
    dev = torch.device("cuda", 0)
    n_ins, x = ctx.n_ins, boxes["x"]
    nx = x.shape[1]
    x_d = torch.from_numpy(x).to(dev)
    xd = torch.full((N_BENCH, nx), float("nan"), dtype=torch.float64, device=dev)
    xd1 = torch.full((N_BENCH, nx), float("nan"), dtype=torch.float64, device=dev)
    npd = torch.zeros((N_BENCH, n_ins), dtype=torch.int64, device=dev)
    fld = torch.zeros((N_BENCH, n_ins), dtype=torch.int32, device=dev)
    np1 = torch.zeros((N_BENCH, n_ins), dtype=torch.int64, device=dev)
    fl1 = torch.zeros((N_BENCH, n_ins), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.calcxd_f64_device(N_BENCH, x_d.data_ptr(), None, xd.data_ptr(), npd.data_ptr(), fld.data_ptr())
    for e in range(N_BENCH):
        ctx.calcxd_f64_device(1, x_d[e].data_ptr(), None, xd1[e].data_ptr(), np1[e].data_ptr(), fl1[e].data_ptr())
    ctx.sync()
    xd, xd1 = xd.cpu().numpy(), xd1.cpu().numpy()
    same = (xd.view(np.int64) == xd1.view(np.int64)).all(axis=1)
    assert same.all(), f"{int((~same).sum())} rows differ, first {np.flatnonzero(~same)[:8]}"
    assert np.array_equal(npd.cpu().numpy(), boxes["ref"]["n_pairs"]) and np.array_equal(fld.cpu().numpy(), boxes["ref"]["flags"])
    assert np.array_equal(np1.cpu().numpy(), boxes["ref"]["n_pairs"]) and np.array_equal(fl1.cpu().numpy(), boxes["ref"]["flags"])
    dyn = D.FloatingBodyDynamics(scene_boxes(orc.OracleContext())[0])   # (its own oracle context: the fixture's keeps the 4096 pair lists)
    for e in np.unique(np.linspace(0, N_BENCH - 1, 256).astype(int)):
        ref = dyn.calcXd(x[e])
        for i in range(0, nx, 3):
            den = max(np.abs(ref[i:i + 3]).max(), 1e-9 * np.abs(ref).max())
            assert np.abs(xd[e, i:i + 3] - ref[i:i + 3]).max() <= TOL * den, (e, i)
