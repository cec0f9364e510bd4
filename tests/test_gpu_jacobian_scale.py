"""The whole Jacobian of calcXd! (pfc_calcxd_jacobian_device, Dual-6) at the benchmark's batch size.

At 4096 boxes.jl environments the Dual tile kernel (16 problems per tile, problems indexed (chunk, environment, instruction)) has 8192 tiles
for a few hundred resident CTAs, so most tiles come from its ticket counter, and the Float64 prefilter runs its grid-stride loop (its grid
is capped at 8 blocks per SM).  Small-batch tests reach neither."""
import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import boxes_env_states, kernel_grids, scene_boxes
from oracle import orc
from pfc_b200 import dynamics as D
from pfc_b200 import scenario as S

pytestmark = pytest.mark.gpu
TOL = 1.0e-9
DP = 16   # problems per Dual tile (kDP in csrc/pfc_dual_chunked.cu)


def _grids(kernels, name):
    return [g for n, g in kernels if name + "(" in n or name + "<" in n]


@pytest.mark.parametrize("bristle,n_env,n_mirror", [(False, 4096, 48), (True, 1500, 12)])
def test_whole_jacobian_at_scale(bristle, n_env, n_mirror):
    """(1) Batch invariance: every environment's Jacobian, value part, pair counts and flags equal, bit for bit, a one-environment call (the
    Dual tile sums each problem's items sequentially in candidate order, whichever tile and CTA it lands in).  (2) The whole Jacobian equals
    the ceil(n_x / 6) pfc_calcxd_dual6_device chunk calls bit for bit (the two modes index tiles differently).  (3) x_dot within 1e-9 of
    pfc_calcxd_f64_device, row by row (a different kernel).  (4) Columns of n_mirror environments -- in the first tile, in the last tile, in
    tiles that only the ticket counter hands out, and random ones -- within 1e-9 of the host mirror with the oracle's Dual-6 wrenches."""
    import torch
    from pfc_b200 import capi
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    m_gpu = scene_boxes(capi.Context(0), max_env=n_env, bristle=bristle)[0]
    ctx = m_gpu.backend
    assert m_gpu.device_dynamics
    nx = S.num_x(m_gpu)
    assert nx == (60 if bristle else 48)
    n_chunk, n_ins = (nx + 5) // 6, ctx.n_ins
    x = boxes_env_states(m_gpu, n_env)
    dev = torch.device("cuda", 0)
    f64 = dict(dtype=torch.float64, device=dev)
    x_d = torch.from_numpy(x).to(dev)
    jac = torch.full((n_env, nx, nx), float("nan"), **f64)
    xd = torch.full((n_env, nx), float("nan"), **f64)
    npd = torch.full((n_env, n_ins), -1, dtype=torch.int64, device=dev)
    fld = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)

    def whole():
        ctx.calcxd_jacobian_device(n_env, x_d.data_ptr(), None, jac.data_ptr(), xd.data_ptr(), npd.data_ptr(), fld.data_ptr())
        ctx.sync()
    torch.cuda.synchronize()
    whole()                           # (the first call at a size may grow the work buffers and repeat itself; the profiled one does not)
    jac.fill_(float("nan"))
    xd.fill_(float("nan"))
    kernels = kernel_grids(whole)
    # boxes.jl: every chunk in one launch, problems (chunk, environment, instruction); bristle scenes: one launch per chunk
    passes = 1 if not bristle else n_chunk
    grids = _grids(kernels, "eval_dual6_tile_kernel")
    assert len(grids) == passes, [n for n, _ in kernels]
    grid = grids[0]
    n_tile = (n_chunk // passes * n_env * n_ins + DP - 1) // DP
    if not bristle:
        assert grid < n_tile // 4        # most tiles come from the ticket counter
    pre, = _grids(kernels, "dual_prefilter_kernel")
    assert pre == 8 * n_sm and (n_env * n_ins + 3) // 4 > pre   # the prefilter's grid-stride loop runs
    jac_h, xd_h = jac.cpu().numpy(), xd.cpu().numpy()
    np_h, fl_h = npd.cpu().numpy(), fld.cpu().numpy()
    assert np.isfinite(jac_h).all() and (fl_h & 1).sum() > n_env

    # (1) one environment per call, queued on the context's stream
    jac1 = torch.full((n_env, nx, nx), float("nan"), **f64)
    xd1 = torch.full((n_env, nx), float("nan"), **f64)
    np1 = torch.full((n_env, n_ins), -1, dtype=torch.int64, device=dev)
    fl1 = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    for e in range(n_env):
        ctx.calcxd_jacobian_device(1, x_d[e].data_ptr(), None, jac1[e].data_ptr(), xd1[e].data_ptr(), np1[e].data_ptr(), fl1[e].data_ptr())
    ctx.sync()
    same = (jac1.cpu().numpy().view(np.int64) == jac_h.view(np.int64)).all(axis=(1, 2))
    assert same.all(), f"{int((~same).sum())} environments differ, first {np.flatnonzero(~same)[:8]}"
    assert np.array_equal(xd1.cpu().numpy().view(np.int64), xd_h.view(np.int64))
    assert np.array_equal(np1.cpu().numpy(), np_h) and np.array_equal(fl1.cpu().numpy(), fl_h)

    # (2) the chunk calls
    xd7 = torch.full((n_env, nx, 7), float("nan"), **f64)
    npc = torch.full((n_env, n_ins), -1, dtype=torch.int64, device=dev)
    flc = torch.zeros((n_env, n_ins), dtype=torch.int32, device=dev)
    for k in range(n_chunk):
        i0, i1 = 6 * k, min(6 * k + 6, nx)
        torch.cuda.synchronize()
        ctx.calcxd_dual6_device(n_env, x_d.data_ptr(), None, i0, xd7.data_ptr(), npc.data_ptr(), flc.data_ptr())
        ctx.sync()
        c = xd7.cpu().numpy()
        assert np.array_equal(jac_h[:, :, i0:i1], c[:, :, 1:1 + (i1 - i0)]), i0
        if k == 0:
            assert np.array_equal(xd_h, c[:, :, 0])
        assert np.array_equal(npc.cpu().numpy(), np_h) and np.array_equal(flc.cpu().numpy(), fl_h)

    # (3) the value part against the Float64 kernels
    xf = torch.full((n_env, nx), float("nan"), **f64)
    torch.cuda.synchronize()
    ctx.calcxd_f64_device(n_env, x_d.data_ptr(), None, xf.data_ptr(), npc.data_ptr(), flc.data_ptr())
    ctx.sync()
    xf = xf.cpu().numpy()
    err = np.abs(xf - xd_h).max(axis=1) / np.abs(xf).max(axis=1)
    assert (err <= TOL).all(), (int(np.argmax(err)), float(err.max()))

    # (4) absolute: host mirror (complex-step rigid-body terms + the oracle's Dual-6 wrenches)
    first, last = [0, 3], [n_env - 4, n_env - 1]
    tile_of = lambda e: (e * n_ins) // DP      # tile of environment e in chunk 0 (the later chunks' tiles come later still)
    late = [e for e in range(n_env) if tile_of(e) >= grid] or list(range(3 * n_env // 4, n_env - 4))
    assert bristle or len(late) > n_env // 4
    rng = np.random.default_rng(5)
    late = sorted(rng.choice(late, n_mirror // 4, replace=False).tolist())
    assert tile_of(first[1]) == 0 and tile_of(last[0]) == tile_of(n_env - 1)
    rest = [e for e in range(n_env) if e not in set(first + last + late)]
    envs = first + last + late + sorted(rng.choice(rest, n_mirror - len(first + last + late), replace=False).tolist())
    dyn = D.FloatingBodyDynamics(scene_boxes(orc.OracleContext(), bristle=bristle)[0])
    for e in envs:
        for i0 in range(0, nx, 6):
            i1 = min(i0 + 6, nx)
            _, cols = dyn.de_jacobian_chunk(x[e], i0, i1)
            for d in range(i1 - i0):
                col = cols[:, d]
                assert np.abs(jac_h[e, :, i0 + d] - col).max() <= TOL * max(np.abs(col).max(), 1e-6 * np.abs(cols).max()), (e, i0, d)
