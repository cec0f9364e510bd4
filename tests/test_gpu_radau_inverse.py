"""pfc_radau_inv_c_device (csrc/pfc_radau.cu) against high-precision references.

The kernel replaces LAPACK getrf! + getri! in the batched Radau step (updateInvC!): C = (h^-1 lambda_i) I - J, inverted by Gauss-Jordan with
a warp pivot search and the row interchanges undone as column interchanges at the end, for 1 <= n <= 96.  The sizes below cover one and
several rows per lane in the pivot search and n * n below and above the 256 threads of a CTA."""
import numpy as np
import pytest

import pfc_b200  # noqa: F401
from helpers import boxes_env_states, scene_boxes

pytestmark = pytest.mark.gpu
SIZES = [1, 2, 5, 31, 32, 33, 47, 48, 60, 64, 95, 96]
EPS = np.finfo(np.float64).eps


def _ctx():
    from pfc_b200 import capi
    return capi.Context(0)


def _inv_c(ctx, neg_J, shift, index=None, info=True):
    """Runs the kernel on torch device buffers: neg_J [n_src][n][n] real, shift [n_mat] complex, index [n_mat] or None -> (inverses
    [n_mat][n][n] complex128, info word or None)."""
    import torch
    dev = torch.device("cuda", 0)
    neg_J = np.ascontiguousarray(neg_J, dtype=np.float64)
    n = neg_J.shape[-1]
    shift = np.ascontiguousarray(np.asarray(shift, dtype=np.complex128).reshape(-1))
    n_mat = shift.shape[0]
    jd = torch.from_numpy(neg_J).to(dev)
    sd = torch.view_as_real(torch.from_numpy(shift)).contiguous().to(dev)
    idx = None if index is None else torch.from_numpy(np.ascontiguousarray(index, dtype=np.int32)).to(dev)
    out = torch.full((n_mat, n, n), complex(float("nan"), float("nan")), dtype=torch.complex128, device=dev)
    inf = torch.zeros(1, dtype=torch.int32, device=dev) if info else None
    torch.cuda.synchronize()
    ctx.radau_inv_c_device(n_mat, n, jd.data_ptr(), sd.data_ptr(), None if idx is None else idx.data_ptr(), out.data_ptr(),
                           None if inf is None else inf.data_ptr())
    ctx.sync()
    return out.cpu().numpy(), (None if inf is None else int(inf.item()))


def _radau_shifts(hs):
    """lambda_i / h for the three stages of the Radau IIA rule of order 5 (radau_table(2)) and every step size in hs."""
    from pfc_b200 import radau as R
    lam = R.radau_table(2).lam
    assert len(lam) == 3
    return np.array([l / h for h in hs for l in lam])


def _random_neg_J(rng, n, scale=10.0):
    return rng.standard_normal((n, n)) * scale


def _check_residual(C, X):
    """||C X - I||_inf <= 16 n eps ||C||_inf ||X||_inf (the backward-stable bound of a pivoted elimination)."""
    n = C.shape[0]
    r = np.abs(C @ X - np.eye(n)).sum(axis=1).max()
    bound = 16 * n * EPS * np.abs(C).sum(axis=1).max() * np.abs(X).sum(axis=1).max()
    assert r <= bound, (n, r, bound)


def _check_elementwise(X, X_ref, tol=1e-12):
    """Every element within tol of the exact inverse's largest element."""
    err = np.abs(X - X_ref).max() / np.abs(X_ref).max()
    assert err <= tol, err


def _mp_inverse(C):
    import mpmath
    with mpmath.workdps(50):
        A = mpmath.matrix([[mpmath.mpc(complex(v)) for v in row] for row in C])
        Ai = A ** -1
        return np.array([[complex(Ai[i, j]) for j in range(C.shape[1])] for i in range(C.shape[0])])


@pytest.mark.parametrize("n", SIZES)
def test_shifted_random_jacobians(n):
    """Random -J with the complex stage shifts lambda_i / h of the order-5 rule for h = 1e-6 .. 1e-1: against numpy's complex128 inverse and
    the residual bound for every matrix, elementwise (to 1e-12 of the largest element) wherever cond(C) < 1e3, and against a 50-digit mpmath
    inverse for two matrices per size up to 48."""
    rng = np.random.default_rng(1000 + n)
    hs = np.logspace(-6, -1, 6)
    shifts = _radau_shifts(hs)
    neg_J = np.stack([_random_neg_J(rng, n) for _ in range(len(shifts))])
    X, info = _inv_c(_ctx(), neg_J, shifts, index=np.arange(len(shifts)))
    assert info == 0
    n_well = 0
    for i, sh in enumerate(shifts):
        C = neg_J[i] + sh * np.eye(n)
        _check_residual(C, X[i])
        if np.linalg.cond(C) < 1e3:
            _check_elementwise(X[i], np.linalg.inv(C))
            n_well += 1
    assert n_well >= len(shifts) // 2
    if n <= 48:
        for i in (2, len(shifts) - 1):      # h = 1e-6 (the shift dominates) and h = 1e-1 (the matrix does)
            C = neg_J[i] + shifts[i] * np.eye(n)
            ref = _mp_inverse(C)
            _check_elementwise(X[i], ref, tol=1e-12 if np.linalg.cond(C) < 1e3 else 1e-12 * np.linalg.cond(C) / 1e3)


@pytest.fixture(scope="module")
def boxes_jacobians():
    """-J of calcXd! for two boxes.jl states: n_x = 48 (regularized friction) and 60 (two bristle instructions)."""
    out = {}
    for bristle in (False, True):
        m = scene_boxes(_ctx(), max_env=2, bristle=bristle)[0]
        x = boxes_env_states(m, 2)
        out[bristle] = -m.backend.calcxd_jacobian(x)["jac"]
    return out


@pytest.mark.parametrize("bristle", [False, True])
def test_boxes_jacobians(boxes_jacobians, bristle):
    """The real Jacobians of test/boxes.jl (48 x 48, and 60 x 60 with bristle friction) with the stage shifts for h = 1e-6 .. 1e-1, shared
    by the stages through `index` as the batched integrator does: residual bound everywhere, elementwise against numpy where cond(C) < 1e3,
    and one matrix against mpmath."""
    neg_J = boxes_jacobians[bristle]
    n = neg_J.shape[-1]
    assert n == (60 if bristle else 48)
    shifts = _radau_shifts(np.logspace(-6, -1, 6))
    index = np.repeat(np.arange(2), len(shifts))
    shifts = np.tile(shifts, 2)
    X, info = _inv_c(_ctx(), neg_J, shifts, index=index)
    assert info == 0
    n_well = 0
    for i, sh in enumerate(shifts):
        C = neg_J[index[i]] + sh * np.eye(n)
        _check_residual(C, X[i])
        if np.linalg.cond(C) < 1e3:
            _check_elementwise(X[i], np.linalg.inv(C))
            n_well += 1
    assert n_well >= 4
    C = neg_J[0] + shifts[3] * np.eye(n)
    if not bristle:
        _check_elementwise(X[3], _mp_inverse(C), tol=1e-12 * max(1.0, np.linalg.cond(C) / 1e3))


@pytest.mark.parametrize("n", SIZES)
def test_pivoting_on_every_step(n):
    """Matrices that need a row interchange at (nearly) every step, with a zero shift: a random permutation matrix (its inverse, the
    transpose, must come out exactly), the anti-diagonal with random entries (inverse: the anti-diagonal of reciprocals), and a zero diagonal
    with random off-diagonal entries (residual bound, numpy)."""
    rng = np.random.default_rng(2000 + n)
    P = np.eye(n)[rng.permutation(n)]
    if n > 1:
        while (np.diag(P) != 0).any():      # a derangement: no pivot is ever found in place
            P = np.eye(n)[rng.permutation(n)]
    d = rng.uniform(0.5, 2.0, n) * rng.choice([-1.0, 1.0], n)
    A = np.fliplr(np.diag(d))
    Z = rng.standard_normal((n, n))
    np.fill_diagonal(Z, 0.0)
    mats = [P, A] + ([Z] if n > 1 else [])
    X, info = _inv_c(_ctx(), np.stack(mats), np.zeros(len(mats)), index=None)
    assert info == 0
    assert np.array_equal(X[0], P.T.astype(np.complex128))
    A_inv = np.flipud(np.diag(1.0 / d))
    assert np.abs(X[1] - A_inv).max() <= 2 * EPS * np.abs(A_inv).max()
    if n > 1:
        _check_residual(Z.astype(np.complex128), X[2])
        if np.linalg.cond(Z) < 1e3:
            _check_elementwise(X[2], np.linalg.inv(Z))


def test_index_gather_more_matrices_than_sources():
    """3 stages x 4096 matrices built from 1000 sources through a non-identity index (repeated, out of order): every matrix bit for bit equal
    to the same inversion with its source copied into place (index = NULL), and a sample of 256 against the residual bound."""
    rng = np.random.default_rng(7)
    n, n_src, n_env = 48, 1000, 4096
    neg_J = rng.standard_normal((n_src, n, n)) * 10.0
    h = 10.0 ** rng.uniform(-6, -1, n_env)
    from pfc_b200 import radau as R
    lam = R.radau_table(2).lam
    shifts = np.concatenate([l / h for l in lam])                 # stage-major, as radau_batched.py queues them
    env_src = rng.integers(0, n_src, n_env)
    index = np.tile(env_src, 3)
    assert len(np.unique(index)) < n_env and (np.diff(index) < 0).any()
    ctx = _ctx()
    X, info = _inv_c(ctx, neg_J, shifts, index=index)
    assert info == 0
    X_flat, _ = _inv_c(ctx, neg_J[index], shifts, index=None)
    assert np.array_equal(X.view(np.float64), X_flat.view(np.float64))
    for i in rng.choice(len(shifts), 256, replace=False):
        _check_residual(neg_J[index[i]] + shifts[i] * np.eye(n), X[i])


def test_singular_flag_null_info_and_arguments():
    """An exactly singular matrix (a zero column survives elimination exactly) sets info bit 0 even among regular ones; regular batches leave
    info at 0; info = NULL is accepted; n_mat = 0 is a no-op; n = 0 and n = 97 are PFC_E_ARG."""
    import torch
    from pfc_b200 import capi
    rng = np.random.default_rng(3)
    ctx = _ctx()
    n = 33
    regular = rng.standard_normal((4, n, n)) + 10.0 * np.eye(n)
    singular = rng.standard_normal((n, n))
    singular[:, 5] = 0.0
    X, info = _inv_c(ctx, np.concatenate([regular, singular[None]]), np.zeros(5))
    assert info & 1
    for i in range(4):
        _check_residual(regular[i].astype(np.complex128), X[i])
    X2, info2 = _inv_c(ctx, regular, np.zeros(4))
    assert info2 == 0 and np.array_equal(X2, X[:4])
    X3, none = _inv_c(ctx, np.concatenate([regular, singular[None]]), np.zeros(5), info=False)
    assert none is None and np.array_equal(X3[:4], X[:4])
    # n_mat = 0: nothing is written
    dev = torch.device("cuda", 0)
    buf = torch.full((2, n, n), 7.0 + 7.0j, dtype=torch.complex128, device=dev)
    jd = torch.zeros((1, n, n), dtype=torch.float64, device=dev)
    sd = torch.zeros((1, 2), dtype=torch.float64, device=dev)
    inf = torch.zeros(1, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ctx.radau_inv_c_device(0, n, jd.data_ptr(), sd.data_ptr(), None, buf.data_ptr(), inf.data_ptr())
    ctx.sync()
    assert (buf.cpu().numpy() == 7.0 + 7.0j).all() and int(inf.item()) == 0
    for bad_n in (0, 97):
        with pytest.raises(capi.PfcError) as exc:
            ctx.radau_inv_c_device(1, bad_n, jd.data_ptr(), sd.data_ptr(), None, buf.data_ptr(), inf.data_ptr())
        assert exc.value.code == -1   # PFC_E_ARG
