"""GPU tests of the small kernels of the C ABI at their edge shapes, each against a reference of higher precision than
the kernel (mpmath, long double or exactly summed reductions, the oracle's analyzers), and of one sweep over whitening
groups of different singular-space dimensions.

    mx_tau_kernel         beta = 1, 40, 1000; tau at 0 and beta; omega at 0, +-1e-300 and where beta |omega| ~ 700-750
    mx_layout_V           every tile count, odd n_omega, n_sv not a multiple of 8: bitwise, zero padding included
    mx_project_data       n_tau from 1 to 10000, n_sv up to 256, data almost inside range(Q)
    mx_gram_schmidt_rows  p up to 512, rows shorter and longer than the CTA, graded and exactly dependent rows
    mx_svd_jacobi         odd sizes, m < n, rank 1, a zero column, the zero matrix; the truncated route with odd p
    mx_analyze            n_alpha from 1 to 1024, both mesh orders, gamma, every LineFit / Bryan option, NaN patterns
    mx_poorman_models     every slot, whitening groups, A_init, odd n_omega, n_omega above 48 KB of shared memory
"""
import ctypes
import math

import numpy as np
import pytest

from oracle import maxent_oracle as mo
from tests import gpu_common as gc

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -52


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


@pytest.fixture(scope="module")
def lib(torch_cuda):
    from maxent_b200 import _lib
    return _lib.load()


def _stream(torch):
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(torch, x):
    return torch.tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


# ----------------------------------------------------------------------------------------------
# mx_tau_kernel
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beta", [1.0, 40.0, 1000.0])
def test_tau_kernel_near_underflow(torch_cuda, lib, beta):
    """K(tau, omega) = -exp(-omega tau) / (1 + exp(-beta omega)) against mpmath at 50 digits.  The exponents are the
    float64 products every float64 evaluation forms (-omega * tau, -beta * omega for omega >= 0; omega * (beta - tau),
    beta * omega below); the reference takes them as given and evaluates the rest exactly.  Within 4 ulp where |K| is
    normal, within 2^-1022 where it is subnormal or underflows; never NaN or Inf."""
    import mpmath
    torch = torch_cuda
    tau = np.concatenate([np.linspace(0.0, beta, 33), [1e-300, beta * 1e-3, beta * (1 - 1e-12)]])
    edge = np.array([700.0, 708.3, 708.4, 709.0, 709.78, 709.79, 710.0, 720.0, 745.0, 745.2, 750.0]) / beta
    omega = np.concatenate([[0.0, 1e-300, -1e-300, 5e-324, -5e-324], edge, -edge,
                            mo.hyperbolic_omega_mesh(-10, 10, 21)])
    t_d, o_d = _dev(torch, tau), _dev(torch, omega)
    K = torch.empty((len(tau), len(omega)), dtype=torch.float64, device="cuda")
    assert lib.mx_tau_kernel(t_d.data_ptr(), o_d.data_ptr(), len(tau), len(omega), beta, K.data_ptr(),
                             _stream(torch)) == 0
    K = K.cpu().numpy()
    assert np.all(np.isfinite(K))
    mpmath.mp.dps = 50
    ref = np.empty_like(K)
    for i, t in enumerate(tau):
        for j, w in enumerate(omega):
            if w >= 0.0:
                x1, x2 = (-w) * t, (-beta) * w
            else:
                x1, x2 = w * (beta - t), beta * w
            ref[i, j] = float(-mpmath.exp(mpmath.mpf(float(x1))) / (1 + mpmath.exp(mpmath.mpf(float(x2)))))
    normal = np.abs(ref) >= 2.0 ** -1022
    err = np.abs(K - ref)
    ulp = np.spacing(np.abs(ref))
    assert np.all(err[normal] <= 4 * ulp[normal]), np.max(err[normal] / ulp[normal])
    assert np.all(err[~normal] <= 2.0 ** -1022)
    assert np.any(~normal) and np.any(normal & (np.abs(ref) < 2.0 ** -1000))        # both sides of the underflow met


# ----------------------------------------------------------------------------------------------
# mx_layout_V
# ----------------------------------------------------------------------------------------------
def _tile_off(n, c):
    """mx_common.cuh tile_off: position of element (row n, column c) of an 8 x 8 tile of V'."""
    q, e, cc, h = n >> 1, n & 1, c >> 1, c & 1
    return 16 * q + 2 * ((4 * e + cc + 2 * q) & 7) + h


@pytest.mark.parametrize("n_sv", [1, 7, 8, 9, 52, 80, 81, 96, 200, 256])
def test_layout_V_inverts_tile_off(torch_cuda, lib, n_sv):
    """V'[n_omega, n_sv] -> [n_kt][NT][64] tiles: every element where the host inverse of tile_off puts it, exact zeros
    in the padding rows (odd n_omega) and columns (n_sv up to NT * 8), bit for bit."""
    torch = torch_cuda
    inv = np.full((64, 2), -1)
    for n in range(8):
        for c in range(8):
            inv[_tile_off(n, c)] = (n, c)
    assert np.all(inv >= 0)                                             # tile_off is a bijection of the 64 slots
    rng = np.random.RandomState(n_sv)
    for n_omega in (1, 7, 8, 1001):
        V = rng.randn(n_omega, n_sv) + 3.0                             # no zeros: a zero in Vt is padding
        NT, n_kt = gc.sweep_tiles(n_sv), (n_omega + 7) // 8
        total = int(lib.mx_layout_V_size(n_omega, n_sv))
        assert total == n_kt * NT * 64
        Vt = torch.full((total,), float("nan"), dtype=torch.float64, device="cuda")
        V_d = _dev(torch, V)
        assert lib.mx_layout_V(V_d.data_ptr(), n_omega, n_sv, Vt.data_ptr(), _stream(torch)) == 0
        o = np.arange(total)
        tile, e = o // 64, o % 64
        k = (tile // NT) * 8 + inv[e, 0]
        j = (tile % NT) * 8 + inv[e, 1]
        inside = (k < n_omega) & (j < n_sv)
        want = np.zeros(total)
        want[inside] = V[k[inside], j[inside]]
        got = Vt.cpu().numpy()
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (n_omega, n_sv)
    for bad in ((0, n_sv), (8, 0), (8, 257), (-1, 8)):
        assert lib.mx_layout_V_size(*bad) < 0


# ----------------------------------------------------------------------------------------------
# mx_project_data
# ----------------------------------------------------------------------------------------------
_PROJECT_CASES = [(n_tau, s) for n_tau in (1, 31, 33, 2000, 10000) for s in (1, 9, 52, 81, 256) if s <= n_tau]


@pytest.mark.parametrize("n_tau,s", _PROJECT_CASES)
def test_project_data_vs_long_double(torch_cuda, lib, n_tau, s):
    """gt = (sqrt(w) Q)^T G and c0 = |sqrt(w) G - Q gt|^2 for orthonormal Q[n_tau, s], error bars over four decades, and
    data y = sqrt(w) G that lie inside range(Q) up to 1e-12 |y| (c0 is then a cancellation: |y|^2 - |gt|^2 ~ 1e-24 |y|^2)
    or far from it.  Reference: the same formula in long double.  gt within 4 eps sqrt(n_tau) sum_i |Qw_ij G_i|; c0 >= 0
    and within 4 eps (s + sqrt(n_tau)) |y|^2, which bounds the rounding of the residual y - Q gt (s products per row,
    each of size <= |y|) and of the sum of its squares, whatever the cancellation."""
    from maxent_b200 import _lib
    torch = torch_cuda
    rng = np.random.RandomState(n_tau * 1000 + s)
    Q, _ = np.linalg.qr(rng.randn(n_tau, s))
    err = 10.0 ** rng.uniform(-6, -2, n_tau)
    sqrtw = 1.0 / err
    Qw = sqrtw[:, None] * Q
    c = rng.randn(3, s)
    y = c @ Q.T
    y[0] += 1e-12 * np.linalg.norm(y[0]) * rng.randn(n_tau) / math.sqrt(n_tau)   # almost inside range(Q)
    y[2] += rng.randn(n_tau)                                                    # far from it
    G = y / sqrtw[None, :]
    Qd, Qwd, swd, Gd = _dev(torch, Q), _dev(torch, Qw), _dev(torch, sqrtw), _dev(torch, G)
    gt = torch.full((3, s), float("nan"), dtype=torch.float64, device="cuda")
    c0 = torch.full((3,), float("nan"), dtype=torch.float64, device="cuda")
    p = _lib.MxProblem()
    p.n_tau, p.n_sv, p.n_omega, p.n_alpha = n_tau, s, 1, 1
    p.Qw, p.Qo, p.sqrtw = Qwd.data_ptr(), Qd.data_ptr(), swd.data_ptr()
    assert lib.mx_project_data(ctypes.byref(p), Gd.data_ptr(), 3, gt.data_ptr(), c0.data_ptr(), _stream(torch)) == 0
    gt, c0 = gt.cpu().numpy(), c0.cpu().numpy()
    L = np.longdouble
    QwL, QL, GL = Qw.astype(L), Q.astype(L), G.astype(L)
    gtL = GL @ QwL                                             # [3, s]
    rL = sqrtw.astype(L)[None, :] * GL - gtL @ QL.T
    c0L = np.sum(rL * rL, axis=1)
    bound_gt = 4 * EPS * math.sqrt(n_tau) * (np.abs(G) @ np.abs(Qw))
    assert np.all(np.abs(gt - gtL.astype(np.float64)) <= bound_gt), np.max(np.abs(gt - gtL.astype(float)) / bound_gt)
    ynorm2 = np.sum((sqrtw[None, :] * G) ** 2, axis=1)
    assert np.all(c0 >= 0.0)
    dc = np.abs(c0 - c0L.astype(np.float64))
    assert np.all(dc <= 4 * EPS * (s + math.sqrt(n_tau)) * ynorm2), (dc, c0L, ynorm2)


# ----------------------------------------------------------------------------------------------
# mx_gram_schmidt_rows
# ----------------------------------------------------------------------------------------------
def _gram_schmidt(torch, lib, Y, drop_rel):
    Yt = _dev(torch, Y)
    rc = lib.mx_gram_schmidt_rows(Yt.data_ptr(), Y.shape[1], Y.shape[0], drop_rel, _stream(torch))
    assert rc == 0
    return Yt.cpu().numpy()


def _check_orthonormal_rows(Qr, chk, tol):
    L = np.longdouble
    QL = Qr.astype(L)
    Gm = (QL[chk] @ QL.T).astype(np.float64)
    keep = np.any(Qr != 0.0, axis=1)
    want = np.zeros_like(Gm)
    want[np.arange(len(chk)), chk] = keep[chk]
    assert np.max(np.abs(Gm - want)) <= tol, np.max(np.abs(Gm - want)) / tol
    return keep


@pytest.mark.parametrize("p", [1, 2, 33, 129, 512])
def test_gram_schmidt_graded_rows(torch_cuda, lib, p):
    """Rows Y_j = sum_{i<j} C_ji X_i + d_j X_j with d_j from 1 down to 1e-12: every row but the first lies within 1e-12 of
    the span of the rows before it (condition ~1e12).  In long double: the rows that come back are orthonormal to
    16 sqrt(len) eps, and Y = R Q with R lower-triangular: the entries of Y Q^T above the diagonal and the residual
    Y_i - sum_{j<=i} R_ij Q_j stay below 16 sqrt(len) eps |Y_i|.  (Every row is checked for p <= 129; 64 of them at
    p = 512, where a full long-double product of 512 x 512 x 5000 would dominate the test.)"""
    torch = torch_cuda
    rng = np.random.RandomState(p)
    for n in sorted({p, 1000, 1025, 5000}):
        if n < p:
            continue
        X = rng.randn(p, n)
        C = np.tril(rng.randn(p, p), -1)
        C[np.diag_indices(p)] = np.logspace(0, -12, p) if p > 1 else 1.0
        Y = C @ X
        Qr = _gram_schmidt(torch, lib, Y, 0.0)
        assert np.all(np.isfinite(Qr))
        chk = np.arange(p) if p <= 129 else np.unique(np.concatenate([np.arange(16), np.arange(p - 16, p),
                                                                        rng.choice(p, 32, replace=False)]))
        tol = 16 * math.sqrt(n) * EPS
        keep = _check_orthonormal_rows(Qr, chk, tol)
        assert np.all(keep), "a graded row was dropped with drop_rel = 0"
        L = np.longdouble
        QL, YL = Qr.astype(L), Y.astype(L)
        R = YL[chk] @ QL.T                                                   # [len(chk), p]
        ynorm = np.sqrt(np.sum(Y[chk] ** 2, axis=1))
        upper = np.arange(p)[None, :] > chk[:, None]
        assert np.all(np.abs(R.astype(float)) * upper <= tol * ynorm[:, None]), (p, n)
        Rl = np.where(upper, L(0), R)
        res = np.sqrt(np.sum(((YL[chk] - Rl @ QL).astype(float)) ** 2, axis=1))
        assert np.all(res <= tol * ynorm), (p, n, np.max(res / ynorm))


def test_gram_schmidt_dependent_rows(torch_cuda, lib):
    """Exactly dependent rows: a zero row and a multiple of an exact unit vector leave a residual of exactly zero and
    come back as zero rows (not 0 * rsqrt(0) = NaN), with drop_rel = 0 as well; a bitwise copy of an earlier row falls
    below drop_rel = 4 eps (the range finder's setting) and is zeroed there.  Every other row is a unit vector
    orthogonal to the rest.  p = 513 rows are refused."""
    torch = torch_cuda
    rng = np.random.RandomState(5)
    p, n = 40, 1000
    Y = rng.randn(p, n)
    Y[0] = 0.0
    Y[0, 17] = 4.0
    Y[3] = 0.0
    Y[3, 17] = -3.0                  # 3 * (-e_17): dependent on row 0 with a zero residual
    Y[7] = 0.0                       # zero row
    Y[12] = Y[9]                     # bitwise copy
    for drop in (0.0, 4 * EPS):
        Qr = _gram_schmidt(torch, lib, Y, drop)
        assert np.all(np.isfinite(Qr))
        assert np.all(Qr[[3, 7]] == 0.0)
        if drop > 0:
            assert np.all(Qr[12] == 0.0)
        keep = _check_orthonormal_rows(Qr, np.arange(p), 16 * math.sqrt(n) * EPS)
        assert np.all(keep[np.setdiff1d(np.arange(p), [3, 7, 12])])     # row 12 at drop_rel = 0: unit or zero
    Yd = torch.zeros((513, 600), dtype=torch.float64, device="cuda")
    assert lib.mx_gram_schmidt_rows(Yd.data_ptr(), 600, 513, 0.0, _stream(torch)) == -1
    assert lib.mx_gram_schmidt_rows(Yd.data_ptr(), 600, 0, 0.0, _stream(torch)) == -1


# ----------------------------------------------------------------------------------------------
# SVD: mx_svd_jacobi and the routes of engine.device_svd
# ----------------------------------------------------------------------------------------------
def _svd_cases():
    rng = np.random.RandomState(12)
    graded = lambda m, n, k: ((np.linalg.qr(rng.randn(m, k))[0] * np.logspace(0, -8, k))
                              @ np.linalg.qr(rng.randn(n, k))[0].T)
    rank1 = np.outer(rng.randn(50), rng.randn(31))
    zcol = rng.randn(60, 21)
    zcol[:, 7] = 0.0
    return [("1x1", np.array([[-2.5]])), ("5x1", rng.randn(5, 1)), ("1x5", rng.randn(1, 5)),
            ("69x69", graded(69, 69, 69)), ("100x69", rng.randn(100, 69)), ("40x69", graded(40, 69, 40)),
            ("rank1", rank1), ("zero column", zcol), ("zero", np.zeros((30, 9))),
            ("200x161", rng.randn(200, 161)), ("400x333", rng.randn(400, 333))]


@pytest.mark.parametrize("case", range(11))
def test_device_svd_edge_shapes(torch_cuda, case):
    """Odd sizes (the dummy player of the Jacobi tournament), m = n, m < n (the transpose route), rank 1, a zero column,
    the zero matrix, and full-rank 161 / 333 columns, which end in the truncated route with an odd p.  Against LAPACK:
    singular values within 64 sqrt(min(m, n)) eps S0, reconstruction within 64 sqrt(max(m, n)) eps S0 (the range finder
    of the truncated route leaves ~1e-13 S0 at 333 columns, the level test_gpu_parity holds a full-rank matrix to), leading vectors
    (S >= 1e-3 S0) orthonormal to 1e-12, exact zeros where the matrix has exact zero columns, nothing NaN; a second call
    gives the same bits."""
    torch = torch_cuda
    from maxent_b200 import engine
    name, K = _svd_cases()[case]
    m, n = K.shape
    Kd = _dev(torch, K)
    U, S, V, info = engine.device_svd(Kd)
    U2, S2, V2, _ = engine.device_svd(Kd)
    assert torch.equal(U, U2) and torch.equal(S, S2) and torch.equal(V, V2), name
    if min(m, n) > engine.SVD_DIRECT_MAX:
        assert info.startswith("range finder + jacobi, all %d" % min(m, n)), info
    U, S, V = U.cpu().numpy(), S.cpu().numpy(), V.cpu().numpy()
    k = min(m, n)
    assert U.shape == (m, k) and S.shape == (k,) and V.shape == (n, k), (name, U.shape, S.shape, V.shape)
    assert np.all(np.isfinite(U)) and np.all(np.isfinite(S)) and np.all(np.isfinite(V)), name
    Sref = np.linalg.svd(K, compute_uv=False)
    S0 = max(Sref[0], np.finfo(float).tiny)
    assert np.all(np.diff(S) <= 0) and np.all(S >= 0), name
    assert np.max(np.abs(S - Sref)) <= 64 * math.sqrt(k) * EPS * S0, (name, np.max(np.abs(S - Sref)) / S0)
    assert np.max(np.abs((U * S) @ V.T - K)) <= 64 * math.sqrt(max(m, n)) * EPS * S0, name
    lead = int(np.sum(Sref >= 1e-3 * Sref[0])) if Sref[0] > 0 else 0
    I = np.eye(lead)
    assert np.max(np.abs(V[:, :lead].T @ V[:, :lead] - I), initial=0.0) < 1e-12, name
    assert np.max(np.abs(U[:, :lead].T @ U[:, :lead] - I), initial=0.0) < 1e-12, name
    if name == "zero":
        assert np.all(S == 0.0) and np.all(U == 0.0)
    if name == "zero column":
        assert S[-1] == 0.0 and np.all(U[:, -1] == 0.0) and np.all(np.abs(V[:, -1]) == np.eye(n)[7])
    if name == "rank1":
        assert np.all(S[1:] <= 64 * math.sqrt(k) * EPS * S0)


# ----------------------------------------------------------------------------------------------
# mx_analyze
# ----------------------------------------------------------------------------------------------
def _nan_patterns(n, chi2, S, logp):
    """Rows 1..9 of the batch: NaN in chi2 / S / logp, leading, trailing, interior, everywhere, one logp left."""
    k = max(1, min(2, n - 1))
    chi2[1, :k] = np.nan
    chi2[2, n - k:] = np.nan
    chi2[3, n // 2] = np.nan
    chi2[4, :] = np.nan
    S[5, :k] = np.nan
    S[5, n // 2] = np.nan
    S[6, :] = np.nan
    logp[7, :] = np.nan
    logp[8, :] = np.nan
    logp[8, (2 * n) // 3] = 0.5
    logp[9, :k] = np.nan
    logp[9, n // 2] = np.nan


def _analyzer_inputs(n, B, rng, ascending):
    if ascending:
        alpha = np.linspace(1e-3, 20.0, n) if n > 1 else np.array([3.0])
    else:
        alpha = mo.log_alpha_mesh(1e-2, 1e3, n) * 50
    la = np.log(alpha)
    brk = np.median(la) + 0.5 * rng.rand(B, 1)
    chi2 = np.exp(np.where(la[None, :] > brk, 2.0 + 1.3 * (la[None, :] - brk), 2.0) + 0.05 * rng.rand(B, n))
    S = -np.exp(0.3 * (8 - la))[None, :] * (1 + 0.1 * rng.rand(B, n))
    logp = -0.5 * (la[None, :] - np.median(la) - rng.rand(B, 1)) ** 2 * 3 + rng.rand(B, n) * 0.1
    A = rng.rand(B, n, 7)
    if B >= 10:
        _nan_patterns(n, chi2, S, logp)
    return alpha, chi2, S, logp, A


def _oracle_or_none(fn):
    try:
        with np.errstate(all="ignore"):
            return fn()
    except ValueError:                   # an all-NaN argmin / argmax: the analyzer reports no result
        return None


def _close_with_nans(got, ref, rtol, cond=0.0):
    """got == ref where ref is NaN, elsewhere within (rtol + 32 eps cond) |ref| + rtol max |ref|: ``cond`` is the
    condition number of the reference's formula in its inputs, so a few ulp of log() on either side stay covered."""
    assert np.array_equal(np.isnan(got), np.isnan(ref)), (got, ref)
    ok = ~np.isnan(ref)
    if ok.any():
        cond = (np.zeros(len(ref)) + cond)[ok]
        tol = (rtol + 32 * EPS * cond) * np.abs(ref[ok]) + rtol * np.max(np.abs(ref[ok]))
        assert np.all(np.abs(got[ok] - ref[ok]) <= tol), np.max(np.abs(got[ok] - ref[ok]) / tol)


def _difference_cond(a, b):
    """|a| + |b| over |a - b|: how much a difference amplifies relative errors of its terms."""
    with np.errstate(all="ignore"):
        return (np.abs(a) + np.abs(b)) / np.abs(a - b)


def _curvature_cond(x, y):
    """Condition number of the three-point curvature d2 / (1 + d1^2)^1.5 at every interior point (NaN elsewhere): the
    mesh steps enter d2 twice, the second difference of y once, the first differences of y through d1^2 (power 3)."""
    c = np.full(len(x), np.nan)
    if len(x) >= 3:
        cx = _difference_cond(x[2:], x[1:-1]) + _difference_cond(x[1:-1], x[:-2])
        with np.errstate(all="ignore"):
            cy2 = (np.abs(y[2:]) + 2 * np.abs(y[1:-1]) + np.abs(y[:-2])) / np.abs(y[2:] - 2 * y[1:-1] + y[:-2])
        cy1 = _difference_cond(y[2:], y[1:-1]) + _difference_cond(y[1:-1], y[:-2])
        c[1:-1] = 2 * cx + cy2 + 3 * cy1
    return c


# four launches cover every (linefit_deg, bryan_by_integration) pair and both gammas
_AN_OPTIONS = [(0, False, 0.2), (1, True, 1.0), (0, True, 1.0), (1, False, 0.2)]


@pytest.mark.parametrize("n_alpha", [1, 2, 3, 4, 5, 6, 60, 129, 257, 1024])
def test_analyzers_vs_oracle_at_edge_meshes(torch_cuda, n_alpha):
    """mx_analyze against the oracle's restatement of python/analyzers/*.py: n_alpha below the five points LineFit needs,
    at and above the 128 threads of the CTA, at the maximum of 1024; descending log and ascending linear meshes; gamma
    0.2 and 1; all four LineFit degree / Bryan integration pairs; NaN patterns in chi2, S and logp.  Every pick identical
    (-1 where the reference raises on an all-NaN slice), A_out slots 0-3 bit for bit A[pick], Bryan to 1e-12; the aux row
    -- curvature and dS/dlog alpha with identical NaN positions to 1e-12, line-fit parameters at the chosen break to
    1e-10.  A spectrum analysed alone gives the bits it gets in a batch of 300.  n_alpha = 1025 is refused."""
    torch = torch_cuda
    from maxent_b200 import engine, _lib
    rng = np.random.RandomState(n_alpha)
    B = 300 if n_alpha <= 60 else 10
    for ascending in (False, True):
        alpha, chi2, S, logp, A = _analyzer_inputs(n_alpha, B, rng, ascending)
        checked = list(range(min(B, 10))) + ([int(b) for b in rng.choice(np.arange(10, B), 6, replace=False)]
                                             if B > 10 else [])
        if n_alpha <= 6:
            checked = list(range(B))
        for deg, integ, gamma in _AN_OPTIONS:
            idx, Aout, aux = engine.analyze(alpha, chi2, S, logp, A, gamma=gamma, linefit_deg=deg,
                                            bryan_by_integration=integ, want_aux=True)
            idx, Aout, aux = idx.cpu().numpy(), Aout.cpu().numpy(), aux.cpu().numpy()
            i1, A1, x1 = engine.analyze(alpha, chi2[:1], S[:1], logp[:1], A[:1], gamma=gamma, linefit_deg=deg,
                                        bryan_by_integration=integ, want_aux=True)
            assert np.array_equal(i1.cpu().numpy()[0], idx[0])
            assert np.array_equal(A1.cpu().numpy()[0], Aout[0], equal_nan=True)
            assert np.array_equal(x1.cpu().numpy()[0], aux[0], equal_nan=True)
            for b in checked:
                where = (n_alpha, ascending, deg, integ, gamma, b)
                lf = _oracle_or_none(lambda: mo.fit_piecewise(np.log(alpha), np.log(chi2[b]), deg))
                want = [-1 if lf is None else lf[0]]
                cv = _oracle_or_none(lambda: mo.curvature(gamma * np.log10(alpha), np.log10(chi2[b]))[0])
                want.append(_oracle_or_none(lambda: int(np.nanargmax(cv))))
                en = _oracle_or_none(lambda: mo.analyze_entropy(alpha, S[b], A[b]))
                want.append(None if en is None else en["alpha_index"])
                want.append(mo.analyze_classic(alpha, logp[b], A[b])["alpha_index"])
                want = [-1 if w is None else int(w) for w in want]
                assert list(idx[b, :4]) == want, (where, idx[b], want)
                for slot in range(4):
                    if want[slot] >= 0:
                        assert np.array_equal(Aout[b, slot], A[b, want[slot]]), (where, slot)
                    else:
                        assert np.all(np.isnan(Aout[b, slot])), (where, slot)
                _close_with_nans(aux[b, 4:4 + n_alpha], cv, 1e-12,
                                 _curvature_cond(gamma * np.log10(alpha), np.log10(chi2[b])))
                # python/analyzers/entropy_analyzer.py:92-95.  The difference of two logarithms of a fine linear mesh
                # cancels (|log alpha| / |d log alpha| ~ 1500 at 1024 points), and so does the curvature's
                dS = np.full(n_alpha, np.nan)
                dS[1:-1] = (S[b, 2:] - S[b, :-2]) / (np.log(alpha[2:]) - np.log(alpha[:-2]))
                cond = np.zeros(n_alpha)
                cond[1:-1] = _difference_cond(np.log(alpha[2:]), np.log(alpha[:-2]))
                _close_with_nans(aux[b, 4 + n_alpha:], dS, 1e-12, cond)
                if lf is not None and idx[b, 0] >= 0:
                    p1, p2 = lf[1]
                    ref = np.array([p1[0], p1[1], p2[0] if deg == 1 else 0.0, p2[-1]])
                    assert np.all(np.abs(aux[b, :4] - ref) <= 1e-10 * np.maximum(1.0, np.abs(ref))), (where, aux[b, :4], ref)
                n_p = int(np.sum(~np.isnan(logp[b])))
                if integ and n_p == 1:
                    # one probability: its trapezoid integral is zero and python/analyzers/bryan_analyzer.py raises
                    # (get_delta of a one-point mesh); there is no reference value to compare with
                    continue
                br = mo.analyze_bryan(alpha, logp[b], A[b], integ)
                if br["A_out"] is None:
                    assert idx[b, 4] == -1 and np.all(np.isnan(Aout[b, 4])), where
                else:
                    assert idx[b, 4] == 0, where
                    np.testing.assert_allclose(Aout[b, 4], br["A_out"], rtol=1e-12, atol=1e-14 * np.max(A[b]))
    with pytest.raises(_lib.MaxEntLibraryError):
        engine.analyze(np.ones(1025), np.ones((1, 1025)), np.ones((1, 1025)), None, None)


def test_linefit_one_point_piece_matches_polyfit(torch_cuda):
    """A degree-1 piece with one point: np.polyfit returns the minimum-norm line of its scaled least-squares problem,
    slope y / (2 x) and intercept y / 2, with a zero residual.  That break point wins when it ties with a later one
    with the exactly determined pieces of a later one (both residuals are exactly zero: np.polyfit returns none), and
    the crossing X -- hence the pick -- depends on that line.  Here the one-point line crosses the second piece near the
    smallest alpha; a flat line at y would cross it beyond the largest."""
    torch = torch_cuda
    from maxent_b200 import engine
    alpha = mo.log_alpha_mesh(1e-2, 1e3, 6) * 50
    chi2 = np.array([[np.nan, 40.0, 7.0, np.nan, np.nan, 3.0]])
    with np.errstate(all="ignore"):
        k, (p1, p2), cost = mo.fit_piecewise(np.log(alpha), np.log(chi2[0]), 1)
    assert cost[2] == cost[3] == 0.0 and k == 5
    idx, _, aux = engine.analyze(alpha, chi2, -np.ones((1, 6)), None, np.zeros((1, 6, 3)), linefit_deg=1, want_aux=True)
    assert int(idx[0, 0]) == k, (int(idx[0, 0]), k)
    np.testing.assert_allclose(aux[0, :4].cpu().numpy(), [p1[0], p1[1], p2[0], p2[1]], rtol=1e-12, atol=1e-14)


# ----------------------------------------------------------------------------------------------
# mx_poorman_models
# ----------------------------------------------------------------------------------------------
def _poorman_call(torch, A_out, slot, rows, delta, d_add, A_init, Vp, group):
    from maxent_b200 import ops
    P, n_omega, n_sv = rows.shape[0], delta.numel(), int(Vp.shape[-1])
    D = torch.full((P, (n_omega + 1) & ~1), float("nan"), dtype=torch.float64, device="cuda")
    v0 = torch.full((P, n_sv), float("nan"), dtype=torch.float64, device="cuda")
    ok = torch.full((P,), -7, dtype=torch.int32, device="cuda")
    ops.poorman_models(A_out, slot, torch.from_numpy(rows.astype(np.int32)), delta, d_add, A_init, Vp,
                       None if group is None else torch.from_numpy(group.astype(np.int32)), D, v0, ok)
    return D.cpu().numpy(), v0.cpu().numpy(), ok.cpu().numpy()


@pytest.mark.parametrize("n_omega", [7, 80, 7000])
@pytest.mark.parametrize("n_sv", [1, 52, 256])
def test_poorman_models_vs_numpy(torch_cuda, n_omega, n_sv):
    """D[p] = (sqrt(A_i A_j) + c) delta bit for bit as numpy forms it (exact zeros behind an odd n_omega), for every
    analyzer slot (slot 4 holds NaN rows where Bryan had no probability), through three whitening groups and with A_init;
    v0[p] = V'_g^T log(arg) against a long-double dot within 1e-15 sum_w |V_wk| (|log arg_w| + 1) (the + 1: log(arg) near
    arg = 1 carries the absolute rounding of arg); ok = 0 exactly where a partner holds NaN.  n_omega = 7000 needs more
    than 48 KB of dynamic shared memory."""
    torch = torch_cuda
    rng = np.random.RandomState(n_omega + n_sv)
    R, P = 14, 12
    delta = mo.omega_delta(mo.hyperbolic_omega_mesh(-8, 8, n_omega))
    A_out = rng.rand(R, 5, n_omega) * 0.4 + 1e-3
    A_out[[2, 9], 4] = np.nan                          # Bryan unavailable for these diagonal spectra
    A_out[5, :, n_omega // 2] = np.nan                 # one NaN point in every slot
    rows = rng.randint(0, R, size=(P, 2))
    rows[0] = (2, 3)
    rows[1] = (4, 5)
    Vp = rng.randn(3, n_omega, n_sv)
    group = rng.randint(0, 3, size=P)
    d_add = 1e-6
    Ad, dd, Vd = _dev(torch, A_out), _dev(torch, delta), _dev(torch, Vp)
    L = np.longdouble
    for slot in range(5):
        for use_init in (False, True):
            A_init = (rng.rand(n_omega) * 0.5) if use_init else None
            D, v0, ok = _poorman_call(torch, Ad, slot, rows, dd, d_add, None if A_init is None else _dev(torch, A_init),
                                      Vd, group)
            Ai, Aj = A_out[rows[:, 0], slot], A_out[rows[:, 1], slot]
            D_np = (np.sqrt(Ai * Aj) + d_add) * delta
            np.testing.assert_array_equal(D[:, :n_omega], D_np)
            assert np.all(D[:, n_omega:] == 0.0)
            bad = np.any(np.isnan(Ai) | np.isnan(Aj), axis=1)
            np.testing.assert_array_equal(ok, (~bad).astype(np.int32))
            H0 = (D_np if A_init is None else A_init[None, :]) * delta
            with np.errstate(invalid="ignore"):
                arg = (H0 + np.sqrt(H0 * H0 + 4 * D_np * D_np)) / (2 * D_np)
            arg = np.where(np.abs(arg) <= 1e-100, 1e-100, arg)
            larg = np.log(arg)
            for p in np.nonzero(~bad)[0]:
                V = Vp[group[p]]
                ref = (larg[p].astype(L) @ V.astype(L)).astype(np.float64)
                tol = 1e-15 * (np.abs(V).T @ (np.abs(larg[p]) + 1.0))
                assert np.all(np.abs(v0[p] - ref) <= tol), (slot, p, np.max(np.abs(v0[p] - ref) / tol))


def test_poorman_models_position_independence(torch_cuda):
    """One spectrum's D, v0 and ok do not depend on P or on its position: the same row alone (P = 1, no group) and in
    the middle of P = 1000 (n_omega = 7000, n_sv = 256), bit for bit."""
    torch = torch_cuda
    rng = np.random.RandomState(3)
    n_omega, n_sv, R, P = 7000, 256, 40, 1000
    om = mo.hyperbolic_omega_mesh(-8, 8, n_omega)
    delta = _dev(torch, mo.omega_delta(om))
    A_out = _dev(torch, rng.rand(R, 5, n_omega) + 1e-3)
    Vp = _dev(torch, rng.randn(n_omega, n_sv))
    rows = rng.randint(0, R, size=(P, 2))
    D1, v1, ok1 = _poorman_call(torch, A_out, 1, rows[517:518], delta, 1e-6, None, Vp, None)
    D, v, ok = _poorman_call(torch, A_out, 1, rows, delta, 1e-6, None, Vp, None)
    assert np.array_equal(D1[0], D[517]) and np.array_equal(v1[0], v[517]) and ok1[0] == ok[517] == 1


# ----------------------------------------------------------------------------------------------
# one sweep over whitening groups of different n_sv
# ----------------------------------------------------------------------------------------------
def _groups_run(variant, marquardt, n_svs, n_tau, n_om, n_alpha):
    from maxent_b200 import engine
    mesh = mo.log_alpha_mesh(0.5, 500, n_alpha)
    probs, Gs, Ks = [], [], []
    for g, s in enumerate(n_svs):
        K, G, om, delta = gc.kernel_problem(s, n_tau, n_om, variant, 40 + g, 2)
        q = engine.SharedProblem(K, 1e-4, mo.flat_default_model(om), delta, variant=variant, reduce_singular_space=1e-9)
        assert q.n_sv == s
        probs.append(q)
        Gs.append(G)
        Ks.append(K)
    index = np.array([0, 1, 1, 0])
    G = np.stack([Gs[0][0], Gs[1][0], Gs[1][1], Gs[0][1]])
    lm = engine.LMParams(marquardt=marquardt)
    return engine, probs, index, G, Ks, om, mesh, lm


@pytest.mark.parametrize("variant", ["normal", "plusminus", "bryan"])
@pytest.mark.parametrize("marquardt", [False, True])
def test_sweep_over_groups_of_different_n_sv(torch_cuda, variant, marquardt):
    """engine.run_sweep(groups=...) over groups of n_sv 26 and 31 (the same four-tile instantiation): the smaller group is
    padded with zero columns of V' and zero xi.  For the plain Levenberg damping of the normal and plus-minus cost
    functions the padded components never move and every spectrum is bitwise the run of its group alone.  Bryan's
    gradient divides by xi (0 / 0 in a padded component) and Marquardt's damping mu diag(J) has exact zero pivots there,
    so a padded launch of either is refused."""
    torch = torch_cuda
    engine, probs, index, G, _, _, mesh, lm = _groups_run(variant, marquardt, (26, 31), 100, 64, 6)
    alpha = mesh * 100
    if variant == "bryan" or marquardt:
        with pytest.raises(ValueError):
            engine.run_sweep(probs[0], G, alpha, lm=lm, groups=(probs, index))
        return
    res = engine.run_sweep(probs[0], G, alpha, lm=lm, groups=(probs, index))
    assert res.n_sv == 31
    for g in range(2):
        sel = np.nonzero(index == g)[0]
        one = engine.run_sweep(probs[g], G[sel], alpha, lm=lm)
        for k, b in enumerate(sel):
            for name in ("A", "chi2", "S", "Q", "n_iter", "alpha_index"):
                assert torch.equal(getattr(res, name)[b], getattr(one, name)[k]), (variant, g, name)
            assert torch.equal(res.v[b, :, :probs[g].n_sv], one.v[k])
            assert not bool(res.v[b, :, probs[g].n_sv:].any())
    assert bool((res.status & 1).all())


@pytest.mark.parametrize("variant", ["normal", "plusminus"])
def test_groups_crossing_the_wide_instantiation(torch_cuda, variant):
    """Groups of n_sv 60 and 90: padded to 90, the smaller group runs on the wide instantiation (12 tiles, Z and J in the
    workspace) instead of its own 8-tile one, so its spectra are held to the tiered oracle contract (1e-8 where the
    oracle reproduces itself, 10x its noise floor elsewhere); the 90 group is bitwise its run alone."""
    torch = torch_cuda
    engine, probs, index, G, Ks, om, mesh, lm = _groups_run(variant, False, (60, 90), 174, 130, 6)
    alpha = mesh * 174
    res = engine.run_sweep(probs[0], G, alpha, lm=lm, groups=(probs, index))
    sel = np.nonzero(index == 1)[0]
    one = engine.run_sweep(probs[1], G[sel], alpha, lm=lm)
    for k, b in enumerate(sel):
        assert torch.equal(res.A[b], one.A[k]) and torch.equal(res.chi2[b], one.chi2[k])
    for b in np.nonzero(index == 0)[0]:
        kw = dict(variant=variant, reduce_singular_space=1e-9, analyzers=False)
        o = mo.maxent_loop(Ks[0], G[b], 1e-4, om, mesh, **kw)
        assert o["n_sv"] == 60
        noise, nchi = gc.oracle_floor(o, lambda f: mo.maxent_loop(Ks[0], G[b] * f, 1e-4, om, mesh, **kw))
        tol = np.maximum(1e-8, 10 * noise)
        dA = gc.rel_A(res.A[b].cpu().numpy(), o["A"])
        assert np.all(dA <= tol), (variant, b, dA / tol)
        assert np.all(np.abs(res.chi2[b].cpu().numpy() / o["chi2"] - 1) <= np.maximum(1e-8, 10 * nchi))
    assert bool((res.status & 1).all())


@pytest.mark.parametrize("cost,marquardt", [("bryan", False), ("normal", True), ("bryan", True)])
def test_preblur_scan_with_bryan_or_marquardt(torch_cuda, cost, marquardt):
    """The preblur b scan with TauMaxEnt(cost_function='bryan') or LevenbergMinimizer(marquardt=True): the b values have
    different n_sv, which one launch cannot pad exactly for these, so they run one launch per b -- and every b gives the
    bits of its run alone."""
    import maxent_b200 as mb
    g = gc.load_golden("g7_preblur_200x100.npz")

    def tau_maxent():
        tm = mb.TauMaxEnt(cost_function=cost, reduce_singular_space=float(g["reduce_singular_space"]))
        tm.set_verbosity(mb.VerbosityFlags.Quiet)
        tm.set_G_tau_data(g["tau"], g["G"])
        tm.omega = mb.DataOmegaMesh(g["omega"])
        tm.alpha_mesh = mb.DataAlphaMesh(g["alpha_mesh"][::3])
        tm.set_error(float(g["err"]) if np.ndim(g["err"]) == 0 else g["err"])
        if marquardt:
            tm.minimizer = mb.LevenbergMinimizer(marquardt=True)
        return tm

    bs = [0.1, 0.2, 0.4]
    scan = mb.preblur_scan(tau_maxent(), bs)
    n_svs = []
    for b in bs:
        t1 = tau_maxent()
        K1 = t1.K
        t1.A_of_H = mb.PreblurA_of_H(b=b, omega=t1.omega)
        t1.K = mb.PreblurKernel(K=K1, b=b)
        r1 = t1.run()
        n_svs.append(len(t1.K.S))
        assert np.all(np.isfinite(scan[b].A)), b
        np.testing.assert_array_equal(scan[b].chi2, r1.chi2)
        np.testing.assert_array_equal(scan[b].A, r1.A)
    assert len(set(n_svs)) > 1, n_svs
