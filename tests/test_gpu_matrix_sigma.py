"""GPU tests of matrix-valued self-energy continuation: mx_matrix_resolvent against the long-double Gauss-Jordan of
oracle/matrix_sigma.py, Matsubara matrices in the batched matrix classes against BatchedTauMaxEnt runs and the oracle
loop, the round trip of the matrix Bethe self-energy without MaxEnt, and BatchedSigmaContinuator with a matrix worker
end to end."""
import numpy as np
import pytest

import maxent_b200 as mb
from maxent_b200 import ops, real_frequency
from maxent_b200.batched_matrix import matsubara_rows
from oracle import matrix_sigma as ms
from oracle import maxent_oracle as mo
from oracle import real_frequency as rf
from tests import gpu_common as gc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _resolve(torch, X, z, C, mode, in_place=False):
    Xd = torch.as_tensor(np.ascontiguousarray(X), device="cuda")
    Y = Xd if in_place else torch.empty_like(Xd)
    Cd = None if C is None else torch.as_tensor(C, dtype=torch.float64, device="cuda")
    ops.matrix_resolvent(Xd, torch.as_tensor(np.asarray(z, dtype=np.complex128), device="cuda"), Cd, mode, Y)
    return Y.cpu().numpy()


def _conditioned(rng, B, M, n, max_cond):
    """B n complex M x M matrices with condition numbers log-uniform in [1, max_cond]: [B, M, M, n]."""
    U, V = ms.random_unitary(B * n, M, rng.integers(1 << 30)), ms.random_unitary(B * n, M, rng.integers(1 << 30))
    cond = 10 ** rng.uniform(0, np.log10(max_cond), B * n)
    sv = cond[:, None] ** -np.linspace(0, 1, M)[None, :] * rng.uniform(0.5, 2.0, (B * n, 1))
    A = np.einsum("pim,pm,pjm->pij", U, sv, np.conj(V))
    return np.moveaxis(A.reshape(B, n, M, M), 1, 3)


def _frob_err(got, ref):
    """Relative Frobenius error per matrix (b, k): [B, n_z]."""
    ref = ref.astype(np.complex128)
    return np.linalg.norm(got - ref, axis=(1, 2)) / np.linalg.norm(ref, axis=(1, 2))


# ---- mx_matrix_resolvent -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 3, 5, 8])
def test_resolvent_against_long_double(torch_cuda, M):
    """Both modes at B n_z = 7 x 37 = 259 (not a multiple of either block size), in place and out of place, against the
    long-double Gauss-Jordan: relative Frobenius error <= 1e-12 per matrix for condition numbers <= 1e3 of the matrix
    that is inverted."""
    torch = torch_cuda
    rng = np.random.default_rng(M)
    B, n = 7, 37
    # z + C exact in binary, so that the shift adds no rounding that the long-double reference does not see
    z = rng.integers(-32, 33, n) / 16 + 1j * rng.uniform(0.01, 1.0, n)
    C = rng.integers(-16, 17, B) / 16
    s = z[None, :] + C[:, None]
    worst = 0.0
    for mode in (0, 1):
        A = _conditioned(rng, B, M, n, 1e3)                         # the matrix the kernel inverts
        X = s[:, None, None, :] * np.eye(M)[None, :, :, None] - A if mode == 0 else A
        ref = ms.resolvent(X, z, C, mode)
        got = _resolve(torch, X, z, C, mode)
        got_in_place = _resolve(torch, X, z, C, mode, in_place=True)
        np.testing.assert_array_equal(got, got_in_place)
        err = _frob_err(got, ref)
        worst = max(worst, float(err.max()))
        assert np.all(err <= 1e-12), (mode, err.max())
    got = _resolve(torch, X, z, None, 1)                            # C = NULL
    assert np.all(_frob_err(got, ms.resolvent(X, z, None, 1)) <= 1e-12)
    print("M = %d: worst relative Frobenius error %.3g (limit 1e-12)" % (M, worst))


def test_resolvent_singular_and_nan(torch_cuda):
    """An exactly singular shifted matrix ([[1, 1], [1, 1]] after the shift) and a NaN entry give all-NaN Y(b,k); every
    other (b, k) is bit for bit the result without them."""
    torch = torch_cuda
    rng = np.random.default_rng(5)
    B, M, n = 3, 2, 6
    z = np.full(n, 0.5 + 0.25j)
    C = np.full(B, 0.25)                                           # z + C = 0.75 + 0.25i, exact in binary
    X = rng.standard_normal((B, M, M, n)) + 1j * rng.standard_normal((B, M, M, n))
    bad = X.copy()
    bad[1, :, :, 2] = (0.75 + 0.25j) * np.eye(M) - np.ones((M, M))   # (z + C) 1 - X = [[1, 1], [1, 1]]
    bad[2, 0, 1, 3] = np.nan
    for mode in (0, 1):
        got = _resolve(torch, bad, z, C, mode)
        clean = _resolve(torch, X, z, C, mode)
        if mode == 0:
            assert np.all(np.isnan(got[1, :, :, 2].real)) and np.all(np.isnan(got[1, :, :, 2].imag))
        assert np.all(np.isnan(got[2, :, :, 3].real)) and np.all(np.isnan(got[2, :, :, 3].imag))
        keep = np.ones((B, n), dtype=bool)
        keep[1, 2] = keep[2, 3] = False
        np.testing.assert_array_equal(np.moveaxis(got, 3, 1)[keep], np.moveaxis(clean, 3, 1)[keep])
    sing = np.ones((1, M, M, 1), dtype=complex)                     # mode 1 inverts X itself
    assert np.all(np.isnan(_resolve(torch, sing, [0.1j], None, 1)))


def test_resolvent_is_independent_of_the_batch(torch_cuda):
    """Permuting the batch, cutting it, or cutting the frequencies changes no bit of any Y(b,k)."""
    torch = torch_cuda
    rng = np.random.default_rng(9)
    B, n = 9, 50
    for M in (3, 6):
        X = rng.standard_normal((B, M, M, n)) + 1j * rng.standard_normal((B, M, M, n))
        z = rng.standard_normal(n) + 1j * rng.uniform(0.1, 1, n)
        C = rng.standard_normal(B)
        for mode in (0, 1):
            full = _resolve(torch, X, z, C, mode)
            perm = rng.permutation(B)
            np.testing.assert_array_equal(_resolve(torch, X[perm], z, C[perm], mode), full[perm])
            np.testing.assert_array_equal(_resolve(torch, X[2:5], z, C[2:5], mode), full[2:5])
            np.testing.assert_array_equal(_resolve(torch, X[..., 10:31], z[10:31], C, mode), full[..., 10:31])


# ---- Matsubara matrices in the batched matrix classes ------------------------------------------------------------------
def _bethe_G_iw(B, M, nu, seed, sigma=1e-5):
    rng = np.random.default_rng(seed)
    t = rng.uniform(0.6, 1.2, (B, M))
    U = ms.random_unitary(B, M, seed + 1)
    G = ms.bethe_matrix_G_aux(1j * nu, t, U)
    return G + sigma * (rng.standard_normal(G.shape) + 1j * rng.standard_normal(G.shape))


def _setup(job, om, n_alpha=24, err=1e-5):
    job.omega = om
    job.alpha_mesh = mb.LogAlphaMesh(0.01, 500, n_alpha)
    job.reduce_singular_space = 1e-11
    if isinstance(job, mb.BatchedElementwiseMaxEnt):
        for w in job._workers():
            w.reduce_singular_space = 1e-11
    job.set_error(err)
    return job


def test_matsubara_matrix_continuation(torch_cuda):
    """BatchedElementwiseMaxEnt on G(i omega_n)[6, 3, 3, n_iw] (complex elements, every element continued): pass 1 is bit
    for bit BatchedTauMaxEnt.set_G_iw_data on the G_ii rows, pass 2 bit for bit BatchedTauMaxEnt('plusminus') on the
    mapped rows, one off-diagonal element agrees with the oracle loop under the contract of gpu_common, and the device
    assembly of A_out equals the host result bit for bit."""
    torch = torch_cuda
    B, M, n_iw, beta = 6, 3, 60, 20.0
    nu = np.pi / beta * (2 * np.arange(n_iw) + 1)
    G = _bethe_G_iw(B, M, nu, seed=3)
    om = mb.HyperbolicOmegaMesh(-4, 4, 120)
    job = _setup(mb.BatchedElementwiseMaxEnt(use_hermiticity=False, use_complex=True), om)
    job.set_G_iw_data(nu, G)
    plans, (r1, r2), (G1, G2), _ = job.run_device()
    diag, off = plans
    ref = _setup(mb.BatchedTauMaxEnt(), om)
    ref.set_G_iw_data(nu, G[diag[:, 0], diag[:, 1], diag[:, 2]])
    out1 = ref.run()
    np.testing.assert_array_equal(r1.A_out.cpu().numpy(), out1.A_out)
    np.testing.assert_array_equal(r1.chi2.cpu().numpy(), out1.chi2)
    np.testing.assert_array_equal(r1.A.cpu().numpy(), out1.device.A.cpu().numpy())
    rows = matsubara_rows(torch.as_tensor(G, device="cuda"), off)
    np.testing.assert_array_equal(G2.cpu().numpy(), rows.cpu().numpy())
    pm = _setup(mb.BatchedTauMaxEnt(cost_function="plusminus"), om)
    pm.set_kernel_iw(nu)
    out2 = pm.run_device(rows, want_A=True, want_v=True, skip_small=True)
    for name in ("A_out", "chi2", "S", "A", "alpha_index"):
        np.testing.assert_array_equal(getattr(r2, name).cpu().numpy(), getattr(out2, name).cpu().numpy(), err_msg=name)

    # one off-diagonal element (b = 0, (0, 1), imaginary part) against the oracle loop on the same stacked rows
    r = int(np.nonzero((off[:, 0] == 0) & (off[:, 1] == 0) & (off[:, 2] == 1) & (off[:, 3] == 1))[0][0])
    K = mb.IOmegaKernel(nu, om).fused_matrix()
    g = rows[r].cpu().numpy()
    mesh, cut = np.asarray(job.alpha_mesh, dtype=np.float64), 1e-11
    svd = mo.kernel_svd(K, cut)
    kw = dict(variant="plusminus", reduce_singular_space=cut, analyzers=False, svd=svd, scale_alpha=n_iw)
    o = mo.maxent_loop(K, g, 1e-5, np.asarray(om), mesh, **kw)
    nA, nc = gc.oracle_floor(o, lambda f: mo.maxent_loop(K, g * f, 1e-5, np.asarray(om), mesh, **kw))
    assert o["n_sv"] == r2.n_sv
    tolA, tolc = np.maximum(gc.RTOL_WELL_DETERMINED, gc.NOISE_FACTOR * nA), np.maximum(gc.RTOL_WELL_DETERMINED,
                                                                                       gc.NOISE_FACTOR * nc)
    rA = gc.rel_A(r2.A[r].cpu().numpy(), o["A"]) / tolA
    rc = np.abs(r2.chi2[r].cpu().numpy() / o["chi2"] - 1) / tolc
    print("oracle element: worst A ratio %.3g, chi2 ratio %.3g" % (rA.max(), rc.max()))
    assert np.all(rA <= 1) and np.all(rc <= 1), (rA.max(), rc.max())

    res = job.run()
    r0 = res.result(0)
    assert r0.matrix_structure == (M, M)
    np.testing.assert_array_equal(r0.data_variable[0, 1, 1], nu)
    for slot in (0, 4):                                             # LineFit, Bryan (unavailable: NaN)
        A = res.A_out_device(slot).cpu().numpy()
        np.testing.assert_array_equal(A[..., 0, :] + 1j * A[..., 1, :], res.A_out[..., slot, :])
    assert np.all(np.isnan(res.A_out[..., 4, :].real))


def _host_sigma(A_out, omega, w, eta, C):
    """The host composition of sigma_w: long-double table, X = T(A') + i T(A''), long-double resolvent mode 1."""
    M_ld = rf.hilbert_table(omega, w, eta)
    LD = np.longdouble
    Tp = A_out.real.astype(np.float64).astype(LD) @ M_ld.T
    Tpp = A_out.imag.astype(np.float64).astype(LD) @ M_ld.T
    X = Tp + 1j * Tpp
    return ms.resolvent(X, np.asarray(w) + 1j * eta, C, 1)


def _per_matrix_err(got, ref):
    ref = ref.astype(np.complex128)
    return np.array([np.max(np.abs(got[b] - ref[b])) / np.max(np.abs(ref[b])) for b in range(len(ref))])


@pytest.mark.parametrize("M", [2, 3])
def test_round_trip_without_maxent(torch_cuda, M):
    """The matrix Bethe self-energy Sigma = U diag(t_m^2 g_sc) U^dagger has G_aux = U diag(g_sc) U^dagger exactly at
    C = 0: its exact A_aux on a 4001-point mesh, through the Hilbert apply and the resolvent (matrix_sigma_w), equals the
    long-double host composition to 1e-11 and Sigma within the discretisation error of that host reference."""
    torch = torch_cuda
    B = 4
    rng = np.random.default_rng(M)
    t = rng.uniform(0.6, 1.2, (B, M))
    U = ms.random_unitary(B, M, 10 + M)
    om = np.linspace(-2.5, 2.5, 4001)
    w = np.linspace(-3, 3, 241)
    eta = 0.05
    A = ms.bethe_matrix_A(om, t, U)
    parts = np.stack([A.real, A.imag], axis=3)                     # [B, M, M, 2, n_omega]
    got = mb.matrix_sigma_w(torch.as_tensor(np.ascontiguousarray(parts), device="cuda"), om, w, eta).cpu().numpy()
    host = _host_sigma(A, om, w, eta, None)
    err = _per_matrix_err(got, host)
    exact = ms.bethe_matrix_sigma(w + 1j * eta, t, U)
    host_err = np.max(np.abs(host.astype(np.complex128) - exact))
    print("M = %d: device vs host %.3g, discretisation error %.3g of max|Sigma| %.3g"
          % (M, err.max(), host_err, np.max(np.abs(exact))))
    assert np.all(err <= 1e-11), err.max()
    assert np.max(np.abs(got - exact)) <= host_err + 1e-11 * np.max(np.abs(exact))
    assert host_err <= 2e-3 * np.max(np.abs(exact))


def _bethe_sigma_iw(B, M, nu, seed, sigma=1e-5, diagonal=False):
    rng = np.random.default_rng(seed)
    t = rng.uniform(0.7, 1.2, (B, M))
    U = np.broadcast_to(np.eye(M), (B, M, M)) if diagonal else ms.random_unitary(B, M, seed + 1)
    S = ms.bethe_matrix_sigma(1j * nu, t, U)
    noise = sigma * (rng.standard_normal(S.shape) + 1j * rng.standard_normal(S.shape))
    if diagonal:
        noise = noise * np.eye(M)[None, :, :, None]
    return S + noise, 0.1 * rng.standard_normal(B)


@pytest.mark.parametrize("M", [2, 3])
def test_sigma_continuator_matrix_end_to_end(torch_cuda, M):
    """BatchedSigmaContinuator(maxent=BatchedPoormanMaxEnt(use_complex=True)) on 16 noisy Bethe self-energies: G_aux_iw
    equals np.linalg.inv to 1e-13, the result is bit for bit a BatchedPoormanMaxEnt run on G_aux_iw, sigma_w equals the
    host composition (result A_out, long-double table and resolvent) to 1e-11, and an unavailable analyzer gives NaN."""
    torch = torch_cuda
    B, n_iw, beta = 16, 100, 40.0
    nu = np.pi / beta * (2 * np.arange(n_iw) + 1)
    S, C = _bethe_sigma_iw(B, M, nu, seed=20 + M)
    om = mb.HyperbolicOmegaMesh(-4, 4, 200)
    sc = mb.BatchedSigmaContinuator(constant_shift=C, maxent=mb.BatchedPoormanMaxEnt(use_complex=True))
    sc.set_S_iw_data(nu, S)
    _setup(sc.maxent, om)
    Gx = sc.G_aux_iw.cpu().numpy()
    s = 1j * nu[None, :] + C[:, None]
    ref = np.moveaxis(np.linalg.inv(s[:, :, None, None] * np.eye(M) - np.moveaxis(S, 3, 1)), 1, 3)
    assert np.max(np.abs(Gx - ref)) <= 1e-13 * np.max(np.abs(ref))
    res = sc.run()
    job = _setup(mb.BatchedPoormanMaxEnt(use_complex=True), om)
    job.set_G_iw_data(nu, Gx)
    r2 = job.run()
    for name in ("A_out", "chi2", "alpha_index"):
        np.testing.assert_array_equal(getattr(res, name), getattr(r2, name), err_msg=name)
    w = np.linspace(-3, 3, 157)
    eta = 0.02
    got = sc.sigma_w(w, eta).cpu().numpy()
    assert got.shape == (B, M, M, len(w))
    host = _host_sigma(res.A_out[..., 0, :], np.asarray(om), w, eta, C)
    nan = np.isnan(res.A_out[..., 0, :]).any(axis=(1, 2, 3))
    assert np.all(np.isnan(got[nan])) and np.all(np.isfinite(got[~nan])), nan
    err = _per_matrix_err(got[~nan], host[~nan])
    print("M = %d: sigma_w vs host composition, worst %.3g over %d matrices" % (M, err.max(), int((~nan).sum())))
    assert np.all(err <= 1e-11), err.max()
    A = res.A_out_device(0).cpu().numpy()
    np.testing.assert_array_equal(A[..., 0, :] + 1j * A[..., 1, :], res.A_out[..., 0, :])
    bryan = sc.sigma_w(w, eta, analyzer="BryanAnalyzer").cpu().numpy()        # no probability: Bryan unavailable
    assert np.all(np.isnan(bryan.real)) and np.all(np.isnan(bryan.imag))


def _scalar_sigma_w(nu, S, C, om, w, eta):
    sc = mb.BatchedSigmaContinuator(constant_shift=C)
    sc.set_S_iw_data(nu, S)
    _setup(sc.maxent, om)
    res = sc.run()
    return sc, res, sc.sigma_w(w, eta).cpu().numpy()


def test_diagonal_sigma_and_M1_match_the_scalar_path(torch_cuda):
    """A diagonal Sigma: the off-diagonal G_aux are exact zeros, continued as zeros (not NaN; with use_hermiticity their
    transposed elements too), so sigma_w is finite, its off-diagonal is zero and its diagonal matches the scalar
    continuator on each element to 1e-12.  M = 1 gives the
    scalar path's G_aux_iw and A_aux bit for bit and its sigma_w to 1e-12."""
    torch = torch_cuda
    B, M, n_iw, beta = 8, 2, 100, 40.0
    nu = np.pi / beta * (2 * np.arange(n_iw) + 1)
    S, C = _bethe_sigma_iw(B, M, nu, seed=31, diagonal=True)
    om = mb.HyperbolicOmegaMesh(-4, 4, 200)
    w = np.linspace(-3, 3, 101)
    eta = 0.02
    sc = mb.BatchedSigmaContinuator(constant_shift=C, maxent=mb.BatchedPoormanMaxEnt(use_complex=True))
    sc.set_S_iw_data(nu, S)
    _setup(sc.maxent, om)
    res = sc.run()
    got = sc.sigma_w(w, eta).cpu().numpy()
    assert np.all(np.isfinite(got))
    assert all(res.zero_elements[b] == [(0, 0, 1), (1, 1, 1), (0, 1)] for b in range(B)), res.zero_elements
    assert np.all(got[:, 0, 1] == 0) and np.all(got[:, 1, 0] == 0)
    # the device assembly is A_out, except that the hermiticity image (1, 0) of the zero element (0, 1) is zero, not NaN
    A = res.A_out_device(0).cpu().numpy()
    want = res.A_out[..., 0, :].copy()
    assert np.all(np.isnan(want[:, 1, 0]))
    want[:, 1, 0] = 0.0
    np.testing.assert_array_equal(A[..., 0, :] + 1j * A[..., 1, :], want)
    for i in range(M):
        ssc, sres, ref = _scalar_sigma_w(nu, S[:, i, i], C, om, w, eta)
        np.testing.assert_array_equal(sc.G_aux_iw.cpu().numpy()[:, i, i], ssc.G_aux_iw)
        np.testing.assert_array_equal(res.A_out[:, i, i, :, :].real, sres.A_out)
        err = np.max(np.abs(got[:, i, i] - ref), axis=1) / np.max(np.abs(ref), axis=1)
        assert np.all(err <= 1e-12), (i, err.max())

    S1 = np.ascontiguousarray(S[:, :1, :1])
    s1 = mb.BatchedSigmaContinuator(constant_shift=C, maxent=mb.BatchedPoormanMaxEnt(use_complex=True))
    s1.set_S_iw_data(nu, S1)
    _setup(s1.maxent, om)
    r1 = s1.run()
    g1 = s1.sigma_w(w, eta).cpu().numpy()
    ssc, sres, ref = _scalar_sigma_w(nu, S[:, 0, 0], C, om, w, eta)
    np.testing.assert_array_equal(s1.G_aux_iw.cpu().numpy()[:, 0, 0], ssc.G_aux_iw)
    np.testing.assert_array_equal(r1.A_out[:, 0, 0].real, sres.A_out)
    err = np.max(np.abs(g1[:, 0, 0] - ref), axis=1) / np.max(np.abs(ref), axis=1)
    assert np.all(err <= 1e-12), err.max()
