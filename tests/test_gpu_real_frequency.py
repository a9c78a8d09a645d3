"""GPU tests of the retarded transform (mx_hilbert_table, mx_hilbert_apply) and BatchedSigmaContinuator, against the
long-double host reference of oracle/real_frequency.py and closed forms of the Bethe lattice."""
import numpy as np
import pytest

import maxent_b200 as mb
from maxent_b200 import ops, real_frequency
from oracle import real_frequency as rf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _table(om, w, eta):
    M, w_d = real_frequency.hilbert_table(om, w, eta)
    return M.cpu().numpy(), w_d


def _row_err(got, ref):
    """max |got - ref| / max |ref| per row (NaN rows compare as 0 when both are NaN)."""
    got, ref = np.asarray(got, dtype=np.complex128), np.asarray(ref).astype(np.complex128)
    return np.max(np.abs(got - ref), axis=1) / np.max(np.abs(ref), axis=1)


@pytest.mark.parametrize("eta", [1e-9, 1e-2, 1.0])
@pytest.mark.parametrize("mesh", ["hyperbolic", "linear"])
def test_table_against_long_double(torch_cuda, eta, mesh):
    """M against the same formula in long double, per row max error <= 1e-12 max|M| (both branches of the device: w on
    the nodes, between them, outside the mesh and far away)."""
    om = np.asarray(mb.HyperbolicOmegaMesh(-10, 10, 400)) if mesh == "hyperbolic" else np.linspace(-3, 3, 401)
    w = np.concatenate([np.linspace(-12, 12, 241), om[::37], 0.5 * (om[1::53] + om[:-1:53]), [-1e4, 3e5]])
    M, _ = _table(om, w, eta)
    ref = rf.hilbert_table(om, w, eta)
    err = _row_err(M, ref)
    print("eta %g %s: worst row error / max|M| = %.3g (limit 1e-12)" % (eta, mesh, err.max()))
    assert np.all(err <= 1e-12), err.max()


@pytest.mark.parametrize("R, n_omega, n_w", [(133, 257, 101), (64, 32, 32), (1, 5, 3), (200, 1001, 77)])
def test_apply_modes_against_host(torch_cuda, R, n_omega, n_w):
    """mx_hilbert_apply in modes 0 / 1 / 2 against the host M A^T plus epilogue (same table), to 1e-12 per row: R not a
    multiple of the tile, odd n_omega and n_w, rows read in place from one analyzer slot of A_out[R, 5, n_omega]
    (lda = 5 n_omega), a NaN row."""
    torch = torch_cuda
    rng = np.random.default_rng(R + n_omega)
    om = np.linspace(-4, 4, n_omega)
    w = np.linspace(-5, 5, n_w)
    eta = 0.05
    M_d, w_d = real_frequency.hilbert_table(om, w, eta)
    M = M_d.cpu().numpy()
    A_out = rng.random((R, 5, n_omega))
    if R > 2:
        A_out[2, 3, n_omega // 2] = np.nan
    A_d = torch.as_tensor(A_out, device="cuda")[:, 3]
    assert A_d.stride(0) == 5 * n_omega
    scale, shift = 0.5 + rng.random(R), rng.standard_normal(R)
    for mode in (0, 1, 2):
        out = torch.empty((R, n_w), dtype=torch.complex128, device="cuda")
        sc = torch.as_tensor(scale, device="cuda") if mode == 1 else None
        ops.hilbert_apply(A_d, M_d, w_d, eta, mode, sc, torch.as_tensor(shift, device="cuda"), out)
        got = out.cpu().numpy()
        ref = rf.hilbert_apply(A_out[:, 3], M, w, eta, mode, scale if mode == 1 else None, shift)
        nan = np.isnan(A_out[:, 3]).any(axis=1)
        assert np.all(np.isnan(got[nan])), mode
        err = _row_err(got[~nan], ref[~nan])
        assert np.all(err <= 1e-12), (mode, err.max())


def test_closed_forms_on_the_device(torch_cuda):
    """The semicircle of half-width 2t on a 4001-point linear mesh: retarded_G equals the long-double reference to 1e-12
    and the closed form within the discretisation error measured with that reference (2.0e-4 of max|G| at eta = 1e-2);
    at eta = 1e-9, Im G = -pi A_lin(w) inside the mesh; for |z| >> mesh, z G -> sum_j delta_j A_j."""
    torch = torch_cuda
    t = 1.0
    om = np.linspace(-2 * t, 2 * t, 4001)
    A = rf.semicircle_A(om, t)
    w = np.linspace(-3, 3, 301)
    G = mb.retarded_G(A, om, w, 1e-2).cpu().numpy()[0]
    ex = rf.semicircle_G(w + 1e-2j, t)
    host = (rf.hilbert_table(om, w, 1e-2) @ A.astype(np.longdouble)).astype(np.complex128)
    assert np.max(np.abs(G - host)) <= 1e-12 * np.max(np.abs(host))
    assert np.max(np.abs(G - ex)) <= 3e-4 * np.max(np.abs(ex))
    w = np.linspace(-1.99, 1.99, 201)
    G = mb.retarded_G(torch.as_tensor(A, device="cuda"), om, w, 1e-9).cpu().numpy()[0]
    assert np.max(np.abs(G.imag + np.pi * rf.linear_interp(om, A, w))) < 1e-8
    w = np.array([1e5, -3e5, 1e7])
    G = mb.retarded_G(A, om, w, 1e-2).cpu().numpy()[0]
    d = np.diff(om)
    delta = np.concatenate([[d[0] / 2], 0.5 * (d[1:] + d[:-1]), [d[-1] / 2]])
    np.testing.assert_allclose(((w + 1e-2j) * G).real, np.sum(delta * A), rtol=1e-9)


@pytest.mark.parametrize("t", [1.0, 0.6])
def test_sigma_round_trip_without_maxent(torch_cuda, t):
    """Sigma(z) = t^2 g_sc(z) (Bethe lattice) makes G_aux = g_sc exactly for both methods (inversion with C = 0; direct
    with Sigma_inf = 0, N = t^2).  The exact A_aux tabulated on the mesh, through mx_hilbert_apply in modes 2 and 1, gives
    back t^2 g_sc(w + i eta) within the discretisation error of the host reference (long double, same table), and equals
    that reference to 1e-12."""
    torch = torch_cuda
    om = np.linspace(-2 * t, 2 * t, 4001)
    A = rf.semicircle_A(om, t)[None, :]
    w = np.linspace(-2.5 * t, 2.5 * t, 251)
    eta = 0.05
    M_d, w_d = real_frequency.hilbert_table(om, w, eta)
    M = rf.hilbert_table(om, w, eta)
    exact = t * t * rf.semicircle_G(w + 1j * eta, t)
    A_d = torch.as_tensor(A, device="cuda")
    for mode, scale in ((2, None), (1, t * t)):
        out = torch.empty((1, len(w)), dtype=torch.complex128, device="cuda")
        sc = None if scale is None else torch.full((1,), scale, dtype=torch.float64, device="cuda")
        ops.hilbert_apply(A_d, M_d, w_d, eta, mode, sc, torch.zeros(1, dtype=torch.float64, device="cuda"), out)
        got = out.cpu().numpy()[0]
        host = rf.hilbert_apply(A, M, w, eta, mode, None if scale is None else [scale], [0.0])[0].astype(np.complex128)
        assert np.max(np.abs(got - host)) <= 1e-12 * np.max(np.abs(host)), mode
        host_err = np.max(np.abs(host - exact))
        print("t %g mode %d: discretisation error %.3g of max|Sigma| %.3g" % (t, mode, host_err, np.max(np.abs(exact))))
        assert np.max(np.abs(got - exact)) <= host_err * (1 + 1e-6) + 1e-13
        assert host_err <= 2e-3 * np.max(np.abs(exact))


@pytest.mark.parametrize("method", ["inversion", "direct"])
def test_sigma_continuator_end_to_end(torch_cuda, method):
    """BatchedSigmaContinuator on noisy t^2 g_sc(i omega_n) for 32 spectra: G_aux_iw equals the numpy construction, A_aux
    is bit for bit a BatchedTauMaxEnt run on that G_aux, sigma_w equals the host composition of A_out, the long-double
    table and the epilogue to 1e-12 per row, and an unavailable analyzer gives NaN rows."""
    torch = torch_cuda
    B, n_iw, beta, t = 32, 120, 40.0, 0.8
    nu = np.pi / beta * (2 * np.arange(n_iw) + 1)
    rng = np.random.default_rng(2)
    S = t * t * rf.semicircle_G(1j * nu, t)[None, :] * (1 + 0.05 * rng.random(B))[:, None]
    S = S + 1e-5 * (rng.standard_normal((B, n_iw)) + 1j * rng.standard_normal((B, n_iw)))
    C = 0.1 * rng.standard_normal(B)
    om = mb.HyperbolicOmegaMesh(-4, 4, 200)
    kw = dict(constant_shift=C) if method == "inversion" else {}
    sc = mb.BatchedSigmaContinuator(method=method, **kw)
    sc.set_S_iw_data(nu, S)
    if method == "inversion":
        np.testing.assert_array_equal(sc.G_aux_iw, 1.0 / (1j * nu[None, :] + C[:, None] - S))
        scale, shift = None, C
    else:
        s_inf, N = real_frequency.fit_tail(nu, S)
        np.testing.assert_array_equal(sc.G_aux_iw, (S - s_inf[:, None]) / N[:, None])
        scale, shift = N, s_inf
        assert np.all((N > 0.98 * t * t) & (N < 1.07 * t * t)), N             # N = t^2 times the factor of each row

    def setup(j):
        j.omega = om
        j.set_alpha_mesh_log(0.01, 500, 24)
        j.reduce_singular_space = 1e-11
        j.set_error(1e-5)
    setup(sc.maxent)
    res = sc.run()
    ref = mb.BatchedTauMaxEnt()
    setup(ref)
    ref.set_G_iw_data(nu, sc.G_aux_iw)
    r2 = ref.run()
    np.testing.assert_array_equal(res.A_out, r2.A_out)
    np.testing.assert_array_equal(res.chi2, r2.chi2)
    w = np.linspace(-3, 3, 157)
    eta = 0.02
    got = sc.sigma_w(w, eta).cpu().numpy()
    assert got.shape == (B, len(w))
    M = rf.hilbert_table(np.asarray(om), w, eta)
    host = rf.hilbert_apply(res.A_out[:, 0], M, w, eta, 2 if method == "inversion" else 1, scale, shift)
    err = _row_err(got, host)
    assert np.all(err <= 1e-12), err.max()
    nan = sc.sigma_w(w, eta, analyzer="BryanAnalyzer").cpu().numpy()          # no probability: Bryan unavailable
    assert np.all(np.isnan(nan.real)) and np.all(np.isnan(nan.imag))
