"""Host-side checks of matrix-valued self-energy continuation: the Matsubara element mapping of the batched matrix
classes, their Matsubara error models, the refusals of BatchedSigmaContinuator with matrix input, the argument checks
of the matrix_resolvent operator and the long-double resolvent reference.  No device needed."""
import numpy as np
import pytest
import torch

import maxent_b200 as mb
from maxent_b200 import _lib, ops
from maxent_b200.batched_matrix import element_plan, matsubara_rows
from oracle import matrix_sigma as ms


def _hermitian_spectra(M, omega, seed=3):
    """A Hermitian A(omega) = A' + i A'' on the mesh: A' symmetric, A'' antisymmetric, [M, M, n_omega] each."""
    rng = np.random.default_rng(seed)
    w = np.asarray(omega)
    c = rng.uniform(-2, 2, (M, M))
    s = rng.uniform(0.3, 1.0, (M, M))
    amp = rng.standard_normal((M, M, 2))
    Ap = amp[..., 0, None] * np.exp(-(w - c[..., None]) ** 2 / s[..., None])
    App = amp[..., 1, None] * np.exp(-(w + c[..., None]) ** 2 / s[..., None])
    return 0.5 * (Ap + Ap.transpose(1, 0, 2)), 0.5 * (App - App.transpose(1, 0, 2))


@pytest.mark.parametrize("herm", [True, False])
def test_matsubara_mapping_is_the_image_of_the_tau_path(herm):
    """G_ij(i nu) = K A'_ij + i K A''_ij with the numpy IOmegaKernel (K delta): the c = 0 rows of matsubara_rows are the
    stacked rows of K A'_ij, the c = 1 rows those of K A''_ij, to 1e-15 of max |G_ij| (the one rounding of forming G from
    the two parts), and a diagonal row is [Re G_ii; Im G_ii] bit for bit."""
    M, n_iw = 3, 40
    nu = np.pi / 20 * (2 * np.arange(n_iw) + 1)
    om = mb.HyperbolicOmegaMesh(-6, 6, 150)
    K = mb.IOmegaKernel(nu, om)
    Kd = K.K_delta if hasattr(K, "K_delta") else K._K_delta
    Ap, App = _hermitian_spectra(M, om)
    KAp, KApp = np.einsum("nw,ijw->ijn", Kd, Ap), np.einsum("nw,ijw->ijn", Kd, App)     # K A'' antisymmetric exactly
    G = (KAp + 1j * KApp)[None]
    G = np.concatenate([G, 2 * G])                                          # B = 2
    diag, off = element_plan(2, M, use_hermiticity=herm, use_complex=True)
    got_d = matsubara_rows(torch.from_numpy(G), diag).numpy()
    for r, (b, i, _, _) in enumerate(diag):
        np.testing.assert_array_equal(got_d[r], np.concatenate([G[b, i, i].real, G[b, i, i].imag]))
    got = matsubara_rows(torch.from_numpy(G), off).numpy()
    for r, (b, i, j, c) in enumerate(off):
        ref = (1 + b) * K.stack(KAp[i, j] if c == 0 else KApp[i, j])
        scale = (1 + b) * max(np.max(np.abs(KAp[i, j])), np.max(np.abs(KApp[i, j])))     # the size of G_ij
        assert np.max(np.abs(got[r] - ref)) <= 1e-15 * scale, (b, i, j, c)


def _iw_job(cls=mb.BatchedPoormanMaxEnt, B=3, M=2, n_iw=6, **kw):
    nu = np.pi / 10 * (2 * np.arange(n_iw) + 1)
    rng = np.random.default_rng(0)
    G = rng.standard_normal((B, M, M, n_iw)) + 1j * rng.standard_normal((B, M, M, n_iw))
    job = cls(use_complex=True, **kw)
    job.set_G_iw_data(nu, G)
    return job, nu, G


def test_set_G_iw_data():
    job, nu, G = _iw_job()
    assert job.tau is None and np.array_equal(job.iomega, nu)
    for w in job._workers():
        assert np.array_equal(w.iomega, nu) and w._n_rows() == 2 * len(nu)
    with pytest.raises(ValueError):
        job.set_G_iw_data(nu, G[:, :, :1])                                   # not square
    with pytest.raises(ValueError):
        job.set_G_iw_data(nu, G[0])                                          # not [B, M, M, n_iw]
    with pytest.raises(Exception):
        job.set_G_iw_data(nu[:-1], G)
    job.set_G_tau_data(np.linspace(0, 10, 6), G.real)                        # back to tau data
    assert job.iomega is None and job.maxent_diagonal.iomega is None


def test_matsubara_error_kinds():
    """The error kinds of the tau path with n_iw in place of n_tau; the workers repeat a per-point error for the Re and
    Im rows; covariances of Matsubara data raise."""
    B, M, n_iw = 3, 2, 6
    job, nu, G = _iw_job(B=B, M=M, n_iw=n_iw)
    kinds = {(): "shared", (n_iw,): "shared", (M, M, n_iw): "element", (B, M, M): "spectrum"}
    for shape, kind in kinds.items():
        job.set_error(np.full(shape, 1e-3) if shape else 1e-3)
        assert job._error_kind(B, M) == kind
    for shape in ((2 * n_iw,), (M, M, 2 * n_iw), (B, M, M + 1)):
        job.set_error(np.ones(shape))
        with pytest.raises(ValueError):
            job._error_kind(B, M)
    e = 1e-3 * (1 + np.arange(M * M * n_iw).reshape(M, M, n_iw))
    job.set_error(e)
    diag, off = element_plan(B, M, True, True)
    job._put_error(job.maxent_offdiagonal, "element", off)
    mode, index, specs = job.maxent_offdiagonal._error_plan(len(off))
    assert mode == "groups"
    for r, (b, i, j, c) in enumerate(off):
        np.testing.assert_array_equal(specs[index[r]][1], np.concatenate([e[i, j], e[i, j]]))
    s = 1e-3 * (1 + np.arange(B * M * M).reshape(B, M, M))
    job.set_error(s)
    job._put_error(job.maxent_diagonal, "spectrum", diag)
    mode, sig, _ = job.maxent_diagonal._error_plan(len(diag))
    assert mode == "sigma" and np.array_equal(sig, s[diag[:, 0], diag[:, 1], diag[:, 2]])
    with pytest.raises(NotImplementedError):
        job.set_cov(np.eye(n_iw))
    tj = mb.BatchedPoormanMaxEnt()
    tj.set_cov(np.eye(n_iw))
    with pytest.raises(NotImplementedError):
        tj.set_G_iw_data(nu, G)


def test_tau_maxent_still_refuses_matrices():
    nu = np.pi / 10 * (2 * np.arange(6) + 1)
    with pytest.raises(NotImplementedError):
        mb.BatchedTauMaxEnt().set_G_iw_data(nu, np.ones((2, 2, 2, 6), dtype=complex))


# ---- BatchedSigmaContinuator with matrix input: every refusal before any device work -----------------------------------
def _S(B=2, M=2, n_iw=8):
    nu = np.pi / 10 * (2 * np.arange(n_iw) + 1)
    return nu, np.ones((B, M, M, n_iw), dtype=complex)


def test_sigma_continuator_matrix_refusals():
    nu, S = _S()
    with pytest.raises(NotImplementedError, match="BatchedPoormanMaxEnt"):           # default scalar worker
        mb.BatchedSigmaContinuator().set_S_iw_data(nu, S)
    for cls in (mb.BatchedElementwiseMaxEnt, mb.BatchedPoormanMaxEnt):
        with pytest.raises(NotImplementedError):                                     # non-square blocks
            mb.BatchedSigmaContinuator(maxent=cls()).set_S_iw_data(nu, S[:, :, :1])
        M = _lib.MX_MAX_MATRIX + 1
        with pytest.raises(NotImplementedError):
            mb.BatchedSigmaContinuator(maxent=cls()).set_S_iw_data(nu, np.ones((1, M, M, len(nu)), dtype=complex))
        with pytest.raises(NotImplementedError):                                     # direct method
            mb.BatchedSigmaContinuator(method="direct", sigma_inf=0.0, norm=1.0, maxent=cls()).set_S_iw_data(nu, S)
        with pytest.raises(ValueError):                                              # scalar data into a matrix worker
            mb.BatchedSigmaContinuator(maxent=cls()).set_S_iw_data(nu, S[:, 0, 0])
        with pytest.raises(ValueError):
            mb.BatchedSigmaContinuator(maxent=cls()).set_S_iw_data(nu[:-1], S)
        with pytest.raises(ValueError):
            mb.BatchedSigmaContinuator(constant_shift=[0.0, 1.0, 2.0], maxent=cls()).set_S_iw_data(nu, S)


# ---- the operator's checks ---------------------------------------------------------------------------------------------
def _resolvent_args(B=3, M=2, n_z=5):
    X = torch.zeros((B, M, M, n_z), dtype=torch.complex128)
    return dict(X=X, z=torch.zeros(n_z, dtype=torch.complex128), C=torch.zeros(B, dtype=torch.float64), mode=0,
                Y=torch.zeros_like(X))


def test_check_matrix_resolvent():
    a = _resolvent_args()
    assert ops.check_matrix_resolvent(**a) == (3, 2, 5)
    assert ops.check_matrix_resolvent(**dict(a, Y=a["X"], C=None, mode=1)) == (3, 2, 5)      # in place
    M = _lib.MX_MAX_MATRIX
    big = torch.zeros((1, M, M, 5), dtype=torch.complex128)
    assert ops.check_matrix_resolvent(**dict(a, X=big, Y=big.clone(), C=None)) == (1, M, 5)
    X9 = torch.zeros((1, M + 1, M + 1, 5), dtype=torch.complex128)
    buf = torch.zeros((4, 2, 2, 5), dtype=torch.complex128)
    bad = [
        dict(X=X9, Y=X9.clone(), C=None),                                         # M = 9
        dict(X=torch.zeros((3, 0, 0, 5), dtype=torch.complex128), Y=torch.zeros((3, 0, 0, 5), dtype=torch.complex128)),
        dict(X=a["X"].real.contiguous()), dict(X=a["X"].to(torch.complex64)), dict(X=a["X"][:, :, :1].contiguous()),
        dict(X=a["X"][0]), dict(X=a["X"].transpose(1, 2)), dict(z=a["z"][:4]), dict(z=a["z"].real.contiguous()),
        dict(C=torch.zeros(2, dtype=torch.float64)), dict(C=torch.zeros(3, dtype=torch.float32)),
        dict(mode=2), dict(mode=-1), dict(Y=a["Y"][:2]), dict(Y=a["Y"].real.contiguous()),
        dict(Y=torch.zeros((3, 2, 2, 5), dtype=torch.complex128).transpose(1, 2)),
        dict(X=buf[:3], Y=buf[1:]),                                               # overlapping, not in place
    ]
    for b in bad:
        with pytest.raises(ValueError):
            ops.check_matrix_resolvent(**dict(a, **b))


def test_operator_registered():
    assert "matrix_resolvent" in ops.OPERATORS
    schema = str(torch.ops.maxent_b200.matrix_resolvent.default._schema)
    assert "(a!)" in schema and schema.endswith("-> ()"), schema
    with pytest.raises(NotImplementedError):                              # CUDA dispatch key only
        ops.matrix_resolvent(**_resolvent_args())


# ---- the long-double reference -----------------------------------------------------------------------------------------
def test_reference_inverts_known_matrices():
    rng = np.random.default_rng(1)
    B, M, n = 4, 5, 6
    X = rng.standard_normal((B, M, M, n)) + 1j * rng.standard_normal((B, M, M, n))
    z = rng.standard_normal(n) + 1j * rng.uniform(0.1, 1, n)
    C = rng.standard_normal(B)
    s = z[None, :] + C[:, None]
    A = np.moveaxis(X, 3, 1)
    eye = np.eye(M)
    Y0 = np.moveaxis(np.linalg.inv(s[..., None, None] * eye - A), 1, 3)
    Y1 = np.moveaxis(s[..., None, None] * eye - np.linalg.inv(A), 1, 3)
    np.testing.assert_allclose(ms.resolvent(X, z, C, 0).astype(complex), Y0, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(ms.resolvent(X, z, C, 1).astype(complex), Y1, rtol=1e-12, atol=1e-12)
    P = np.zeros((1, 3, 3, 1), dtype=complex)                            # a permutation needs the pivot search
    P[0, [0, 1, 2], [1, 2, 0], 0] = [2.0, 1j, -0.5]
    Pinv = np.zeros_like(P)
    Pinv[0, [1, 2, 0], [0, 1, 2], 0] = [0.5, -1j, -2.0]
    assert np.array_equal(ms.resolvent(P, [0.0], None, 1).astype(complex), -Pinv)
    S = np.ones((1, 2, 2, 2), dtype=complex)                             # singular; a NaN entry
    S[0, 0, 0, 1] = np.nan
    Y = ms.resolvent(S, [0.0, 0.0], None, 1)
    assert np.all(np.isnan(Y.astype(complex).real))


def test_bethe_matrix_closed_form():
    """U diag(g_sc) U^dagger is (z - Sigma)^-1 of Sigma = U diag(t^2 g_sc) U^dagger."""
    z = np.linspace(-3, 3, 11) + 0.05j
    t = np.array([[1.0, 0.6], [0.8, 1.2]])
    U = ms.random_unitary(2, 2, seed=4)
    S = ms.bethe_matrix_sigma(z, t, U)
    G = ms.resolvent(S, z, None, 0).astype(complex)
    np.testing.assert_allclose(G, ms.bethe_matrix_G_aux(z, t, U), rtol=0, atol=1e-13)
