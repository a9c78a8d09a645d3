"""Host-side checks of the Matsubara batch, the retarded transform and BatchedSigmaContinuator: the long-double reference
of the transform against closed forms, the argument checks made before every launch, the error models of Matsubara
data and the self-energy algebra.  No device needed."""
import numpy as np
import pytest
import torch

import maxent_b200 as mb
from maxent_b200 import ops, real_frequency
from oracle import real_frequency as rf


def _delta(om):
    d = np.diff(om)
    out = np.zeros_like(om)
    out[:-1] += d / 2
    out[1:] += d / 2
    return out


# ---- the host reference against closed forms --------------------------------------------------------------------------
@pytest.mark.parametrize("eta, tol", [(1e-2, 3e-4), (1e-1, 4e-5), (1.0, 6e-6)])
def test_reference_semicircle(eta, tol):
    """Semicircle of half-width 2t on a 4001-point linear mesh: G(z) = (z - sqrt(z - 2t) sqrt(z + 2t)) / (2 t^2) up to
    the discretisation of A (linear between nodes; measured 2.0e-4, 2.2e-5, 3.7e-6 of max|G| at eta 1e-2, 0.1, 1)."""
    t = 1.0
    om = np.linspace(-2 * t, 2 * t, 4001)
    w = np.linspace(-3, 3, 301)
    G = (rf.hilbert_table(om, w, eta) @ rf.semicircle_A(om, t).astype(np.longdouble)).astype(np.complex128)
    ex = rf.semicircle_G(w + 1j * eta, t)
    assert np.max(np.abs(G - ex)) <= tol * np.max(np.abs(ex))


def test_reference_spectral_limit_and_moment():
    """At eta = 1e-9, Im G(w) = -pi A_lin(w) inside the mesh (measured 1.6e-9); for |z| >> mesh,
    z G(z) -> sum_j delta_j A_j (the first moment of the semicircle vanishes: the rest is O(1/z^2))."""
    om = np.linspace(-2, 2, 4001)
    A = rf.semicircle_A(om)
    w = np.linspace(-1.99, 1.99, 201)
    G = (rf.hilbert_table(om, w, 1e-9) @ A.astype(np.longdouble)).astype(np.complex128)
    assert np.max(np.abs(G.imag + np.pi * rf.linear_interp(om, A, w))) < 1e-8
    w = np.array([1e5, -3e5, 1e7])
    G = (rf.hilbert_table(om, w, 1e-2) @ A.astype(np.longdouble)).astype(np.complex128)
    np.testing.assert_allclose(((w + 1e-2j) * G).real, np.sum(_delta(om) * A), rtol=1e-9)


def test_reference_branches_agree():
    """The direct form and the series of the reference meet continuously at their switch (|q| = 1e3)."""
    x = np.array([0.0, 0.01])
    M = rf.hilbert_table(x, 0.01 + 0.01 * np.array([1e3 - 1e-9, 1e3 + 1e-9]), 1e-6)
    np.testing.assert_allclose(M[0].astype(np.complex128), M[1].astype(np.complex128), rtol=1e-11)


# ---- argument checks before the launches -------------------------------------------------------------------------------
def _apply_args(R=5, n_omega=7, n_w=3):
    A = torch.zeros((R, n_omega), dtype=torch.float64)
    M = torch.zeros((n_w, n_omega), dtype=torch.complex128)
    w = torch.zeros(n_w, dtype=torch.float64)
    out = torch.zeros((R, n_w), dtype=torch.complex128)
    return A, M, w, out


def test_hilbert_apply_checks():
    A, M, w, out = _apply_args()
    assert ops.check_hilbert_apply(A, M, w, 0.1, 0, None, None, out) == (7, 5, 7, 3)
    A_out = torch.zeros((5, 5, 7), dtype=torch.float64)
    assert ops.check_hilbert_apply(A_out[:, 3], M, w, 0.1, 2, None, None, out) == (35, 5, 7, 3)
    bad = [
        dict(eta=0.0), dict(eta=-1.0), dict(eta=float("nan")), dict(mode=3), dict(mode=-1),
        dict(A=A.to(torch.float32)), dict(A=A.t().contiguous().t()), dict(A=A[None]),
        dict(A=torch.as_strided(torch.zeros(40, dtype=torch.float64), (5, 7), (3, 1))),      # rows overlap
        dict(A=torch.zeros((5, 6), dtype=torch.float64)), dict(M=M.real.contiguous()), dict(M=M.t()),
        dict(w=w[:2]), dict(scale=torch.zeros(4, dtype=torch.float64)), dict(shift=torch.zeros(5, dtype=torch.float32)),
        dict(out=out[:4]), dict(out=out.real.contiguous()), dict(out=torch.zeros((3, 5), dtype=torch.complex128).t()),
    ]
    for b in bad:
        kw = dict(A=A, M=M, w=w, eta=0.1, mode=0, scale=None, shift=None, out=out)
        kw.update(b)
        with pytest.raises(ValueError):
            ops.check_hilbert_apply(**kw)


def test_hilbert_table_checks():
    om = torch.linspace(-1, 1, 7, dtype=torch.float64)
    w = torch.zeros(3, dtype=torch.float64)
    M = torch.zeros((3, 7), dtype=torch.complex128)
    assert ops.check_hilbert_table(om, w, 1e-3, M) == (7, 3)
    for kw in (dict(eta=0.0), dict(eta=-1e-3), dict(eta=float("inf")), dict(M=M[:2]), dict(M=M.real.contiguous()),
               dict(omega=om[:1]), dict(omega=om.to(torch.float32)), dict(w=w[::2])):
        args = dict(omega=om, w=w, eta=1e-3, M=M)
        args.update(kw)
        with pytest.raises(ValueError):
            ops.check_hilbert_table(**args)


def test_front_end_checks_before_any_device():
    with pytest.raises(ValueError):
        mb.retarded_G(np.zeros((2, 5)), np.linspace(-1, 1, 5), [0.0], 0.0)
    with pytest.raises(ValueError):
        mb.retarded_G(np.zeros((2, 5)), np.linspace(-1, 1, 5), [0.0], -1e-3)
    with pytest.raises(ValueError):
        mb.retarded_G(np.zeros((2, 5)), np.array([0.0, 1.0, 1.0, 2.0, 3.0]), [0.0], 1e-3)     # not increasing
    with pytest.raises(ValueError):
        mb.retarded_G(np.zeros((2, 5)), np.array([0.0]), [0.0], 1e-3)
    with pytest.raises(ValueError):
        mb.BatchedSigmaContinuator(method="other")


def test_operators_registered():
    for name in ("hilbert_table", "hilbert_apply"):
        assert name in ops.OPERATORS
        schema = str(getattr(torch.ops.maxent_b200, name).default._schema)
        assert "(a!)" in schema and schema.endswith("-> ()"), schema


# ---- Matsubara data in BatchedTauMaxEnt --------------------------------------------------------------------------------
def _iw_job(B=4, n_iw=6):
    nu = np.pi / 10 * (2 * np.arange(n_iw) + 1)
    G = (np.arange(B * n_iw) + 1j * np.arange(B * n_iw)[::-1]).reshape(B, n_iw) * 1e-2
    j = mb.BatchedTauMaxEnt()
    j.set_G_iw_data(nu, G)
    return j, nu, G


def test_G_iw_is_stacked():
    j, nu, G = _iw_job()
    np.testing.assert_array_equal(j.G, np.concatenate([G.real, G.imag], axis=1))
    assert j._n_rows() == 12 and j._n_data(j._n_rows()) == 6
    jt = mb.BatchedTauMaxEnt()
    jt.set_G_iw_data(nu, torch.from_numpy(G))
    np.testing.assert_array_equal(jt.G.numpy(), j.G)
    with pytest.raises(Exception):
        j.set_G_iw_data(nu[:-1], G)
    with pytest.raises(NotImplementedError):
        j.set_G_iw_data(nu, G.reshape(2, 2, 6))


def test_matsubara_error_models_map_onto_the_stacked_rows():
    j, nu, G = _iw_job(B=4, n_iw=6)
    j.set_error(1e-3)
    assert j._error_plan(4)[0] == "shared"
    e = np.linspace(1, 2, 6) * 1e-3
    j.set_error(e)
    mode, _, _ = j._error_plan(4)
    err, per = j._row_error()
    assert mode == "shared" and not per
    np.testing.assert_array_equal(err, np.concatenate([e, e]))
    j.set_error(np.array([1e-3, 2e-3, 3e-3, 4e-3]))                     # [B]
    mode, sig, _ = j._error_plan(4)
    assert mode == "sigma" and np.array_equal(sig, [1e-3, 2e-3, 3e-3, 4e-3])
    E = np.stack([e, e, 2 * e, e])                                       # [B, n_iw]: two whitening groups
    j.set_error(E)
    mode, index, specs = j._error_plan(4)
    assert mode == "groups" and len(specs) == 2
    for b in range(4):
        np.testing.assert_array_equal(specs[index[b]][1], np.concatenate([E[b], E[b]]))
    j.set_error(np.ones((4, 12)))                                        # stacked rows are not an error model
    with pytest.raises(Exception):
        j._error_plan(4)


def test_matsubara_rejections():
    j, nu, G = _iw_job()
    with pytest.raises(NotImplementedError):
        j.set_cov(np.eye(12))
    jt = mb.BatchedTauMaxEnt()
    with pytest.raises(NotImplementedError):
        jt.set_G_tau_data(np.linspace(0, 10, 6), G)                       # complex G(tau)
    with pytest.raises(NotImplementedError):
        jt.set_G_tau_data(np.linspace(0, 10, 6), torch.from_numpy(G))
    jt.set_cov(np.eye(12))
    with pytest.raises(NotImplementedError):
        jt.set_kernel_iw(nu)


# ---- BatchedSigmaContinuator: the self-energy algebra on the host ------------------------------------------------------
def _sigma(B=5, n_iw=40, t=0.8, beta=20.0):
    nu = np.pi / beta * (2 * np.arange(n_iw) + 1)
    S = t * t * rf.semicircle_G(1j * nu, 1.0 * t)[None, :] * (1 + 0.1 * np.arange(B))[:, None]
    return nu, S


def test_G_aux_construction():
    nu, S = _sigma()
    C = np.array([0.0, 0.1, -0.2, 0.3, 0.0])
    sc = mb.BatchedSigmaContinuator(method="inversion", constant_shift=C)
    sc.set_S_iw_data(nu, S)
    np.testing.assert_array_equal(sc.G_aux_iw, 1.0 / (1j * nu[None, :] + C[:, None] - S))
    np.testing.assert_array_equal(sc.maxent.G, np.concatenate([sc.G_aux_iw.real, sc.G_aux_iw.imag], axis=1))
    sd = mb.BatchedSigmaContinuator(method="direct", sigma_inf=0.5, norm=np.arange(1.0, 6.0))
    sd.set_S_iw_data(nu, S)
    np.testing.assert_array_equal(sd.G_aux_iw, (S - 0.5) / np.arange(1.0, 6.0)[:, None])


def test_tail_fit_recovers_an_exact_tail():
    rng = np.random.RandomState(4)
    B, n_iw = 6, 200
    nu = np.pi / 40 * (2 * np.arange(n_iw) + 1)
    a = rng.rand(4, B) + [[0.0], [0.5], [0.0], [0.0]]
    S = (a[0][:, None] + a[2][:, None] / (1j * nu) ** 2) + (a[1][:, None] + a[3][:, None] / (1j * nu) ** 2) / (1j * nu)
    s_inf, N = real_frequency.fit_tail(nu, S)
    np.testing.assert_allclose(s_inf, a[0], rtol=0, atol=1e-10)
    np.testing.assert_allclose(N, a[1], rtol=0, atol=1e-10)
    sd = mb.BatchedSigmaContinuator(method="direct")
    sd.set_S_iw_data(nu, S)
    np.testing.assert_allclose(sd._shift, a[0], atol=1e-10)
    np.testing.assert_allclose(sd._scale, a[1], atol=1e-10)


def test_sigma_continuator_rejections():
    nu, S = _sigma()
    sd = mb.BatchedSigmaContinuator(method="direct", sigma_inf=0.0, norm=[1.0, -1.0, 1.0, 0.0, 2.0])
    with pytest.raises(ValueError, match=r"\[1, 3\]"):
        sd.set_S_iw_data(nu, S)
    with pytest.raises(ValueError, match=r"\[0, 1, 2, 3, 4\]"):
        mb.BatchedSigmaContinuator(method="direct").set_S_iw_data(nu, -S)        # fitted N < 0
    with pytest.raises(NotImplementedError):                                     # matrix-valued Sigma
        mb.BatchedSigmaContinuator().set_S_iw_data(nu, np.stack([S, S], axis=1).reshape(5, 2, 1, -1))
    with pytest.raises(ValueError):
        mb.BatchedSigmaContinuator(constant_shift=[0.0, 1.0]).set_S_iw_data(nu, S)      # not one per spectrum
    with pytest.raises(ValueError):
        mb.BatchedSigmaContinuator().set_S_iw_data(nu[:-1], S)
    sc = mb.BatchedSigmaContinuator()
    sc.set_S_iw_data(nu, S)
    with pytest.raises(NotImplementedError):                                     # covariance of Matsubara data
        sc.maxent.set_cov(np.eye(2 * len(nu)))
    with pytest.raises(Exception):
        sc.sigma_w([0.0], 0.1)                                                   # before run()
