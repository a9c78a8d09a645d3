"""Host references of the matrix steps of the inversion method for matrix-valued self-energies
(csrc/mx_resolvent.cu, BatchedSigmaContinuator with a matrix worker), in long double.

``resolvent`` is Gauss-Jordan with partial pivoting by modulus in np.clongdouble, vectorised over every (b, k):

    mode 0: Y(b,k) = ((z_k + C_b) 1 - X(b,k))^-1,    mode 1: Y(b,k) = (z_k + C_b) 1 - X(b,k)^-1,

with X[B, M, M, n_z] (frequency innermost, the device layout).  A matrix with a non-finite entry or an exactly zero pivot
gives NaN, as on the device.

``bethe_matrix_*`` is a closed form to check the whole chain against: Sigma(z) = U diag(t_m^2 g_sc(z; t_m)) U^dagger with
a unitary U and the Bethe-lattice (semicircle) g_sc of half-width 2 t_m.  Since g_sc = 1 / (z - t^2 g_sc), at C = 0 the
auxiliary Green function is exactly G_aux(z) = (z 1 - Sigma(z))^-1 = U diag(g_sc(z; t_m)) U^dagger, whose spectral
function is A_aux(omega) = U diag(A_sc(omega; t_m)) U^dagger.
"""
import numpy as np

from oracle import real_frequency as rf

LD = np.longdouble


def _inverse(A):
    """Inverse of every matrix A[..., M, M] (clongdouble) by Gauss-Jordan on [A | 1] with partial pivoting by modulus;
    NaN for a matrix with a non-finite entry or an exactly zero pivot."""
    M = A.shape[-1]
    aug = np.concatenate([A, np.broadcast_to(np.eye(M, dtype=A.dtype), A.shape)], axis=-1).copy()
    bad = ~np.all(np.isfinite(A), axis=(-2, -1))
    aug[bad] = 0
    idx = np.indices(A.shape[:-2])
    for k in range(M):
        p = k + np.argmax(np.abs(aug[..., k:, k]), axis=-1)
        row_k, row_p = aug[..., k, :].copy(), aug[(*idx, p)].copy()
        aug[..., k, :] = row_p
        aug[(*idx, p)] = row_k
        piv = aug[..., k, k].copy()
        bad |= piv == 0
        piv = np.where(piv == 0, 1, piv)
        aug[..., k, :] /= piv[..., None]
        for r in range(M):
            if r != k:
                aug[..., r, :] -= aug[..., r, k][..., None] * aug[..., k, :]
    inv = aug[..., M:]
    inv[bad] = np.nan
    return inv


def resolvent(X, z, C, mode):
    """The long-double counterpart of mx_matrix_resolvent: X[B, M, M, n_z] complex, z[n_z] complex, C[B] real or None.
    Returns Y[B, M, M, n_z] as np.clongdouble."""
    X = np.asarray(X).astype(np.clongdouble)
    B, M, _, n_z = X.shape
    s = np.asarray(z).astype(np.clongdouble)[None, :] + (
        np.zeros(B, dtype=LD) if C is None else np.asarray(C, dtype=np.float64).astype(LD))[:, None]
    A = np.moveaxis(X, 3, 1)                                   # [B, n_z, M, M]
    eye = np.eye(M, dtype=np.clongdouble)
    Y = _inverse(s[..., None, None] * eye - A) if mode == 0 else s[..., None, None] * eye - _inverse(A)
    return np.moveaxis(Y, 1, 3)


def random_unitary(B, M, seed):
    """B Haar-like unitary M x M matrices (QR of complex Gaussians)."""
    rng = np.random.default_rng(seed)
    Z = rng.standard_normal((B, M, M)) + 1j * rng.standard_normal((B, M, M))
    Q, R = np.linalg.qr(Z)
    d = np.diagonal(R, axis1=-2, axis2=-1)
    return Q * (d / np.abs(d))[:, None, :]


def _rotate(U, diag):
    """U diag(d) U^dagger for U[B, M, M] and d[B, M, n]: [B, M, M, n]."""
    return np.einsum("bim,bmk,bjm->bijk", U, diag, np.conj(U))


def bethe_matrix_sigma(z, t, U):
    """Sigma_b(z) = U_b diag(t_bm^2 g_sc(z; t_bm)) U_b^dagger at the complex frequencies z[n]: [B, M, M, n] complex."""
    g = np.stack([np.stack([rf.semicircle_G(z, tm) for tm in tb]) for tb in np.asarray(t)])
    return _rotate(U, np.asarray(t)[..., None] ** 2 * g)


def bethe_matrix_G_aux(z, t, U):
    """G_aux = (z 1 - Sigma)^-1 = U diag(g_sc(z; t_m)) U^dagger of bethe_matrix_sigma (C = 0): [B, M, M, n] complex."""
    g = np.stack([np.stack([rf.semicircle_G(z, tm) for tm in tb]) for tb in np.asarray(t)])
    return _rotate(U, g)


def bethe_matrix_A(omega, t, U):
    """The spectral function of G_aux, U diag(A_sc(omega; t_m)) U^dagger (Hermitian): [B, M, M, n_omega] complex."""
    a = np.stack([np.stack([rf.semicircle_A(omega, tm) for tm in tb]) for tb in np.asarray(t)])
    return _rotate(U, a.astype(np.complex128))
