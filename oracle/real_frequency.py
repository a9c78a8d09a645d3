"""Host references of the retarded transform (maxent_b200/real_frequency.py, csrc/mx_hilbert.cu), in long double.

G(z) = int dx A(x) / (z - x) for A linear between the mesh nodes and zero outside them; per segment [x_a, x_b],
h = x_b - x_a, q = (z - x_b) / h, u = (z - x_a) / h, L = log(u / q):

    int = c_a A_a + c_b A_b,   c_a = 1 - q L,   c_b = u L - 1.

Evaluated in np.longdouble: directly where |q| <= 1e3, by the series of log1p(1/q) beyond (c_a = sum (-1)^(n+1) t^n /
(n+1), c_b = sum (-1)^(n+1) t^n / (n (n+1)), t = 1/q), where the direct form would cancel more than three digits.  The
switch sits elsewhere than the device kernel's (|q| = 10), so each branch of one is checked against the other's.
"""
import numpy as np

LD = np.longdouble
_FAR_Q = 1.e3
_TERMS = 10                         # |t|^10 <= 1e-30


def _segment_coeffs(x_a, x_b, w, eta):
    h = x_b - x_a
    q = (w - x_b) / h + 1j * (eta / h)
    u = (w - x_a) / h + 1j * (eta / h)
    far = np.abs(q) > _FAR_Q
    qn = np.where(far, 1.0, q)
    L = np.log(np.where(far, 1.0, u) / qn)
    c_a = 1 - qn * L
    c_b = np.where(far, 1.0, u) * L - 1
    t = 1 / np.where(far, q, 1.0)
    sa = np.zeros_like(t)
    sb = np.zeros_like(t)
    for n in range(_TERMS, 0, -1):
        s = 1 if n & 1 else -1
        sa = t * (sa + LD(s) / (n + 1))
        sb = t * (sb + LD(s) / (n * (n + 1)))
    return np.where(far, sa, c_a), np.where(far, sb, c_b)


def hilbert_table(omega, w, eta):
    """M[n_w, n_omega] (complex long double) with G(w_k + i eta) = sum_j M[k, j] A_j."""
    om = np.asarray(omega, dtype=np.float64).astype(LD)
    wk = np.asarray(w, dtype=np.float64).astype(LD)[:, None]
    eta = LD(float(eta))
    c_a, c_b = _segment_coeffs(om[None, :-1], om[None, 1:], wk, eta)
    M = np.zeros((wk.shape[0], len(om)), dtype=np.clongdouble)
    M[:, :-1] += c_a
    M[:, 1:] += c_b
    return M


def hilbert_apply(A, M, w, eta, mode, scale=None, shift=None):
    """out[R, n_w] = epilogue(A M^T) of mx_hilbert_apply in long double: mode 0 G, mode 1 scale G + shift, mode 2
    z + shift - 1/G, z = w + i eta."""
    A = np.asarray(A, dtype=np.float64).astype(LD)
    G = A @ np.asarray(M).astype(np.clongdouble).T
    R = A.shape[0]
    sc = np.ones(R, dtype=LD) if scale is None else np.asarray(scale, dtype=np.float64).astype(LD)
    sh = np.zeros(R, dtype=LD) if shift is None else np.asarray(shift, dtype=np.float64).astype(LD)
    if mode == 0:
        return G
    if mode == 1:
        return sc[:, None] * G + sh[:, None]
    z = np.asarray(w, dtype=np.float64).astype(LD) + 1j * LD(float(eta))
    return z[None, :] + sh[:, None] - 1 / G


def semicircle_A(x, t=1.0):
    """Spectral function of the Bethe lattice (half-width 2t), normalised to 1."""
    x = np.asarray(x, dtype=np.float64)
    return np.sqrt(np.maximum(4 * t * t - x * x, 0.0)) / (2 * np.pi * t * t)


def semicircle_G(z, t=1.0):
    """Its retarded Green function G(z) = (z - sqrt(z - 2t) sqrt(z + 2t)) / (2 t^2) for Im z > 0."""
    z = np.asarray(z, dtype=np.complex128)
    return (z - np.sqrt(z - 2 * t) * np.sqrt(z + 2 * t)) / (2 * t * t)


def linear_interp(omega, A, x):
    """A linear between the nodes of omega, zero outside the mesh (the spectrum the transform assumes)."""
    om = np.asarray(omega, dtype=np.float64)
    return np.interp(x, om, A, left=0.0, right=0.0)
