"""Back to the real axis: the retarded transform of many spectra and the batched self-energy continuation.

``retarded_G(A, omega, w, eta)`` is G_r(w + i eta) = int dx A_r(x) / (w + i eta - x) for spectra A_r given on the omega
mesh -- what ``get_G_w_from_A_w`` (python/maxent_util.py) computes on TRIQS containers.  A_r is taken linear between the
mesh nodes and zero outside [omega_0, omega_{n-1}] (the spectrum whose integral the trapezoid weights of the mesh give),
for which the transform is exact: G = A M^T with a complex table M[n_w, n_omega] that depends on (mesh, w, eta) only.
The table is built on the device once per (mesh, w, eta) (``mx_hilbert_table``) and cached here; the product runs on the
FP64 tensor cores (``mx_hilbert_apply``), with the self-energy algebra of the continuators fused into its epilogue.

``BatchedSigmaContinuator`` is the array-based counterpart of the reference's ``DirectSigmaContinuator`` and
``InversionSigmaContinuator`` (python/sigma_continuator.py) for a batch of scalar self-energies Sigma_b(i omega_n):
auxiliary Green function, batched MaxEnt continuation on the Matsubara axis (``BatchedTauMaxEnt.set_G_iw_data``) and
Sigma_b(w + i eta) from the analyzer's A_aux without a trip to the host.  With a matrix worker (``BatchedElementwiseMaxEnt``
or ``BatchedPoormanMaxEnt``) it continues matrix-valued self-energies Sigma_b(i omega_n)[M, M] by inversion: the two
matrix inversions run on the device (``mx_matrix_resolvent``), the continuation element by element in between.
"""
import numpy as np

from . import _lib
from .batched import ANALYZER_NAMES, BatchedTauMaxEnt
from .batched_matrix import BatchedElementwiseMaxEnt

_TABLE_CACHE = {}
_TABLE_CACHE_SIZE = 4


def _mesh(omega):
    om = np.array(omega, dtype=np.float64).reshape(-1)
    if len(om) < 2 or not np.all(np.isfinite(om)) or not np.all(np.diff(om) > 0):
        raise ValueError("the omega mesh must hold at least two finite, strictly increasing points")
    return om


def _frequencies(w):
    w = np.array(w, dtype=np.float64).reshape(-1)
    if len(w) < 1 or not np.all(np.isfinite(w)):
        raise ValueError("w must hold at least one finite frequency")
    return w


def _eta(eta):
    eta = float(eta)
    if not (np.isfinite(eta) and eta > 0.0):
        raise ValueError("eta must be a finite number > 0, got %r" % (eta,))
    return eta


def _device(device):
    import torch
    if not torch.cuda.is_available():
        raise _lib.MaxEntLibraryError("maxent_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda" if device is None else device)


def hilbert_table(omega, w, eta, device=None):
    """The table M[n_w, n_omega] (complex128, on the device) with G(w_k + i eta) = sum_j M[k, j] A_j, and w on the
    device: (M, w_dev).  Cached per (mesh, w, eta, device)."""
    import torch
    from . import ops
    om, w, eta = _mesh(omega), _frequencies(w), _eta(eta)
    dev = _device(device)
    key = (om.tobytes(), w.tobytes(), eta, str(dev))
    hit = _TABLE_CACHE.get(key)
    if hit is not None:
        return hit
    with torch.cuda.device(dev):
        om_d = torch.as_tensor(om, device=dev)
        w_d = torch.as_tensor(w, device=dev)
        M = torch.empty((len(w), len(om)), dtype=torch.complex128, device=dev)
        ops.hilbert_table(om_d, w_d, eta, M)
    while len(_TABLE_CACHE) >= _TABLE_CACHE_SIZE:
        _TABLE_CACHE.pop(next(iter(_TABLE_CACHE)))
    _TABLE_CACHE[key] = (M, w_d)
    return M, w_d


def _rows(A, n_omega, device):
    """A as a float64 device matrix [R, n_omega] with unit column stride (a strided view is kept as it is)."""
    import torch
    if not torch.is_tensor(A):
        A = torch.from_numpy(np.ascontiguousarray(A, dtype=np.float64))
    if A.dim() == 1:
        A = A[None, :]
    if A.dim() != 2 or A.shape[1] != n_omega:
        raise ValueError("A must be [R, %d] (one spectrum per row on the omega mesh), got %s" % (n_omega, tuple(A.shape)))
    if A.is_complex():
        raise ValueError("A must be real")
    A = A.to(device=device, dtype=torch.float64)
    return A if A.shape[1] <= 1 or A.stride(1) == 1 else A.contiguous()


def _apply(A, M, w_d, eta, mode, scale=None, shift=None):
    import torch
    from . import ops
    out = torch.empty((A.shape[0], M.shape[0]), dtype=torch.complex128, device=M.device)
    with torch.cuda.device(M.device):
        ops.hilbert_apply(A, M, w_d, eta, mode, scale, shift, out)
    return out


def retarded_G(A, omega, w, eta):
    """G_r(w_k + i eta) = int dx A_r(x) / (w_k + i eta - x) of the spectra A[R, n_omega] (numpy or tensor) given on the
    mesh ``omega``, for A_r linear between the nodes and zero outside the mesh: a complex128 tensor [R, n_w] on the
    device of A (the current CUDA device for host input).  No normalisation is applied to A."""
    import torch
    om = _mesh(omega)
    dev = A.device if torch.is_tensor(A) and A.is_cuda else None
    M, w_d = hilbert_table(om, w, eta, device=dev)
    return _apply(_rows(A, len(om), M.device), M, w_d, _eta(eta), 0)


def _per_spectrum(x, B, what):
    x = np.asarray(x)
    if np.iscomplexobj(x):
        raise ValueError("%s must be real" % what)
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 0:
        return np.full(B, float(x))
    if x.shape != (B,):
        raise ValueError("%s must be a scalar or one value per spectrum (%d), got shape %s" % (what, B, x.shape))
    return x.copy()


def fit_tail(iomega, S_iw, n_tail=None):
    """High-frequency fit of scalar self-energies S_iw[B, n_iw] over the last ``n_tail`` Matsubara frequencies (default:
    the last 10 %, at least 4), per spectrum by least squares: Re S = a0 + a2 / nu^2 and -nu Im S = a1 + a3 / nu^2.
    Returns (sigma_inf, norm) = (a0, a1), each [B]."""
    nu = np.asarray(iomega, dtype=np.float64).reshape(-1)
    S = np.asarray(S_iw)
    n_iw = len(nu)
    n = max(4, int(np.ceil(0.1 * n_iw))) if n_tail is None else int(n_tail)
    if not 2 <= n <= n_iw:
        raise ValueError("the tail fit needs 2 <= n_tail <= n_iw (%d), got %d" % (n_iw, n))
    x = nu[-n:]
    X = np.stack([np.ones(n), 1.0 / x ** 2], axis=1)
    a_re = np.linalg.lstsq(X, S[:, -n:].real.T, rcond=None)[0]
    a_im = np.linalg.lstsq(X, (-x[:, None] * S[:, -n:].imag.T), rcond=None)[0]
    return a_re[0], a_im[0]


class BatchedSigmaContinuator(object):
    """Continuation of B scalar self-energies Sigma_b(i omega_n) through an auxiliary Green function
    (python/sigma_continuator.py, without the TRIQS containers):

    * ``method='inversion'`` (InversionSigmaContinuator): G_aux(i w) = 1 / (i w + C - Sigma(i w)) and
      Sigma(z) = z + C - 1 / G_aux(z), with ``constant_shift`` C a scalar or one value per spectrum (default 0);
    * ``method='direct'`` (DirectSigmaContinuator): G_aux(i w) = (Sigma(i w) - Sigma_inf) / N and
      Sigma(z) = N G_aux(z) + Sigma_inf; ``sigma_inf`` and ``norm`` are scalars or [B] arrays, fitted per spectrum on the
      last ``n_tail`` frequencies when not given (``fit_tail``).

    ``self.maxent`` is the ``BatchedTauMaxEnt`` that continues G_aux on the Matsubara axis: set its error, omega mesh,
    alpha mesh and cost function there, as with the reference's TauMaxEnt on Gaux_iw.  ``run()`` returns its
    ``BatchedMaxEntResult``; ``sigma_w(w, eta)`` maps the analyzer's A_aux(omega) back to Sigma_b(w + i eta) on the
    device.  A_aux is used as the continuation returns it: it is NOT renormalised before the transform.

    Matrix-valued self-energies S_iw[B, M, M, n_iw] (M <= 8) need a matrix worker, ``maxent=BatchedElementwiseMaxEnt(...)``
    or ``BatchedPoormanMaxEnt(...)``, and ``method='inversion'``: G_aux(i w) = ((i w + C) 1 - Sigma(i w))^-1 per matrix,
    element-wise continuation of G_aux, and Sigma(z) = (z + C) 1 - G_aux(z)^-1 with G_aux(z) = T(A_aux') + i T(A_aux'')
    assembled from the element spectra; ``run()`` returns a ``BatchedMatrixMaxEntResult`` and ``sigma_w`` [B, M, M, n_w].
    Covariance matrices of Matsubara data are not supported."""

    def __init__(self, method="inversion", constant_shift=0.0, sigma_inf=None, norm=None, n_tail=None, maxent=None):
        if method not in ("inversion", "direct"):
            raise ValueError("method must be 'inversion' or 'direct', got %r" % (method,))
        if method == "inversion" and (sigma_inf is not None or norm is not None):
            raise ValueError("sigma_inf and norm belong to method='direct'")
        self.method = method
        self.constant_shift = constant_shift
        self.sigma_inf = sigma_inf
        self.norm = norm
        self.n_tail = n_tail
        self.maxent = BatchedTauMaxEnt() if maxent is None else maxent
        self.iomega = None
        self.G_aux_iw = None
        self.result = None
        self._scale = self._shift = None
        self._matrix = False

    def set_S_iw_data(self, iomega, S_iw):
        """iomega[n_iw] (real Matsubara frequencies), S_iw[B, n_iw] (complex, numpy or tensor; [B, M, M, n_iw] with a
        matrix worker): builds G_aux_iw and hands it to ``self.maxent``."""
        nu = np.array(iomega, dtype=np.float64)
        if nu.ndim != 1 or len(nu) < 1:
            raise ValueError("iomega must be a vector of Matsubara frequencies")
        if isinstance(self.maxent, BatchedElementwiseMaxEnt):
            return self._set_matrix_S_iw(nu, S_iw)
        S = S_iw.detach().cpu().numpy() if hasattr(S_iw, "detach") else np.asarray(S_iw)
        if S.ndim == 1:
            S = S[None, :]
        if S.ndim != 2:
            raise NotImplementedError("matrix-valued self-energies S_iw[B, M, M, n_iw] need a matrix worker: "
                                      "BatchedSigmaContinuator(maxent=BatchedElementwiseMaxEnt(...)) or "
                                      "maxent=BatchedPoormanMaxEnt(...); the default worker takes S_iw[B, n_iw]")
        if S.shape[1] != len(nu):
            raise ValueError("iomega and S_iw don't have the same length (%d, %d)" % (len(nu), S.shape[1]))
        S = S.astype(np.complex128)
        B = S.shape[0]
        if self.method == "inversion":
            C = _per_spectrum(self.constant_shift, B, "constant_shift")
            G_aux = 1.0 / (1j * nu[None, :] + C[:, None] - S)
            self._scale, self._shift = None, C
        else:
            fit = fit_tail(nu, S, self.n_tail) if self.sigma_inf is None or self.norm is None else None
            s_inf = fit[0] if self.sigma_inf is None else _per_spectrum(self.sigma_inf, B, "sigma_inf")
            N = fit[1] if self.norm is None else _per_spectrum(self.norm, B, "norm")
            bad = np.nonzero(~(N > 0))[0]
            if len(bad):
                raise ValueError("the norm N of G_aux must be > 0; it is not for spectra %s" % bad.tolist())
            G_aux = (S - s_inf[:, None]) / N[:, None]
            self._scale, self._shift = N, s_inf
        self.iomega = nu
        self.G_aux_iw = G_aux
        self.result = None
        self._matrix = False
        self.maxent.set_G_iw_data(nu, G_aux)

    def _set_matrix_S_iw(self, nu, S_iw):
        """Matrix-valued Sigma with a matrix worker: G_aux_iw = ((i nu + C) 1 - Sigma)^-1 on the device
        (mx_matrix_resolvent mode 0), kept there as a complex128 tensor [B, M, M, n_iw]."""
        import torch
        from . import ops
        S = S_iw if torch.is_tensor(S_iw) else np.asarray(S_iw)
        shape = tuple(S.shape)
        if len(shape) != 4:
            raise ValueError("a matrix worker continues matrix-valued self-energies S_iw[B, M, M, n_iw], got shape %s"
                             % (shape,))
        if self.method != "inversion":
            raise NotImplementedError("method='direct' is not supported for matrix-valued self-energies (it needs a matrix "
                                      "normalisation of Sigma - Sigma_inf): use method='inversion'")
        B, M, n_iw = shape[0], shape[1], shape[3]
        if shape[2] != M:
            raise NotImplementedError("non-square blocks S_iw[B, %d, %d, n_iw] are not supported" % (shape[1], shape[2]))
        if not 1 <= M <= _lib.MX_MAX_MATRIX:
            raise NotImplementedError("blocks of M = %d orbitals are not supported (1 <= M <= %d)" % (M, _lib.MX_MAX_MATRIX))
        if n_iw != len(nu):
            raise ValueError("iomega and S_iw don't have the same length (%d, %d)" % (len(nu), n_iw))
        C = _per_spectrum(self.constant_shift, B, "constant_shift")
        dev = _device(self.maxent.maxent_diagonal.device)
        X = (S if torch.is_tensor(S) else torch.from_numpy(np.ascontiguousarray(S)))
        X = X.to(device=dev, dtype=torch.complex128).contiguous()
        z = torch.complex(torch.zeros(n_iw, dtype=torch.float64), torch.from_numpy(nu)).to(dev)
        G_aux = torch.empty_like(X)
        with torch.cuda.device(dev):
            ops.matrix_resolvent(X, z, torch.as_tensor(C, device=dev), 0, G_aux)
        self.iomega = nu
        self.G_aux_iw = G_aux
        self.result = None
        self._scale, self._shift, self._matrix = None, C, True
        self.maxent.set_G_iw_data(nu, G_aux)

    def run(self):
        """The batched continuation of G_aux_iw: a BatchedMaxEntResult (A_out = A_aux of every analyzer), a
        BatchedMatrixMaxEntResult with a matrix worker."""
        if self.G_aux_iw is None:
            raise Exception("no data: call set_S_iw_data")
        self.result = self.maxent.run()
        return self.result

    def sigma_w(self, w, eta, analyzer="LineFitAnalyzer"):
        """Sigma_b(w + i eta), complex128 tensor [B, n_w] on the device, from the analyzer's A_aux(omega) of ``run()``
        (read from the device result in place).  Spectra without that analyzer's pick (alpha_index -1: analyzer not
        available, or G_aux below G_threshold) are NaN rows.

        Matrix-valued Sigma: [B, M, M, n_w].  A_aux of every element is the result's A_out (zero below G_threshold,
        NaN without a pick), assembled on the device; a matrix with a NaN element is NaN at every frequency."""
        import torch
        if self.result is None:
            raise Exception("call run() first")
        if analyzer not in ANALYZER_NAMES:
            raise ValueError("unknown analyzer %r (one of %s)" % (analyzer, ", ".join(ANALYZER_NAMES)))
        slot = ANALYZER_NAMES.index(analyzer)
        if self._matrix:
            return self._matrix_sigma_w(w, _eta(eta), slot)
        dev = self.result.device
        eta = _eta(eta)
        M, w_d = hilbert_table(np.asarray(self.result.omega), w, eta, device=dev.A_out.device)
        A = dev.A_out[:, slot, :]
        put = lambda x: None if x is None else torch.as_tensor(x, dtype=torch.float64, device=M.device)
        mode = 2 if self.method == "inversion" else 1
        out = _apply(A, M, w_d, eta, mode, put(self._scale), put(self._shift))
        return out.masked_fill_((dev.alpha_index[:, slot] < 0)[:, None], complex(float("nan"), float("nan")))

    def _matrix_sigma_w(self, w, eta, slot):
        res = self.result
        return matrix_sigma_w(res.A_out_device(slot), np.asarray(res.omega), w, eta, self._shift)


def matrix_sigma_w(A, omega, w, eta, shift=None):
    """Sigma_b(z_k) = (z_k + C_b) 1 - G_b(z_k)^-1 at z_k = w_k + i eta, complex128 [B, M, M, n_w] on A's device, for
    matrix spectra A[B, M, M, n_omega] (real elements) or [B, M, M, 2, n_omega] (real and imaginary part of Hermitian
    A = A' + i A'') given as float64 device tensors on the mesh ``omega``: G(z) = T(A') + i T(A''), T the retarded
    transform of every part (mx_hilbert_apply mode 0), and the inverse per matrix and frequency (mx_matrix_resolvent
    mode 1, in place).  ``shift`` C is None or [B].  A matrix with a NaN element is NaN at every frequency."""
    import torch
    from . import ops
    om, eta = _mesh(omega), _eta(eta)
    B, M, n_omega = int(A.shape[0]), int(A.shape[1]), int(A.shape[-1])
    if A.dim() not in (4, 5) or int(A.shape[2]) != M or n_omega != len(om) or (A.dim() == 5 and int(A.shape[3]) != 2):
        raise ValueError("A must be [B, M, M, (2,) %d], got %s" % (len(om), tuple(A.shape)))
    M_d, w_d = hilbert_table(om, w, eta, device=A.device)
    n_w = int(M_d.shape[0])
    T = _apply(_rows(A.reshape(-1, n_omega), n_omega, M_d.device), M_d, w_d, eta, 0)
    if A.dim() == 5:
        T = torch.view_as_real(T).reshape(B, M, M, 2, n_w, 2)
        X = torch.complex(T[:, :, :, 0, :, 0] - T[:, :, :, 1, :, 1], T[:, :, :, 0, :, 1] + T[:, :, :, 1, :, 0])
        X = X.contiguous()
    else:
        X = T.reshape(B, M, M, n_w)
    z = torch.complex(w_d, torch.full_like(w_d, eta))
    C = None if shift is None else torch.as_tensor(_per_spectrum(shift, B, "shift"), device=X.device)
    with torch.cuda.device(X.device):
        ops.matrix_resolvent(X, z, C, 1, X)
    return X
