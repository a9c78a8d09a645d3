"""Host driver of the fused alpha sweep: prepares the state shared by a batch of spectra
(kernel SVD, truncation, whitening rotation, V' re-tiling, initial v) and calls the C ABI.

PyTorch is used for device memory, streams and the one-time small dense factorisations only; the
hot path (projection, alpha sweep, analyzers) runs in libmaxent_b200.so.  Nothing here runs the
algorithm on the CPU: a missing library or a missing CUDA device is an error.

Reference seam: MaxEntLoop.run (python/maxent_loop.py:144-302).
"""
import ctypes

import numpy as np

from . import _lib

_F64 = None


def _torch():
    import torch
    return torch


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


class LMParams(object):
    """LevenbergMinimizer parameters (python/minimizers/levenberg_minimizer.py:92-121)."""

    def __init__(self, maxiter=1000, miniter=0, mu0=1.e-18, nu=1.3, max_mu=1.e20,
                 conv_max_derivative=1.e-4, conv_rel_change=1.e-16, conv_abs_change=-1.0, marquardt=False):
        if nu <= 1.0:
            raise Exception('If nu <= 1, there will be an infinite loop.')   # levenberg_minimizer.py:139-140
        self.maxiter, self.miniter, self.mu0, self.nu, self.max_mu = maxiter, miniter, mu0, nu, max_mu
        self.conv_max_derivative, self.conv_rel_change = conv_max_derivative, conv_rel_change
        self.conv_abs_change, self.marquardt = conv_abs_change, bool(marquardt)

    def c_struct(self):
        return _lib.MxLMParams(int(self.maxiter), int(self.miniter), float(self.mu0), float(self.nu),
                               float(self.max_mu), float(self.conv_max_derivative), float(self.conv_rel_change),
                               float(self.conv_abs_change), int(self.marquardt), 0)


class SharedProblem(object):
    """Everything a batch of spectra shares: K = U S V^T truncated at `reduce_singular_space`
    (python/kernels.py:101-122), rotated so that chi2 is diagonal in the singular space:

        M = diag(1/err) K V_s = Q Xi P^T ,  V' = V_s P ,  chi2(H) = |Xi V'^T H - Q^T G/err|^2 + c0

    (for a scalar err: Q = U_s, Xi = S_s/err, P = 1).  The Levenberg iterates are invariant under
    this rotation because mu*1 is."""

    def __init__(self, K, err, D, delta, variant="normal", reduce_singular_space=1.e-14, device=None,
                 svd="jacobi", A_init=None, max_nsv=None, engine=0, rank_floor=5.e-16, usv=None,
                 orthonormal_U=True):
        """``usv`` = (U, S, V) already truncated by the caller (a ``kernels.KernelSVD`` after
        ``reduce_singular_space``); ``orthonormal_U=False`` when U was rotated by a non-square T
        (TauMaxEnt.set_cov with dropped eigenvalues), which forces the general whitening branch."""
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.MaxEntLibraryError("maxent_b200 needs a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        self.device = torch.device("cuda" if device is None else device)
        f64 = torch.float64
        dev = self.device
        with torch.cuda.device(dev):
            K = torch.as_tensor(np.ascontiguousarray(K, dtype=np.float64) if not torch.is_tensor(K) else K,
                                dtype=f64, device=dev).contiguous()
            n_tau, n_omega = K.shape
            self.n_tau, self.n_omega = int(n_tau), int(n_omega)
            self.variant = variant
            # ---- SVD of the kernel (KernelSVD.svd, python/kernels.py:53-64) ----
            if usv is not None:
                U, S, V = [torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64) if not torch.is_tensor(x) else x,
                                           dtype=f64, device=dev).contiguous() for x in usv]
                reduce_singular_space, rank_floor = None, 0.0          # the caller has applied its cut
            else:
                U, S, V = self._svd(K, svd)
            # reduce_singular_space is an ABSOLUTE threshold (python/kernels.py:101-122).  Below
            # rank_floor * S[0] the computed singular triplets are rounding noise (which of them pass an absolute
            # 1e-14 depends on the SVD implementation, and their left vectors are not orthonormal any more), so the
            # cut is honoured only down to the numerical rank -- the one documented deviation (DESIGN.md); the
            # optimum A_alpha does not depend on those directions (SURVEY.md Appendix A, last item).
            thr = -1.0 if reduce_singular_space is None else float(reduce_singular_space)
            self.n_sv_requested = int((S >= thr).sum())
            thr = max(thr, float(rank_floor) * float(S[0]))
            keep = torch.nonzero(S >= thr).flatten()
            self.n_sv_uncapped = int(keep.numel())
            if max_nsv is not None and keep.numel() > int(max_nsv):
                keep = keep[:int(max_nsv)]               # explicit request of the caller: continue in a smaller space
            if keep.numel() > _lib.MX_MAX_NSV:
                # the reference keeps every S >= threshold (python/kernels.py:101-122); silently continuing in a
                # truncated space would return a different A(omega), so this is an error, not a fallback
                raise _lib.MaxEntLibraryError(
                    "the kernel keeps %d singular values >= %g (numerical rank floor %g * S[0]); the fused path supports "
                    "n_sv <= %d -- raise reduce_singular_space, or pass max_nsv=%d to truncate explicitly"
                    % (keep.numel(), thr, rank_floor, _lib.MX_MAX_NSV, _lib.MX_MAX_NSV))
            U, S, V = U[:, keep].contiguous(), S[keep].contiguous(), V[:, keep].contiguous()
            self.U, self.S, self.V = U, S, V
            s = int(S.numel())
            self.n_sv = s
            # ---- whitening rotation ----
            err_np = np.asarray(err, dtype=np.float64) * np.ones(self.n_tau)
            err_t = torch.as_tensor(err_np, dtype=f64, device=dev)
            sqrtw = 1.0 / err_t
            if orthonormal_U and np.all(err_np == err_np[0]):
                Q, Xi, P = U, S / err_np[0], None
            else:
                M = (sqrtw[:, None] * (K @ V)).contiguous()
                Q, Xi, P = self._svd(M, svd)
                # A covariance estimated from few samples (TauMaxEnt.set_cov drops its null space, python/tau_maxent.py:
                # 253-288) leaves k = n_tau' < s rows: M = Q[k, k] Xi[k] P[s, k]^T has rank <= k, and the singular space
                # the kernels work in shrinks to it (directions of V outside the row space of M do not enter chi2; the
                # entropy pulls them to the default model, where v' = 0 keeps them).
                k = int(Xi.numel())
                if k < s:
                    # Complete P to an orthonormal s x s rotation with zero singular values: the extra directions do
                    # not enter chi2 (zero rows of Xi, zero columns of Q) but keep their entropy term, exactly as in the
                    # reference, whose v lives in the full s-dimensional space of the unrotated kernel
                    # (python/kernels.py:160-180 rotates U only).
                    if variant == "bryan":
                        raise NotImplementedError("BryanCostFunction with fewer data rows (%d) than singular values (%d): "
                                                  "its Hessian is singular" % (k, s))
                    Pc = torch.linalg.svd(P, full_matrices=True)[0][:, k:]
                    P = torch.cat([P, Pc], dim=1).contiguous()
                    Xi = torch.cat([Xi, torch.zeros(s - k, dtype=f64, device=dev)])
            # The left vectors of singular values near the rounding floor come out of a one-sided Jacobi (or any
            # SVD) with an orthogonality error ~ eps * S[0] / S[i]; chi2 = |Xi y - Q^T g|^2 + |(1 - Q Q^T) g|^2
            # needs Q^T Q = 1.  Re-orthogonalised Gram-Schmidt in order of decreasing singular value leave the
            # well-determined columns untouched (to rounding) and move the others by an amount whose effect on
            # K H is ~ 1e-2 * S[i] -- far below the data error.
            Q = self._reorthonormalize(Q)
            if Q.shape[1] < s:                                           # rank-deficient whitening: zero columns for Xi = 0
                Q = torch.cat([Q, torch.zeros((Q.shape[0], s - Q.shape[1]), dtype=f64, device=dev)], dim=1)
            self.P = P
            self.Vp = V if P is None else (V @ P).contiguous()
            self.Q = Q.contiguous()
            self.Qw = (sqrtw[:, None] * Q).contiguous()
            self.sqrtw = sqrtw.contiguous()
            self.xi = Xi.contiguous()
            self.D = torch.as_tensor(np.asarray(D, dtype=np.float64), dtype=f64, device=dev).contiguous()
            self.delta = torch.as_tensor(np.asarray(delta, dtype=np.float64), dtype=f64, device=dev).contiguous()
            self.A_init = None if A_init is None else _dev_f64(A_init, dev)
            self.v0 = (self.Vp.transpose(0, 1) @ _log_initial_arg(self.D, self.A_init, self.delta, variant)).contiguous()
            self.Vt = _layout_V(self.lib, self.Vp)
            self.engine = int(engine)
            self.config = _lib.sweep_config(s, self.engine)

    def _reorthonormalize(self, Q):
        """Columns of Q made orthonormal in order, on the device in one launch (mx_gram_schmidt_rows)."""
        torch = _torch()
        Qt = Q.transpose(0, 1).contiguous()
        stream = ctypes.c_void_p(torch.cuda.current_stream(Q.device).cuda_stream)
        with torch.cuda.device(Q.device):
            _lib.check(self.lib.mx_gram_schmidt_rows(_ptr(Qt), int(Qt.shape[1]), int(Qt.shape[0]), 0.0, stream),
                       "mx_gram_schmidt_rows")
        return Qt.transpose(0, 1).contiguous()

    def _svd(self, K, method):
        torch = _torch()
        if not hasattr(self, "svd_sweeps"):
            self.svd_sweeps = None
        if method == "jacobi":
            U, S, V, info = device_svd(K)
            if self.svd_sweeps is None:
                self.svd_sweeps = info
            return U, S, V
        elif method == "torch":
            U, S, Vh = torch.linalg.svd(K, full_matrices=False)
            return U.contiguous(), S.contiguous(), Vh.transpose(0, 1).contiguous()
        raise ValueError("svd must be 'jacobi' or 'torch'")

    def v_to_reference_basis(self, v):
        """v' (rotated basis) -> v in the basis of the truncated SVD of K."""
        return v if self.P is None else v @ self.P.transpose(0, 1)


def _log_initial_arg(D, A_init, delta, variant):
    """log of the argument of the entropy's inverse at the initial H0 = (A_init or D) * delta, with D [..., n_omega]
    (python/maxent_loop.py:196-203; quirk: D*delta although D holds delta).  The initial vector is V'^T of it."""
    torch = _torch()
    H0 = (D if A_init is None else A_init) * delta
    if variant == "plusminus":
        arg = (H0 + torch.sqrt(H0 ** 2 + 4 * D ** 2)) / (2 * D)         # functions.py:793-796
    else:
        arg = H0 / D                                                     # functions.py:753-755
    return torch.log(torch.where(arg.abs() <= 1e-100, torch.full_like(arg, 1e-100), arg))


def _layout_V(lib, Vp):
    """V'[n_omega, n_sv] re-tiled for the sweep kernel (mx_layout_V)."""
    torch = _torch()
    n_omega, s = int(Vp.shape[0]), int(Vp.shape[1])
    n = int(lib.mx_layout_V_size(n_omega, s))
    if n < 0:
        raise _lib.MaxEntLibraryError("n_sv=%d outside the fused path (max %d)" % (s, _lib.MX_MAX_NSV))
    Vt = torch.empty(n, dtype=torch.float64, device=Vp.device)
    _lib.check(lib.mx_layout_V(_ptr(Vp), n_omega, s, _ptr(Vt), _stream(Vp.device)), "mx_layout_V")
    return Vt


def _require_cuda():
    torch = _torch()
    if not torch.cuda.is_available():
        raise _lib.MaxEntLibraryError("maxent_b200 needs a CUDA device (no CPU fallback)")
    return torch


def tau_kernel_host(tau, omega, beta, device=None):
    """TauKernel values (python/kernels.py:244-266) computed by mx_tau_kernel; numpy in, numpy out."""
    torch = _require_cuda()
    lib = _lib.load()
    dev = torch.device("cuda" if device is None else device)
    with torch.cuda.device(dev):
        t_d = torch.as_tensor(np.ascontiguousarray(tau, dtype=np.float64), device=dev)
        o_d = torch.as_tensor(np.ascontiguousarray(omega, dtype=np.float64), device=dev)
        K = torch.empty((t_d.numel(), o_d.numel()), dtype=torch.float64, device=dev)
        _lib.check(lib.mx_tau_kernel(_ptr(t_d), _ptr(o_d), int(t_d.numel()), int(o_d.numel()), float(beta), _ptr(K),
                                     _stream(dev)), "mx_tau_kernel")
        return K.cpu().numpy()


def matmul_host(A, B, device=None):
    """A @ B on the device (plain library GEMM, problem set-up only: K diag(delta) B of the preblur kernel);
    numpy in, numpy out."""
    torch = _require_cuda()
    dev = torch.device("cuda" if device is None else device)
    with torch.cuda.device(dev):
        return (torch.as_tensor(np.ascontiguousarray(A, dtype=np.float64), device=dev)
                @ torch.as_tensor(np.ascontiguousarray(B, dtype=np.float64), device=dev)).cpu().numpy()


SVD_DIRECT_MAX = 160      # matrices with min(m, n) up to this get the full one-sided Jacobi (mx_svd_jacobi)
SVD_FIRST_RANK = 128      # first guess of the number of leading triplets of a larger matrix (mx_svd_truncated)
SVD_RANGE_MAX = 512       # columns the range finder of mx_svd_truncated handles (one-CTA Gram-Schmidt)
SVD_FLOOR = 1.e-15        # a returned singular value below SVD_FLOOR * S[0] is at the rounding floor of the matrix
SVD_SEED = 0x6d6178656e74  # the random range finder is reproducible


def device_svd(K):
    """SVD of a device tensor K[m, n] for KernelSVD.svd (python/kernels.py:53-64): (U[m, k], S[k], V[n, k], info).

    Small matrices (min(m, n) <= SVD_DIRECT_MAX): full one-sided Jacobi, k = min(m, n).  Larger ones: the leading
    triplets only (mx_svd_truncated), with k doubled until at least eight of the returned singular values sit at the
    rounding floor -- then K = U S V^T holds to eps * S[0] and nothing above the floor is missing; a matrix that is
    not numerically rank deficient ends at k = min(m, n), i.e. with the full SVD (through the same range finder up to
    SVD_RANGE_MAX columns, plain Jacobi on K above).  ``info`` says which route ran."""
    torch = _torch()
    lib = _lib.load()
    dev = K.device
    f64 = torch.float64
    m, n = int(K.shape[0]), int(K.shape[1])
    kmin = min(m, n)
    stream = _stream(dev)

    def full():
        tr = m < n
        Kk = K.transpose(0, 1).contiguous() if tr else K.contiguous()
        m2, n2 = int(Kk.shape[0]), int(Kk.shape[1])
        U = torch.empty((m2, n2), dtype=f64, device=dev)
        S = torch.empty((n2,), dtype=f64, device=dev)
        V = torch.empty((n2, n2), dtype=f64, device=dev)
        work = torch.empty((m2 * n2 + n2 * n2 + n2 + 64,), dtype=f64, device=dev)
        _lib.check(lib.mx_svd_jacobi(_ptr(Kk), m2, n2, _ptr(U), _ptr(S), _ptr(V), _ptr(work), 60, None, stream),
                   "mx_svd_jacobi")
        return ((V, S, U) if tr else (U, S, V)) + ("jacobi, all %d columns" % n2,)

    if kmin <= SVD_DIRECT_MAX:
        return full()
    Kc = K.contiguous()
    p = SVD_FIRST_RANK
    while min(p, kmin) <= SVD_RANGE_MAX:
        p = min(p, kmin)
        U = torch.empty((m, p), dtype=f64, device=dev)
        S = torch.empty((p,), dtype=f64, device=dev)
        V = torch.empty((n, p), dtype=f64, device=dev)
        nwork = int(lib.mx_svd_truncated_work_doubles(m, n, p))
        work = torch.empty((nwork,), dtype=f64, device=dev)
        _lib.check(lib.mx_svd_truncated(_ptr(Kc), m, n, p, _ptr(U), _ptr(S), _ptr(V), _ptr(work), SVD_SEED, stream),
                   "mx_svd_truncated")
        if p == kmin:
            # not rank deficient: the range finder spans everything, K Q has graded columns -- the form in which a
            # one-sided Jacobi converges in a few sweeps (on K itself, columns of equal norm and a condition number of
            # 1e12, sixty sweeps are not enough beyond ~200 columns)
            return U, S, V, "range finder + jacobi, all %d columns" % p
        Sh = S.cpu()
        if int((Sh > SVD_FLOOR * float(Sh[0])).sum()) <= p - 8:
            return U, S, V, "truncated, %d leading triplets" % p
        p *= 2
    return full()


def svd_jacobi_host(K, device=None):
    """KernelSVD.svd on the device (python/kernels.py:53-64): numpy in, numpy (U[m, k], S[k], V[n, k]) out; see
    ``device_svd`` for k."""
    torch = _require_cuda()
    dev = torch.device("cuda" if device is None else device)
    with torch.cuda.device(dev):
        Kd = torch.as_tensor(np.ascontiguousarray(K, dtype=np.float64), device=dev)
        U, S, V, _ = device_svd(Kd)
        return U.cpu().numpy(), S.cpu().numpy(), V.cpu().numpy()


class SweepResult(object):
    """Device tensors produced by one call of the fused sweep (+ analyzers).  ``problems`` and ``index`` (host [B], None
    for a launch of one problem) say which SharedProblem every spectrum ran with: ``problem(b)``."""
    __slots__ = ("alpha", "v", "A", "chi2", "S", "Q", "logp", "n_iter", "n_qeval", "n_solve", "status",
                 "alpha_index", "A_out", "n_sv", "n_trial", "n_batch", "phase_cycles", "alpha_scale", "problems", "index")

    def problem(self, b):
        return self.problems[0 if self.index is None else int(self.index[b])]


def _stream(dev):
    torch = _torch()
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _dev_f64(x, dev):
    """Host array / tensor -> contiguous float64 tensor on `dev` (asynchronous when the source is pinned)."""
    torch = _torch()
    if torch.is_tensor(x):
        return x.to(device=dev, dtype=torch.float64, non_blocking=True).contiguous()
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)


def _problem_args(prob, alpha, lm, chi2_factor, probability=False, n_sv=None, Vt=None, xi=None, D=None, v0=None,
                  vt_index=None, vt_stride=0, alpha_rows=None):
    """The problem description as the leading arguments of the torch operators (maxent_b200/ops.py): the state of
    ``prob``, in a singular space of ``n_sv`` dimensions, with the per-spectrum rows that are given in place of its own
    (MxProblem.per_spectrum_model bits: D with v0, xi, Vt with vt_index, alpha)."""
    flags = ((_lib.PER_SPECTRUM_MODEL if D is not None else 0) | (_lib.PER_SPECTRUM_XI if xi is not None else 0)
             | (_lib.PER_SPECTRUM_VT if vt_index is not None else 0)
             | (_lib.PER_SPECTRUM_ALPHA if alpha_rows is not None else 0))
    dims = [prob.n_tau, prob.n_omega, prob.n_sv if n_sv is None else n_sv, int(alpha.numel()), _lib.VARIANTS[prob.variant],
            int(bool(probability)), prob.engine, flags, int(lm.maxiter), int(lm.miniter), int(lm.marquardt), int(vt_stride)]
    params = [float(chi2_factor), float(lm.mu0), float(lm.nu), float(lm.max_mu), float(lm.conv_max_derivative),
              float(lm.conv_rel_change), float(lm.conv_abs_change)]
    return (prob.Vt if Vt is None else Vt, prob.Qw, prob.Q, prob.sqrtw, prob.xi if xi is None else xi,
            prob.D if D is None else D, prob.delta, alpha if alpha_rows is None else alpha_rows,
            prob.v0 if D is None else v0, vt_index, dims, params)


def _ops():
    from . import ops
    return ops


def project_data(prob, G):
    """mx_project_data: gt[B, n_sv] = (sqrt(W) Q)^T G and c0[B] = the part of chi2 outside the kept
    singular space (NormalChi2.f uses the full kernel, python/functions.py:358-360)."""
    torch = _torch()
    dev = prob.device
    with torch.cuda.device(dev):
        G = _dev_f64(G, dev)
        B = int(G.shape[0])
        alpha = torch.ones((1,), dtype=torch.float64, device=dev)
        gt = torch.empty((B, prob.n_sv), dtype=torch.float64, device=dev)
        c0 = torch.empty((B,), dtype=torch.float64, device=dev)
        _ops().project_data(*_problem_args(prob, alpha, LMParams(), 1.0), G, gt, c0)
    return gt, c0


def analyze(alpha, chi2, S, logp, A, gamma=0.2, linefit_deg=0, bryan_by_integration=False, device=None,
            want_aux=False):
    """mx_analyze on arrays (python/analyzers/*.py): returns alpha_index[B, 5] (int32, -1 = not available)
    and A_out[B, 5, n_omega] (None if A is None); with ``want_aux`` also aux[B, 4 + 2 n_alpha]
    (line-fit parameters, curvature, dS/dlog alpha)."""
    torch = _require_cuda()
    _lib.load()                              # a missing library is an error here, not inside the operator
    dev = torch.device("cuda" if device is None else device)
    if torch.is_tensor(chi2) and chi2.is_cuda:
        dev = chi2.device
    with torch.cuda.device(dev):
        alpha, chi2, S = _dev_f64(alpha, dev), _dev_f64(chi2, dev), _dev_f64(S, dev)
        logp = None if logp is None else _dev_f64(logp, dev)
        A = None if A is None else _dev_f64(A, dev)
        B, n_alpha = int(chi2.shape[0]), int(chi2.shape[1])
        n_omega = int(A.shape[2]) if A is not None else 0
        idx = torch.full((B, _lib.N_ANALYZERS), -1, dtype=torch.int32, device=dev)
        A_out = torch.empty((B, _lib.N_ANALYZERS, n_omega), dtype=torch.float64, device=dev) if A is not None else None
        aux = torch.empty((B, 4 + 2 * n_alpha), dtype=torch.float64, device=dev) if want_aux else None
        _ops().analyze(alpha, chi2, S, logp, A, float(gamma), int(linefit_deg), bool(bryan_by_integration),
                       idx, A_out, aux)
    if want_aux:
        return idx, A_out, aux
    return idx, A_out




def run_sweep(prob, G, alpha_eff, probability=False, lm=None, chi2_factor=1.0, want_A=True, want_v=True,
              analyze_results=True, gamma=0.2, linefit_deg=0, bryan_by_integration=False, time_kernel=False, D=None,
              phase_timers=False, sigma=None, groups=None, alpha_scale=None, v0=None):
    """Fused alpha sweep for a batch G[B, n_tau] sharing `prob`.  `alpha_eff` = alpha * scale_alpha, descending.
    G may live on the host (numpy / pinned tensor: copied asynchronously) or on the device.
    Everything stays on the device; returns a SweepResult of torch tensors.

    Error models per spectrum (TauMaxEnt.set_error / set_cov per data set, python/tau_maxent.py:227-288), still ONE
    launch of the sweep: ``sigma`` [B] gives every spectrum its own scalar error bar (``prob`` built with err = 1);
    ``groups`` = (problems, index[B]) gives every spectrum one of several SharedProblems that differ in the error vector
    or covariance (hence in the whitening rotation V'); G[b] is then the data of spectrum b in the (rotated) data space
    of its group, rows padded to the longest.  ``prob`` must be problems[0].  ``sigma`` and ``groups`` exclude each
    other.  ``alpha_scale`` [B] (with ``groups``) multiplies the alpha mesh per spectrum (scale_alpha = 'Ndata' when
    groups keep different numbers of data rows; the analyzers are invariant under a common factor on alpha and see the
    unscaled mesh).

    Default models per spectrum: ``D`` [B, n_omega] (incl. delta omega), with or without ``groups``; every spectrum's
    initial vector is computed in the basis of its own group's V'.  With ``v0`` [B, n_sv] the rows are already built on
    the device (``D`` then [B, ldD] in the MX_PER_SPECTRUM_MODEL layout, e.g. by mx_poorman_models)."""
    torch = _torch()
    dev = prob.device
    f64, i32 = torch.float64, torch.int32
    lm = LMParams() if lm is None else lm
    ops = _ops()
    probs, index = ([prob], None) if groups is None else groups
    if index is not None:
        if sigma is not None:
            raise ValueError("sigma and groups cannot be combined: every group carries its own error vector")
        index = np.asarray(index.cpu() if torch.is_tensor(index) else index)
    n_omega, s = prob.n_omega, max(q.n_sv for q in probs)
    if probs[0] is not prob or any(q.n_omega != n_omega or q.variant != prob.variant for q in probs):
        raise ValueError("the problems of all groups must share the omega mesh and the cost function")
    if any(q.n_sv != s for q in probs) and (prob.variant == "bryan" or lm.marquardt):
        # Groups with different singular-space dimensions (different kernels, e.g. the b values of a preblur scan) are
        # padded with zero columns of V' (and zero xi, v0, g~) up to the largest.  The padded components never move
        # (their rows of Z, J and f are exactly zero) and add exact zeros to every sum.  Not for the Bryan cost function
        # (its gradient divides by xi: 0 / 0 in a padded component) nor for Marquardt's damping mu diag(J) (an exact
        # zero pivot in a padded row): those need one launch per n_sv.
        raise ValueError("groups of different n_sv cannot share a launch with the Bryan cost function or "
                         "Marquardt's damping: run each n_sv separately")
    with torch.cuda.device(dev):
        G = _dev_f64(G, dev)
        if G.dim() == 1:
            G = G[None, :]
        B = int(G.shape[0])
        alpha = _dev_f64(np.asarray(alpha_eff, dtype=np.float64) if not torch.is_tensor(alpha_eff) else alpha_eff, dev)
        n_alpha = int(alpha.numel())
        zeros = lambda *shape: torch.zeros(shape, dtype=f64, device=dev)
        # the spectra of every problem: the whole batch for a single problem, the rows of its group otherwise
        if index is None:
            if G.shape[1] != prob.n_tau:
                raise ValueError("G has %d data points, kernel has %d" % (G.shape[1], prob.n_tau))
            parts = [(prob, slice(None))]
        else:
            index_d = torch.as_tensor(index, device=dev).to(torch.int64)
            parts = []
            for g, q in enumerate(probs):
                sel = np.nonzero(index == g)[0]
                if len(sel):
                    parts.append((q, torch.as_tensor(sel, device=dev)))
        if sigma is not None:                    # Xi_b = Xi / sigma_b, data divided by sigma_b (prob carries err = 1)
            sg = _dev_f64(sigma, dev).reshape(-1)
            if sg.numel() != B:
                raise ValueError("sigma has %d entries for %d spectra" % (sg.numel(), B))
            G = (G / sg[:, None]).contiguous()
        # ---- projection: every problem with its own Q, 1/err and data rows, in its own singular space ----
        gt = torch.empty((B, s), dtype=f64, device=dev) if index is None else zeros(B, s)
        c0 = torch.empty((B,), dtype=f64, device=dev)
        for q, sel in parts:
            if index is None:
                Gq, gq, cq = G, gt, c0
            else:
                Gq = G[sel][:, :q.n_tau].contiguous()
                gq, cq = torch.empty((len(sel), q.n_sv), dtype=f64, device=dev), torch.empty((len(sel),), dtype=f64, device=dev)
            ops.project_data(*_problem_args(q, alpha, lm, chi2_factor), Gq, gq, cq)
            if index is not None:
                gt[sel, :q.n_sv], c0[sel] = gq, cq
        # ---- per-spectrum rows, zero-padded to the common n_sv ----
        xi = Vt = vt_index = alpha_rows = None
        vt_stride = 0
        if sigma is not None:
            xi = (prob.xi[None, :] / sg[:, None]).contiguous()
        if index is not None:
            xi = zeros(B, s)
            for q, sel in parts:
                xi[sel, :q.n_sv] = q.xi
            tiled = [q.Vt if q.n_sv == s else _layout_V(q.lib, torch.cat([q.Vp, zeros(n_omega, s - q.n_sv)], dim=1))
                     for q in probs]
            vt_stride = max(int(t.numel()) for t in tiled)
            Vt = zeros(len(probs), vt_stride)
            for g, t in enumerate(tiled):
                Vt[g, :t.numel()] = t
            vt_index = index_d.to(i32).contiguous()
            if alpha_scale is not None:          # alpha * (data rows of the spectrum's group), python/maxent_loop.py:216-220
                alpha_rows = (alpha[None, :] * _dev_f64(alpha_scale, dev).reshape(-1, 1)).contiguous()
        ld = (n_omega + 1) & ~1
        D_rows = v0_rows = None
        if v0 is not None:                       # rows built on the device already
            if D is None or tuple(D.shape) != (B, ld) or v0.shape[0] != B or v0.shape[1] > s:
                raise ValueError("ready-made model rows must be D[%d, %d] and v0[%d, <= %d]" % (B, ld, B, s))
            D_rows, v0_rows = _dev_f64(D, dev), zeros(B, s)
            v0_rows[:, :v0.shape[1]] = _dev_f64(v0, dev)
        elif D is not None or index is not None:
            D_rows, v0_rows = zeros(B, ld), zeros(B, s)
            if D is None:                        # the shared model, with the initial vector of every spectrum's group
                D_rows[:, :n_omega] = prob.D
                for q, sel in parts:
                    v0_rows[sel, :q.n_sv] = q.v0
            else:                                # one default model per spectrum, v0 in its own group's basis
                D = _dev_f64(D, dev)
                if tuple(D.shape) != (B, n_omega):
                    raise ValueError("D must be [%d, %d]" % (B, n_omega))
                D_rows[:, :n_omega] = D
                for q, sel in parts:
                    v0_rows[sel, :q.n_sv] = _log_initial_arg(D[sel], q.A_init, q.delta, q.variant) @ q.Vp
        # ---- launch ----
        pargs = _problem_args(prob, alpha, lm, chi2_factor, probability, n_sv=s, Vt=Vt, xi=xi, D=D_rows, v0=v0_rows,
                              vt_index=vt_index, vt_stride=vt_stride, alpha_rows=alpha_rows)
        r = SweepResult()
        r.alpha, r.n_sv, r.problems, r.index, r.alpha_scale = alpha, s, probs, index, alpha_scale
        r.v = torch.empty((B, n_alpha, s), dtype=f64, device=dev) if want_v else None
        r.A = torch.empty((B, n_alpha, n_omega), dtype=f64, device=dev) if want_A else None
        r.chi2 = torch.empty((B, n_alpha), dtype=f64, device=dev)
        r.S = torch.empty((B, n_alpha), dtype=f64, device=dev)
        r.Q = torch.empty((B, n_alpha), dtype=f64, device=dev)
        r.logp = torch.full((B, n_alpha), float("nan"), dtype=f64, device=dev)
        r.n_iter = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.n_qeval = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.n_solve = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.status = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.n_trial = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.n_batch = torch.zeros((B, n_alpha), dtype=i32, device=dev)
        r.phase_cycles = torch.zeros((B, 8), dtype=torch.int64, device=dev) if phase_timers else None
        ws_bytes = int(prob.lib.mx_sweep_workspace_bytes(ctypes.byref(ops.problem_struct(*pargs)), B))
        if ws_bytes < 0:
            _lib.check(ws_bytes, "mx_sweep_workspace_bytes")
        ws = getattr(prob, "_workspace", None)
        if ws is None or ws.numel() < ws_bytes:
            ws = prob._workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        if time_kernel:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        ops.alpha_sweep(*pargs, gt, c0, r.v, r.A, r.chi2, r.S, r.Q, r.logp, r.n_iter, r.n_qeval, r.n_solve, r.status,
                        r.n_trial, r.n_batch, r.phase_cycles, ws)
        if time_kernel:
            ev1.record()
            ev1.synchronize()
            return ev0.elapsed_time(ev1)
        r.alpha_index = r.A_out = None
        if analyze_results:
            r.alpha_index = torch.full((B, _lib.N_ANALYZERS), -1, dtype=i32, device=dev)
            r.A_out = torch.empty((B, _lib.N_ANALYZERS, n_omega), dtype=f64, device=dev) if want_A else None
            ops.analyze(alpha, r.chi2, r.S, r.logp if probability else None, r.A, float(gamma), int(linefit_deg),
                        bool(bryan_by_integration), r.alpha_index, r.A_out, None)
        return r
