"""PyTorch custom operators over the C ABI (include/maxent_b200.h).

    torch.ops.maxent_b200.project_data    -> mx_project_data
    torch.ops.maxent_b200.alpha_sweep     -> mx_alpha_sweep
    torch.ops.maxent_b200.analyze         -> mx_analyze
    torch.ops.maxent_b200.poorman_models  -> mx_poorman_models
    torch.ops.maxent_b200.hilbert_table   -> mx_hilbert_table
    torch.ops.maxent_b200.hilbert_apply   -> mx_hilbert_apply
    torch.ops.maxent_b200.matrix_resolvent -> mx_matrix_resolvent

The operators are registered for the CUDA dispatch key ONLY: calling one with host tensors raises
``NotImplementedError`` from the dispatcher -- there is no CPU implementation of the hot path.  They are thin:
every operator packs its tensor arguments into the plain-pointer structs of the ABI, takes the current stream
of the tensors' device and calls the shared library; outputs are caller-allocated tensors the operator writes
(``Tensor(a!)`` in the schema), so nothing is allocated and nothing synchronises inside an operator.

Reference seam these replace: the body of MaxEntLoop.run (python/maxent_loop.py:205-302) and
MaxEntResult.analyze (python/maxent_result.py:795-818).
"""
import ctypes
import math

import torch

from . import _lib

# dims  = [n_tau, n_omega, n_sv, n_alpha, variant, want_probability, per_spectrum_model, maxiter, miniter, marquardt,
#          vt_stride]
# param = [chi2_factor, mu0, nu, max_mu, conv_max_derivative, conv_rel_change, conv_abs_change]
_PROBLEM = ("Tensor Vt, Tensor Qw, Tensor Qo, Tensor sqrtw, Tensor xi, Tensor D, Tensor delta, Tensor alpha, "
            "Tensor v0, Tensor? vt_index, int[] dims, float[] params")

_library = torch.library.Library("maxent_b200", "DEF")
_library.define("project_data(" + _PROBLEM + ", Tensor G, Tensor(a!) gt, Tensor(b!) c0) -> ()")
_library.define("alpha_sweep(" + _PROBLEM + ", Tensor gt, Tensor c0, Tensor(a!)? v, Tensor(b!)? A, Tensor(c!) chi2, "
                "Tensor(d!) S, Tensor(e!) Q, Tensor(f!) logp, Tensor(g!) n_iter, Tensor(h!) n_qeval, Tensor(i!) n_solve, "
                "Tensor(j!) status, Tensor(k!) n_trial, Tensor(l!) n_batch, Tensor(m!)? phase_cycles, "
                "Tensor(n!) workspace) -> ()")
_library.define("analyze(Tensor alpha, Tensor chi2, Tensor S, Tensor? logp, Tensor? A, float gamma, int linefit_deg, "
                "bool bryan_by_integration, Tensor(a!) alpha_index, Tensor(b!)? A_out, Tensor(c!)? aux) -> ()")
_library.define("poorman_models(Tensor A_out, int slot, Tensor rows, Tensor delta, float d_add, Tensor? A_init, Tensor Vp, "
                "Tensor? group, Tensor(a!) D, Tensor(b!) v0, Tensor(c!) ok) -> ()")
_library.define("hilbert_table(Tensor omega, Tensor w, float eta, Tensor(a!) M) -> ()")
_library.define("hilbert_apply(Tensor A, Tensor M, Tensor w, float eta, int mode, Tensor? scale, Tensor? shift, "
                "Tensor(a!) out) -> ()")
_library.define("matrix_resolvent(Tensor X, Tensor z, Tensor? C, int mode, Tensor(a!) Y) -> ()")


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _f64c(*ts):
    for t in ts:
        if t is not None and (t.dtype != torch.float64 or not t.is_contiguous()):
            raise ValueError("maxent_b200 operators take contiguous float64 tensors")


def problem_struct(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0, vt_index, dims, params):
    """The MxProblem of the C ABI that the leading arguments of project_data / alpha_sweep describe."""
    if len(dims) != 11 or len(params) != 7:
        raise ValueError("dims must hold 11 integers and params 7 floats (see maxent_b200/ops.py)")
    if vt_index is not None and (vt_index.dtype != torch.int32 or not vt_index.is_contiguous()):
        raise ValueError("vt_index must be a contiguous int32 tensor")
    _f64c(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0)
    lm = _lib.MxLMParams(int(dims[7]), int(dims[8]), float(params[1]), float(params[2]), float(params[3]),
                         float(params[4]), float(params[5]), float(params[6]), int(dims[9]), 0)
    return _lib.MxProblem(int(dims[0]), int(dims[1]), int(dims[2]), int(dims[3]), int(dims[4]), int(dims[5]),
                          int(dims[6]), float(params[0]), _ptr(Vt), _ptr(Qw), _ptr(Qo), _ptr(sqrtw),
                          _ptr(xi), _ptr(D), _ptr(delta), _ptr(alpha), _ptr(v0), lm, _ptr(vt_index), int(dims[10]))


def _project_data(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0, vt_index, dims, params, G, gt, c0):
    p = problem_struct(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0, vt_index, dims, params)
    _f64c(G, gt, c0)
    with torch.cuda.device(G.device):
        _lib.check(_lib.load().mx_project_data(ctypes.byref(p), _ptr(G), int(G.shape[0]), _ptr(gt), _ptr(c0),
                                               _stream(G)), "mx_project_data")


def _alpha_sweep(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0, vt_index, dims, params, gt, c0, v, A, chi2, S, Q, logp,
                 n_iter, n_qeval, n_solve, status, n_trial, n_batch, phase_cycles, workspace):
    p = problem_struct(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0, vt_index, dims, params)
    _f64c(gt, c0, v, A, chi2, S, Q, logp)
    out = _lib.MxSweepOut(_ptr(v), _ptr(A), _ptr(chi2), _ptr(S), _ptr(Q), _ptr(logp), _ptr(n_iter), _ptr(n_qeval),
                          _ptr(n_solve), _ptr(status), _ptr(n_trial), _ptr(n_batch), _ptr(phase_cycles))
    with torch.cuda.device(gt.device):
        _lib.check(_lib.load().mx_alpha_sweep(ctypes.byref(p), _ptr(gt), _ptr(c0), int(gt.shape[0]), ctypes.byref(out),
                                              _ptr(workspace), int(workspace.numel() * workspace.element_size()),
                                              _stream(gt)), "mx_alpha_sweep")


def _analyze(alpha, chi2, S, logp, A, gamma, linefit_deg, bryan_by_integration, alpha_index, A_out, aux):
    _f64c(alpha, chi2, S, logp, A, A_out, aux)
    B, n_alpha = int(chi2.shape[0]), int(chi2.shape[1])
    n_omega = int(A.shape[2]) if A is not None else 0
    with torch.cuda.device(chi2.device):
        _lib.check(_lib.load().mx_analyze(_ptr(alpha), _ptr(chi2), _ptr(S), _ptr(logp), _ptr(A), B, n_alpha, n_omega,
                                          float(gamma), int(linefit_deg), int(bool(bryan_by_integration)),
                                          _ptr(alpha_index), _ptr(A_out), _ptr(aux), _stream(chi2)), "mx_analyze")


def _poorman_models(A_out, slot, rows, delta, d_add, A_init, Vp, group, D, v0, ok):
    """``rows`` [P, 2] and ``group`` [P] are HOST tensors: every index the kernel dereferences is checked here before
    they are uploaded (rows within the R spectra of A_out[R, 5, n_omega], group within the G buffers of
    Vp[G, n_omega, n_sv]), so the check needs nothing back from the device."""
    _f64c(A_out, delta, A_init, Vp, D, v0)
    for t in (rows, group, ok):
        if t is not None and (t.dtype != torch.int32 or not t.is_contiguous()):
            raise ValueError("rows, group and ok must be contiguous int32 tensors")
    if rows.is_cuda or (group is not None and group.is_cuda):
        raise ValueError("rows and group must be host tensors (their bounds are checked before the upload)")
    if A_out.dim() != 3 or A_out.shape[1] != _lib.N_ANALYZERS or not 0 <= int(slot) < _lib.N_ANALYZERS:
        raise ValueError("A_out must be [R, %d, n_omega] and slot an analyzer index" % _lib.N_ANALYZERS)
    R, n_omega = int(A_out.shape[0]), int(A_out.shape[2])
    if Vp.dim() == 2:
        Vp = Vp[None]
    G, n_sv = int(Vp.shape[0]), int(Vp.shape[2])
    P = int(rows.shape[0])
    ldD = (n_omega + 1) & ~1
    if rows.shape != (P, 2) or Vp.shape[1] != n_omega or delta.numel() != n_omega:
        raise ValueError("rows must be [P, 2], Vp [G, n_omega, n_sv] and delta [n_omega]")
    if A_init is not None and A_init.numel() != n_omega:
        raise ValueError("A_init must have n_omega points")
    if D.shape != (P, ldD) or v0.shape != (P, n_sv) or ok.shape != (P,):
        raise ValueError("D must be [P, %d] (n_omega rounded up to even), v0 [P, n_sv], ok [P]" % ldD)
    if (group is None and G != 1) or (group is not None and group.shape != (P,)):
        raise ValueError("group must be [P] (or None with a single V' buffer)")
    if P == 0:
        return
    if int(rows.min()) < 0 or int(rows.max()) >= R or (group is not None and (int(group.min()) < 0 or int(group.max()) >= G)):
        raise ValueError("rows must lie in [0, %d) and group in [0, %d)" % (R, G))
    rows = rows.to(A_out.device, non_blocking=True)
    group = None if group is None else group.to(A_out.device, non_blocking=True)
    with torch.cuda.device(A_out.device):
        _lib.check(_lib.load().mx_poorman_models(_ptr(A_out), int(slot), _ptr(rows), P, _ptr(delta), float(d_add),
                                                 _ptr(A_init), _ptr(Vp), _ptr(group), n_omega, n_sv,
                                                 _ptr(D), _ptr(v0), _ptr(ok), _stream(A_out)), "mx_poorman_models")


def _vector(t, n, what):
    if t.dtype != torch.float64 or not t.is_contiguous() or t.shape != (n,):
        raise ValueError("%s must be a contiguous float64 tensor of shape (%d,)" % (what, n))


def _eta(eta):
    if not (math.isfinite(eta) and eta > 0.0):
        raise ValueError("eta must be a finite number > 0, got %r" % (eta,))


def check_hilbert_table(omega, w, eta, M):
    """Every size mx_hilbert_table uses, checked before the launch: omega[n_omega >= 2], w[n_w] contiguous float64,
    M complex128 [n_w, n_omega] contiguous, eta > 0.  Returns (n_omega, n_w).  (That omega increases strictly is the
    caller's guarantee: real_frequency checks it on the host mesh.)"""
    n_omega, n_w = int(omega.numel()), int(w.numel())
    if n_omega < 2:
        raise ValueError("the omega mesh needs at least two points")
    _vector(omega, n_omega, "omega")
    _vector(w, n_w, "w")
    _eta(eta)
    if M.dtype != torch.complex128 or not M.is_contiguous() or M.shape != (n_w, n_omega):
        raise ValueError("M must be a contiguous complex128 tensor of shape (%d, %d)" % (n_w, n_omega))
    if len({t.device for t in (omega, w, M)}) != 1:
        raise ValueError("omega, w and M must be on one device")
    return n_omega, n_w


def check_hilbert_apply(A, M, w, eta, mode, scale, shift, out):
    """Every index and size mx_hilbert_apply uses, checked before the launch.  A is [R, n_omega] float64 with unit column
    stride and any row stride lda >= n_omega (e.g. A_out[:, slot] of an analyzer output [B, 5, n_omega], read in place);
    torch keeps every view inside its storage.  M complex128 [n_w, n_omega], w float64 [n_w], scale and shift
    float64 [R] or None, out complex128 [R, n_w], all contiguous and on A's device; mode 0 / 1 / 2, eta > 0.
    Returns (lda, R, n_omega, n_w)."""
    if A.dtype != torch.float64 or A.dim() != 2 or (A.shape[1] > 1 and A.stride(1) != 1):
        raise ValueError("A must be a float64 matrix [R, n_omega] with contiguous rows")
    R, n_omega = int(A.shape[0]), int(A.shape[1])
    if n_omega < 1:
        raise ValueError("A has no omega points")
    lda = int(A.stride(0)) if R > 1 else max(int(A.stride(0)), n_omega)
    if lda < n_omega:
        raise ValueError("the rows of A overlap (row stride %d < n_omega %d)" % (lda, n_omega))
    if M.dtype != torch.complex128 or not M.is_contiguous() or M.dim() != 2 or int(M.shape[1]) != n_omega:
        raise ValueError("M must be a contiguous complex128 tensor [n_w, %d]" % n_omega)
    n_w = int(M.shape[0])
    if n_w < 1:
        raise ValueError("M has no frequencies")
    _vector(w, n_w, "w")
    _eta(eta)
    if int(mode) not in (0, 1, 2):
        raise ValueError("mode must be 0 (G), 1 (scale G + shift) or 2 (z + shift - 1/G)")
    for t, what in ((scale, "scale"), (shift, "shift")):
        if t is not None:
            _vector(t, R, what)
    if out.dtype != torch.complex128 or not out.is_contiguous() or out.shape != (R, n_w):
        raise ValueError("out must be a contiguous complex128 tensor of shape (%d, %d)" % (R, n_w))
    if len({t.device for t in (A, M, w, scale, shift, out) if t is not None}) != 1:
        raise ValueError("the tensors of hilbert_apply must be on one device")
    return lda, R, n_omega, n_w


def _hilbert_table(omega, w, eta, M):
    n_omega, n_w = check_hilbert_table(omega, w, eta, M)
    with torch.cuda.device(M.device):
        _lib.check(_lib.load().mx_hilbert_table(_ptr(omega), n_omega, _ptr(w), n_w, float(eta), _ptr(M), _stream(M)),
                   "mx_hilbert_table")


def _hilbert_apply(A, M, w, eta, mode, scale, shift, out):
    lda, R, n_omega, n_w = check_hilbert_apply(A, M, w, eta, mode, scale, shift, out)
    if R == 0:
        return
    with torch.cuda.device(out.device):
        _lib.check(_lib.load().mx_hilbert_apply(_ptr(A), lda, R, _ptr(M), n_omega, n_w, _ptr(w), float(eta), int(mode),
                                                _ptr(scale), _ptr(shift), _ptr(out), _stream(out)), "mx_hilbert_apply")


def check_matrix_resolvent(X, z, C, mode, Y):
    """Every size mx_matrix_resolvent uses, checked before the launch: X complex128 [B, M, M, n_z] contiguous with
    1 <= M <= MX_MAX_MATRIX, z complex128 [n_z] contiguous, C float64 [B] contiguous or None, Y like X (Y may be X itself,
    but may not overlap it otherwise), all on one device; mode 0 ((z + C) 1 - X)^-1 or 1 (z + C) 1 - X^-1.
    Returns (B, M, n_z)."""
    if X.dtype != torch.complex128 or X.dim() != 4 or not X.is_contiguous():
        raise ValueError("X must be a contiguous complex128 tensor [B, M, M, n_z]")
    B, M, n_z = int(X.shape[0]), int(X.shape[1]), int(X.shape[3])
    if int(X.shape[2]) != M:
        raise ValueError("X must hold square matrices [B, M, M, n_z], got %s" % (tuple(X.shape),))
    if not 1 <= M <= _lib.MX_MAX_MATRIX:
        raise ValueError("the matrices must be M x M with 1 <= M <= %d, got M = %d" % (_lib.MX_MAX_MATRIX, M))
    if z.dtype != torch.complex128 or not z.is_contiguous() or z.shape != (n_z,):
        raise ValueError("z must be a contiguous complex128 tensor of shape (%d,)" % n_z)
    if C is not None:
        _vector(C, B, "C")
    if int(mode) not in (0, 1):
        raise ValueError("mode must be 0 (((z + C) 1 - X)^-1) or 1 ((z + C) 1 - X^-1)")
    if Y.dtype != torch.complex128 or not Y.is_contiguous() or Y.shape != X.shape:
        raise ValueError("Y must be a contiguous complex128 tensor of shape %s" % (tuple(X.shape),))
    if len({t.device for t in (X, z, C, Y) if t is not None}) != 1:
        raise ValueError("the tensors of matrix_resolvent must be on one device")
    nbytes = X.numel() * X.element_size()
    if Y.data_ptr() != X.data_ptr() and abs(Y.data_ptr() - X.data_ptr()) < nbytes:
        raise ValueError("Y overlaps X without being X")
    return B, M, n_z


def _matrix_resolvent(X, z, C, mode, Y):
    B, M, n_z = check_matrix_resolvent(X, z, C, mode, Y)
    if B == 0 or n_z == 0:
        return
    with torch.cuda.device(Y.device):
        _lib.check(_lib.load().mx_matrix_resolvent(_ptr(X), B, M, n_z, _ptr(z), _ptr(C), int(mode), _ptr(Y), _stream(Y)),
                   "mx_matrix_resolvent")


_library.impl("project_data", _project_data, "CUDA")
_library.impl("alpha_sweep", _alpha_sweep, "CUDA")
_library.impl("analyze", _analyze, "CUDA")
_library.impl("poorman_models", _poorman_models, "CUDA")
_library.impl("hilbert_table", _hilbert_table, "CUDA")
_library.impl("hilbert_apply", _hilbert_apply, "CUDA")
_library.impl("matrix_resolvent", _matrix_resolvent, "CUDA")

project_data = torch.ops.maxent_b200.project_data
alpha_sweep = torch.ops.maxent_b200.alpha_sweep
analyze = torch.ops.maxent_b200.analyze
poorman_models = torch.ops.maxent_b200.poorman_models
hilbert_table = torch.ops.maxent_b200.hilbert_table
hilbert_apply = torch.ops.maxent_b200.hilbert_apply
matrix_resolvent = torch.ops.maxent_b200.matrix_resolvent
OPERATORS = ("project_data", "alpha_sweep", "analyze", "poorman_models", "hilbert_table", "hilbert_apply",
             "matrix_resolvent")
