"""PyTorch custom operators over the C ABI (include/maxent_b200.h).

    torch.ops.maxent_b200.project_data    -> mx_project_data
    torch.ops.maxent_b200.alpha_sweep     -> mx_alpha_sweep
    torch.ops.maxent_b200.analyze         -> mx_analyze
    torch.ops.maxent_b200.poorman_models  -> mx_poorman_models

The operators are registered for the CUDA dispatch key ONLY: calling one with host tensors raises
``NotImplementedError`` from the dispatcher -- there is no CPU implementation of the hot path.  They are thin:
every operator packs its tensor arguments into the plain-pointer structs of the ABI, takes the current stream
of the tensors' device and calls the shared library; outputs are caller-allocated tensors the operator writes
(``Tensor(a!)`` in the schema), so nothing is allocated and nothing synchronises inside an operator.

Reference seam these replace: the body of MaxEntLoop.run (python/maxent_loop.py:205-302) and
MaxEntResult.analyze (python/maxent_result.py:795-818).
"""
import ctypes

import torch

from . import _lib

# dims  = [n_tau, n_omega, n_sv, n_alpha, variant, want_probability, engine, per_spectrum_model, maxiter, miniter,
#          marquardt, vt_stride]
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
    if len(dims) != 12 or len(params) != 7:
        raise ValueError("dims must hold 12 integers and params 7 floats (see maxent_b200/ops.py)")
    if vt_index is not None and (vt_index.dtype != torch.int32 or not vt_index.is_contiguous()):
        raise ValueError("vt_index must be a contiguous int32 tensor")
    _f64c(Vt, Qw, Qo, sqrtw, xi, D, delta, alpha, v0)
    lm = _lib.MxLMParams(int(dims[8]), int(dims[9]), float(params[1]), float(params[2]), float(params[3]),
                         float(params[4]), float(params[5]), float(params[6]), int(dims[10]), 0)
    return _lib.MxProblem(int(dims[0]), int(dims[1]), int(dims[2]), int(dims[3]), int(dims[4]), int(dims[5]),
                          int(dims[6]), int(dims[7]), float(params[0]), _ptr(Vt), _ptr(Qw), _ptr(Qo), _ptr(sqrtw),
                          _ptr(xi), _ptr(D), _ptr(delta), _ptr(alpha), _ptr(v0), lm, _ptr(vt_index), int(dims[11]))


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


_library.impl("project_data", _project_data, "CUDA")
_library.impl("alpha_sweep", _alpha_sweep, "CUDA")
_library.impl("analyze", _analyze, "CUDA")
_library.impl("poorman_models", _poorman_models, "CUDA")

project_data = torch.ops.maxent_b200.project_data
alpha_sweep = torch.ops.maxent_b200.alpha_sweep
analyze = torch.ops.maxent_b200.analyze
poorman_models = torch.ops.maxent_b200.poorman_models
OPERATORS = ("project_data", "alpha_sweep", "analyze", "poorman_models")
