"""Host-side logic of the drop-in interface (no GPU, no compute calls): export surface, attribute
forwarding, descriptor -> kernel-variant mapping, result assembly, log formatting.  Modelled on the
reference's own host-level tests (test/python/logtaker.py, matrix_maxent_result.py, pickle_maxent_result.py,
elementwise_set_G.py, alpha_meshes.py, omega_meshes.py)."""
import io
import pickle
from contextlib import redirect_stdout

import numpy as np
import pytest

import maxent_b200 as mb
from maxent_b200 import _lib

# SURVEY.md Appendix C: what ``from triqs_maxent import *`` gives and the hot path needs
EXPORTS = """BaseAlphaMesh DataAlphaMesh LinearAlphaMesh LogAlphaMesh Analyzer AnalyzerResult BryanAnalyzer
Chi2CurvatureAnalyzer ClassicAnalyzer EntropyAnalyzer LineFitAnalyzer BryanCostFunction MaxEntCostFunction
BaseDefaultModel DataDefaultModel FileDefaultModel FlatDefaultModel CallableMethodCheck DiagonalMaxEnt
ElementwiseMaxEnt PoormanMaxEnt AbsoluteEntropy CachedFunction Chi2 ComplexChi2 ComplexPlusMinusEntropy
ComplexPlusMinusH_of_v DoublyDerivableFunction Entropy GenericA_of_H GenericFunction GenericH_of_v IdentityA_of_H
IdentityH_of_v InvertibleFunction NoExpH_of_v NormalChi2 NormalEntropy NormalH_of_v NullFunction PlusMinusEntropy
PlusMinusH_of_v PreblurA_of_H ShiftedAbsoluteEntropy cached safelog view_complex view_real DataKernel IOmegaKernel
Kernel KernelSVD PreblurKernel TauKernel Logtaker VerbosityFlags MaxEntLoop MaxEntResult MaxEntResultData
LevenbergMinimizer ConvergenceMethod AndConvergenceMethod OrConvergenceMethod MaxDerivativeConvergenceMethod
NullConvergenceMethod FunctionChangeConvergenceMethod RelativeFunctionChangeConvergenceMethod BaseOmegaMesh
DataOmegaMesh HyperbolicOmegaMesh LinearOmegaMesh LorentzianOmegaMesh LorentzianSmallerOmegaMesh
NormalLogProbability TauMaxEnt get_preblur check_der numder get_G_tau_from_A_w get_G_w_from_A_w SigmaContinuator
DirectSigmaContinuator InversionSigmaContinuator if_no_triqs if_triqs_1 if_triqs_2 require_triqs
assert_text_files_equal show_version show_git_hash""".split()


def test_export_surface():
    missing = [n for n in EXPORTS if not hasattr(mb, n)]
    assert not missing, missing


def test_logtaker_masks_and_format():
    """test/python/logtaker.py: which message shows under which verbosity mask."""
    F = mb.VerbosityFlags
    masks = [F.Quiet, F.Header, F.ElementInfo, F.Timing, F.AlphaLoop, F.SolverDetails, F.Errors,
             F.Header | F.Timing, F.Default]
    buf = io.StringIO()
    with redirect_stdout(buf):
        log = mb.Logtaker()
        for i, m in enumerate(masks):
            log.verbose = m
            log.message(F.Quiet, "=== Test #{} ===", i)
            log.message(F.Header, "header")
            log.message(F.ElementInfo, "element")
            log.message(F.Timing, "timing")
            log.message(F.AlphaLoop, "alpha")
            log.message(F.SolverDetails, "solver")
            log.error_message("oops {}", 3)
            log.message(F.Timing | F.Header, "header+timing")
    # solver details rewrite the line ("\r" prefix, no newline): normalise before comparing
    text = buf.getvalue().replace("\r", "").replace("solver\n", "solver").replace("solver", "solver\n")
    blocks = [b.strip().splitlines()[1:] for b in text.split("=== Test")[1:]]
    assert blocks[0] == []
    assert blocks[1] == ["header"] and blocks[2] == ["element"] and blocks[3] == ["timing"] and blocks[4] == ["alpha"]
    assert blocks[5] == ["solver"] and blocks[6] == ["ERROR: oops 3"]
    assert blocks[7] == ["header", "timing", "header+timing"]
    assert blocks[8] == ["header", "element", "timing", "alpha", "ERROR: oops 3", "header+timing"]
    assert log.get_error_messages() == ["oops 3"] * 9
    with pytest.raises(NotImplementedError):
        log.verbosity_message("x")


def test_convergence_trees_map_to_device_thresholds():
    m = mb.LevenbergMinimizer()
    p = m.lm_params()
    assert (p.maxiter, p.miniter, p.mu0, p.nu, p.max_mu) == (1000, 0, 1e-18, 1.3, 1e20)
    assert (p.conv_max_derivative, p.conv_rel_change) == (1e-4, 1e-16)
    tree = mb.MaxDerivativeConvergenceMethod(1e-6) & mb.RelativeFunctionChangeConvergenceMethod(1e-12)
    assert isinstance(tree, mb.AndConvergenceMethod) and tree.thresholds() == (1e-6, 1e-12, -1.0)
    assert mb.MaxDerivativeConvergenceMethod(1e-3).thresholds() == (1e-3, -1.0, -1.0)
    assert (mb.NullConvergenceMethod() | mb.MaxDerivativeConvergenceMethod(1.0)).thresholds()[0] == np.inf
    q = mb.LevenbergMinimizer(convergence=mb.FunctionChangeConvergenceMethod(1e-3) | mb.MaxDerivativeConvergenceMethod(1e-5),
                              marquardt=True).lm_params()
    assert (q.conv_max_derivative, q.conv_rel_change, q.conv_abs_change, q.marquardt) == (1e-5, -1.0, 1e-3, True)
    assert q.c_struct().marquardt == 1 and q.c_struct().conv_abs_change == 1e-3
    assert p.c_struct().marquardt == 0 and p.c_struct().conv_abs_change == -1.0
    with pytest.raises(NotImplementedError):
        mb.LevenbergMinimizer(J_squared=True).lm_params()
    with pytest.raises(Exception):
        mb.LevenbergMinimizer(nu=1.0).lm_params()          # levenberg_minimizer.py:139-140
    c = p.c_struct()
    assert isinstance(c, _lib.MxLMParams) and c.maxiter == 1000


def test_cost_function_variants():
    assert mb.MaxEntCostFunction().variant() == "normal"
    assert mb.MaxEntLoop(cost_function='plusminus').cost_function.variant() == "plusminus"
    assert mb.MaxEntLoop(cost_function='bryan').cost_function.variant() == "bryan"
    with pytest.raises(Exception):
        mb.MaxEntLoop(cost_function='nonsense')
    for bad in (mb.MaxEntCostFunction(d_dv=True), mb.MaxEntCostFunction(dA_projection=1),
                mb.MaxEntCostFunction(S=mb.PlusMinusEntropy()), mb.BryanCostFunction(S=mb.PlusMinusEntropy(),
                                                                                   H_of_v=mb.PlusMinusH_of_v())):
        with pytest.raises(NotImplementedError):
            bad.variant()
    for cls in (mb.ComplexPlusMinusEntropy, mb.NoExpH_of_v, mb.ComplexPlusMinusH_of_v):
        with pytest.raises(NotImplementedError):
            cls()
    # Matsubara kernel and complex misfit: host objects as in the reference (python/kernels.py:283-346), real A on the fused path
    om_iw = mb.HyperbolicOmegaMesh(-5, 5, 30)
    iw = (2 * np.arange(16) + 1) * np.pi / 10.0
    Kiw = mb.IOmegaKernel(iw, om_iw, beta=10.0)
    np.testing.assert_allclose(Kiw.K, 1.0 / (1j * iw[:, None] - np.asarray(om_iw)[None, :]), rtol=1e-15)
    np.testing.assert_allclose(Kiw.K_delta, Kiw.K * om_iw.delta[None, :], rtol=1e-15)
    assert Kiw.fused_matrix().shape == (32, 30) and np.all(Kiw.fused_matrix()[16:] == Kiw.K.imag)
    np.testing.assert_array_equal(Kiw.stack(np.array([1 + 2j, 3 - 1j])), [1, 3, 2, -1])
    assert mb.MaxEntCostFunction(chi2=mb.ComplexChi2(K=Kiw)).variant() == "normal"
    with pytest.raises(NotImplementedError):
        Kiw.transform(np.eye(16))
    om = mb.HyperbolicOmegaMesh(-5, 5, 40)
    pre = mb.PreblurA_of_H(b=0.3, omega=om)
    assert mb.MaxEntCostFunction(A_of_H=pre).variant() == "normal"
    B = mb.get_preblur(om, 0.3)
    np.testing.assert_allclose(B @ om.delta, np.ones(40), rtol=1e-12)            # exact after the second normalisation
    np.testing.assert_allclose((om.delta @ B)[5:-5], np.ones(30), rtol=1e-2)     # approximate for the first
    pre.b = 0.5
    assert not np.allclose(pre._B, B)
    with pytest.raises(NotImplementedError):
        mb.MaxEntCostFunction()(np.zeros(3))                # no host evaluation of Q(v)


def test_loop_defaults_and_forwarding():
    ml = mb.MaxEntLoop()
    assert [a.name for a in ml.analyzers] == ['LineFitAnalyzer', 'Chi2CurvatureAnalyzer', 'EntropyAnalyzer']
    assert isinstance(ml.alpha_mesh, mb.LogAlphaMesh) and len(ml.alpha_mesh) == 20
    assert ml.reduce_singular_space == 1e-14 and ml.G_threshold == 1e-10 and ml.scale_alpha == 'Ndata'
    mp = mb.MaxEntLoop(probability='normal')
    assert isinstance(mp.probability, mb.NormalLogProbability)
    assert [a.name for a in mp.analyzers][3:] == ['BryanAnalyzer', 'ClassicAnalyzer']
    omega = mb.LinearOmegaMesh(-2, 2, 7)
    K = mb.DataKernel(np.arange(5.0), omega, np.random.RandomState(0).rand(5, 7))
    ml.K = K
    ml.D = mb.FlatDefaultModel(omega)
    ml.G = np.ones(5)
    ml.err = 0.1 * np.ones(5)
    assert ml.cost_function.chi2.K is K and ml.cost_function.H_of_v.K is K and ml.K is K
    assert ml.cost_function.S.D is ml.D and ml.cost_function.H_of_v.D is ml.D
    assert ml.omega is omega and np.all(ml.data_variable == np.arange(5.0))
    np.testing.assert_allclose(K.K_delta, K.K * omega.delta[None, :])
    ml.check_consistency()
    ml.G = np.ones(4)
    with pytest.raises(AssertionError):
        ml.check_consistency()


def test_tau_maxent_attribute_shadowing_without_touching_the_device():
    tm = mb.TauMaxEnt()
    assert tm.maxent_loop.omega is tm.omega and len(tm.omega) == 100
    tau = np.linspace(0, 10, 21)
    tm.set_G_tau_data(tau, -0.5 * np.ones(21))
    tm.set_error(1e-3)
    assert np.all(tm.tau == tau) and np.all(tm.maxent_loop.data_variable == tau)
    assert np.all(tm.err == 1e-3) and tm.err.shape == (21,)
    assert np.all(tm.cost_function.G_orig == tm.G)
    tm.alpha_mesh = mb.LogAlphaMesh(0.1, 10, 4)
    assert tm.maxent_loop.alpha_mesh is tm.alpha_mesh
    tm.omega = mb.HyperbolicOmegaMesh(-5, 5, 30)
    assert len(tm.K.omega) == 30 and len(tm.D.D) == 30 and len(tm.cost_function.A_of_H.omega) == 30
    assert tm.K._dirty                                  # values are produced on the device at first use
    with pytest.raises(Exception):
        tm.set_error(np.ones(5))
    with pytest.raises(Exception):
        tm.set_error(1j)
    with pytest.raises(AssertionError):
        tm.set_G_tau_data(tau, np.ones(3))
    with pytest.raises(NotImplementedError):
        tm.set_G_iw(None)


def test_elementwise_setters():
    """test/python/elementwise_set_G.py: the element loaders and the error plumbing."""
    ew = mb.ElementwiseMaxEnt(use_hermiticity=True)
    tau = np.linspace(0, 5, 11)
    G = np.random.RandomState(1).rand(2, 2, 11)
    ew.set_G_tau_data(tau, G)
    assert ew.shape == (2, 2)
    ew.set_G_element(ew.maxent_offdiagonal, ew.G_mat, (0, 1), True)
    np.testing.assert_array_equal(ew.maxent_offdiagonal.G, G[0, 1])
    ew.set_error(0.01)
    assert ew.get_error((0, 1)) == 0.01
    ew.set_error(np.full(11, 0.02))
    assert ew.get_error((1, 0)).shape == (11,)
    e3 = np.random.RandomState(2).rand(2, 2, 11)
    ew.set_error(e3)
    np.testing.assert_array_equal(ew.get_error((1, 0)), e3[1, 0])
    ew.alpha_mesh = mb.LogAlphaMesh(0.5, 50, 6)
    assert len(ew.maxent_diagonal.alpha_mesh) == 6 and len(ew.maxent_offdiagonal.alpha_mesh) == 6
    assert len(ew.alpha_mesh) == 6
    with pytest.raises(Exception):
        ew.G                                               # differs between the two workers
    assert ew.maxent_diagonal.cost_function.variant() == "normal"
    assert ew.maxent_offdiagonal.cost_function.variant() == "plusminus"
    ew.prepare_maxent_result()
    assert ew.maxent_result.matrix_structure == (2, 2) and ew.maxent_result.element_wise
    with pytest.raises(TypeError):
        mb.DiagonalMaxEnt().run_offdiagonal()


def _record(n_alpha, n_om, n_sv, seed):
    r = np.random.RandomState(seed)
    return dict(alpha=np.logspace(2, 0, n_alpha), v=r.rand(n_alpha, n_sv), chi2=r.rand(n_alpha), S=-r.rand(n_alpha),
                Q=r.rand(n_alpha), A=r.rand(n_alpha, n_om), H=r.rand(n_alpha, n_om), probability=np.full(n_alpha, np.nan),
                omega=mb.LinearOmegaMesh(-1, 1, n_om), G=r.rand(9), G_orig=r.rand(9), data_variable=np.arange(9.0),
                G_rec=r.rand(n_alpha, 9), n_iter=np.arange(n_alpha), converged=np.ones(n_alpha, bool))


def test_matrix_result_shapes_and_hermiticity():
    """test/python/matrix_maxent_result.py: shapes of the assembled arrays, NaN padding, hermiticity fill."""
    res = mb.MaxEntResult(matrix_structure=(2, 2), element_wise=True, use_hermiticity=True)
    res.add_sweep(_record(6, 5, 4, 0), matrix_element=(0, 0))
    res.add_sweep(_record(6, 5, 3, 1), matrix_element=(0, 1))
    assert res.alpha.shape == (6,) and res.chi2.shape == (2, 2, 6) and res.A.shape == (2, 2, 6, 5)
    assert res.v.shape == (2, 2, 6, 4) and np.all(np.isnan(res.v[0, 1, :, 3])) and not np.any(np.isnan(res.v[0, 0]))
    assert np.all(np.isnan(res.chi2[1, 1])) and np.all(np.isnan(res.chi2[1, 0]))
    np.testing.assert_array_equal(res.A[1, 0], res.A[0, 1])          # filled from the transposed element
    assert np.all(np.isnan(res.A[1, 1]))
    assert res.G.shape == (2, 2, 9) and res.G_rec.shape == (2, 2, 6, 9)
    assert res.matrix_structure == (2, 2) and res.effective_matrix_structure == (2, 2)
    # A_out: computed / hermitian partner / zero element / missing
    res._results_from_analyzers[0][0]['LineFitAnalyzer'] = mb.AnalyzerResult(A_out=np.ones(5), name='LineFitAnalyzer')
    res._results_from_analyzers[0][1]['LineFitAnalyzer'] = mb.AnalyzerResult(A_out=2 * np.ones(5), name='LineFitAnalyzer')
    res.zero_elements.append((1, 1))
    A_out = res.A_out
    assert A_out.shape == (2, 2, 5)
    assert np.all(A_out[0, 0] == 1) and np.all(A_out[0, 1] == 2) and np.all(A_out[1, 0] == 2) and np.all(A_out[1, 1] == 0)
    # complex elements: extra axis of length 2, conjugation on the lower triangle
    rc = mb.MaxEntResult(matrix_structure=(2, 2), complex_elements=True)
    rc.add_sweep(_record(4, 5, 3, 2), matrix_element=(0, 1), complex_index=0)
    rc.add_sweep(_record(4, 5, 3, 3), matrix_element=(0, 1), complex_index=1)
    assert rc.effective_matrix_structure == (2, 2, 2) and rc.A.shape == (2, 2, 2, 4, 5)
    np.testing.assert_array_equal(rc.A[1, 0, 0], rc.A[0, 1, 0])
    np.testing.assert_array_equal(rc.A[1, 0, 1], -rc.A[0, 1, 1])


def test_result_data_twin_and_pickle():
    """test/python/pickle_maxent_result.py: result.data keeps the arrays; pickle round trip."""
    res = mb.MaxEntResult()
    rec = _record(5, 4, 3, 7)
    res.add_sweep(rec)
    res._results_from_analyzers['LineFitAnalyzer'] = mb.AnalyzerResult(A_out=rec['A'][2], alpha_index=2,
                                                                       name='LineFitAnalyzer', info='x')
    res._default_analyzer_name = 'LineFitAnalyzer'
    np.testing.assert_array_equal(res.A_out, rec['A'][2])
    data = res.data
    assert type(data) is mb.MaxEntResultData
    for f in ('alpha', 'chi2', 'S', 'Q', 'A', 'H', 'v', 'G', 'G_rec', 'omega'):
        np.testing.assert_array_equal(getattr(data, f), getattr(res, f))
    assert isinstance(data.omega, mb.DataOmegaMesh) and isinstance(data.alpha, mb.DataAlphaMesh)
    np.testing.assert_array_equal(data.A_out, res.A_out)
    assert data.analyzer_results['LineFitAnalyzer'].maxent_result is data
    again = pickle.loads(pickle.dumps(data))
    np.testing.assert_array_equal(again.chi2, res.chi2)
    np.testing.assert_array_equal(again.get_A_out('LineFitAnalyzer'), res.A_out)
    res.exclude(['A', 'H'])
    small = res.data
    assert not hasattr(small, 'A') and hasattr(small, 'chi2')
    with pytest.raises(AttributeError):
        res.include(['nonsense'])
    # add_result: alpha by alpha
    class Sol(object):
        pass
    r2 = mb.MaxEntResult()
    for i in range(3):
        s = Sol()
        for name in ('alpha', 'v', 'chi2', 'S', 'Q', 'H', 'A', 'G_rec'):
            setattr(s, name, rec[name][i])
        for name in ('omega', 'G', 'G_orig', 'data_variable'):
            setattr(s, name, rec[name])
        r2.add_result(s, log_probability=None if i else -3.0)
    np.testing.assert_array_equal(r2.chi2, rec['chi2'][:3])
    assert r2.probability[0] == -3.0 and np.isnan(r2.probability[1])
    # plot data providers (python/maxent_result.py:468-582): (x, y, options) tuples
    x, y, opt = res.plot_A(alpha_index=2)
    np.testing.assert_array_equal(x, res.omega)
    np.testing.assert_array_equal(y, res.A[2])
    assert opt['n_alpha_index'] == 5 and opt['x_label'] == r'$\omega$' and not opt['log_x']
    x, y, opt = res.plot_G()
    np.testing.assert_array_equal(x, res.data_variable)
    np.testing.assert_array_equal(y, res.G_orig)
    curves = res.plot_G_rec(alpha_index=1)
    assert len(curves) == 2 and curves[1][2]['plot_G'] is True
    np.testing.assert_array_equal(curves[1][1], res.G_rec[1])
    assert len(res.plot_G_rec(alpha_index=1, plot_G=False)) == 1


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry refuses loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    tm = mb.TauMaxEnt()
    tm.set_G_tau_data(np.linspace(0, 10, 21), -0.5 * np.ones(21))
    tm.set_error(1e-3)
    with pytest.raises(_lib.MaxEntLibraryError):
        tm.run()
    with pytest.raises(_lib.MaxEntLibraryError):
        mb.TauKernel(np.linspace(0, 1, 5), mb.LinearOmegaMesh(-1, 1, 5)).K
    with pytest.raises(_lib.MaxEntLibraryError):
        mb.LineFitAnalyzer().analyze(_mock_result())


def _mock_result():
    res = mb.MaxEntResult()
    res.add_sweep(_record(8, 4, 3, 5))
    return res


def test_file_setters(tmp_path):
    """set_G_tau_file / set_cov_file read text files like the reference (python/tau_maxent.py:198-225,290-301)."""
    tau = np.linspace(0, 4, 9)
    G = -np.exp(-tau)
    err = 0.01 * (1 + tau)
    f = tmp_path / "g.dat"
    np.savetxt(str(f), np.column_stack([tau, G, err]))
    tm = mb.TauMaxEnt()
    tm.set_G_tau_file(str(f), tau_col=0, G_col=1, err_col=2)
    np.testing.assert_allclose(tm.tau, tau)
    np.testing.assert_allclose(tm.G, G)
    np.testing.assert_allclose(tm.err, err)
    tm2 = mb.TauMaxEnt()
    tm2.set_G_tau_file(str(f))
    assert tm2.err is None and len(tm2.G) == 9
    ew = mb.ElementwiseMaxEnt()
    ew.set_G_tau_filenames([[str(f), str(f)], [str(f), str(f)]])
    assert ew.shape == (2, 2)
    ew.set_G_element(ew.maxent_diagonal, ew.G_mat, (1, 1), True)
    np.testing.assert_allclose(ew.maxent_diagonal.G, G)
    ew.set_G_tau_filename_pattern(str(tmp_path / "g_{i}_{j}.dat"), (3, 3))
    assert ew.shape == (3, 3)


def test_batched_front_end_accepts_a_levenberg_minimizer():
    """BatchedTauMaxEnt(minimizer=...) takes the same LevenbergMinimizer object MaxEntLoop does."""
    import maxent_b200 as mb
    from maxent_b200 import engine
    job = mb.BatchedTauMaxEnt(minimizer=mb.LevenbergMinimizer(marquardt=True, maxiter=77))
    assert isinstance(job.minimizer, engine.LMParams) and job.minimizer.marquardt and job.minimizer.maxiter == 77
    assert isinstance(mb.BatchedTauMaxEnt().minimizer, engine.LMParams)
    assert isinstance(mb.BatchedTauMaxEnt(minimizer=engine.LMParams(nu=1.5)).minimizer, engine.LMParams)


def test_batched_whitening_groups_are_planned_on_the_whole_batch(monkeypatch):
    """BatchedTauMaxEnt numbers the whitening groups of err[B, n_tau] in the sorted order of the vectors, those of
    cov[B, n, n] in the order of first appearance and those of set_error_groups as given.  A run that leaves a spectrum
    below G_threshold out of the launch keeps the groups of the whole batch, so the next run of the same job gives every
    spectrum its own error vector again.  SharedProblem and run_sweep are replaced by recorders: no device is used."""
    import torch
    import maxent_b200 as mb
    from maxent_b200 import batched, engine
    n_tau = 4
    job = mb.BatchedTauMaxEnt(scale_alpha=None)
    job.set_G_tau_data(np.linspace(0, 1, n_tau), np.ones((1, n_tau)))
    vec = np.array([3e-3, 1e-3, 2e-3])
    which = np.array([0, 1, 2, 1])
    job.set_error(np.repeat(vec[which][:, None], n_tau, axis=1))
    mode, index, specs = job._error_plan(4)
    assert mode == "groups" and index.tolist() == [2, 0, 1, 0] and [s[1][0] for s in specs] == [1e-3, 2e-3, 3e-3]
    job.set_error_groups(vec[:, None] * np.ones(n_tau), which)
    mode, index, specs = job._error_plan(4)
    assert mode == "groups" and index.tolist() == which.tolist() and [s[1][0] for s in specs] == vec.tolist()
    C = [np.diag(np.full(n_tau, c)) for c in (4.0, 1.0, 9.0)]
    job.set_cov(np.stack([C[k] for k in which]))
    mode, index, specs = job._error_plan(4)
    assert mode == "groups" and index.tolist() == which.tolist() and [s[1][0] for s in specs] == [2.0, 1.0, 3.0]

    class Problem(object):
        def __init__(self, K, err, *args, **kwargs):
            self.err = np.atleast_1d(np.asarray(err, dtype=np.float64))
            self.n_tau, self.n_omega, self.n_sv, self.device, self.U, self.S, self.V = n_tau, 3, 2, torch.device("cpu"), 0, 0, 0

    def run_sweep(prob, G, alpha, groups=None, **kwargs):
        B, n_alpha = int(G.shape[0]), len(alpha)
        r = engine.SweepResult()
        for name in ("chi2", "S", "Q", "logp"):
            setattr(r, name, torch.zeros((B, n_alpha), dtype=torch.float64))
        for name in ("n_iter", "n_qeval", "n_solve", "status", "n_trial", "n_batch"):
            setattr(r, name, torch.zeros((B, n_alpha), dtype=torch.int32))
        r.alpha_index = torch.zeros((B, 5), dtype=torch.int32)
        r.A, r.A_out = torch.zeros((B, n_alpha, 3), dtype=torch.float64), torch.zeros((B, 5, 3), dtype=torch.float64)
        r.v = None
        r.alpha, r.n_sv, r.phase_cycles, r.alpha_scale = torch.as_tensor(alpha), 2, None, None
        r.problems, r.index = groups
        launched.append([r.problem(b).err[0] for b in range(B)])
        return r

    base = Problem(np.ones((n_tau, 3)), 1.0)
    monkeypatch.setattr(engine, "SharedProblem", Problem)
    monkeypatch.setattr(engine, "run_sweep", run_sweep)
    monkeypatch.setattr(batched.BatchedTauMaxEnt, "prepare", lambda self: base)
    job._K_dev, job._D_host = torch.ones((n_tau, 3), dtype=torch.float64), np.ones(3)
    job.omega, job.alpha_mesh = batched.DataOmegaMesh(np.linspace(-1, 1, 3)), [2.0, 1.0]
    job.set_error(np.repeat(vec[which][:, None], n_tau, axis=1))
    G = torch.ones((4, n_tau), dtype=torch.float64)
    G[0] = 0.0                                       # the only spectrum of its group is below G_threshold
    launched = []
    res = job.run_device(G, skip_small=True)
    assert launched == [[1e-3, 2e-3, 1e-3]]
    assert [res.problem(b).err[0] for b in (1, 2, 3)] == [1e-3, 2e-3, 1e-3]
    launched = []
    res = job.run_device(torch.ones((4, n_tau), dtype=torch.float64), skip_small=True)
    assert launched == [vec[which].tolist()]
    assert [res.problem(b).err[0] for b in range(4)] == vec[which].tolist()


def test_meshes_and_default_model_match_the_reference_exactly():
    """Tier T0 (SURVEY.md 8(c)): omega meshes with their integration weights, alpha meshes and the flat default model
    are the reference's arrays (tests/golden/g0_meshes.npz, written by oracle/make_golden.py from the real
    python/omega_meshes.py, alpha_meshes.py, default_models.py); the oracle's TauKernel agrees to 1e-15
    (test/python/tau_kernel.py:27-69).  Copies keep the mesh attributes (test/python/omega_meshes.py:62-73)."""
    import copy
    import os
    import maxent_b200 as mb
    from oracle import maxent_oracle as mo
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "g0_meshes.npz"))
    for name in ("LinearOmegaMesh", "LorentzianOmegaMesh", "LorentzianSmallerOmegaMesh", "HyperbolicOmegaMesh"):
        for (lo, hi, n) in ((-10, 10, 10), (-7.5, 12.25, 57)):
            mesh = getattr(mb, name)(omega_min=lo, omega_max=hi, n_points=n)
            key = "%s_%d" % (name, n)
            np.testing.assert_array_equal(np.asarray(mesh), g[key], err_msg=key)
            np.testing.assert_array_equal(np.asarray(mesh.delta), g[key + "_delta"], err_msg=key)
            np.testing.assert_array_equal(mb.FlatDefaultModel(omega=mesh).D, g[key + "_flatD"], err_msg=key)
            for c in (mesh.copy(), copy.deepcopy(mesh)):
                assert np.all(c == mesh) and (c.omega_min, c.omega_max, c.n_points) == (lo, hi, n)
    np.testing.assert_array_equal(np.asarray(mb.LogAlphaMesh(alpha_min=0.0001, alpha_max=20, n_points=20)), g["LogAlphaMesh"])
    np.testing.assert_array_equal(np.asarray(mb.LogAlphaMesh(0.01, 2000, 60)), g["LogAlphaMesh_60"])
    np.testing.assert_array_equal(np.asarray(mb.LinearAlphaMesh(alpha_min=0.0001, alpha_max=20, n_points=20)), g["LinearAlphaMesh"])
    # oracle side of the same tier
    np.testing.assert_array_equal(mo.hyperbolic_omega_mesh(-7.5, 12.25, 57), g["HyperbolicOmegaMesh_57"])
    np.testing.assert_array_equal(mo.omega_delta(g["HyperbolicOmegaMesh_57"]), g["HyperbolicOmegaMesh_57_delta"])
    np.testing.assert_array_equal(mo.log_alpha_mesh(0.01, 2000, 60), g["LogAlphaMesh_60"])
    K = mo.tau_kernel(g["kernel_tau"], g["kernel_omega"], 7.5)
    assert np.max(np.abs(K - g["kernel_K"])) < 1e-15
    np.testing.assert_allclose(K * mo.omega_delta(g["kernel_omega"])[None, :], g["kernel_K_delta"], rtol=0, atol=1e-15)
    # default model given on another grid, and the preblur matrix
    om = mb.DataOmegaMesh(g["kernel_omega"])
    np.testing.assert_allclose(mb.DataDefaultModel(g["ddm_default"], g["ddm_omega_in"], om).D, g["ddm_D"], rtol=1e-15, atol=0)
    np.testing.assert_allclose(mb.DataDefaultModel(np.exp(-g["kernel_omega"]**2) + 0.1, om, om).D, g["ddm_D_same_grid"],
                               rtol=1e-15, atol=0)
    np.testing.assert_allclose(mb.get_preblur(om, 0.4), g["preblur_B"], rtol=1e-14, atol=1e-300)


def test_caller_side_utilities(tmp_path, capsys):
    """numder / check_der (python/maxent_util.py:170-237), the TRIQS switches of a USE_TRIQS=OFF build
    (python/triqs_support.py.in:31-78) and the version report."""
    import maxent_b200 as mb
    x0 = np.array([[0.3, -1.2], [2.0, 0.5]])
    f = lambda x: np.sum(np.sin(x) * x)
    d = lambda x: (np.cos(x) * x + np.sin(x))[None]
    J = mb.numder(f, x0)
    assert J.shape == (1, 2, 2) and np.max(np.abs(J - d(x0))) < 1e-8
    vec = lambda x: np.array([x[0] * x[1], x[0] ** 2, np.exp(x[1])])
    Jv = mb.numder(vec, np.array([1.5, -0.5]))
    assert Jv.shape == (3, 2)
    np.testing.assert_allclose(Jv, [[-0.5, 1.5], [3.0, 0.0], [0.0, np.exp(-0.5)]], atol=1e-8)
    assert mb.check_der(f, d, x0, name="ok")
    assert not mb.check_der(f, lambda x: 1.01 * d(x), x0, name="wrong")
    assert "wrong" in capsys.readouterr().out
    assert mb.check_der(f, lambda x: (1 + 1e-10) * d(x), x0, renorm=True) and mb.check_der(f, d, x0, renorm=5.0)
    assert mb.if_no_triqs() and not mb.if_triqs_1() and not mb.if_triqs_2()
    with pytest.raises(NotImplementedError, match="only available with TRIQS"):
        mb.get_G_tau_from_A_w(np.ones(3), np.linspace(-1, 1, 3), 10.0, 11)
    with pytest.raises(NotImplementedError):
        mb.get_G_w_from_A_w(np.ones(3), np.linspace(-1, 1, 3))
    assert "TRIQS support" in mb.get_G_w_from_A_w.__doc__
    for make in (lambda: mb.SigmaContinuator(), lambda: mb.DirectSigmaContinuator(None),
                 lambda: mb.InversionSigmaContinuator(None, constant_shift=1.0)):
        with pytest.raises(NotImplementedError, match="only available with TRIQS"):
            make()
    a, b = tmp_path / "a.txt", tmp_path / "b.txt"
    a.write_text("x  \ny\n\n"); b.write_text("x\ny\n")
    mb.assert_text_files_equal(str(a), str(b))
    b.write_text("x\nz\n")
    with pytest.raises(AssertionError):
        mb.assert_text_files_equal(str(a), str(b))
    mb.show_version(); mb.show_git_hash()
    assert "maxent_b200 version" in capsys.readouterr().out
