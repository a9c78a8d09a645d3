"""The MaxEnt loop: for every alpha of the mesh minimise Q_alpha, then analyze.

``MaxEntLoop.run(result=None, matrix_element=None, complex_index=None)`` is the seam where the fused
B200 path replaces the reference (python/maxent_loop.py:144-302): the reference's Python loop

    for alpha in alpha_mesh:  v = minimizer.minimize(cost_function, v); result.add_result(...)

becomes ONE call of the C ABI (``mx_project_data`` -> ``mx_alpha_sweep``), which runs the warm-started
Levenberg-Marquardt solves for all alphas on the device, followed by ``mx_analyze`` through the analyzer
objects.  Constructor arguments, attribute forwarding (``K, G, err, D, omega, data_variable, chi2, S,
H_of_v, A_of_H``), alpha scaling, the G_threshold skip, the consistency check and the log lines follow
the reference; combinations the kernels do not implement raise ``NotImplementedError`` (no host loop).

Not reproduced: the "Minimal chi2" header line (an unregularised lstsq, python/maxent_loop.py:187-193,
SURVEY.md N8 -- a log line only) and the Ctrl-C menu (one kernel launch cannot be interrupted per alpha)."""
from datetime import datetime

import numpy as np

from .alpha_meshes import LogAlphaMesh
from .analyzers import (LineFitAnalyzer, Chi2CurvatureAnalyzer, EntropyAnalyzer, BryanAnalyzer, ClassicAnalyzer)
from .cost_functions import MaxEntCostFunction, BryanCostFunction
from .functions import PlusMinusEntropy, PlusMinusH_of_v, PreblurA_of_H
from .logtaker import Logtaker, VerbosityFlags
from .maxent_result import MaxEntResult
from .minimizers import LevenbergMinimizer
from .probabilities import NormalLogProbability


def _bytes(x):
    return None if x is None else np.ascontiguousarray(x, dtype=np.float64).tobytes()


class MaxEntLoop(object):

    def __init__(self, cost_function=None, minimizer=None, alpha_mesh=None, probability=None, analyzers=None,
                 logtaker=None, G_threshold=1.e-10, reduce_singular_space=1.e-14, A_init=None,
                 interactive=True, scale_alpha='Ndata'):
        if cost_function is None:
            cost_function = MaxEntCostFunction()
        elif isinstance(cost_function, str):
            kind = cost_function.lower()
            if kind == 'normal':
                cost_function = MaxEntCostFunction()
            elif kind == 'plusminus':
                cost_function = MaxEntCostFunction(S=PlusMinusEntropy(), H_of_v=PlusMinusH_of_v())
            elif kind == 'bryan':
                cost_function = BryanCostFunction()
            else:
                raise Exception('Unknown cost_function str {}.'.format(cost_function))
        self.cost_function = cost_function
        self.minimizer = LevenbergMinimizer() if minimizer is None else minimizer
        self.alpha_mesh = LogAlphaMesh() if alpha_mesh is None else alpha_mesh
        self.logtaker = Logtaker() if logtaker is None else logtaker
        if isinstance(probability, str):
            if probability.lower() != 'normal':
                raise Exception('Unknown probability str {}.'.format(probability))
            probability = NormalLogProbability()
        self.probability = probability
        if analyzers is None:
            analyzers = [LineFitAnalyzer(), Chi2CurvatureAnalyzer(), EntropyAnalyzer()]
            if self.probability is not None:
                analyzers += [BryanAnalyzer(), ClassicAnalyzer()]
        self.analyzers = analyzers
        self.G_threshold = G_threshold
        self.interactive = interactive
        self.A_init = A_init
        self.reduce_singular_space = reduce_singular_space
        self.scale_alpha = scale_alpha
        self.device = None                     # torch device of the sweep (None: current CUDA device)
        self._problem_cache = {}

    # ---- the fused run ----------------------------------------------------------------------------
    def _scale(self):
        if self.scale_alpha is None:
            return 1.0
        if isinstance(self.scale_alpha, str):
            if self.scale_alpha.lower() != "ndata":
                raise Exception("Unknown value {} for scale_alpha".format(self.scale_alpha))
            s = len(self.G)
            self.logtaker.message(VerbosityFlags.Header,
                                  'scaling alpha by a factor {} (number of data points)'.format(s))
            return s
        self.logtaker.message(VerbosityFlags.Header, 'scaling alpha by a factor {}'.format(self.scale_alpha))
        return self.scale_alpha

    def shared_problem(self, variant=None):
        """The device-side state shared by every spectrum continued with this kernel / error / default model
        (engine.SharedProblem); the last few are cached so that elementwise runs alternate cheaply."""
        from . import engine
        variant = self.cost_function.variant() if variant is None else variant
        K = self.K
        err = np.asarray(self.err, dtype=np.float64) * np.ones(len(self.G))
        if getattr(K, "is_complex", False):
            err = K.stack(err)                               # the same error bar for real and imaginary part
        # the default model is NOT part of the key: jobs that differ only in D share the device problem and are
        # continued in one launch with one default model per spectrum (PoormanMaxEnt's off-diagonal pass)
        key = (id(K), K._svd_version, variant, _bytes(err), _bytes(self.omega.delta), _bytes(self.A_init),
               str(self.device))
        prob = self._problem_cache.get(key)
        if prob is not None and prob.kernel_ref is not K:     # id() of a collected kernel can be reused by a new object
            prob = None
        if prob is None:
            while len(self._problem_cache) >= 4:
                self._problem_cache.pop(next(iter(self._problem_cache)))
            prob = engine.SharedProblem(K.fused_matrix(), err, self.D.D, self.omega.delta, variant=variant, device=self.device,
                                        A_init=self.A_init, usv=(K.U, K.S, K.V), orthonormal_U=K._T is None)
            prob.D_host = np.array(self.D.D, dtype=np.float64)
            prob.kernel_ref = K                                # strong reference: the cache entry belongs to THIS kernel object
            self._problem_cache[key] = prob
        return prob

    def snapshot(self, matrix_element=None, complex_index=None):
        """Freeze the current data set (G, error model, kernel, default model) as one *job* of the sweep.
        Several jobs that share their device problem are continued in ONE launch by ``run_jobs`` -- this is how
        ``ElementwiseMaxEnt`` batches matrix elements."""
        cplx = getattr(self.K, "is_complex", False)
        if np.iscomplexobj(self.G) and not cplx:
            raise NotImplementedError("complex data need a complex kernel (IOmegaKernel); complex matrix elements of "
                                      "G(tau) go through ElementwiseMaxEnt(use_complex=True)")
        # complex Matsubara data enter the real fused path as the stacked rows [Re G; Im G] (kernels.IOmegaKernel)
        G = self.K.stack(np.asarray(self.G)) if cplx else np.array(self.G, dtype=np.float64)
        job = dict(G=G, matrix_element=matrix_element, complex_index=complex_index, problem=None)
        if np.max(np.abs(G)) < self.G_threshold:
            return job                                       # skipped (python/maxent_loop.py:174-179)
        assert self.err is not None, 'No error specified'
        variant = self.cost_function.variant()          # NotImplementedError for combinations off the fused path
        if self.probability is not None and not isinstance(self.probability, NormalLogProbability):
            raise NotImplementedError("only NormalLogProbability is evaluated by the fused kernel")
        self.K.reduce_singular_space(self.reduce_singular_space)
        self.check_consistency()
        blur = self.A_of_H._B if isinstance(self.A_of_H, PreblurA_of_H) else None     # A = B H (functions.py:991-993)
        job.update(problem=self.shared_problem(variant), scale=self._scale(), omega=self.omega, blur=blur,
                   D=np.array(self.D.D, dtype=np.float64),
                   G_orig=np.array(self.cost_function.G_orig, dtype=complex if cplx else np.float64),
                   data_variable=np.array(self.data_variable, dtype=np.float64), K_delta=self.K.K_delta)
        if cplx:
            job["G_report"] = np.array(self.G, dtype=complex)
        return job

    def run_jobs(self, jobs, result=None):
        """Continue the given jobs; consecutive groups that share a device problem and alpha scaling go
        through one ``mx_project_data`` / ``mx_alpha_sweep`` call each.  Returns the result."""
        from . import engine
        lm = self.minimizer.lm_params()
        if result is None:
            result = MaxEntResult()
        if result._default_analyzer_name is None:
            try:
                result._default_analyzer_name = self.analyzers[0].name
            except Exception:
                pass
        live = []
        for job in jobs:
            if job["problem"] is None:
                if job["matrix_element"] is not None:
                    result.zero_elements.append(job["matrix_element"])
                self.logtaker.error_message('G below threshold, not performing the calculation.')
            else:
                live.append(job)
        groups = []
        for job in live:
            if groups and groups[-1][0]["problem"] is job["problem"] and groups[-1][0]["scale"] == job["scale"]:
                groups[-1].append(job)
            else:
                groups.append([job])
        # Consecutive groups that differ only in their device problem (other kernel, other error model: e.g. the b values
        # of a preblur scan, doc/guide/preblur_example.py:46-75) and use the problem's own default model go through ONE
        # launch of the sweep as whitening groups (engine.run_sweep(groups=...)).  Groups of different n_sv are padded to
        # the largest, which is not exact for the Bryan cost function nor for Marquardt's damping: there only problems of
        # the same n_sv share a launch.
        merged = []
        for group in groups:
            p0 = group[0]["problem"]
            own_D = all(np.array_equal(job["D"], job["problem"].D_host) for job in group)
            last = merged[-1] if merged else None
            if (last is not None and last["multi_ok"] and own_D and last["jobs"][0]["scale"] == group[0]["scale"]
                    and last["jobs"][0]["problem"].variant == p0.variant and last["jobs"][0]["problem"].n_omega == p0.n_omega
                    and last["jobs"][0]["problem"].n_tau == p0.n_tau
                    and (last["jobs"][0]["problem"].n_sv == p0.n_sv or not (p0.variant == "bryan" or lm.marquardt))
                    and np.array_equal(last["jobs"][0]["problem"].D_host, p0.D_host)):
                last["jobs"].extend(group)
            else:
                merged.append(dict(jobs=list(group), multi_ok=own_D))
        want_p = self.probability is not None
        for entry in merged:
            group = entry["jobs"]
            prob, scale = group[0]["problem"], group[0]["scale"]
            alpha_eff = np.asarray(self.alpha_mesh, dtype=np.float64) * scale
            for job in group:
                job.get("result", result).start_timing(matrix_element=job["matrix_element"], complex_index=job["complex_index"])
            probs = []
            for job in group:
                if not any(job["problem"] is q for q in probs):
                    probs.append(job["problem"])
            Gs = np.stack([job["G"] for job in group])
            if len(probs) > 1:
                index = np.array([next(i for i, q in enumerate(probs) if q is job["problem"]) for job in group])
                res = engine.run_sweep(prob, Gs, alpha_eff, probability=want_p, lm=lm,
                                       chi2_factor=self.cost_function.chi2_factor, want_A=True, want_v=True,
                                       analyze_results=False, groups=(probs, index))
            else:
                D_rows = np.stack([job["D"] for job in group])
                if np.all(D_rows == prob.D_host[None, :]):
                    D_rows = None                            # the model the problem was built with: shared mode
                res = engine.run_sweep(prob, Gs, alpha_eff, probability=want_p, lm=lm,
                                       chi2_factor=self.cost_function.chi2_factor, want_A=True, want_v=True,
                                       analyze_results=False, D=D_rows)
            H_all = (res.A * prob.delta).cpu().numpy()          # the sweep writes H / delta (IdentityA_of_H)
            v_host = [job["problem"].v_to_reference_basis(res.v[b][..., :job["problem"].n_sv]).cpu().numpy()
                      for b, job in enumerate(group)]
            host = dict(A=res.A.cpu().numpy(), v=v_host,
                        chi2=res.chi2.cpu().numpy(), S=res.S.cpu().numpy(), Q=res.Q.cpu().numpy(),
                        logp=res.logp.cpu().numpy(), status=res.status.cpu().numpy(), n_iter=res.n_iter.cpu().numpy())
            width = str(int(np.ceil(np.log10(max(len(alpha_eff), 1)))))
            for b, job in enumerate(group):
                elem, cidx = job["matrix_element"], job["complex_index"]
                A, H = host["A"][b], H_all[b]
                if job["blur"] is not None:                  # preblur: the spectral function is the blurred hidden image
                    import torch
                    Bd = torch.as_tensor(np.ascontiguousarray(job["blur"]), device=res.A.device)
                    A = ((res.A[b] * prob.delta) @ Bd.transpose(0, 1)).cpu().numpy()
                conv = (host["status"][b] & 1).astype(bool)
                n_iter = host["n_iter"][b]
                record = dict(alpha=alpha_eff, v=host["v"][b], chi2=host["chi2"][b], S=host["S"][b], Q=host["Q"][b],
                              A=A, H=H,
                              probability=host["logp"][b] if want_p else np.full(len(alpha_eff), np.nan),
                              omega=job["omega"], G=job.get("G_report", job["G"]), G_orig=job["G_orig"],
                              data_variable=job["data_variable"], G_rec=np.dot(A, np.asarray(job["K_delta"]).T),
                              n_iter=n_iter, converged=conv, n_sv=job["problem"].n_sv)
                target = job.get("result", result)               # a job may bring its own result object (preblur_scan)
                if target._default_analyzer_name is None:
                    target._default_analyzer_name = result._default_analyzer_name
                run_time = target.end_timing(matrix_element=elem, complex_index=cidx)
                # the reference's per-alpha report (python/maxent_loop.py:248-255), printed from the device counters
                for i, a in enumerate(alpha_eff):
                    self.logtaker.message(VerbosityFlags.AlphaLoop,
                                          "alpha[{:" + width + "d}] = {:16.8e}, chi2 = {:16.8e}, n_iter={:8d}{}",
                                          i, a, record['chi2'][i], int(n_iter[i]), ' ' if conv[i] else '!')
                self.minimizer.n_iter_last = int(n_iter[-1]) if len(n_iter) else 0
                self.minimizer.n_iter += int(n_iter.sum())
                self.minimizer.converged = bool(conv[-1]) if len(n_iter) else False
                if not np.all(conv):
                    self.logtaker.message(VerbosityFlags.AlphaLoop,
                                          "\n! ... The minimizer did not converge. Results might be wrong.\n")
                self.logtaker.message(VerbosityFlags.Timing, "MaxEnt loop finished in {}", run_time)
                target.add_sweep(record, matrix_element=elem, complex_index=cidx)
                target.analyze(self.analyzers, matrix_element=elem, complex_index=cidx)
        return result

    def run(self, result=None, matrix_element=None, complex_index=None):
        """Run the alpha sweep for the current G and write it into ``result`` (a new ``MaxEntResult`` if None).
        Returns the result, or None when max|G| < G_threshold (the element is then listed in
        ``result.zero_elements``)."""
        if np.max(np.abs(np.asarray(self.G))) < self.G_threshold:
            if result is not None and matrix_element is not None:
                result.zero_elements.append(matrix_element)
            self.logtaker.error_message('G below threshold, not performing the calculation.')
            return None
        self.logtaker.welcome_message()
        return self.run_jobs([self.snapshot(matrix_element, complex_index)], result)

    # ---- helpers ------------------------------------------------------------------------------------
    def check_consistency(self):
        """All components must talk about the same kernel, default model and meshes (python/maxent_loop.py:306-337)."""
        cf = self.cost_function
        assert cf.H_of_v.K is cf.chi2.K, "H_of_v and chi2 use different kernels"
        assert cf.H_of_v.D is cf.S.D, "H_of_v and S use different default models"
        assert np.all(np.asarray(self.K.omega) == np.asarray(self.omega))
        assert np.all(np.asarray(self.D.omega) == np.asarray(self.omega))
        assert np.all(np.asarray(cf.A_of_H.omega) == np.asarray(self.omega))
        assert len(self.D.D) == len(self.omega)
        assert np.shape(self.K.K)[1] == len(self.omega), "kernel and omega mesh have different sizes"
        assert np.shape(self.K.K)[0] == len(self.G), "kernel and data have different sizes"
        assert np.ndim(self.err) == 0 or len(self.err) == len(self.G), "error and data have different sizes"

    def set_verbosity(self, verbosity=None, add=None, remove=None, change_callback=True):
        if verbosity is not None:
            self.logtaker.verbose = verbosity
        if add is not None:
            self.logtaker.verbose |= add
        if remove is not None:
            self.logtaker.verbose &= ~remove
        if change_callback:
            if self.logtaker.verbose & VerbosityFlags.SolverDetails:
                self.minimizer.verbose_callback = self.logtaker.solver_verbose_callback
            else:
                self.minimizer.verbose_callback = None


def _forward(name):
    """Property ``name`` of the loop = the same property of its cost function, with ``get_/set_`` methods."""
    def getter(self):
        return getattr(self.cost_function, "get_" + name)()

    def setter(self, value, **kwargs):
        getattr(self.cost_function, "set_" + name)(value, **kwargs)
    getter.__name__, setter.__name__ = "get_" + name, "set_" + name
    setattr(MaxEntLoop, "get_" + name, getter)
    setattr(MaxEntLoop, "set_" + name, setter)
    setattr(MaxEntLoop, name, property(getter, lambda self, value: setter(self, value)))


for _name in ("K", "G", "err", "omega", "data_variable", "D", "chi2", "S", "H_of_v", "A_of_H"):
    _forward(_name)
